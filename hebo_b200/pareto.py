"""Device non-dominated filter (K <= 8 objectives, minimised, optionally constrained) through the C ABI.

Replaces the rank-0 extraction NSGA-II performs on the final population
(HEBO/hebo/acq_optimizers/evolution_optimizer.py:141-149) for candidate batches of any size; with a constraint violation
``cv`` only feasible rows (cv <= 0) form the front, and with none feasible the least-infeasible row is returned
(GeneralBO, HEBO/hebo/optimizers/general.py:23-204).
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib

_ws_cache = {}


def _workspace(dev: torch.device, need: int, tag: str = "front") -> torch.Tensor:
    key = (dev.index, tag)
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        _ws_cache[key] = ws
    return ws


def pareto_front_device(F: torch.Tensor, cv: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """F [m, K] float32 CUDA tensor (1 <= K <= 8; a column slice of a wider row-major tensor is read in place), cv [m] or
    None -> (idx int32 [m] whose first `count` entries are the ascending indices of the non-dominated feasible rows -- or
    the single least-infeasible row when none is feasible -- count int32 [1]), both on the device; NO host
    synchronisation."""
    lib = _lib.lib()
    assert F.is_cuda and F.dim() == 2 and 1 <= F.shape[1] <= 8
    m, K = F.shape
    dev = F.device
    ws = _workspace(dev, int(lib.hb_pareto_workspace_bytes(m)))
    idx = torch.empty(m, dtype=torch.int32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    if K == 3 and cv is None:                  # the 3-objective MACE front
        F = F.to(torch.float32).contiguous()
        with torch.cuda.device(dev):
            st = lib.hb_pareto_front3(_lib.ptr(F), m, _lib.ptr(idx), _lib.ptr(cnt), _lib.ptr(ws), ws.numel(),
                                      _lib.stream_ptr())
        _lib.check(st, "hb_pareto_front3")
        return idx, cnt
    if F.dtype != torch.float32 or F.stride(1) != 1 or F.stride(0) < K:
        F = F.to(torch.float32).contiguous()
    if cv is not None:
        assert cv.is_cuda and cv.numel() == m
        cv = cv.reshape(-1).to(torch.float32).contiguous()
    with torch.cuda.device(dev):
        st = lib.hb_pareto_front(_lib.ptr(F), m, K, F.stride(0) if m else K, _lib.ptr(cv), _lib.ptr(idx), _lib.ptr(cnt),
                                 _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
    _lib.check(st, "hb_pareto_front")
    return idx, cnt


def pareto_front(F: torch.Tensor, cv: Optional[torch.Tensor] = None) -> torch.Tensor:
    """F [m, K] float32 CUDA tensor (and optional cv [m]) -> ascending int64 indices (on the device) of the non-dominated
    feasible rows (one host read of the count)."""
    idx, cnt = pareto_front_device(F, cv)
    return idx[:int(cnt.item())].to(torch.int64)


FRONT_W = 8     # floats per row of a front buffer (include/hebo_b200.h "multi-GPU front exchange")


def front_pack(F: torch.Tensor, mu, var, idx: torch.Tensor, cnt: torch.Tensor, row_offset: int, capacity: int) -> torch.Tensor:
    """Fixed-capacity front buffer [(capacity + 1), 8] of the rows idx[:cnt] (hb_front_pack; no host sync)."""
    lib = _lib.lib()
    dev = F.device
    out = torch.empty(capacity + 1, FRONT_W, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        st = lib.hb_front_pack(_lib.ptr(F), _lib.ptr(mu), _lib.ptr(var), _lib.ptr(idx), _lib.ptr(cnt), int(row_offset),
                               int(capacity), _lib.ptr(out), _lib.stream_ptr())
    _lib.check(st, "hb_front_pack")
    return out


def front_merge(all_buf: torch.Tensor, world: int, capacity: int) -> torch.Tensor:
    """All-gathered buffers [world, capacity + 1, 8] -> merged front buffer [(world * capacity + 1), 8] (hb_front_merge)."""
    lib = _lib.lib()
    dev = all_buf.device
    ws = _workspace(dev, int(lib.hb_front_merge_workspace_bytes(world, capacity)), "merge")
    out = torch.empty(world * capacity + 1, FRONT_W, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        st = lib.hb_front_merge(_lib.ptr(all_buf), world, capacity, _lib.ptr(out), _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
    _lib.check(st, "hb_front_merge")
    return out


def front_wait(buf: torch.Tensor) -> torch.Tensor:
    """Make the current stream wait for a front buffer that an overlapped exchange is still producing
    (``dist.gather_merge_fronts(overlap=True)``); a no-op for any other tensor.  Returns buf."""
    ready = getattr(buf, "_hb_ready", None)
    if ready is not None and buf.is_cuda:
        cur = torch.cuda.current_stream(buf.device)
        cur.wait_event(ready)
        buf.record_stream(cur)              # allocated on the exchange stream's pool
    return buf


def front_read(buf: torch.Tensor):
    """Host view of a front buffer: (global ids int64 [K], F [K,3], (mu, sigma) [K,2]).  This is the ONE device->host
    read of a scoring step; raises if any rank's front overflowed the gather capacity (never silently truncated)."""
    host = front_wait(buf).cpu()
    k, over = int(host[0, 0]), bool(host[0, 1] != 0)
    if over or k > host.shape[0] - 1:
        raise RuntimeError(f"local Pareto front larger than the gather capacity ({host.shape[0] - 1} rows per buffer)")
    body = host[1:k + 1]
    gid = body[:, 5].to(torch.int64) + (body[:, 6].to(torch.int64) << 24)
    return gid, body[:, :3].contiguous(), body[:, 3:5].contiguous()
