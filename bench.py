#!/usr/bin/env python
"""bench.py -- acquisition candidates/sec (+ suggest() ms) at n=4096, d=32 on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...        # the reference's CPU path (oracle port) on the host cores
    python bench.py ... --dump-outputs DIR      # also write the last timed step's result to DIR/*.npy

Metric (BASELINE.json): "acquisition candidates/sec + suggest() ms at n=4096 d=32; 1/2/4/8 GPU".
One STEP = one pass of the scoring hot path over one candidate batch: fused posterior (mu, sigma^2) + MACE
(LCB, -logEI, -logPI) + 3-objective Pareto front over m_per_gpu candidates per rank (+ the front all-gather
and merge when N > 1), model already fitted, candidates resident in HBM.  `value` = N * m_per_gpu / step time
(weak scaling: per-GPU work fixed).  `e2e` = EXACTLY the same pass fed from pinned HOST candidates (H2D inside the timed
region) with the resulting global front (ids, objectives, mu, sigma) read back to the host.
Timing: CUDA events on the launching stream per step, max over ranks, L2 flushed (256 MiB write) between
steps and excluded from the timed intervals.  No step waits for the host: kernels + one collective are enqueued, the
front buffer is read once.

Extra keys: `parity` (mu / sigma / objectives / front of a 2368-candidate sample against the fp64 oracle rebuilt on the host
cores, N = 1), `guard_flagged_frac` (rows the precision guard re-contracted on the FP32 pipe), `dense_regime` (a second
workload, n=4096 d=8, where most candidates sit inside the data and the guard fires), `suggest` (suggest() ms with the
fit / scoring split), `roofline`, `cpu_baseline`.

--dump-outputs DIR writes what the last timed step of the headline workload returned to its caller, the global Pareto
front: DIR/front_ids.npy (global candidate row, float64), DIR/front_objectives.npy ([K, 3] LCB, -logEI, -logPI, float32)
and DIR/front_mu_sigma.npy ([K, 2], float32).  All inputs are seeded, so two builds run with the same arguments can be
compared output for output.  bench.py writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

sys.dont_write_bytecode = True        # no __pycache__ in the (possibly read-only) source tree
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_OBS, DIM, Q = 4096, 32, 8
KERNEL = "matern32"
M_HEADLINE = 10000            # north-star suggest() workload: q=8, 10k candidates
M_PER_GPU = 131072            # BASELINE config 5 shard size (1M candidates / 8 GPUs); weak scaling keeps it fixed
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel (32768 x 4096 chunk) from the committed
# `ncu --set full` capture under profiles/ (r02_vnorm_h16_kernel_ncu_full_32768x4096.txt).  Algorithmic operand bytes per
# launch: 32768*4096*4 (K* h0/h1) + 4096*4096*4/2 (Linv h0/h1, lower half) = 5.7e8.
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "r02_vnorm_h16_traffic.json")


def synth(n, d, seed, fn="hartmann6"):
    """Hartmann-6 embedded in d dims (or Ackley-d) + 0.05 N(0,1) (BASELINE.md section 4), X ~ U(-1,1)^d."""
    g = torch.Generator().manual_seed(seed)
    X = torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1
    if fn == "ackley":
        z = (X.numpy() + 1) * 7.5 - 5
        y = (-20 * np.exp(-0.2 * np.sqrt((z ** 2).sum(1) / d)) - np.exp(np.cos(2 * np.pi * z).sum(1) / d) + 20 + np.e)
        y = y + 0.05 * torch.randn(n, generator=g, dtype=torch.float64).numpy()
        return X.float(), y
    A = np.array([[10, 3, 17, 3.5, 1.7, 8], [0.05, 10, 17, 0.1, 8, 14], [3, 3.5, 1.7, 10, 17, 8], [17, 8, 0.05, 10, 0.1, 14]])
    P = 1e-4 * np.array([[1312, 1696, 5569, 124, 8283, 5886], [2329, 4135, 8307, 3736, 1004, 9991],
                         [2348, 1451, 3522, 2883, 3047, 6650], [4047, 8828, 8732, 5743, 1091, 381]])
    al = np.array([1.0, 1.2, 3.0, 3.2])
    x = (X.numpy()[:, :6] + 1) * 0.5
    y = -(al[None] * np.exp(-(A[None] * (x[:, None, :] - P[None]) ** 2).sum(-1))).sum(1)
    y = y + 0.05 * torch.randn(n, generator=g, dtype=torch.float64).numpy()
    return X.float(), y


def candidates(m, d, seed):
    eng = torch.quasirandom.SobolEngine(d, scramble=True, seed=seed)
    return (eng.draw(m) * 2 - 1).float()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None
        self.frozen = False

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            if not self.frozen:
                self.rows.append((time.perf_counter(), line.strip()))

    def window(self, t0, t1):
        """keep only the samples that arrived inside the timed region [t0, t1]"""
        self.frozen = True
        rows = list(self.rows)
        inside = [r for (ts, r) in rows if t0 <= ts <= t1 + 0.02]
        self.rows = inside if inside else [r for (_, r) in rows[-3:]]

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads() -> int:
    """Usable host cores: scheduler affinity capped by the cgroup CPU quota (os.cpu_count() over-reports in
    containers and oversubscribes the BLAS thread pool)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return float(p["bf16_tflops"]), float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst bf16)"
    return 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------ CPU reference path
def cpu_reference(steps, warmup, sample_m, threads, fit_epochs=2, n=N_OBS, d=DIM, seed=1234 + 5):
    """The reference's CPU path restated by the oracle (gpytorch is not installable here): fp32 torch on the host
    cores.  Scores `sample_m` candidates per step at the full n, d; also times `fit_epochs` MLL epochs."""
    from oracle import gp_oracle as O
    O.KERNEL_FORM = "mm"          # the reference's (gpytorch) matmul-form distance: its actual CPU code path
    torch.set_num_threads(threads)
    X, y = synth(n, d, seed)
    yt = torch.from_numpy(O.hebo_y_transform(y)).float().reshape(-1)
    t0 = time.perf_counter()
    f = O.make_fitted(X, yt, kind=KERNEL, dtype=torch.float32, rng=np.random.RandomState(0))
    t_factor = time.perf_counter() - t0
    Xs = candidates(sample_m, d, 99)
    xi1, xi2 = torch.randn(sample_m, 1), torch.randn(sample_m, 1)
    tau, kappa = float(yt.min()), O.kappa_schedule(n, Q, d)

    def step():
        mu, var = O.predict(f, Xs)
        F = O.mace(mu, var, float(f.noise), tau, kappa, 1e-4, xi1, xi2)
        O.pareto_front(F.numpy())
        return F
    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        F = step()
        ts.append(time.perf_counter() - t0)
    # fit: time a couple of MLL forward+backward epochs (autograd, like the reference) and extrapolate to 100
    t_epoch = None
    if fit_epochs:
        t0 = time.perf_counter()
        for _ in range(fit_epochs):
            O.neg_mll_autograd(f.Xt, f._yt, f.hp, KERNEL)
        t_epoch = (time.perf_counter() - t0) / fit_epochs
    O.KERNEL_FORM = "direct"
    ms = float(np.mean(ts)) * 1e3
    rate = sample_m / (ms / 1e3)
    return dict(value=rate, ms_per_step=ms, fit_epoch_s=t_epoch, factor_s=t_factor,
                suggest_ms_est=None if t_epoch is None else (100 * t_epoch + M_HEADLINE / rate) * 1e3,
                finite=bool(torch.isfinite(F).all()))


def parity_sample(gp, X, yt, tau, kappa, dev):
    """mu / sigma / MACE objectives / Pareto front of the CUDA path against the fp64 oracle on a sample of the bench
    workload: 2048 Sobol candidates + 256 rows within 1e-3 of training points + 64 exact training points.  The oracle is
    rebuilt on the host cores at the hypers the CUDA fit ended on (test infrastructure; this leg is the checker only)."""
    from oracle import gp_oracle as O
    from hebo_b200.pareto import pareto_front
    n, d = X.shape
    g = torch.Generator().manual_seed(77)
    near = X[torch.randperm(n, generator=g)[:256]] + 1e-3 * torch.randn(256, d, generator=g)
    exact = X[torch.randperm(n, generator=g)[:64]].clone()
    Xs = torch.cat([candidates(2048, d, 4242), near, exact], 0).float()
    m = Xs.shape[0]
    xi1, xi2 = torch.randn(m, 1, generator=g), torch.randn(m, 1, generator=g)
    F, mu, var = gp.predict_mace(Xs.to(dev), tau, kappa, 1e-4, xi1, xi2, return_mu_var=True)
    front_gpu = pareto_front(F).cpu().numpy()
    F, mu, var = F.cpu().double().numpy(), mu.cpu().double().numpy(), var.cpu().double().numpy()
    dt = torch.float64
    sc, mn = gp.xscaler.scale_.to(dt), gp.xscaler.min_.to(dt)
    ym, ys = float(gp.yscaler.mean[0]), float(gp.yscaler.std[0])
    f = O.FittedGP(sc * X.to(dt) + mn, O.Hypers.unpack(gp.raw.to(dt), gp.noise_lb), gp.kernel, sc, mn, ym, ys)
    f._yt = (yt.to(dt).reshape(-1) - ym) / ys
    O.refactor(f)
    mu64, var64 = O.predict(f, Xs.to(dt))
    F64 = O.mace(mu64, var64, float(f.noise), tau, kappa, 1e-4, xi1, xi2).numpy()
    mu64, var64 = mu64.numpy().reshape(-1), var64.numpy().reshape(-1)
    emu = np.abs(mu - mu64) / np.maximum(np.abs(mu64), ys)
    esg = np.abs(np.sqrt(var) - np.sqrt(var64)) / np.sqrt(var64)
    ratio = var64 / (float(f.hp.outputscale) * ys ** 2)
    reg = ratio >= 0.02
    front64 = O.pareto_front(F64)
    return {"mu": float(emu.max()), "sigma": float(esg[reg].max()), "sigma_on_training_points": float(esg[~reg].max()) if (~reg).any() else None,
            "lcb_abs": float(np.abs(F[:, 0] - F64[:, 0]).max()), "front_equal": bool(np.array_equal(front_gpu, front64)),
            "front_size": int(front64.size),
            "argmin_mu_equal": int(np.argmin(mu[front64])) == int(np.argmin(mu64[front64])),
            "argmax_sigma_equal": int(np.argmax(var[front64])) == int(np.argmax(var64[front64])),
            "sample": "2048 Sobol + 256 near-training + 64 exact-training candidates vs oracle/gp_oracle.py in fp64 at the fitted hypers; "
                      "criteria 1e-4 (mu scale-relative, sigma relative; rows with sigma^2 < 0.02 s listed separately, cap 2e-4)"}


def dump_outputs(out_dir, front):
    """front = pareto.front_read(...) of the last timed step: (global ids, F [K, 3], (mu, sigma) [K, 2])."""
    os.makedirs(out_dir, exist_ok=True)
    gid, F, mu_sigma = front
    np.save(os.path.join(out_dir, "front_ids.npy"), gid.numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "front_objectives.npy"), F.numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "front_mu_sigma.npy"), mu_sigma.numpy().astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--m-per-gpu", type=int, default=M_PER_GPU)
    ap.add_argument("--no-suggest", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-dense", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's Pareto front to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the CUDA path's result: use it with --impl b200")
    steps, warmup = args.steps, max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    REF_SAMPLE = 2048
    config = {"workload": f"n{N_OBS}_d{DIM}_q{Q}_{KERNEL}_score+front_m{args.m_per_gpu}_per_gpu",
              "n": N_OBS, "d": DIM, "q": Q, "kernel": KERNEL, "m_per_gpu": args.m_per_gpu, "m_suggest": M_HEADLINE,
              "l2": "flushed between steps (256 MiB write), flush excluded from the timed intervals",
              "exchange": ("single GPU: no exchange" if world == 1 else
                           "front pack -> ONE all-gather -> merge of step i on an exchange stream under the scoring of step i+1; the "
                           "timed region (one event pair around the K steps minus the flush durations) closes after every step's "
                           "merged front is complete"),
              "parallelism": f"candidate-sharded x{max(world, 1)}; fit on rank 0 + state broadcast",
              "reference_arm": f"oracle port (torch fp32 CPU, all usable host threads), {REF_SAMPLE} candidates per step at the full "
                               f"n={N_OBS}, d={DIM} (a bounded sample of the same workload; rate = candidates / s)"}

    # ---------------------------------------------------------------- reference arm (CPU oracle port)
    if args.impl == "reference":
        if rank != 0:
            return
        threads = host_threads()
        r = cpu_reference(max(1, steps), warmup, REF_SAMPLE, threads)
        line = {"metric": "acquisition candidates/sec (posterior+MACE+front) at n=4096 d=32", "value": r["value"],
                "unit": "candidates/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "impl": "reference", "config": config,
                "cpu_baseline": {"value": r["value"], "unit": "candidates/s", "cores": threads, "kind": "port",
                                 "sample": f"{REF_SAMPLE} of the candidates per step at full n={N_OBS}, d={DIM} (oracle/gp_oracle.py, torch fp32 CPU; "
                                           "the reference itself pins torch to 1 thread, hebo.py:28 -- all threads is the generous reading)",
                                 "fit_epoch_s": r["fit_epoch_s"], "suggest_ms_est": r["suggest_ms_est"],
                                 "suggest_ms_est_note": "100 x (mean of 2 timed MLL forward+backward epochs) + 10000 candidates at the measured rate"},
                "e2e": {"value": r["value"], "unit": "candidates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ---------------------------------------------------------------- B200 arm
    import torch.distributed as dist
    import hebo_b200
    from hebo_b200 import _lib, dist as hdist
    from hebo_b200.pareto import FRONT_W, front_read, front_wait
    from hebo_b200.suggest import HEBO, hebo_y_transform, kappa_schedule
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.lib()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()          # started before the fit: nvidia-smi needs ~1 s before its first row; only rows that arrive
                                 # inside the timed region are kept (ClockSampler.window)
    CAP = 4096                   # rows per front buffer (a larger local front raises at read time, never truncates)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k, pipelined=False):
        """K steps between barriers.  Per-step CUDA events on the launching stream (the L2 flush between steps is outside
        them); max over ranks.  pipelined=True (N > 1 device step, whose front exchange runs on a separate stream under the
        NEXT step's scoring): ONE event pair around all K steps, the stream made to wait for every step's merged front before
        the closing event, minus the flush durations (own events) -- so the exchange that is still in flight after the last
        scoring kernel is inside the timed region.  Returns (ms, wall ms, what the last step returned)."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        barrier()
        t0 = time.perf_counter()
        if pipelined:
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
            outs = []
            for a, b in ev:
                a.record()
                flush.fill_(1)
                b.record()
                outs.append(fn())
            for o in outs:
                front_wait(o)
            end.record()
            last = outs[-1]
        else:
            for a, b in ev:
                flush.fill_(1)
                a.record()
                last = fn()
                b.record()
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        ms = sum(a.elapsed_time(b) for a, b in ev)
        if pipelined:
            ms = start.elapsed_time(end) - ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), wall, last

    def run_workload(n, d, seed, m, k_steps, k_warm, profile, fn="hartmann6"):
        """fit on rank 0 (+ broadcast), then time the device step and the end-to-end step over m candidates per rank"""
        X, y = synth(n, d, seed, fn)
        yt = hebo_y_transform(y)
        np.random.seed(0)
        torch.manual_seed(0)
        gp = hebo_b200.GP(d, 0, 1, lr=0.01, num_epochs=100, noise_lb=8e-4, pred_likeli=False, kernel=KERNEL,
                          device=str(dev), rng="device")
        fit_ms = None
        if rank == 0:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            gp.fit(X, None, yt)
            torch.cuda.synchronize()
            fit_ms = (time.perf_counter() - t0) * 1e3
        if world > 1:
            hdist.broadcast_state(gp, 0)
        tau = float(yt.min())
        kappa = kappa_schedule(n, Q, d)
        lo = rank * m
        Xs_host = candidates(m, d, 1000 + rank).pin_memory()
        Xs_dev = Xs_host.to(dev)

        def step_dev():
            # fused posterior + MACE over this rank's shard, device front, fixed-capacity pack, (N > 1: ONE all-gather + device
            # merge); everything is enqueued, nothing waits for the host
            return hdist.sharded_score_front(gp, Xs_dev, lo, tau, kappa, 1e-4, seed=7, capacity=CAP, overlap=world > 1)

        def step_e2e():
            # the same work fed from HOST buffers: pinned candidates in (uploaded chunk by chunk under the scoring by the
            # plugin call itself), the front (ids, objectives, mu, sigma) read back
            return front_read(hdist.sharded_score_front(gp, Xs_host, lo, tau, kappa, 1e-4, seed=7, capacity=CAP))

        for _ in range(k_warm):
            step_dev()
            step_e2e()
        g0 = (C.c_uint64 * 2)()
        lib.hb_guard_stats(g0, 1)
        t_region0 = time.perf_counter()
        lib.hb_launch_count(1)
        if profile:
            lib.hb_profile_enable(1)
        total_ms, wall_ms, last_dev = timed(step_dev, k_steps, pipelined=world > 1)
        launches = int(lib.hb_launch_count(1))
        kms, kn = C.c_double(0), C.c_int32(0)
        if profile:
            lib.hb_profile_collect(C.byref(kms), C.byref(kn))
            lib.hb_profile_enable(0)
        gs = (C.c_uint64 * 2)()
        lib.hb_guard_stats(gs, 1)
        e2e_ms, _, _ = timed(step_e2e, k_steps)
        t_region1 = time.perf_counter()
        front = front_read(last_dev)
        return dict(gp=gp, X=X, yt=yt, tau=tau, kappa=kappa, total_ms=total_ms, wall_ms=wall_ms, e2e_ms=e2e_ms, launches=launches,
                    kms=kms.value, kn=kn.value, guard_frac=(gs[1] / gs[0]) if gs[0] else 0.0, fit_ms=fit_ms, region=(t_region0, t_region1),
                    front=front, front_size=int(front[0].numel()))

    m = args.m_per_gpu
    w = run_workload(N_OBS, DIM, 1234 + 5, m, steps, warmup, True)
    if rank == 0 and sampler.proc is not None:
        sampler.window(*w["region"])
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, w["front"])
    gp = w["gp"]
    ms_per_step = w["total_ms"] / steps
    value = world * m / (ms_per_step / 1e3)
    e2e_value = world * m / (w["e2e_ms"] / steps / 1e3)

    # ---- second workload (N = 1 only): the dense low-d regime, where most candidates sit inside the data
    dense = None
    if world == 1 and not args.no_dense:
        nd_steps = max(3, steps // 2)
        wd = run_workload(N_OBS, 8, 1234 + 9, m, nd_steps, 3, False, fn="ackley")
        dense = {"workload": f"ackley_n{N_OBS}_d8_q{Q}_{KERNEL}_score+front_m{m}_per_gpu", "value": m / (wd["total_ms"] / nd_steps / 1e3),
                 "unit": "candidates/s", "ms_per_step": wd["total_ms"] / nd_steps, "e2e": m / (wd["e2e_ms"] / nd_steps / 1e3),
                 "guard_flagged_frac": wd["guard_frac"], "steps": nd_steps, "front": wd["front_size"]}
        del wd

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (posterior variance contraction V = K* Linv^T, row sum of squares)
    bf16_peak, hbm_peak, which = peaks()
    flop_per_cand = float(N_OBS) * N_OBS                     # n^2 term of BASELINE.md's per-candidate figure
    n_chunks = math.ceil(m / gp.m_chunk)
    flop_per_launch = flop_per_cand * m / n_chunks
    k_avg_ms = w["kms"] / max(1, w["kn"])
    achieved = flop_per_launch / (k_avg_ms / 1e3) / 1e12 if k_avg_ms > 0 else None
    traffic = None
    if os.path.exists(TRAFFIC_FILE):
        traffic = json.load(open(TRAFFIC_FILE)).get("dram_bytes_per_launch")
    roofline = {"bound": "tensor",
                "kernel": "vnorm_h16_kernel (posterior variance V = K* Linv^T, row ||.||^2; tcgen05 cta_group::2 kind::f16 on a "
                          "two-level fp16 operand split, fp32 accumulate)",
                "achieved": achieved, "peak": bf16_peak, "unit": "TFLOP/s", "frac": (achieved / bf16_peak) if achieved else None,
                "traffic": traffic, "peak_source": which, "launches_timed": w["kn"], "avg_launch_ms": k_avg_ms,
                "candidates_per_launch": m // n_chunks, "share_of_step": w["kms"] / w["total_ms"] if w["total_ms"] > 0 else None,
                "note": "algorithmic flops = n^2 per candidate (triangular trsm form). The kernel issues 3 fp16 MMAs (h0*h0, h0*h1, "
                        "h1*h0) per algorithmic MAC for ~2^-22 operand precision, so frac <= 1/3 of the measured bf16 peak by "
                        "construction; tensor-pipe busy % is in profiles/"}

    # ---- suggest() ms at the north-star point (n=4096, d=32, q=8, 10k candidates), fit/score split
    suggest = None
    if not args.no_suggest:
        opt = HEBO(-torch.ones(DIM), torch.ones(DIM), n_candidates=M_HEADLINE, device=str(dev), scramble_seed=1)
        opt.observe(w["X"], synth(N_OBS, DIM, 1234 + 5)[1])
        ts = []
        for _ in range(3):
            np.random.seed(0)
            opt.suggest(Q)
            ts.append(dict(opt.last_timing))
        best = min(ts[1:], key=lambda r: r["total_ms"])       # the first call pays workspace allocation / lazy module loads
        suggest = {"total_ms": best["total_ms"], "fit_ms": best["fit_ms"], "score_select_ms": best["score_ms"],
                   "split_ms": {k: round(v, 3) for k, v in best.items() if k.endswith("_ms") and k not in ("fit_ms", "total_ms", "score_ms")},
                   "epochs": 100, "m": M_HEADLINE, "q": Q, "front": best["front"], "runs": len(ts),
                   "all_total_ms": [round(r["total_ms"], 2) for r in ts]}

    cpu, parity = None, None
    if not args.no_cpu_baseline:
        threads = min(host_threads(), 32)
        r = cpu_reference(3, 1, REF_SAMPLE, threads)
        cpu = {"value": r["value"], "unit": "candidates/s", "cores": threads, "kind": "port",
               "sample": f"{REF_SAMPLE} candidates per step x3 at full n={N_OBS}, d={DIM}; fit: 2 MLL fwd+bwd epochs timed, x100 for suggest_ms_est",
               "fit_epoch_s": r["fit_epoch_s"], "suggest_ms_est": r["suggest_ms_est"]}
        if world == 1:
            parity = parity_sample(gp, w["X"], w["yt"], w["tau"], w["kappa"], dev)

    line = {"metric": "acquisition candidates/sec (posterior+MACE+front) at n=4096 d=32", "value": value,
            "unit": "candidates/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "candidates/s", "h2d_bytes_per_step": int(m * DIM * 4),
                    "d2h_bytes_per_step": int((max(world, 1) * CAP + 1) * FRONT_W * 4) if world > 1 else int((CAP + 1) * FRONT_W * 4),
                    "ms_per_step": w["e2e_ms"] / steps,
                    "result": "global Pareto front buffer (ids, F[3], mu, sigma) read to the host on every rank"},
            "gpu_launches": w["launches"], "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
            "guard_flagged_frac": w["guard_frac"], "dense_regime": dense, "suggest": suggest,
            "fit_ms_first_call_cold": w["fit_ms"], "wall_ms_incl_flush": w["wall_ms"], "front_size": w["front_size"]}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
