"""Torch restatement of GeneralAcq.eval (HEBO/hebo/acquisitions/acq.py:233-242) for the CPU and GPU tests: the
reference's fp32 operation order, with the N(0,1) draw xi [m, O] passed in instead of drawn.  Pinned to the reference's
own outputs by tests/golden/ref_general_acq.npz (written by oracle/make_golden_general.py)."""
from __future__ import annotations

import numpy as np
import torch


def general_acq(py, ps2, noise, xi, num_obj: int, kappa: float, c_kappa: float, use_noise: bool) -> torch.Tensor:
    """py, ps2 [m, O] fp32, noise [O] (model.noise), xi [m, O] -> out [m, O] fp32."""
    py = torch.as_tensor(py, dtype=torch.float32).clone()
    ps2 = torch.as_tensor(ps2, dtype=torch.float32)
    ps = ps2.sqrt().clamp(min=torch.finfo(torch.float32).eps)
    if use_noise:
        py += torch.as_tensor(noise, dtype=torch.float32).sqrt() * torch.as_tensor(xi, dtype=torch.float32)
    out = torch.ones(py.shape)
    out[:, :num_obj] = py[:, :num_obj] - kappa * ps[:, :num_obj]
    out[:, num_obj:] = py[:, num_obj:] - c_kappa * ps[:, num_obj:]
    return out


def constraint_violation(out: torch.Tensor, num_obj: int) -> np.ndarray:
    """cv = sum_j max(0, g_j) accumulated in fp32 in ascending j (a NaN propagates)."""
    G = np.asarray(out, dtype=np.float32)[:, num_obj:]
    cv = np.zeros(G.shape[0], dtype=np.float32)
    for j in range(G.shape[1]):
        g = G[:, j]
        cv = (cv + np.where(np.isnan(g), g, np.maximum(g, np.float32(0)))).astype(np.float32)
    return cv
