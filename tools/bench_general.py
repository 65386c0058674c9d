"""Timings of the multi-objective / constrained path on one GPU, printed as one JSON object (card name and power limit
read in the same run):

  * scoring step (O posteriors + GeneralAcq epilogue + constrained front) at n = 4096, d = 32, m = 131072 for O = 2 (2 + 0)
    and O = 3 (2 + 1): ms and candidates/s;
  * hb_pareto_front for K in {2, 3, 4, 6, 8}, with and without cv, m = 131072: ms and sieve-survivor count (stage 2);
  * GeneralBO.suggest() at n = 256, O = 3 (2 + 1), both acquisition optimisers;
  * the unchanged 3-objective entry points hb_pareto_front3 (m = 131072) and hb_nsga2_survive (pop = 100), repeated so
    their spread is visible.

    python tools/bench_general.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True
import hebo_b200                                        # noqa: E402
from hebo_b200 import _lib                              # noqa: E402
from hebo_b200.acq import GeneralAcq                    # noqa: E402
from hebo_b200.general import GeneralBO                 # noqa: E402
from hebo_b200.pareto import pareto_front_device        # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [s.strip() for s in q.split(",")]
        return dict(gpu=name, power_limit=pl, max_sm_clock=clk)
    except Exception as e:                      # the timing itself never depends on it
        return dict(gpu=torch.cuda.get_device_name(0), power_limit=f"unavailable ({e})")


def timed(fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return dict(median_ms=float(np.median(ts)), min_ms=float(np.min(ts)), max_ms=float(np.max(ts)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_general needs a GPU"
    torch.manual_seed(0)
    np.random.seed(0)
    res = dict(card())
    lib = _lib.lib()
    # ---- scoring step
    n, d, m = 4096, 32, 131072
    X = torch.rand(n, d) * 2 - 1
    Y = torch.stack([torch.sin(3 * X[:, 0]) + X[:, 1], (X[:, :4] ** 2).sum(1), X[:, 2] - 0.3 * X[:, 3]], 1)
    Xs = (torch.rand(m, d) * 2 - 1).cuda()
    step = {}
    for no, nc in [(2, 0), (2, 1)]:
        O = no + nc
        model = hebo_b200.MultiTaskModel(d, 0, O, num_epochs=2, pred_likeli=False, rng="device")
        model.fit(X, None, Y[:, :O])
        acq = GeneralAcq(model, no, nc, kappa=2.0, c_kappa=0.5, use_noise=True)

        def one():
            out, cv = acq.evaluate(Xs, None, device_out=True, return_cv=True, seed=1)
            return pareto_front_device(out[:, :no], cv if nc else None)
        t = timed(one, reps=10)
        step[f"O{O}_{no}+{nc}"] = dict(t, candidates_per_s=m / (t["median_ms"] * 1e-3))
    res["score_step_n4096_d32_m131072"] = step
    # ---- fronts
    ws = torch.empty(int(lib.hb_pareto_workspace_bytes(m)), dtype=torch.uint8, device="cuda")
    idx = torch.empty(m, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    fronts = {}
    g = torch.Generator().manual_seed(3)
    for K in (2, 3, 4, 6, 8):
        Fk = torch.rand(m, K, generator=g).cuda()
        cv = torch.where(torch.rand(m, generator=g) < 0.5, torch.rand(m, generator=g), torch.zeros(m)).cuda()
        for tag, c in (("no_cv", None), ("cv", cv)):
            def call():
                _lib.check(lib.hb_pareto_front(_lib.ptr(Fk), m, K, K, _lib.ptr(c), _lib.ptr(idx), _lib.ptr(cnt), _lib.ptr(ws), ws.numel(),
                                               _lib.stream_ptr()), "front")
            t = timed(call)
            ru = lambda x, a: (x + a - 1) // a * a                    # workspace layout of pareto.cu carve_pareto: the nA slot
            off = ru(m, 256) + ru((m + 255) // 256 * 4 + 4, 256) + ru(m, 256) * 4 + ru(4096 * 4, 256) + 256
            fronts[f"K{K}_{tag}"] = dict(t, front=int(cnt), sieve_survivors=int(ws[off:off + 4].view(torch.int32)[0]))
    res["pareto_front_m131072_uniform"] = fronts
    # ---- unchanged 3-objective entry points
    F3 = torch.rand(m, 3, generator=g).cuda()

    def f3():
        _lib.check(lib.hb_pareto_front3(_lib.ptr(F3), m, _lib.ptr(idx), _lib.ptr(cnt), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "f3")
    res["pareto_front3_m131072_runs"] = [timed(f3, reps=50) for _ in range(5)]
    P, D = 100, 6
    Xp, C = torch.rand(P, D).cuda(), torch.rand(P, D).cuda()
    Fp, FC = torch.randn(P, 3).cuda(), torch.randn(P, 3).cuda()
    Xn, Fn = torch.empty(P, D, device="cuda"), torch.empty(P, 3, device="cuda")
    Xcn, Xen = torch.empty(P, D - 1, device="cuda"), torch.empty(P, 1, dtype=torch.int32, device="cuda")

    def surv():
        _lib.check(lib.hb_nsga2_survive(_lib.ptr(Xp), _lib.ptr(Fp), _lib.ptr(C), _lib.ptr(FC), P, D, D - 1, _lib.ptr(Xn), _lib.ptr(Fn),
                                        _lib.ptr(Xcn), _lib.ptr(Xen), _lib.stream_ptr()), "surv")
    res["nsga2_survive_pop100_runs"] = [timed(surv, reps=50) for _ in range(5)]
    # ---- GeneralBO.suggest at n = 256, O = 3
    space = [{"name": f"x{i}", "type": "num", "lb": -1, "ub": 1} for i in range(6)]
    sug = {}
    for optname in ("sobol", "nsga2"):
        opt = GeneralBO(space, 2, 1, acq_optimizer=optname, scramble_seed=0)
        Xo = opt.space.sample(256)
        xv = Xo.values.astype(float)
        opt.observe(Xo, np.stack([(xv ** 2).sum(1), ((xv - 0.5) ** 2).sum(1), xv[:, 0] + xv[:, 1] - 0.5], 1))
        opt.suggest(8)
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            opt.suggest(8)
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        sug[optname] = dict(median_ms=float(np.median(ts)), runs_ms=ts)
    res["general_bo_suggest_n256_O3"] = sug
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
