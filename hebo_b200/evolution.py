"""NSGA-II acquisition optimiser for box-bounded continuous spaces (tensor/array form).

The reference optimises the MACE objectives with pymoo's NSGA-II (HEBO/hebo/acq_optimizers/evolution_optimizer.py:107-160:
pop 100, `iters` generations of 100 offspring, MixedVariableMating = random parent selection + SBX crossover +
polynomial mutation, duplicate elimination, rank-and-crowding survival; the result is the non-dominated part of the
final population).  pymoo is a third-party dependency that is not installed here, so this is a restatement of the
published algorithm (Deb et al. 2002) with pymoo 0.6 operator defaults as recalled in SURVEY.md Appendix C
(SBX eta=15, pair probability 0.9, per-variable 0.5; PM eta=20, per-variable min(0.5, 1/d)); parity with pymoo's random
stream is neither possible nor claimed.  The bookkeeping (200 x 3 objective values per generation) runs vectorised on the
host like pymoo's; every generation's offspring are scored in ONE call of `acq_fn` (the fused posterior+MACE pass on the
device), which replaces the per-individual marshalling of evolution_optimizer.py:84-105.

`hebo_b200.suggest.HEBO(acq_optimizer="nsga2")` runs the DEVICE version below (`DeviceNSGA2`: population, mating, typed
repair, duplicate elimination and rank-and-crowding survival in CUDA kernels, hebo_b200/csrc/nsga.cu; no per-generation
host round trip); the numpy functions in this file restate the same operators on the host and serve as the checker of
those kernels (tests/test_evolution.py, tests/test_gpu_nsga.py).  The default optimiser of suggest() is the one-pass Sobol
mega-batch.
"""
from __future__ import annotations

from typing import Callable, Optional

import numpy as np


def dominance_matrix(F: np.ndarray) -> np.ndarray:
    """D[i, j] = True iff row i dominates row j (all <=, one <), minimisation."""
    le = (F[:, None, :] <= F[None, :, :]).all(-1)
    lt = (F[:, None, :] < F[None, :, :]).any(-1)
    return le & lt


def fast_non_dominated_sort(F: np.ndarray) -> np.ndarray:
    """Front index (0 = non-dominated) of every row."""
    n = F.shape[0]
    D = dominance_matrix(F)
    n_dom = D.sum(0).astype(np.int64)          # how many rows dominate j
    rank = np.full(n, -1, dtype=np.int64)
    current = np.flatnonzero(n_dom == 0)
    r = 0
    while current.size:
        rank[current] = r
        n_dom[current] = -1                    # never selected again
        n_dom -= D[current].sum(0)             # remove their dominance (entries already at -1 only go lower)
        current = np.flatnonzero(n_dom == 0)
        r += 1
    return rank


def crowding_distance(F: np.ndarray) -> np.ndarray:
    """Crowding distance inside ONE front (boundary points get +inf)."""
    n, m = F.shape
    if n <= 2:
        return np.full(n, np.inf)
    dist = np.zeros(n)
    for k in range(m):
        order = np.argsort(F[:, k], kind="stable")
        f = F[order, k]
        span = f[-1] - f[0]
        d = np.zeros(n)
        d[0] = d[-1] = np.inf
        if span > 0:
            d[1:-1] = (f[2:] - f[:-2]) / span
        dist[order] += d
    return dist


def rank_and_crowding_survival(F: np.ndarray, n_survive: int) -> np.ndarray:
    """Indices of the survivors: whole fronts in rank order, the last one truncated by descending crowding distance."""
    rank = fast_non_dominated_sort(F)
    keep = []
    for r in range(rank.max() + 1):
        front = np.flatnonzero(rank == r)
        if len(keep) + front.size <= n_survive:
            keep.extend(front.tolist())
        else:
            cd = crowding_distance(F[front])
            order = np.argsort(-cd, kind="stable")
            keep.extend(front[order[: n_survive - len(keep)]].tolist())
        if len(keep) >= n_survive:
            break
    return np.asarray(keep, dtype=np.int64)


def constraint_violation(G: np.ndarray) -> np.ndarray:
    """cv = sum_j max(0, g_j) per row (pymoo 0.6 calc_cv as recalled; pymoo is not installed).  A NaN propagates."""
    G = np.asarray(G)
    return np.where(np.isnan(G), G, np.maximum(G, 0)).sum(1) if G.shape[1] else np.zeros(G.shape[0], dtype=G.dtype)


def constrained_front(F: np.ndarray, cv: Optional[np.ndarray] = None) -> np.ndarray:
    """Ascending indices of the non-dominated FEASIBLE rows of F [m, K] (cv <= 0; a NaN objective or cv excludes a row).
    With no feasible row: the single row of least cv, lowest index on ties (pymoo's filter_optimum(least_infeasible=True)
    behind res.X, as recalled).  The host restatement of hb_pareto_front."""
    F = np.asarray(F, dtype=np.float64)
    m = F.shape[0]
    ok = ~np.isnan(F).any(1)
    if cv is not None:
        cv = np.asarray(cv, dtype=np.float64).reshape(-1)
        ok &= ~np.isnan(cv)
    feas = ok & (cv <= 0) if cv is not None else ok
    idx = np.flatnonzero(feas)
    if idx.size:
        # rows in ascending objective sum (a dominator's sum is smaller), in blocks: each row is tested against the front
        # found so far and against its own block
        order = idx[np.argsort(F[idx].sum(1), kind="stable")]
        front = np.zeros(0, dtype=np.int64)
        for b in range(0, order.size, 1024):
            blk = order[b:b + 1024]
            Fb = F[blk]
            dom = np.zeros(blk.size, dtype=bool)
            for f0 in range(0, front.size, 1024):
                Ff = F[front[f0:f0 + 1024]]
                dom |= ((Ff[:, None, :] <= Fb[None]).all(-1) & (Ff[:, None, :] < Fb[None]).any(-1)).any(0)
            blk = blk[~dom]                                  # (a block row the front dominates dominates nothing new)
            front = np.concatenate([front, blk[~dominance_matrix(F[blk]).any(0)]])
        return np.sort(front)
    if cv is None or not ok.any():
        return np.zeros(0, dtype=np.int64)
    cand = np.flatnonzero(ok)
    return cand[[int(np.argmin(np.maximum(cv[cand], 0)))]]                 # argmin: first of the ties


def constrained_rank_and_crowding_survival(F: np.ndarray, cv: Optional[np.ndarray], n_survive: int) -> np.ndarray:
    """Survivors of the merged population under pymoo's filter_infeasible rule (Survival.do, as recalled): feasible rows
    (cv <= 0, finite objectives) by rank-and-crowding for min(n_feasible, n_survive) slots, then the other rows in
    ascending cv (lower index first), rows with a non-finite objective or a NaN cv last.  Ascending indices.  Without cv: the
    unconstrained survival with every non-finite row at +inf.  The host restatement of hb_nsga2_survive_k."""
    F = np.asarray(F, dtype=np.float64)
    finite = np.isfinite(F).all(1)
    Fi = np.where(finite[:, None], F, np.inf)
    if cv is None:
        return np.sort(rank_and_crowding_survival(Fi, n_survive))
    cv = np.asarray(cv, dtype=np.float64).reshape(-1)
    bad = ~finite | np.isnan(cv)
    feas = ~bad & (cv <= 0)
    fi = np.flatnonzero(feas)
    keep = fi[rank_and_crowding_survival(Fi[fi], min(fi.size, n_survive))].tolist() if fi.size else []
    rest = np.flatnonzero(~feas)
    key = np.where(bad[rest], 0.0, cv[rest])
    order = np.lexsort((rest, key, bad[rest]))                              # (bad, cv, index)
    keep += rest[order[: n_survive - len(keep)]].tolist()
    return np.sort(np.asarray(keep, dtype=np.int64))


class EvolutionOpt:
    def __init__(self, lb, ub, acq_fn: Callable[[np.ndarray], np.ndarray], pop: int = 100, iters: int = 100,
                 seed: Optional[int] = None, sbx_eta: float = 15.0, sbx_prob: float = 0.9, sbx_prob_var: float = 0.5,
                 pm_eta: float = 20.0, pm_prob_var: Optional[float] = None):
        self.lb = np.asarray(lb, dtype=np.float64).reshape(-1)
        self.ub = np.asarray(ub, dtype=np.float64).reshape(-1)
        assert self.lb.shape == self.ub.shape and (self.ub > self.lb).all()
        self.d = self.lb.size
        self.acq_fn = acq_fn
        self.pop, self.iters = int(pop), int(iters)
        self.rng = np.random.default_rng(seed)
        self.sbx_eta, self.sbx_prob, self.sbx_prob_var = sbx_eta, sbx_prob, sbx_prob_var
        self.pm_eta = pm_eta
        self.pm_prob_var = min(0.5, 1.0 / self.d) if pm_prob_var is None else pm_prob_var
        self.n_evals = 0

    # ------------------------------------------------------------------ variation operators
    def _sbx(self, P1: np.ndarray, P2: np.ndarray):
        """Simulated binary crossover with bounds (Deb & Agrawal); returns two children per parent pair."""
        rng, eta = self.rng, self.sbx_eta
        n, d = P1.shape
        lo, hi = self.lb[None, :], self.ub[None, :]
        y1, y2 = np.minimum(P1, P2), np.maximum(P1, P2)
        diff = y2 - y1
        do = (rng.random((n, 1)) < self.sbx_prob) & (rng.random((n, d)) < self.sbx_prob_var) & (diff > 1e-14)
        safe = np.where(diff > 1e-14, diff, 1.0)
        u = rng.random((n, d))

        def betaq(beta):
            alpha = 2.0 - np.power(beta, -(eta + 1.0))
            inner = np.where(u <= 1.0 / alpha, u * alpha, 1.0 / np.maximum(2.0 - u * alpha, 1e-300))
            return np.power(inner, 1.0 / (eta + 1.0))
        c1 = 0.5 * ((y1 + y2) - betaq(1.0 + 2.0 * (y1 - lo) / safe) * diff)
        c2 = 0.5 * ((y1 + y2) + betaq(1.0 + 2.0 * (hi - y2) / safe) * diff)
        swap = rng.random((n, d)) < 0.5
        c1, c2 = np.where(swap, c2, c1), np.where(swap, c1, c2)
        C1 = np.where(do, c1, P1)
        C2 = np.where(do, c2, P2)
        return np.clip(C1, lo, hi), np.clip(C2, lo, hi)

    def _pm(self, X: np.ndarray) -> np.ndarray:
        """Polynomial mutation (Deb & Goyal)."""
        rng, eta = self.rng, self.pm_eta
        lo, hi = self.lb[None, :], self.ub[None, :]
        span = hi - lo
        do = rng.random(X.shape) < self.pm_prob_var
        u = rng.random(X.shape)
        d1, d2 = (X - lo) / span, (hi - X) / span
        mp = 1.0 / (eta + 1.0)
        low = np.power(2.0 * u + (1.0 - 2.0 * u) * np.power(1.0 - d1, eta + 1.0), mp) - 1.0
        high = 1.0 - np.power(2.0 * (1.0 - u) + 2.0 * (u - 0.5) * np.power(1.0 - d2, eta + 1.0), mp)
        dq = np.where(u < 0.5, low, high)
        return np.clip(np.where(do, X + dq * span, X), lo, hi)

    def _offspring(self, X: np.ndarray, n_off: int) -> np.ndarray:
        """Random mating until n_off non-duplicate children exist (a bounded number of rounds, like pymoo's infill)."""
        kids = np.zeros((0, self.d))
        for _ in range(10):
            need = n_off - kids.shape[0]
            if need <= 0:
                break
            n_pairs = (need + 1) // 2
            a = self.rng.integers(0, X.shape[0], n_pairs)
            b = self.rng.integers(0, X.shape[0], n_pairs)
            c1, c2 = self._sbx(X[a], X[b])
            new = self._pm(np.concatenate([c1, c2], 0))
            # duplicate elimination against the population, the accepted children and inside the new batch
            ref = np.concatenate([X, kids], 0)
            dup = (np.abs(new[:, None, :] - ref[None, :, :]).max(-1) <= 1e-16).any(1)
            _, first = np.unique(new.round(16), axis=0, return_index=True)
            uniq = np.zeros(new.shape[0], dtype=bool)
            uniq[first] = True
            kids = np.concatenate([kids, new[~dup & uniq]], 0)
        return kids[:n_off]

    # ------------------------------------------------------------------ main loop
    def _eval(self, X: np.ndarray) -> np.ndarray:
        F = np.asarray(self.acq_fn(X.astype(np.float32)), dtype=np.float64).reshape(X.shape[0], -1)
        self.n_evals += X.shape[0]
        return np.where(np.isfinite(F), F, np.inf)

    def optimize(self, initial_suggest: Optional[np.ndarray] = None, return_pop: bool = False) -> np.ndarray:
        X = self.lb + (self.ub - self.lb) * self.rng.random((self.pop, self.d))      # evolution_optimizer.py:44-55 (uniform)
        if initial_suggest is not None:
            init = np.clip(np.asarray(initial_suggest, dtype=np.float64).reshape(-1, self.d), self.lb, self.ub)
            X = np.concatenate([init, X], 0)[: self.pop]                              # :56-57 prepend + truncate
        F = self._eval(X)
        for _ in range(self.iters - 1):                                               # ('n_gen', iters): gen 1 = the initial pop
            kids = self._offspring(X, self.pop)
            if kids.shape[0] == 0:
                break
            Fk = self._eval(kids)
            Xa, Fa = np.concatenate([X, kids], 0), np.concatenate([F, Fk], 0)
            keep = rank_and_crowding_survival(Fa, self.pop)
            X, F = Xa[keep], Fa[keep]
        self.pop_X, self.pop_F = X, F
        if return_pop:
            return X
        nd = fast_non_dominated_sort(F) == 0                                          # res.X: non-dominated members
        return X[nd]


class DeviceNSGA2:
    """NSGA-II with the population resident on the GPU (include/hebo_b200.h "device NSGA-II").

    kinds [D]: 'real' | 'int' | 'choice' per optimisation column (numeric columns first, then the categorical ones:
    evolution_optimizer.py:26-41); lb / ub [D]; fixed: {column index: value} (fix_input, :97-101).  `score(Xc, Xe, gen)`
    returns the objectives F [pop, num_obj] of a batch as a device tensor (the fused posterior + MACE call for the default
    num_obj = 3), or a pair (F, cv) with the constraint violation cv [pop] (GeneralAcq): survival then follows pymoo's
    filter_infeasible rule and the result is the constrained front (hb_nsga2_survive_k, hb_pareto_front)."""

    KIND = {"real": 0, "int": 1, "choice": 2}

    def __init__(self, kinds, lb, ub, num_numeric: int, score: Callable, pop: int = 100, iters: int = 100,
                 seed: Optional[int] = None, fixed: Optional[dict] = None, device="cuda", num_obj: int = 3):
        import torch
        self.torch = torch
        self.num_obj = int(num_obj)
        assert 1 <= self.num_obj <= 8
        self.D, self.d, self.pop, self.iters = len(kinds), int(num_numeric), int(pop), int(iters)
        assert 2 * self.pop <= 512 and self.pop >= 2
        dev = torch.device(device)
        self.dev = dev
        self.kind = torch.tensor([self.KIND[k] for k in kinds], dtype=torch.int32, device=dev)
        self.lb = torch.as_tensor(np.asarray(lb, dtype=np.float32)).to(dev)
        self.ub = torch.as_tensor(np.asarray(ub, dtype=np.float32)).to(dev)
        fx = np.full(self.D, np.nan, dtype=np.float32)
        for k, v in (fixed or {}).items():
            fx[k] = v
        self.fixed = torch.from_numpy(fx).to(dev)
        self.score = score
        self.seed = int(np.random.randint(0, 2 ** 31 - 1)) if seed is None else int(seed)
        self.n_evals = 0

    def _bufs(self):
        t, dev, P, D, d = self.torch, self.dev, self.pop, self.D, self.d
        return (t.empty(P, D, device=dev), t.empty(P, max(d, 1), device=dev)[:, :d].contiguous() if d else t.empty(P, 0, device=dev),
                t.empty(P, D - d, dtype=t.int32, device=dev))

    def optimize(self, initial_suggest=None):
        """Returns (Xc [K, d] fp32, Xe [K, e] int32, F [K, num_obj]) of the non-dominated members of the final population
        (res.X of evolution_optimizer.py:141-149; with constraints the feasible front, or the least-infeasible member when
        none is feasible), all on the device.  With constraints `self.pop_cv` holds the final population's cv."""
        from . import _lib
        from .pareto import pareto_front
        t, lib, P, D, d, K = self.torch, _lib.lib(), self.pop, self.D, self.d, self.num_obj
        st = _lib.stream_ptr
        X, Xc, Xe = self._bufs()
        Xn, Xcn, Xen = self._bufs()
        C, Cc, Ce = self._bufs()
        init = None if initial_suggest is None else t.as_tensor(np.asarray(initial_suggest, dtype=np.float32).reshape(-1, D)).to(self.dev)
        n_init = 0 if init is None else min(init.shape[0], P)
        pc = lambda x: _lib.ptr(x) if x.numel() else None

        def scored(xc, xe, gen):
            out = self.score(xc, xe, gen)
            F, cv = out if isinstance(out, tuple) else (out, None)
            F = F.contiguous()
            assert F.shape[1] == K, f"score returned {F.shape[1]} objectives, expected {K}"
            return F, (None if cv is None else cv.reshape(-1).contiguous())
        with t.cuda.device(self.dev):
            _lib.check(lib.hb_nsga2_init(_lib.ptr(X), P, D, d, _lib.ptr(self.kind), _lib.ptr(self.lb), _lib.ptr(self.ub), _lib.ptr(self.fixed),
                                         _lib.ptr(init), n_init, self.seed, pc(Xc), pc(Xe), st()), "hb_nsga2_init")
            F, cv = scored(Xc, Xe, 0)
            Fn = t.empty_like(F)
            cvn = None if cv is None else t.empty_like(cv)
            self.n_evals = P
            for gen in range(1, self.iters):                       # ('n_gen', iters): generation 1 is the initial population
                _lib.check(lib.hb_nsga2_mate(_lib.ptr(X), P, D, d, _lib.ptr(self.kind), _lib.ptr(self.lb), _lib.ptr(self.ub),
                                             _lib.ptr(self.fixed), self.seed, gen, _lib.ptr(C), pc(Cc), pc(Ce), st()), "hb_nsga2_mate")
                FC, cvc = scored(Cc, Ce, gen)
                if K == 3 and cv is None:                          # the MACE path
                    _lib.check(lib.hb_nsga2_survive(_lib.ptr(X), _lib.ptr(F), _lib.ptr(C), _lib.ptr(FC), P, D, d, _lib.ptr(Xn), _lib.ptr(Fn),
                                                    pc(Xcn), pc(Xen), st()), "hb_nsga2_survive")
                else:
                    _lib.check(lib.hb_nsga2_survive_k(_lib.ptr(X), _lib.ptr(F), _lib.ptr(cv), _lib.ptr(C), _lib.ptr(FC), _lib.ptr(cvc), P, D, d,
                                                      K, _lib.ptr(Xn), _lib.ptr(Fn), _lib.ptr(cvn), pc(Xcn), pc(Xen), st()),
                               "hb_nsga2_survive_k")
                X, Xn, Xc, Xcn, Xe, Xen, F, Fn, cv, cvn = Xn, X, Xcn, Xc, Xen, Xe, Fn, F, cvn, cv
                self.n_evals += P
        self.pop_X, self.pop_F, self.pop_cv = X, F, cv
        idx = pareto_front(F, cv)
        return Xc[idx], Xe[idx], F[idx]
