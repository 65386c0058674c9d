"""GeneralAcq epilogue, K-objective constrained front and survival, GeneralBO end to end (hebo_b200/csrc/posterior.cu
general_acq_kernel, pareto.cu, nsga.cu) against the host restatements and the reference's stored outputs."""
import os

import numpy as np
import pandas as pd
import pytest
import torch

import hebo_b200
from hebo_b200 import _lib
from hebo_b200.acq import GeneralAcq
from hebo_b200.evolution import constrained_front, constrained_rank_and_crowding_survival, dominance_matrix
from hebo_b200.general import GeneralBO
from hebo_b200.pareto import pareto_front, pareto_front_device
from oracle.general_acq_oracle import constraint_violation, general_acq

pytestmark = pytest.mark.gpu


def _assert_acq_close(out, ref, mu, var, noise, xi, no, kappa, c_kappa, use_noise):
    """Equal to the reference up to one ulp of ps carried through k ps, plus one rounding each of k ps, py and the result:
    the device sqrtf is correctly rounded, torch's CPU sqrt is occasionally one ulp off (the same allowance as the sigma
    column of the front buffers); every other step is the same IEEE fp32 operation in the same order."""
    mu, var, xi = (np.asarray(a, dtype=np.float32) for a in (mu, var, xi))
    O = mu.shape[1]
    k = np.where(np.arange(O) < no, np.float32(kappa), np.float32(c_kappa)).astype(np.float32)
    ps = np.maximum(np.sqrt(var), np.float32(1.1920929e-07))
    py = np.abs(mu) + (np.abs(np.sqrt(np.asarray(noise, dtype=np.float32))[None, :] * xi) if use_noise else 0)
    kps = (np.abs(k)[None, :] * ps).astype(np.float32)
    tol = (np.abs(k)[None, :].astype(np.float64) * np.spacing(ps) + np.spacing(kps) + np.spacing(py.astype(np.float32))
           + np.spacing(np.abs(ref.numpy())))
    assert (np.abs(out.double().numpy() - ref.double().numpy()) <= tol).all()


def _epilogue(mu, var, no, nc, noise, kappa, c_kappa, use_noise, xi=None, seed=0):
    m = mu.shape[0]
    O = no + nc
    mu_d = torch.as_tensor(mu).t().contiguous().cuda()
    var_d = torch.as_tensor(var).t().contiguous().cuda()
    nz = torch.as_tensor(noise, dtype=torch.float32).cuda()
    xi_d = None if xi is None else torch.as_tensor(xi, dtype=torch.float32).contiguous().cuda()
    out = torch.empty(m, O, device="cuda")
    cv = torch.empty(m, device="cuda")
    _lib.check(_lib.lib().hb_general_acq_epilogue(_lib.ptr(mu_d), _lib.ptr(var_d), m, no, nc, _lib.ptr(nz), float(kappa), float(c_kappa),
                                                  int(use_noise), _lib.ptr(xi_d), seed, 0, _lib.ptr(out), _lib.ptr(cv),
                                                  _lib.stream_ptr()), "general_acq")
    return out.cpu(), cv.cpu()


def test_epilogue_matches_the_reference_outputs_and_cv_is_exact():
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_general_acq.npz"))
    for i in range(int(z["n_cases"])):
        c = {k[len(f"c{i}_"):]: z[k] for k in z.files if k.startswith(f"c{i}_")}
        no, nc, kappa, c_kappa, use_noise = c["conf"]
        out, cv = _epilogue(c["mu"], c["var"], int(no), int(nc), c["noise"], kappa, c_kappa, bool(use_noise), c["xi"])
        ref = torch.from_numpy(c["out"])
        _assert_acq_close(out, ref, c["mu"], c["var"], c["noise"], c["xi"], int(no), kappa, c_kappa, bool(use_noise))
        assert np.array_equal(cv.numpy(), constraint_violation(out, int(no))), i


def test_epilogue_philox_is_deterministic_and_independent():
    m, no, nc = 200000, 2, 3
    mu, var = torch.zeros(m, 5), torch.full((m, 5), 1e-20)
    a, _ = _epilogue(mu, var, no, nc, [1.0] * 5, 0.0, 0.0, True, seed=7)
    b, _ = _epilogue(mu, var, no, nc, [1.0] * 5, 0.0, 0.0, True, seed=7)
    c, _ = _epilogue(mu, var, no, nc, [1.0] * 5, 0.0, 0.0, True, seed=8)
    assert torch.equal(a, b) and not torch.equal(a, c)
    z = a.double()
    assert float(z.mean(0).abs().max()) < 0.01 and float((z.var(0) - 1).abs().max()) < 0.02
    corr = torch.corrcoef(z.t())
    assert float((corr - torch.eye(5, dtype=torch.float64)).abs().max()) < 0.01          # across outputs
    assert abs(float(torch.corrcoef(torch.stack([z[1:, 0], z[:-1, 0]]))[0, 1])) < 0.01    # across rows


def test_dummy_model_case_of_the_reference():
    from hebo_b200.base import BaseModel

    class Dummy(BaseModel):
        support_multi_output = True

        def __init__(self):
            super().__init__(3, 0, 7)

        def fit(self, *a):
            pass

        def predict(self, x, _):
            return torch.zeros(x.shape[0], 7), torch.ones(x.shape[0], 7)

        @property
        def noise(self):
            return torch.zeros(7)
    acq = GeneralAcq(Dummy(), 3, 4, kappa=3, c_kappa=4, use_noise=True)
    v = acq(torch.randn(10, 3), torch.ones(10, 3).long())
    assert (v[:, :3] + 3).abs().max() < 1e-6 and (v[:, 3:] + 4).abs().max() < 1e-6
    assert acq.num_obj == 3 and acq.num_constr == 4


def _front_cases(K, m, rng):
    F = rng.normal(size=(m, K)).astype(np.float32)
    if m > 5000:                                                                    # correlated objectives: a short front
        F = (rng.normal(size=(m, 1)) + 0.3 * F).astype(np.float32)
    elif K >= 2:
        F[:, -1] = (-F[:, :-1].sum(1) + 0.3 * F[:, -1]).astype(np.float32)            # a real trade-off surface
    if m >= 8:
        F[5] = F[2]                                                                 # duplicates
        F[6, 0] = np.nan
    cv_mixed = np.where(rng.random(m) < 0.5, rng.random(m).astype(np.float32), 0).astype(np.float32)
    if m >= 8:
        cv_mixed[4] = np.nan
    cv_inf = (rng.random(m) + 0.5).astype(np.float32)
    if m >= 8:
        cv_inf[[3, 7]] = cv_inf.min() / 2
    return F, {"none": None, "mixed": cv_mixed, "infeasible": cv_inf}


@pytest.mark.parametrize("K", [1, 2, 3, 4, 6, 8])
@pytest.mark.parametrize("m", [1, 7, 4096, 4097, 300000])
def test_pareto_front_equals_constrained_front(K, m):
    rng = np.random.default_rng(K * 1000 + m % 997)
    F, cases = _front_cases(K, m, rng)
    Fd = torch.from_numpy(F).cuda()
    for name, cv in cases.items():
        cvd = None if cv is None else torch.from_numpy(cv).cuda()
        got = pareto_front(Fd, cvd).cpu().numpy()
        assert np.array_equal(got, constrained_front(F, cv)), (name, K, m)
    if K == 3:
        i3, c3 = pareto_front_device(Fd)
        lib = _lib.lib()
        ws = torch.empty(int(lib.hb_pareto_workspace_bytes(m)), dtype=torch.uint8, device="cuda")
        idx = torch.empty(m, dtype=torch.int32, device="cuda")
        cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
        _lib.check(lib.hb_pareto_front(_lib.ptr(Fd), m, 3, 3, None, _lib.ptr(idx), _lib.ptr(cnt), _lib.ptr(ws), ws.numel(),
                                       _lib.stream_ptr()), "front")
        assert int(cnt) == int(c3) and torch.equal(idx[:int(cnt)], i3[:int(c3)])


@pytest.mark.parametrize("K,O", [(2, 5), (3, 7), (1, 2)])
def test_pareto_front_reads_a_column_slice_in_place(K, O):
    rng = np.random.default_rng(O)
    out = torch.from_numpy(rng.normal(size=(20000, O)).astype(np.float32)).cuda()
    cv = torch.clamp(out[:, K:], min=0).sum(1).contiguous()
    got = pareto_front(out[:, :K], cv).cpu().numpy()
    assert np.array_equal(got, constrained_front(out[:, :K].cpu().numpy(), cv.cpu().numpy()))


def test_pareto_front_rejects_bad_arguments():
    lib = _lib.lib()
    F = torch.zeros(16, 9, device="cuda")
    ws = torch.empty(int(lib.hb_pareto_workspace_bytes(16)), dtype=torch.uint8, device="cuda")
    idx, cnt = torch.empty(16, dtype=torch.int32, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
    for K, ldf in [(0, 9), (9, 9), (4, 3)]:
        assert lib.hb_pareto_front(_lib.ptr(F), 16, K, ldf, None, _lib.ptr(idx), _lib.ptr(cnt), _lib.ptr(ws), ws.numel(), None) == _lib.HB_ERR_INVALID
    assert lib.hb_pareto_front(None, 16, 2, 2, None, _lib.ptr(idx), _lib.ptr(cnt), _lib.ptr(ws), ws.numel(), None) == _lib.HB_ERR_INVALID
    assert lib.hb_general_acq_epilogue(None, None, 16, 1, 0, None, 1.0, 0.0, 0, None, 0, 0, None, None, None) == _lib.HB_ERR_INVALID
    assert lib.hb_nsga2_survive_k(*([None] * 6), 8, 2, 1, 9, *([None] * 6)) == _lib.HB_ERR_INVALID


def _survive(X, F, CV, C, FC, CVC, P, D, d, K):
    dev = "cuda"
    Xn, Fn, CVn = torch.empty(P, D, device=dev), torch.empty(P, K, device=dev), torch.empty(P, device=dev)
    Xcn, Xen = torch.empty(P, d, device=dev), torch.empty(P, D - d, dtype=torch.int32, device=dev)
    t = [None if a is None else a.contiguous().cuda() for a in (X, F, CV, C, FC, CVC)]
    _lib.check(_lib.lib().hb_nsga2_survive_k(*[_lib.ptr(a) for a in t], P, D, d, K, _lib.ptr(Xn), _lib.ptr(Fn),
                                             _lib.ptr(CVn) if CV is not None else None, _lib.ptr(Xcn), _lib.ptr(Xen),
                                             _lib.stream_ptr()), "survive_k")
    torch.cuda.synchronize()
    return Xn.cpu(), Fn.cpu(), CVn.cpu(), Xcn.cpu(), Xen.cpu()


@pytest.mark.parametrize("K", [1, 2, 3, 5])
@pytest.mark.parametrize("constrained", [False, True])
@pytest.mark.parametrize("P,D,seed", [(100, 5, 0), (64, 3, 1), (7, 2, 2), (256, 4, 3)])
def test_survival_k_equals_the_host_rule(K, constrained, P, D, seed):
    g = torch.Generator().manual_seed(seed + 10 * K)
    X, C = torch.rand(P, D, generator=g), torch.rand(P, D, generator=g)
    F, FC = torch.randn(P, K, generator=g), torch.randn(P, K, generator=g)
    if K >= 2:
        F[:, -1] = -F[:, :-1].sum(1) + 0.2 * F[:, -1]
        FC[:, -1] = -FC[:, :-1].sum(1) + 0.2 * FC[:, -1] + 0.1
    if P >= 64:
        C[3] = X[5]                                              # a duplicate child
        FC[7, :] = float("nan")                                  # NaN objectives
        F[:, 0] = torch.round(F[:, 0] * 4) / 4                   # ties
    CV = CVC = None
    if constrained:
        CV = torch.where(torch.rand(P, generator=g) < 0.6, torch.rand(P, generator=g), torch.zeros(P))
        CVC = torch.where(torch.rand(P, generator=g) < 0.6, torch.rand(P, generator=g), torch.zeros(P))
        if P >= 64:
            CVC[9] = float("nan")
            CV[11] = CV[12]
    d = D - 1
    Xn, Fn, CVn, Xcn, Xen = _survive(X, F, CV, C, FC, CVC, P, D, d, K)
    Fa = torch.cat([F, FC], 0).double().numpy()
    if P >= 64:
        Fa[P + 3] = np.inf
    cva = None if CV is None else torch.cat([CV, CVC]).double().numpy()
    keep = constrained_rank_and_crowding_survival(Fa, cva, P)
    Xa = torch.cat([X, C], 0)
    assert torch.equal(Xn, Xa[keep])
    Fe = np.where(np.isfinite(Fa), Fa, np.inf)[keep]
    if constrained and P >= 64:
        Fe[keep == P + 3] = np.inf
    assert torch.equal(Fn.double(), torch.from_numpy(Fe))
    if constrained:
        assert torch.equal(CVn, torch.cat([CV, CVC])[keep])
    assert torch.equal(Xcn, Xa[keep][:, :d]) and torch.equal(Xen.reshape(-1), Xa[keep][:, d].round().int())


@pytest.mark.parametrize("P,D,seed", [(100, 5, 0), (64, 3, 1), (7, 2, 2), (256, 4, 3)])
def test_survival_k3_unconstrained_is_bit_identical_to_the_mace_entry(P, D, seed):
    g = torch.Generator().manual_seed(seed)
    X, C = torch.rand(P, D, generator=g), torch.rand(P, D, generator=g)
    F, FC = torch.randn(P, 3, generator=g), torch.randn(P, 3, generator=g)
    if P >= 64:
        C[3] = X[5]
        FC[7, 1] = float("nan")
    d = D - 1
    a = _survive(X, F, None, C, FC, None, P, D, d, 3)
    dev = "cuda"
    Xn, Fn = torch.empty(P, D, device=dev), torch.empty(P, 3, device=dev)
    Xcn, Xen = torch.empty(P, d, device=dev), torch.empty(P, 1, dtype=torch.int32, device=dev)
    Xd, Fd, Cd, FCd = X.cuda(), F.cuda(), C.cuda(), FC.cuda()
    _lib.check(_lib.lib().hb_nsga2_survive(_lib.ptr(Xd), _lib.ptr(Fd), _lib.ptr(Cd), _lib.ptr(FCd), P, D, d, _lib.ptr(Xn),
                                           _lib.ptr(Fn), _lib.ptr(Xcn), _lib.ptr(Xen), _lib.stream_ptr()), "survive")
    torch.cuda.synchronize()
    assert torch.equal(a[0], Xn.cpu()) and torch.equal(a[1], Fn.cpu()) and torch.equal(a[3], Xcn.cpu()) and torch.equal(a[4], Xen.cpu())


def test_general_acq_multitask_device_path_equals_predict_through_the_restatement():
    torch.manual_seed(0)
    n, d, m = 600, 4, 40000
    X = torch.rand(n, d) * 2 - 1
    y = torch.stack([torch.sin(3 * X[:, 0]) + X[:, 1], (X ** 2).sum(1), X[:, 2] - 0.3 * X[:, 3]], 1)
    model = hebo_b200.MultiTaskModel(d, 0, 3, num_epochs=10, pred_likeli=False)
    model.fit(X, None, y)
    Xs = torch.rand(m, d) * 2 - 1
    acq = GeneralAcq(model, 2, 1, kappa=1.7, c_kappa=0.6, use_noise=True)
    torch.manual_seed(5)
    out, cv = acq.evaluate(Xs, None, return_cv=True)
    torch.manual_seed(5)
    xi = torch.randn(m, 3)
    py, ps2 = model.predict(Xs, None)
    ref = general_acq(py, ps2, model.noise, xi, 2, 1.7, 0.6, True)
    assert out.shape == (m, 3) and not out.is_cuda
    _assert_acq_close(out, ref, py, ps2, model.noise, xi, 2, 1.7, 0.6, True)
    assert np.array_equal(cv.numpy(), constraint_violation(out, 2))
    outd = acq.evaluate(Xs.cuda(), None)
    assert outd.is_cuda and outd.shape == (m, 3)


def _hv2(Y, ref):
    """Exact 2-D hypervolume (minimisation) of the points of Y dominating ref."""
    Y = np.asarray(Y, dtype=np.float64)
    Y = Y[(Y < ref).all(1)]
    if Y.shape[0] == 0:
        return 0.0
    Y = Y[np.argsort(Y[:, 0])]
    hv, best1 = 0.0, ref[1]
    for y0, y1 in Y:
        if y1 < best1:
            hv += (ref[0] - y0) * (best1 - y1)
            best1 = y1
    return hv


@pytest.mark.parametrize("optimizer", ["sobol", "nsga2"])
@pytest.mark.parametrize("q", [1, 4, 50])
def test_general_mo_constrained_opt(optimizer, q):
    """HEBO/test/test_optimizer.py:136-151 shape: 1-D, 2 objectives + 1 constraint, evo_pop 20."""
    np.random.seed(q)
    torch.manual_seed(q)

    def f(param):
        x = param[["x0"]].values.astype(float)
        return np.hstack([x ** 2, (x - 3) * 2, -10 - x])
    opt = GeneralBO([{"name": "x0", "type": "num", "lb": -1, "ub": 4.0}], 2, 1, rand_sample=4, acq_optimizer=optimizer,
                    evo_pop=20, evo_iters=30, n_candidates=2048, scramble_seed=q)
    for _ in range(2):
        rec = opt.suggest(q)
        assert len(rec) == q and bool(((rec["x0"] >= -1) & (rec["x0"] <= 4)).all())
        opt.observe(rec, f(rec))
    assert opt.y.shape == (2 * q, 3)


def _binh_korn(df):
    x, yv = df["x"].values.astype(float), df["y"].values.astype(float)
    pen = np.array([{"a": 0.0, "b": 4.0, "c": 10.0}[c] for c in df["c"]])
    f1 = 4 * x ** 2 + 4 * yv ** 2 + pen
    f2 = (x - 5) ** 2 + (yv - 5) ** 2 + pen
    g1 = (x - 5) ** 2 + yv ** 2 - 25
    g2 = 7.7 - (x - 8) ** 2 - (yv + 3) ** 2
    return np.stack([f1 / 50, f2 / 50, g1 / 25, g2 / 25], 1)


@pytest.mark.parametrize("optimizer", ["sobol", "nsga2"])
def test_constrained_binh_korn_on_a_mixed_space(optimizer):
    np.random.seed(1)
    torch.manual_seed(1)
    space = [{"name": "x", "type": "num", "lb": 0, "ub": 5}, {"name": "y", "type": "num", "lb": 0, "ub": 3},
             {"name": "k", "type": "int", "lb": 0, "ub": 4}, {"name": "c", "type": "cat", "categories": ["a", "b", "c"]}]
    opt = GeneralBO(space, 2, 2, acq_optimizer=optimizer, evo_pop=40, evo_iters=30, n_candidates=4096, scramble_seed=3,
                    model_config={"num_epochs": 60})
    for it in range(10):
        fix = {"c": "a"} if it == 9 else None
        rec = opt.suggest(4, fix_input=fix)
        assert len(rec) == 4 and set(rec["c"]) <= {"a", "b", "c"}
        assert bool(((rec["x"] >= 0) & (rec["x"] <= 5) & (rec["y"] >= 0) & (rec["y"] <= 3)).all())
        assert all(float(v).is_integer() and 0 <= v <= 4 for v in rec["k"])
        if fix:
            assert set(rec["c"]) == {"a"}
        y = _binh_korn(rec)
        if it == 5:
            y[0, 1] = np.inf
        opt.observe(rec, y)
        if it == 0:
            start = opt.y.copy()
    assert opt.y.shape[0] == 39
    by = opt.best_y
    assert by.shape[0] >= 1 and (by[:, 2:] <= 0).all() and not dominance_matrix(by[:, :2]).any()
    ref = np.array([3.0, 3.0])
    start_pf = start[(start[:, 2:] <= 0).all(1), :2]
    assert _hv2(by[:, :2], ref) > _hv2(start_pf, ref)


@pytest.mark.parametrize("optimizer", ["sobol", "nsga2"])
def test_single_objective_with_a_disc_constraint(optimizer):
    """Branin subject to (x1 - 2.5)^2 + (x2 - 7.5)^2 <= 9 (no unconstrained minimum lies in the disc; the constrained
    optimum, 4.78 on a 1501^2 grid, sits on its boundary): the best feasible observation is within 1.5 of it."""
    np.random.seed(2)
    torch.manual_seed(2)

    def f(df):
        x1, x2 = df["x1"].values.astype(float), df["x2"].values.astype(float)
        b = (x2 - 5.1 / (4 * np.pi ** 2) * x1 ** 2 + 5 / np.pi * x1 - 6) ** 2 + 10 * (1 - 1 / (8 * np.pi)) * np.cos(x1) + 10
        g = ((x1 - 2.5) ** 2 + (x2 - 7.5) ** 2 - 9) / 9
        return np.stack([b, g], 1)
    g1, g2 = np.meshgrid(np.linspace(-5, 10, 1501), np.linspace(0, 15, 1501))
    grid = pd.DataFrame({"x1": g1.ravel(), "x2": g2.ravel()})
    v = f(grid)
    best = v[v[:, 1] <= 0, 0].min()
    opt = GeneralBO([{"name": "x1", "type": "num", "lb": -5, "ub": 10}, {"name": "x2", "type": "num", "lb": 0, "ub": 15}],
                    1, 1, acq_optimizer=optimizer, evo_pop=40, evo_iters=40, n_candidates=4096, scramble_seed=4,
                    model_config={"num_epochs": 60})
    for _ in range(12):
        rec = opt.suggest(3)
        opt.observe(rec, f(rec))
    by = opt.best_y
    assert by.shape[0] >= 1 and (by[:, 1] <= 0).all()
    assert by[:, 0].min() < best + 1.5, (by[:, 0].min(), best)
