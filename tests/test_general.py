"""GeneralAcq / constrained front / constrained survival / GeneralBO: host logic and the oracle, CPU only."""
import numpy as np
import pandas as pd
import pytest
import torch

from hebo_b200.evolution import (constrained_front, constrained_rank_and_crowding_survival, constraint_violation,
                                 dominance_matrix, rank_and_crowding_survival)
from hebo_b200.general import GeneralBO, general_kappa
from oracle.general_acq_oracle import general_acq


def _ref_cases():
    import os
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_general_acq.npz"))
    return [{k[len(f"c{i}_"):]: z[k] for k in z.files if k.startswith(f"c{i}_")} for i in range(int(z["n_cases"]))]


def test_general_acq_restatement_equals_the_reference_outputs():
    for c in _ref_cases():
        no, nc, kappa, c_kappa, use_noise = c["conf"]
        out = general_acq(c["mu"], c["var"], c["noise"], c["xi"], int(no), float(kappa), float(c_kappa), bool(use_noise))
        ref = torch.from_numpy(c["out"])
        assert out.shape == ref.shape == (c["mu"].shape[0], int(no + nc))
        ulp = (out.view(torch.int32).long() - ref.view(torch.int32).long()).abs().max()
        assert int(ulp) <= 1


def brute_front(F, cv):
    """Definition: feasible rows (cv <= 0, no NaN) not dominated by any feasible row; else the least-cv row."""
    m = F.shape[0]
    ok = [not np.isnan(F[i]).any() and (cv is None or not np.isnan(cv[i])) for i in range(m)]
    feas = [i for i in range(m) if ok[i] and (cv is None or cv[i] <= 0)]
    if feas:
        return np.array([i for i in feas if not any((F[j] <= F[i]).all() and (F[j] < F[i]).any() for j in feas)], dtype=np.int64)
    cand = [i for i in range(m) if ok[i]]
    if cv is None or not cand:
        return np.zeros(0, dtype=np.int64)
    best = min(cand, key=lambda i: (max(cv[i], 0.0), i))
    return np.array([best])


@pytest.mark.parametrize("K", [1, 2, 3, 5])
@pytest.mark.parametrize("case", ["none", "mixed", "infeasible", "nan", "ties"])
def test_constrained_front_matches_brute_force(K, case):
    rng = np.random.default_rng(K * 10 + len(case))
    m = 60
    F = rng.integers(0, 5, size=(m, K)).astype(float) if case == "ties" else rng.normal(size=(m, K))
    cv = None
    if case in ("mixed", "ties", "nan"):
        cv = np.maximum(rng.normal(size=m), 0) * (rng.random(m) < 0.5)
    if case == "infeasible":
        cv = rng.random(m) + 0.1
        cv[[7, 30]] = cv.min() / 2                                 # tie at the least cv: lowest index wins
    if case == "nan":
        F[3, 0] = np.nan
        cv[5] = np.nan
    if case == "ties":
        F[10] = F[11]                                               # exact duplicates both stay
    got = constrained_front(F, cv)
    assert np.array_equal(got, brute_front(F, cv))
    if case == "infeasible":
        assert got.tolist() == [7]


def test_constrained_front_all_nan_is_empty():
    F = np.full((4, 2), np.nan)
    assert constrained_front(F, np.ones(4)).size == 0 and constrained_front(F).size == 0


def brute_survival(F, cv, n):
    finite = np.isfinite(F).all(1)
    bad = ~finite | np.isnan(cv)
    feas = np.flatnonzero(~bad & (cv <= 0))
    keep = []
    if feas.size:
        Ff = F[feas]
        keep = feas[rank_and_crowding_survival(Ff, min(feas.size, n))].tolist()
    rest = sorted(np.flatnonzero(~(~bad & (cv <= 0))).tolist(), key=lambda i: (bool(bad[i]), 0.0 if bad[i] else cv[i], i))
    keep += rest[: n - len(keep)]
    return np.sort(np.array(keep, dtype=np.int64))


@pytest.mark.parametrize("K", [1, 2, 3, 5])
@pytest.mark.parametrize("frac", [0.0, 0.3, 0.8, 1.0])
def test_constrained_survival_matches_the_filter_infeasible_rule(K, frac):
    rng = np.random.default_rng(K + int(frac * 10))
    N, n = 80, 40
    F = rng.normal(size=(N, K))
    F[:, 0] = np.round(F[:, 0] * 3) / 3                             # ties
    cv = np.where(rng.random(N) < frac, rng.random(N) + 0.01, 0.0)
    cv[[4, 9]] = cv[4]                                              # equal cv: index order
    F[12, K - 1] = np.nan                                           # non-finite objective: last
    cv[13] = np.nan                                                 # NaN cv: last
    F[14] = np.inf                                                  # a duplicate child arrives as +inf
    got = constrained_rank_and_crowding_survival(F, cv, n)
    assert got.size == n and np.array_equal(got, brute_survival(F, cv, n))
    n_feas = int(((cv <= 0) & np.isfinite(F).all(1)).sum())
    assert int(((cv[got] <= 0) & np.isfinite(F[got]).all(1)).sum()) == min(n_feas, n)
    if frac == 0.0:
        assert not {12, 13, 14} & set(got.tolist())                         # enough finite rows: the bad ones never survive


def test_unconstrained_survival_is_the_existing_rule():
    rng = np.random.default_rng(5)
    F = rng.normal(size=(50, 3))
    F[3, 1] = np.nan
    Fi = np.where(np.isfinite(F).all(1)[:, None], F, np.inf)
    assert np.array_equal(constrained_rank_and_crowding_survival(F, None, 25), np.sort(rank_and_crowding_survival(Fi, 25)))


def test_constraint_violation():
    G = np.array([[-1.0, 2.0], [0.5, 0.25], [np.nan, -1.0], [-1.0, -2.0]])
    cv = constraint_violation(G)
    assert cv[0] == 2.0 and cv[1] == 0.75 and np.isnan(cv[2]) and cv[3] == 0.0
    assert constraint_violation(np.zeros((3, 0))).tolist() == [0.0, 0.0, 0.0]


SPACE = [{"name": "x", "type": "num", "lb": -1, "ub": 4.0}, {"name": "n", "type": "int", "lb": 0, "ub": 5},
         {"name": "c", "type": "cat", "categories": ["a", "b"]}]


def test_general_bo_start_up_phase_fix_input_and_iter():
    np.random.seed(0)
    opt = GeneralBO(SPACE, num_obj=2, num_constr=1, rand_sample=6)
    assert opt.rand_sample == 6 and GeneralBO(SPACE, 2, 1).rand_sample == 4           # 1 + number of parameters
    rec = opt.suggest(5, fix_input={"c": "b", "n": 3})
    assert isinstance(rec, pd.DataFrame) and len(rec) == 5 and list(rec.columns) == ["x", "n", "c"]
    assert set(rec["c"]) == {"b"} and set(rec["n"]) == {3} and bool(((rec["x"] >= -1) & (rec["x"] <= 4)).all())
    rec = opt.suggest(3)
    assert opt.iter == 2 and len(rec) == 3


def test_general_bo_kappa_schedule():
    opt = GeneralBO(SPACE, 2, 1, kappa=None, c_kappa=None)
    opt.iter = 7
    k, ck = opt._kappas()
    ref = np.sqrt(0.1 * 2 * ((2.0 + 3 / 2.0) * np.log(7) + np.log(3 * np.pi ** 2 / (3 * 0.01))))
    assert k == pytest.approx(ref, rel=1e-12) and ck == k == general_kappa(3, 7)
    assert GeneralBO(SPACE, 2, 1, kappa=1.5, c_kappa=0.5)._kappas() == (1.5, 0.5)


def test_general_bo_observe_filters_and_pareto_bookkeeping():
    opt = GeneralBO(SPACE, num_obj=2, num_constr=1)
    X = pd.DataFrame({"x": [0.0, 1.0, 2.0, 3.0, 0.5, 1.5], "n": [0, 1, 2, 3, 4, 5], "c": ["a", "b", "a", "b", "a", "b"]})
    y = np.array([[1.0, 1.0, -1.0],        # feasible, non-dominated
                  [0.5, 2.0, -0.1],        # feasible, non-dominated
                  [2.0, 2.0, -1.0],        # feasible, dominated
                  [0.0, 0.0, 0.5],         # infeasible (would dominate everything)
                  [np.inf, 0.0, -1.0],     # dropped
                  [0.2, 3.0, np.nan]])     # dropped
    opt.observe(X, y)
    assert opt.y.shape == (4, 3) and opt.Xc.shape[0] == 4
    mask = opt.get_pf(opt.y, return_optimal=True)
    assert mask.tolist() == [True, True, False, False]
    assert np.array_equal(opt.best_y, opt.y[:2])
    bx = opt.best_x
    assert bx["x"].tolist() == [0.0, 1.0] and bx["c"].tolist() == ["a", "b"]
    D = dominance_matrix(opt.best_y[:, :2])
    assert not D.any()
    opt2 = GeneralBO(SPACE, num_obj=1, num_constr=1)
    opt2.observe(X.iloc[:2], np.array([[1.0, 0.5], [0.0, 0.1]]))
    assert opt2.best_y.shape == (0, 2) and len(opt2.best_x) == 0             # nothing feasible yet


def test_general_bo_ref_point_and_model_name_are_rejected():
    with pytest.raises(NotImplementedError, match="hypervolume"):
        GeneralBO(SPACE, 2, 0, ref_point=np.array([1.0, 1.0]))
    with pytest.raises(ValueError):
        GeneralBO(SPACE, 2, 0, model_name="rf")
