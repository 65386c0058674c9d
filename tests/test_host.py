"""CPU tests of the host-side mirror of the reference interface (no GPU, no kernels)."""
import numpy as np
import pytest
import torch

import hebo_b200
from hebo_b200 import scalers
from hebo_b200.base import BaseModel
from tests.util import load_golden, assert_mace_close


def test_scalers_match_reference_vectors():
    g = load_golden("ref_scalers.npz")
    X, y = torch.from_numpy(g["X"]), torch.from_numpy(g["y"])
    mm = scalers.MinMaxScaler((-1, 1)).fit(X)
    np.testing.assert_allclose(mm.scale_.numpy(), g["scale"], rtol=1e-6)
    np.testing.assert_allclose(mm.min_.numpy(), g["min"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(mm.transform(X).numpy(), g["Xt"], rtol=1e-6, atol=1e-6)
    ss = scalers.StandardScaler().fit(y)
    np.testing.assert_allclose(ss.mean.numpy(), g["mean"], rtol=1e-6)
    np.testing.assert_allclose(ss.std.numpy(), g["std"], rtol=1e-6)
    np.testing.assert_allclose(ss.transform(y).numpy(), g["yt"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(ss.inverse_transform(ss.transform(y)).numpy(), y.numpy(), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(mm.inverse_transform(mm.transform(X)).numpy(), X.numpy(), rtol=1e-4, atol=1e-4)


def test_filter_nan_rules():
    x = torch.randn(6, 2)
    y = torch.randn(6, 1)
    y[0] = np.nan
    y[3] = np.inf
    xf, xef, yf = scalers.filter_nan(x, None, y, "all")
    assert xf.shape[0] == 4 and xef is None and torch.isfinite(yf).all()
    with pytest.raises(AssertionError):
        scalers.filter_nan(x, None, torch.full((6, 1), np.nan), "all")


def test_gp_constructor_contract_and_conf_keys():
    gp = hebo_b200.GP(3, 0, 1, lr=0.01, num_epochs=100, noise_lb=8e-4, pred_likeli=False, verbose=False)
    assert isinstance(gp, BaseModel)
    assert gp.support_grad and not gp.support_ts and not gp.support_multi_output and not gp.support_warm_start
    assert gp.kernel == "matern32"                      # reference default nu = 1.5 (gp_util.py:46)
    assert (gp.lr, gp.num_epochs, gp.noise_lb, gp.pred_likeli) == (0.01, 100, 8e-4, False)
    d = hebo_b200.GP(3, 0, 1)
    assert (d.lr, d.num_epochs, d.noise_lb, d.pred_likeli, d.optimizer) == (3e-2, 100, 1e-5, True, "psgld")
    assert hebo_b200.GP(3, 0, 1, kernel="matern52").kern_id == 1
    with pytest.raises(NotImplementedError):
        gp.sample_f()
    with pytest.raises(AssertionError):
        hebo_b200.GP(0, 0, 1)
    with pytest.raises(AssertionError):
        hebo_b200.GP(1, 1, 1)                           # num_uniqs is mandatory with enum columns (base_model.py:27-30)
    # mixed / enum-only / non-ARD models (test_base_model.py:41-73 shapes): parameter layout in registration order
    mixed = hebo_b200.GP(2, 2, 1, num_uniqs=[5, 9])
    assert mixed.emb_sizes == [3, 5] and mixed.De == 8 and mixed.T == 5 * 3 + 9 * 5     # layers.py:19: min(50, 1 + v // 2)
    lay = mixed._param_layout()
    assert (lay["tab"], lay["mean"], lay["os"], lay["ls"], lay["n_ls"], lay["le"], lay["P"]) == (1, 61, 62, 63, 2, 65, 66)
    assert hebo_b200.GP(0, 1, 1, num_uniqs=[4])._param_layout()["P"] == 1 + 4 * 3 + 2 + 0 + 1
    assert hebo_b200.GP(3, 0, 1, ard_kernel=False)._param_layout()["P"] == 4
    assert hebo_b200.GP(1, 1, 1, num_uniqs=[4], emb_sizes=[2]).T == 8

    class FakeKern:            # stands in for gpytorch ScaleKernel(MaternKernel(nu=2.5)) passed as conf['kern']
        class base_kernel:
            nu = 2.5
    assert hebo_b200.GP(2, 0, 1, kern=FakeKern()).kernel == "matern52"


def test_langevin_draws_follow_reference_rng_order():
    gp = hebo_b200.GP(5, 0, 1, num_epochs=30)
    torch.manual_seed(123)
    lang = gp._draw_langevin(8, 5)
    torch.manual_seed(123)
    for ep in range(30):
        if ep + 1 > 3:
            exp = torch.cat([torch.randn(1), torch.randn(()).reshape(1), torch.randn(()).reshape(1), torch.randn(1, 5)[0]])
            assert torch.equal(lang[ep], exp)
        else:
            assert float(lang[ep].abs().sum()) == 0.0


def test_langevin_draws_of_a_mixed_model_follow_registration_order_and_shapes():
    """sgld.py:70 draws randn_like per parameter tensor: raw_noise [1], embedding tables [num_uniq, emb] (numel >= 16 takes
    torch's vectorised normal fill, so the SHAPE matters), mean [], raw_outputscale [], raw_lengthscale [1,d], emb ls [1,1]."""
    gp = hebo_b200.GP(2, 2, 1, num_uniqs=[5, 9], num_epochs=20)
    P = gp._param_layout()["P"]
    torch.manual_seed(7)
    lang = gp._draw_langevin(P, 2)
    torch.manual_seed(7)
    for ep in range(20):
        if ep + 1 > 2:
            exp = torch.cat([torch.randn(1), torch.randn(5, 3).reshape(-1), torch.randn(9, 5).reshape(-1), torch.randn(()).reshape(1),
                             torch.randn(()).reshape(1), torch.randn(1, 2)[0], torch.randn(1, 1)[0]])
            assert torch.equal(lang[ep], exp)
        else:
            assert float(lang[ep].abs().sum()) == 0.0


@pytest.mark.gpu
def test_generic_mace_path_matches_reference_vectors():
    """MACE over a non-B200 model pushes model.predict through the CUDA epilogue (acq.py:151-171 arithmetic), drawing the
    two N(0,1) tensors from torch's CPU generator in the reference's order."""
    g = load_golden("ref_mace.npz")

    class Fake(BaseModel):
        def __init__(self, mu, var, noise):
            super().__init__(1, 0, 1)
            self.mu, self.var, self._n = mu, var, noise

        def fit(self, *a):
            pass

        def predict(self, x, xe):
            return self.mu.clone(), self.var.clone()

        @property
        def noise(self):
            return self._n

    for ci in range(4):
        mu, var = torch.from_numpy(g[f"c{ci}_mu"]), torch.from_numpy(g[f"c{ci}_var"])
        tau, kappa, noise, eps = g[f"c{ci}_par"]
        acq = hebo_b200.MACE(Fake(mu, var, torch.tensor([float(noise)])), best_y=np.float32(tau), kappa=float(kappa))
        assert acq.num_obj == 3 and acq.num_constr == 0
        torch.manual_seed(1000 + ci)
        F = acq(torch.zeros(mu.shape[0], 1), None)
        assert F.shape == (mu.shape[0], 3)
        assert_mace_close(F.numpy(), g[f"c{ci}_F"], mu.numpy(), var.numpy(), float(noise), float(np.float32(tau)),
                          float(eps), g[f"c{ci}_xi2"], what=f"case {ci}")


def test_mean_sigma_lcb_contract():
    class Fake(BaseModel):
        def fit(self, *a):
            pass

        def predict(self, x, xe):
            return x.sum(1, keepdim=True), torch.full((x.shape[0], 1), 4.0)

    m = Fake(2, 0, 1)
    x = torch.randn(7, 2)
    assert torch.equal(hebo_b200.Mean(m)(x, None), x.sum(1, keepdim=True))
    assert torch.equal(hebo_b200.Sigma(m)(x, None), torch.full((7, 1), -2.0))
    assert torch.allclose(hebo_b200.LCB(m, kappa=3.0)(x, None), x.sum(1, keepdim=True) - 6.0)
    for a in (hebo_b200.Mean(m), hebo_b200.Sigma(m), hebo_b200.LCB(m)):
        assert a.num_obj == 1 and a.num_constr == 0


def test_fp16_two_level_split_error_bound():
    """Numerics of the tensor path's operand format (hebo_b200/csrc/h16.cuh), emulated in numpy:
    x * 2^k = h0 + h1 / 2048 with h0 = rn_fp16(x 2^k), h1 = rn_fp16((x 2^k - h0) 2048) keeps 2^-22 relative precision in
    the fp16 normal range and ~1.5e-11 absolute precision (in units where the matrix maximum is 2^9..2^10) below it."""
    rng = np.random.default_rng(0)
    mags = 10.0 ** rng.uniform(-12, 0, size=200000)
    x = (rng.choice([-1.0, 1.0], size=mags.size) * mags).astype(np.float32)
    x[:10] = [0.0, 1.0, -1.0, 0.999, 6.1e-5, 6.0e-8, 3e-8, 1e-11, -2.5e-7, 0.5]
    maxabs = float(np.abs(x).max())
    e = int(np.frexp(maxabs)[1])
    scale = np.float32(2.0 ** (10 - e))                      # pow2_scale(maxabs, 10): the maximum lands in [512, 1024)
    xs = x * scale
    assert 512.0 <= float(np.abs(xs).max()) < 1024.0
    h0 = xs.astype(np.float16)
    r = xs - h0.astype(np.float32)                           # exact in fp32
    h1 = (r * np.float32(2048.0)).astype(np.float16)
    assert np.isfinite(h0).all() and np.isfinite(h1).all()
    rec = (h0.astype(np.float64) + h1.astype(np.float64) / 2048.0) / float(scale)
    err = np.abs(rec - x.astype(np.float64))
    normal = np.abs(xs) >= 6.2e-5                            # fp16 normal range after scaling
    assert (err[normal] <= 2.0 ** -22 * np.abs(x[normal])).all()
    assert (err[~normal] * float(scale) <= 2.0 ** -35).all()  # below the normal range: absolute, ~1.5e-11 of the scaled unit


# ------------------------------------------------------------------------------------------------ typed design space
SPEC = [{"name": "lr", "type": "pow", "lb": 1e-4, "ub": 1e-1}, {"name": "n", "type": "int", "lb": 1, "ub": 9},
        {"name": "b", "type": "bool"}, {"name": "w", "type": "pow_int", "lb": 8, "ub": 512, "base": 2},
        {"name": "e", "type": "int_exponent", "lb": 32, "ub": 1024, "base": 2},
        {"name": "s", "type": "step_int", "lb": 4, "ub": 16, "step": 4},
        {"name": "c", "type": "cat", "categories": ["a", "b", "c"]}, {"name": "x", "type": "num", "lb": -1, "ub": 2}]
FRAME = {"lr": [1e-3, 1e-1], "n": [3, 9], "b": [True, False], "w": [16, 300], "e": [64, 1024], "s": [8, 16], "c": ["b", "a"],
         "x": [0.5, -1.0]}


def test_design_space_types_round_trip_like_the_reference():
    """hebo_b200.space against the semantics of HEBO/hebo/design_space/*.py (transform / inverse_transform / bounds / the
    pymoo variable kind of evolution_optimizer.py:26-41), incl. a cross-check with what the reference's own classes
    compute on the same spec (tests/golden/ref_design_space.npz)."""
    import pandas as pd
    from hebo_b200.space import DesignSpace
    sp = DesignSpace().parse(SPEC)
    assert sp.numeric_names == ["lr", "n", "b", "w", "e", "s", "x"] and sp.enum_names == ["c"]       # numeric first, then enum
    assert sp.var_kinds == ["real", "int", "int", "real", "int", "int", "real", "choice"] and sp.num_uniqs == [3]
    assert torch.allclose(sp.opt_lb, torch.tensor([-4., 1., 0., 3., 5., 0., -1., 0.], dtype=torch.float64))
    assert torch.allclose(sp.opt_ub, torch.tensor([-1., 9., 1., 9., 10., 3., 2., 2.], dtype=torch.float64))
    df = pd.DataFrame(FRAME)
    xc, xe = sp.transform(df)
    assert xc.dtype == torch.float32 and xe.dtype == torch.int64 and xe.reshape(-1).tolist() == [1, 0]
    assert torch.allclose(xc[0], torch.tensor([-3., 3., 1., 4., 6., 1., 0.5]))
    back = sp.inverse_transform(xc, xe)
    assert back["n"].tolist() == [3, 9] and back["b"].tolist() == [True, False] and back["w"].tolist() == [16, 300]
    assert back["e"].tolist() == [64, 1024] and back["s"].tolist() == [8, 16] and back["c"].tolist() == ["b", "a"]
    assert np.allclose(back["lr"].values, [1e-3, 1e-1], rtol=1e-5) and np.allclose(back["x"].values, [0.5, -1.0])
    np.random.seed(0)
    smp = sp.sample(50)
    xs, es = sp.transform(smp)
    lo, hi = sp.opt_lb.float(), sp.opt_ub.float()
    assert bool(((torch.cat([xs, es.float()], 1) >= lo - 1e-5) & (torch.cat([xs, es.float()], 1) <= hi + 1e-5)).all())
    ref = load_golden("ref_design_space.npz")                # the reference's own DesignSpace on SPEC / FRAME
    assert torch.allclose(torch.from_numpy(ref["xc"]), xc) and torch.equal(torch.from_numpy(ref["xe"]), xe)
    assert ref["para_names"].tolist() == sp.para_names
    assert torch.allclose(torch.from_numpy(ref["opt_lb"]), sp.opt_lb) and torch.allclose(torch.from_numpy(ref["opt_ub"]), sp.opt_ub)
    for col in sp.para_names:
        rb_str, rb_num = ref[f"inv_{col}_str"].tolist(), ref[f"inv_{col}_num"]
        assert rb_str == [str(v) for v in back[col].tolist()] or (rb_num.size and np.allclose(rb_num, back[col].values.astype(float)))


def test_standalone_hebo_host_logic_typed_space():
    """quasi_sample / observe / duplicate check / fix_input of hebo_b200.suggest.HEBO on a mixed space (no GPU involved:
    fewer observations than rand_sample, hebo.py:122-124)."""
    import pandas as pd
    from hebo_b200.suggest import HEBO
    opt = HEBO(SPEC, scramble_seed=3)
    assert opt.rand_sample == 9 and opt.d == 7 and opt.e == 1
    df = opt.suggest(5)
    assert isinstance(df, pd.DataFrame) and list(df.columns) == opt.space.para_names and len(df) == 5
    assert all(v in ("a", "b", "c") for v in df["c"]) and all(float(v).is_integer() for v in df["n"]) and all(v in (4, 8, 12, 16) for v in df["s"])
    fx = opt.suggest(4, fix_input={"c": "b", "n": 7})
    assert set(fx["c"]) == {"b"} and set(fx["n"]) == {7}
    y = np.arange(5, dtype=float).reshape(-1, 1)
    y[2] = np.inf                                           # dropped at observe (hebo.py:211-215)
    opt.observe(df, y)
    assert opt.Xc.shape == (4, 7) and opt.Xe.shape == (4, 1) and opt.best_y == 0.0 and len(opt.best_x) == 1
    assert opt.get_best_id() == 0
    xc, xe = opt.Xc[:2].clone(), opt.Xe[:2].clone()
    xc2 = torch.cat([xc, xc[:1] + 0.25], 0)
    assert opt._unique_mask(xc2, torch.cat([xe, xe[:1]], 0)).tolist() == [False, False, True]
    assert opt.model_config["num_uniqs"] == [3] and opt.model_config["num_epochs"] == 100
    box = HEBO([-1.0, 0.0], [1.0, 2.0], scramble_seed=1)     # tensor front end
    t = box.suggest(3)
    assert torch.is_tensor(t) and t.shape == (3, 2) and bool(((t >= box.lb) & (t <= box.ub)).all())
