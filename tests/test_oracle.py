"""CPU tests: the oracle against the committed golden vectors, among them the outputs of the reference's own
acq.py / scalers.py / sgld.py / KumarWarp recorded by oracle/make_golden.py."""
import math

import numpy as np
import pytest
import torch

from oracle import gp_oracle as O
from tests.util import load_golden

GP_CASES = ["c1_branin", "c2_ackley", "c3_hartmann_warp", "c4_hetero", "rbf"]


def test_mace_restatement_matches_reference_vectors():
    """fp32 restatement of acq.py:146-171 reproduces the reference's own MACE.eval outputs."""
    g = load_golden("ref_mace.npz")
    for ci in range(4):
        mu, var = torch.from_numpy(g[f"c{ci}_mu"]), torch.from_numpy(g[f"c{ci}_var"])
        xi1, xi2 = torch.from_numpy(g[f"c{ci}_xi1"]), torch.from_numpy(g[f"c{ci}_xi2"])
        tau, kappa, noise, eps = g[f"c{ci}_par"]
        F = O.mace(mu, var, float(noise), float(np.float32(tau)), float(kappa), float(eps), xi1, xi2).numpy()
        Fr = g[f"c{ci}_F"]
        assert F.shape == Fr.shape == (mu.shape[0], 3)
        same_nan = np.isnan(F) == np.isnan(Fr)
        assert same_nan.all()
        # same torch kernels on the same ISA reproduce bit-exactly; across ISAs the fp32 erf/exp/log differ in
        # the last ulp, which the ill-conditioned tail amplifies (tests/util.py PHI_BUDGET): compare off-tail
        z = (np.float32(tau) - eps - mu.numpy().reshape(-1) - math.sqrt(2 * noise) * xi2.numpy().reshape(-1)) / np.sqrt(var.numpy().reshape(-1)).clip(1.19e-7)
        ok = (z > -4) | (z < -6.5)
        np.testing.assert_allclose(F[ok], Fr[ok], rtol=2e-3, atol=2e-3)
        np.testing.assert_allclose(F[:, 0], Fr[:, 0], rtol=1e-6, atol=1e-6)


def test_scaler_restatement_matches_reference_vectors():
    g = load_golden("ref_scalers.npz")
    sc, mn = O.minmax_fit(g["X"])
    np.testing.assert_allclose(sc, g["scale"], rtol=1e-6)
    np.testing.assert_allclose(mn, g["min"], rtol=1e-6, atol=1e-7)
    mean, std = O.standard_fit(g["y"])
    np.testing.assert_allclose(mean, g["mean"], rtol=1e-6)
    np.testing.assert_allclose(std, g["std"], rtol=1e-6)


def test_mace_live_against_reference_source():
    """The reference's MACE on a seeded batch (tests/golden/ref_mace_seeded.npz), its xi drawn by the reference itself
    after torch.manual_seed(11): the oracle, given the same draws in the same order, reproduces its objectives."""
    g = load_golden("ref_mace_seeded.npz")
    mu, var, Fr = torch.from_numpy(g["mu"]), torch.from_numpy(g["var"]), torch.from_numpy(g["F"])
    best_y, kappa, noise = g["par"]
    torch.manual_seed(11)
    xi1, xi2 = torch.randn(777, 1), torch.randn(777, 1)
    F = O.mace(mu, var, float(noise), float(np.float32(best_y)), float(kappa), 1e-4, xi1, xi2)
    # not bit-equal: the reference gathers rows before log() (acq.py:169-170), which changes ATen's
    # vector/scalar-tail split and with it the last ulps of erf/exp/log
    torch.testing.assert_close(F, Fr, rtol=2e-4, atol=2e-4)


@pytest.mark.parametrize("kind", ["matern32", "matern52", "rbf"])
def test_closed_form_gradient_matches_autograd(kind):
    X, y = O.synthetic_problem("ackley", 48, 4, 5)
    f = O.make_fitted(X, y, kind=kind, rng=np.random.RandomState(0))
    g = torch.Generator().manual_seed(1)
    vec = f.hp.pack() + 0.3 * torch.randn(7, generator=g, dtype=torch.float64)
    hp = O.Hypers.unpack(vec, 8e-4)
    nd = 1e-2 * (1 + (f.Xt ** 2).sum(1))
    for noise_diag in (None, nd):
        l1, g1 = O.neg_mll_autograd(f.Xt, f._yt, hp, kind, noise_diag=noise_diag)
        l2, g2, _ = O.neg_mll_closed_form(f.Xt, f._yt, hp, kind, noise_diag=noise_diag)
        assert abs(float(l1 - l2)) < 1e-12
        assert float((g1 - g2).abs().max()) < 1e-11


def test_psgld_matches_torch_rmsprop_plus_langevin():
    torch.manual_seed(0)
    p = torch.nn.Parameter(torch.randn(6, dtype=torch.float64))
    opt = torch.optim.RMSprop([p], lr=0.01, alpha=0.99, eps=1e-8)
    vec = p.detach().clone()
    st = O.PSGLDState(torch.zeros_like(vec))
    for step in range(8):
        g = torch.randn(6, dtype=torch.float64)
        xi = torch.randn(6, dtype=torch.float64)
        p.grad = g.clone()
        opt.step()
        if step + 1 > 3:   # sgld.py:63-70
            avg = opt.state[p]["square_avg"].sqrt().add(1e-8)
            with torch.no_grad():
                p.add_(0.1 * (2 * 0.01 / avg).sqrt() * xi)
        vec = O.psgld_step(vec, g, st, 0.01, 0.1, 3, xi)
    assert float((vec - p.detach()).abs().max()) < 1e-14


@pytest.mark.parametrize("case", GP_CASES)
def test_oracle_reproduces_gp_goldens(case):
    """The committed gp_*.npz fixtures are what the current oracle code computes (guards against drift)."""
    g = load_golden(f"gp_{case}.npz")
    kind = str(g["kind"])
    X = torch.from_numpy(g["X"]).double()
    yt = torch.from_numpy(g["y_transformed"]).double()
    f = O.make_fitted(X, yt, kind=kind, rng=np.random.RandomState(0))
    Xt = f.Xt
    if g["warp_a"].size:
        Xt = O.kumaraswamy_warp(f.Xt, torch.from_numpy(g["warp_a"]), torch.from_numpy(g["warp_b"]))
    nd = torch.from_numpy(g["noise_diag"]) if g["noise_diag"].size else None
    for which in ("0", "1"):
        hp = O.Hypers.unpack(torch.from_numpy(g["raw" + which]), 8e-4)
        loss, grad, _ = O.neg_mll_closed_form(Xt, f._yt, hp, kind, noise_diag=nd)
        assert abs(float(loss) - float(g["loss" + which])) < 1e-9
        np.testing.assert_allclose(grad.numpy(), g["grad" + which], rtol=1e-7, atol=1e-10)
    # posterior at the post-fit hypers
    f.Xt, f.hp, f.noise_diag = Xt, O.Hypers.unpack(torch.from_numpy(g["raw1"]), 8e-4), nd
    O.refactor(f)
    Xs = torch.from_numpy(g["Xs"]).double()
    if g["warp_a"].size:
        Xs_model = O.kumaraswamy_warp(f.x_scale * Xs + f.x_min, torch.from_numpy(g["warp_a"]), torch.from_numpy(g["warp_b"]))
        f.x_scale, f.x_min = torch.ones_like(f.x_scale), torch.zeros_like(f.x_min)
        mu, var = O.predict(f, Xs_model)
    else:
        mu, var = O.predict(f, Xs)
    np.testing.assert_allclose(mu.numpy().reshape(-1), g["mu"], rtol=1e-8, atol=1e-9)
    np.testing.assert_allclose(var.numpy().reshape(-1), g["var"], rtol=1e-7, atol=1e-12)
    F = O.mace(mu, var, float(g["noise"]), float(g["tau"]), float(g["kappa"]), 1e-4,
               torch.from_numpy(g["xi1"]), torch.from_numpy(g["xi2"])).numpy()
    np.testing.assert_allclose(F, g["F"], rtol=1e-7, atol=1e-9)
    assert np.array_equal(O.pareto_front(F), g["front"])


def test_pareto_front_against_bruteforce_and_edge_cases():
    rng = np.random.RandomState(1)
    F = rng.randn(700, 3)
    F[:, 2] = 0.5 * F[:, 0] + 0.5 * F[:, 2]
    assert np.array_equal(O.pareto_front(F), O.pareto_front_bruteforce(F))
    dup = np.vstack([F[:5], F[:5]])                       # duplicates never dominate each other
    assert np.array_equal(O.pareto_front(dup), O.pareto_front_bruteforce(dup))
    one = np.array([[1.0, 2.0, 3.0]])
    assert np.array_equal(O.pareto_front(one), [0])
    chain = np.array([[3., 3., 3.], [2., 2., 2.], [1., 1., 1.]])
    assert np.array_equal(O.pareto_front(chain), [2])


def test_kappa_schedule_and_lengthscale_init():
    # hebo.py:156-160 at n=64 obs, q=1, D=2
    k = O.kappa_schedule(64, 1, 2)
    assert abs(k - math.sqrt((3.0) * math.log(64) + math.log(3 * math.pi ** 2 / 0.03))) < 1e-12
    X = torch.linspace(-1, 1, 11, dtype=torch.float64).reshape(-1, 1)
    ls = O.init_lengthscales(X, rng=np.random.RandomState(0))
    assert abs(float(ls[0]) - float(torch.pdist(X).median())) < 1e-15


def test_psgld_step_against_the_reference_optimizer_class():
    """oracle.psgld_step vs the reference's real pSGLD (HEBO/hebo/models/nn/sgld.py:49-70; its parameters after each
    step are in tests/golden/ref_psgld.npz): same parameters after 25 steps over three parameter tensors with the
    reference's own torch.randn_like draws replayed as the oracle's xi."""
    ref = load_golden("ref_psgld.npz")
    shapes = [(1,), (), (1, 5)]
    A = torch.from_numpy(ref["A"]).split([int(np.prod(s)) for s in shapes])
    vec = torch.from_numpy(ref["p0"])

    def loss_of(ps):                # a smooth non-quadratic test loss
        return sum(((a * p.reshape(-1)) ** 2).sum() + torch.cos(p.reshape(-1)).sum() for a, p in zip(A, ps))
    n, lr, steps = ref["par"]
    n, steps = int(n), int(steps)
    assert ref["traj"].shape == (steps, vec.numel())
    st = O.PSGLDState(torch.zeros_like(vec))
    for ep in range(steps):
        # oracle step with the same draws
        torch.manual_seed(100 + ep)
        xi = None
        if ep + 1 > steps // 10:
            xi = torch.cat([torch.randn(s, dtype=torch.float64).reshape(-1) for s in shapes])
        v = vec.clone().requires_grad_(True)
        off, ps = 0, []
        for s in shapes:
            k = int(np.prod(s)) if len(s) else 1
            ps.append(v[off:off + k].reshape(s))
            off += k
        (gr,) = torch.autograd.grad(loss_of(ps), v)
        vec = O.psgld_step(vec, gr, st, float(lr), 1.0 / n, steps // 10, xi)
        ref_vec = torch.from_numpy(ref["traj"][ep])
        assert float((vec - ref_vec).abs().max()) < 1e-13, ep


def test_kumaraswamy_warp_against_the_reference_layer():
    """oracle.warp_oracle.warp / exponents vs the reference's KumarWarp layer (mono_layers/layers.py:85-117; its exponents
    and outputs are in tests/golden/ref_kumar_warp.npz): a, b = 0.01 + 9.99 sigmoid(raw), w(u) = 1 - (1 - clamp(u)^a)^b on
    u = (x + 1) / 2."""
    from oracle import warp_oracle as W
    ref = load_golden("ref_kumar_warp.npz")
    a, b = torch.from_numpy(ref["a"]), torch.from_numpy(ref["b"])
    assert torch.equal(W.exponents(torch.from_numpy(ref["raw_a"])), a)
    assert torch.equal(W.exponents(torch.from_numpy(ref["raw_b"])), b)
    X = torch.from_numpy(ref["X"])
    assert float(X.min()) == -1.0 and float(X.max()) == 1.0          # the clamp at eps / 1 - eps is exercised
    ours = W.warp(X, a, b)
    assert float((ours - torch.from_numpy(ref["out"])).abs().max()) < 1e-15
