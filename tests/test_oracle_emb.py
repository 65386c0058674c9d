"""Categorical (embedding) GP oracle -- groundwork for SURVEY section 8(f) row 2: closed-form gradient vs autograd, CPU."""
import torch

from oracle import emb_oracle as E
from tests.util import load_golden


def problem(n=60, d=3, num_uniqs=(4, 7), seed=0):
    g = torch.Generator().manual_seed(seed)
    Xt = torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1
    Xe = torch.stack([torch.randint(0, u, (n,), generator=g) for u in num_uniqs], 1)
    y = torch.sin(3 * Xt[:, 0]) + 0.5 * (Xe[:, 0] == 1).double() - 0.3 * (Xe[:, 1] % 3).double() \
        + 0.05 * torch.randn(n, generator=g, dtype=torch.float64)
    yt = (y - y.mean()) / y.std()
    return Xt, Xe, yt, list(num_uniqs)


def test_embedding_sizes_and_concatenation_follow_the_reference():
    assert E.default_emb_sizes([2, 3, 10, 200]) == [2, 2, 6, 50]          # layers.py:19
    Xt, Xe, yt, nu = problem()
    hp = E.init_emb_hypers(Xt, Xe, yt, nu)
    emb = E.embed(Xe, hp.tables)
    assert emb.shape == (Xt.shape[0], sum(E.default_emb_sizes(nu)))
    assert torch.equal(emb[5, :hp.tables[0].shape[1]], hp.tables[0][Xe[5, 0]])
    assert hp.pack().numel() == 1 + sum(t.numel() for t in hp.tables) + 3 + Xt.shape[1]
    assert torch.equal(hp.like(hp.pack()).pack(), hp.pack())


def test_closed_form_gradient_matches_autograd_for_every_parameter_group():
    Xt, Xe, yt, nu = problem()
    hp = E.init_emb_hypers(Xt, Xe, yt, nu, seed=3)
    # move away from the symmetric initial point
    g = torch.Generator().manual_seed(9)
    vec = hp.pack() + 0.3 * torch.randn(hp.pack().numel(), generator=g, dtype=torch.float64)
    hp = hp.like(vec)
    la, ga = E.neg_mll_emb_autograd(Xt, Xe, yt, hp)
    lc, gc = E.neg_mll_emb_closed_form(Xt, Xe, yt, hp)
    assert abs(float(la - lc)) < 1e-12
    assert float((ga - gc).abs().max()) < 1e-10 * max(1.0, float(ga.abs().max()))
    n_tab = sum(t.numel() for t in hp.tables)
    assert float(ga[1:1 + n_tab].abs().max()) > 1e-6                      # the embedding weights do receive gradient


def test_unused_categories_get_zero_gradient_and_prediction_is_consistent():
    Xt, Xe, yt, nu = problem(num_uniqs=(5, 3))
    Xe[:, 0] = Xe[:, 0].clamp(max=3)                                      # category 4 of column 0 never occurs
    hp = E.init_emb_hypers(Xt, Xe, yt, nu, seed=1)
    _, gc = E.neg_mll_emb_closed_form(Xt, Xe, yt, hp)
    t0 = hp.tables[0]
    g_t0 = gc[1:1 + t0.numel()].reshape(t0.shape)
    assert float(g_t0[4].abs().max()) == 0.0
    mu, var = E.predict_emb(Xt, Xe, yt, hp, Xt[:7], Xe[:7])
    assert float((mu - yt[:7]).abs().max()) < 0.5 and (var > 0).all() and (var < float(hp.outputscale)).all()
    # the same numeric point with another category is a different input
    Xe2 = Xe[:7].clone()
    Xe2[:, 1] = (Xe2[:, 1] + 1) % 3
    mu2, var2 = E.predict_emb(Xt, Xe, yt, hp, Xt[:7], Xe2)
    assert float((var2 - var).min()) > 0.0


def test_embedding_lookup_matches_the_reference_module():
    """Pins `embed` against the reference's real EmbTransform (HEBO/hebo/models/layers.py:14-34; its sizes, tables and
    output are in tests/golden/ref_emb.npz): same default sizes, same column order, same concatenation."""
    ref = load_golden("ref_emb.npz")
    nu = ref["num_uniqs"].tolist()
    assert ref["emb_sizes"].tolist() == E.default_emb_sizes(nu) and int(ref["num_out"]) == sum(E.default_emb_sizes(nu))
    tables = [torch.from_numpy(ref[f"table{i}"]) for i in range(len(nu))]
    assert torch.equal(E.embed(torch.from_numpy(ref["Xe"]), tables), torch.from_numpy(ref["out"]))


def test_general_layouts_closed_form_vs_autograd():
    """Enum-only (no numeric columns), numeric-only with one shared lengthscale (ard_kernel=False) and the Matern-5/2 /
    RBF numeric kernels of a mixed model: closed form == autograd for every parameter."""
    Xt, Xe, yt, nu = problem(n=50, d=3)
    g = torch.Generator().manual_seed(5)

    def check(hp, Xt_, Xe_, kind="matern32"):
        hp = hp.like(hp.pack() + 0.3 * torch.randn(hp.pack().numel(), generator=g, dtype=torch.float64))
        la, ga = E.neg_mll_emb_autograd(Xt_, Xe_, yt, hp, kind=kind)
        lc, gc = E.neg_mll_emb_closed_form(Xt_, Xe_, yt, hp, kind=kind)
        assert abs(float(la - lc)) < 1e-12 and float((ga - gc).abs().max()) < 1e-10 * max(1.0, float(ga.abs().max()))
        return hp
    base = E.init_emb_hypers(Xt, Xe, yt, nu, seed=2)
    for kind in ("matern52", "rbf"):
        check(base, Xt, Xe, kind)
    # enum only
    hp_e = E.EmbHypers(base.raw_noise, base.tables, base.mean, base.raw_os, torch.zeros(0, dtype=torch.float64), base.raw_ls_e)
    hp_e = check(hp_e, Xt[:, :0], Xe)
    assert hp_e.pack().numel() == 1 + sum(t.numel() for t in base.tables) + 2 + 1
    # numeric only, shared lengthscale
    hp_s = E.EmbHypers(base.raw_noise, [], base.mean, base.raw_os, torch.zeros(1, dtype=torch.float64), base.raw_ls_e)
    hp_s = check(hp_s, Xt, Xe[:, :0])
    assert hp_s.pack().numel() == 4
    # pSGLD over the packed vector runs and lowers the loss
    hp1, losses = E.fit_psgld_emb(Xt, Xe, yt, base, lr=0.01, num_epochs=15, record=True)
    assert losses[-1] < losses[0] and hp1.pack().numel() == base.pack().numel()
