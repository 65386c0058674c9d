"""Generates the committed golden fixtures under tests/golden/ (needs a copy of the reference HEBO at
``oracle.ref_loader.REF_ROOT``; nothing else does).

    python -m oracle.make_golden

Two kinds of vectors:
  * ``ref_*.npz``  -- outputs of the REFERENCE's own code loaded by path (HEBO/hebo/acquisitions/acq.py
    MACE.eval, models/scalers.py, models/nn/sgld.py pSGLD, models/nn/mono_layers/layers.py KumarWarp,
    models/layers.py EmbTransform, design_space/*.py DesignSpace) on seeded inputs.  These pin the oracle's
    restatements (tests/test_oracle.py, tests/test_oracle_emb.py), the host design space (tests/test_host.py)
    and the CUDA MACE epilogue (tests/test_gpu_parity.py).
  * ``gp_*.npz``   -- fp64 outputs of the oracle's restatement of the gpytorch exact-GP maths (no gpytorch
    install exists to generate them from; "parity unpinned" at that boundary, see oracle/gp_oracle.py)
    for small seeded versions of the BASELINE configs: loss, gradient, 100-epoch pSGLD trajectory end
    point, posterior mean/variance, MACE objectives, Pareto front, argmin mu / argmax sigma.
Test infrastructure; never imported by hebo_b200/.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import gp_oracle as O
from . import ref_loader

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def gen_ref_mace():
    ref = ref_loader.load_reference()

    class Dummy(ref.BaseModel):
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

    cases = {}
    g = torch.Generator().manual_seed(20260922)
    for ci, (m, tau, kappa, noise, shift) in enumerate([(512, -0.5, 2.3, 0.013, 0.0), (512, -2.0, 3.7, 1e-3, 0.0),
                                                        (512, -1.0, 2.0, 0.05, 25.0), (256, 0.3, 4.4, 8e-4, 0.0)]):
        mu = torch.randn(m, 1, generator=g) * 1.5
        var = torch.rand(m, 1, generator=g) ** 4 * 2 + 1e-8
        if shift:
            mu[: m // 4] += shift          # z << -6 : log-approximation branch (acq.py:161-164)
        var[m // 2: m // 2 + 8] = 1e-16    # sigma clamp (acq.py:153)
        model = Dummy(mu, var, torch.tensor([noise]))
        acq = ref.MACE(model, best_y=np.float32(tau), kappa=kappa)
        torch.manual_seed(1000 + ci)
        F = acq(torch.zeros(m, 1), None)
        torch.manual_seed(1000 + ci)
        xi1 = torch.randn(m, 1)
        xi2 = torch.randn(m, 1)
        cases[f"c{ci}_mu"] = mu.numpy()
        cases[f"c{ci}_var"] = var.numpy()
        cases[f"c{ci}_xi1"] = xi1.numpy()
        cases[f"c{ci}_xi2"] = xi2.numpy()
        cases[f"c{ci}_par"] = np.array([tau, kappa, noise, 1e-4], dtype=np.float64)
        cases[f"c{ci}_F"] = F.numpy()
    np.savez_compressed(os.path.join(OUT, "ref_mace.npz"), **cases)


def gen_ref_scalers():
    ref = ref_loader.load_reference()
    g = torch.Generator().manual_seed(7)
    X = torch.randn(40, 5, generator=g) * torch.tensor([1.0, 10.0, 0.1, 3.0, 1.0]) + torch.tensor([0., 5., -2., 0., 1.])
    X[:, 4] = 0.75                      # constant column: sklearn's zero-range handling
    y = torch.randn(40, 1, generator=g) * 3 + 2
    mm = ref.TorchMinMaxScaler((-1, 1)).fit(X)
    ss = ref.TorchStandardScaler().fit(y)
    np.savez_compressed(os.path.join(OUT, "ref_scalers.npz"), X=X.numpy(), y=y.numpy(), scale=mm.scale_.numpy(),
                        min=mm.min_.numpy(), Xt=mm.transform(X).numpy(), mean=ss.mean.numpy(), std=ss.std.numpy(),
                        yt=ss.transform(y).numpy())


def gen_ref_mace_seeded():
    """The reference's MACE on one seeded batch, its xi drawn by the reference itself after torch.manual_seed(11)
    (tests/test_oracle.py replays that draw for the oracle)."""
    ref = ref_loader.load_reference()

    class Dummy(ref.BaseModel):
        def __init__(self, mu, var):
            super().__init__(1, 0, 1)
            self.mu, self.var = mu, var

        def fit(self, *a):
            pass

        def predict(self, x, xe):
            return self.mu.clone(), self.var.clone()

        @property
        def noise(self):
            return torch.tensor([0.02])

    torch.manual_seed(3)
    mu, var = torch.randn(777, 1), torch.rand(777, 1) + 1e-3
    acq = ref.MACE(Dummy(mu, var), best_y=np.float32(-0.3), kappa=2.9)
    torch.manual_seed(11)
    F = acq(torch.zeros(777, 1), None)
    np.savez_compressed(os.path.join(OUT, "ref_mace_seeded.npz"), mu=mu.numpy(), var=var.numpy(), F=F.numpy(),
                        par=np.array([-0.3, 2.9, 0.02], dtype=np.float64))


def gen_ref_psgld():
    """Parameters after each of 25 steps of the reference's pSGLD (models/nn/sgld.py, its unrelated imports stubbed) on
    the loss sum_i ||a_i * p_i||^2 + sum cos(p_i), noise drawn by the reference after torch.manual_seed(100 + step)."""
    mod = ref_loader.load_file("_hebo_ref_nn.sgld", "models/nn/sgld.py",
                               stubs=[("_hebo_ref_nn", ()), ("_hebo_ref_nn.deep_ensemble", ("BaseNet", "DeepEnsemble")),
                                      ("matplotlib", ()), ("matplotlib.pyplot", ())])
    g = torch.Generator().manual_seed(0)
    params = [torch.nn.Parameter(torch.randn(s, generator=g, dtype=torch.float64)) for s in [(1,), (), (1, 5)]]
    A = [torch.rand(p.numel(), generator=g, dtype=torch.float64) + 0.5 for p in params]
    p0 = torch.cat([p.detach().reshape(-1).clone() for p in params])
    n, lr, steps = 40, 0.01, 25
    opt = mod.pSGLD(params, lr=lr, factor=1.0 / n, pretrain_step=steps // 10)
    traj = []
    for ep in range(steps):
        torch.manual_seed(100 + ep)
        opt.zero_grad()
        sum(((a * p.reshape(-1)) ** 2).sum() + torch.cos(p.reshape(-1)).sum() for a, p in zip(A, params)).backward()
        opt.step()
        traj.append(torch.cat([p.detach().reshape(-1) for p in params]))
    np.savez_compressed(os.path.join(OUT, "ref_psgld.npz"), p0=p0.numpy(), A=torch.cat(A).numpy(),
                        traj=torch.stack(traj).numpy(), par=np.array([n, lr, steps], dtype=np.float64))


def gen_ref_kumar_warp():
    """The reference's KumarWarp layer (models/nn/mono_layers/layers.py) at seeded raw exponents, on [-1, 1] inputs
    mapped to [0, 1] and back."""
    mod = ref_loader.load_file("_hebo_ref_mono_layers", "models/nn/mono_layers/layers.py")
    d = 6
    layer = mod.KumarWarp(d).double()
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        layer._a.copy_(torch.randn(d, generator=g, dtype=torch.float64))
        layer._b.copy_(torch.randn(d, generator=g, dtype=torch.float64))
    X = torch.rand(200, d, generator=g, dtype=torch.float64) * 2 - 1
    X[0], X[1] = -1.0, 1.0                               # the clamp at eps / 1 - eps
    out = 2.0 * layer((X + 1.0) * 0.5).detach() - 1.0
    np.savez_compressed(os.path.join(OUT, "ref_kumar_warp.npz"), raw_a=layer._a.detach().numpy(),
                        raw_b=layer._b.detach().numpy(), a=layer.a.detach().numpy(), b=layer.b.detach().numpy(),
                        X=X.numpy(), out=out.numpy())


def gen_ref_emb():
    """The reference's EmbTransform (models/layers.py): default sizes, its randomly initialised tables, and its output
    on seeded category indices."""
    mod = ref_loader.load_file("_hebo_ref_layers", "models/layers.py")
    nu = [4, 7, 2, 120]
    torch.manual_seed(0)
    tr = mod.EmbTransform(nu)
    g = torch.Generator().manual_seed(0)
    Xe = torch.stack([torch.randint(0, u, (33,), generator=g) for u in nu], 1)
    tables = {f"table{i}": m.weight.detach().double().numpy() for i, m in enumerate(tr.emb)}
    np.savez_compressed(os.path.join(OUT, "ref_emb.npz"), num_uniqs=np.array(nu), emb_sizes=np.array(tr.emb_sizes),
                        num_out=tr.num_out, Xe=Xe.numpy(), out=tr(Xe).detach().double().numpy(), **tables)


def gen_ref_design_space():
    """The reference's DesignSpace on tests/test_host.py's SPEC: names, optimisation bounds, transform of a fixed frame
    and inverse transform of this package's own transform of it (each column as str(value), and as float where it is
    numeric)."""
    import pandas as pd
    from hebo_b200.space import DesignSpace
    from tests.test_host import FRAME, SPEC
    df = pd.DataFrame(FRAME)
    ref = ref_loader.load_design_space()().parse(SPEC)
    rc, re_ = ref.transform(df)
    xc, xe = DesignSpace().parse(SPEC).transform(df)
    rb = ref.inverse_transform(xc, xe)
    cols = {}
    for col in ref.para_names:
        cols[f"inv_{col}_str"] = np.array([str(v) for v in rb[col].tolist()])
        num = pd.to_numeric(rb[col], errors="coerce").to_numpy(dtype=np.float64)
        cols[f"inv_{col}_num"] = num if np.isfinite(num).all() else np.zeros(0)
    np.savez_compressed(os.path.join(OUT, "ref_design_space.npz"), xc=rc.numpy(), xe=re_.numpy(),
                        para_names=np.array(ref.para_names), opt_lb=ref.opt_lb.double().numpy(),
                        opt_ub=ref.opt_ub.double().numpy(), **cols)


def gen_gp(name, fn, n, d, m, q, kind, seed, warp=False, hetero=False):
    X, y = O.synthetic_problem(fn, n, d, seed)
    X = X.float().double()
    yt_np = O.hebo_y_transform(y.numpy())                        # hebo.py:128-135 on the host
    yt = torch.from_numpy(yt_np).double().reshape(-1)
    g = torch.Generator().manual_seed(seed + 1)
    rng = np.random.RandomState(seed)
    f = O.make_fitted(X, yt, kind=kind, dtype=torch.float64, rng=rng)
    warp_a = warp_b = None
    Xt = f.Xt
    if warp:
        warp_a = torch.rand(d, generator=g, dtype=torch.float64) * 1.5 + 0.5
        warp_b = torch.rand(d, generator=g, dtype=torch.float64) * 1.5 + 0.5
        Xt = O.kumaraswamy_warp(f.Xt, warp_a, warp_b)
        f.Xt = Xt
        f.hp = O.init_hypers(Xt, f._yt, 8e-4, rng=np.random.RandomState(seed))
    nd = None
    if hetero:
        nd = 1e-2 * (1 + (Xt ** 2).sum(1) / d)
        f.noise_diag = nd
    hp0 = f.hp
    loss0, grad0, _ = O.neg_mll_closed_form(Xt, f._yt, hp0, kind, noise_diag=nd)
    lang = torch.randn(100, d + 3, generator=g, dtype=torch.float64)
    lang[:10] = 0
    hp1, losses = O.fit_psgld(Xt, f._yt, hp0, kind, lr=0.01, num_epochs=100, langevin=lang, noise_diag=nd, record=True)
    loss1, grad1, _ = O.neg_mll_closed_form(Xt, f._yt, hp1, kind, noise_diag=nd)
    f.hp = hp1
    O.refactor(f)
    # candidates: scrambled Sobol in [-1,1] plus near-duplicates of training rows and out-of-range rows
    sob = torch.quasirandom.SobolEngine(d, scramble=True, seed=seed).draw(m).double() * 2 - 1
    k = m // 8
    sob[:k] = X[:k] + 1e-3 * torch.randn(k, d, generator=g, dtype=torch.float64)
    sob[k:2 * k] = sob[k:2 * k] * 1.3
    Xs = sob.float().double()
    if warp:
        Xs_model = O.kumaraswamy_warp(f.x_scale * Xs + f.x_min, warp_a, warp_b)
        # predict() applies the MinMax transform itself: undo it so the oracle path matches xtrans+warp
        fw = O.FittedGP(f.Xt, f.hp, kind, torch.ones(d, dtype=torch.float64), torch.zeros(d, dtype=torch.float64),
                        f.y_mean, f.y_std, noise_diag=nd)
        fw.L, fw.alpha = f.L, f.alpha
        mu, var = O.predict(fw, Xs_model)
    else:
        mu, var = O.predict(f, Xs)
    best = int(torch.argmin(yt))
    if warp:
        tau = float(O.predict(fw, Xt[best:best + 1])[0])
    else:
        tau = float(O.predict(f, X[best:best + 1])[0])
    kappa = O.kappa_schedule(n, q, d)
    xi1 = torch.randn(m, 1, generator=g)
    xi2 = torch.randn(m, 1, generator=g)
    F = O.mace(mu, var, float(f.noise), tau, kappa, 1e-4, xi1, xi2)
    front = O.pareto_front(F.numpy())
    np.savez_compressed(
        os.path.join(OUT, f"gp_{name}.npz"), X=X.numpy().astype(np.float32), y_transformed=yt_np.reshape(-1),
        kind=kind, raw0=hp0.pack().numpy(), raw1=hp1.pack().numpy(), loss0=float(loss0), grad0=grad0.numpy(),
        loss1=float(loss1), grad1=grad1.numpy(), losses=np.array(losses), langevin=lang.numpy().astype(np.float32),
        Xs=Xs.numpy().astype(np.float32), mu=mu.numpy().reshape(-1), var=var.numpy().reshape(-1), tau=tau, kappa=kappa,
        xi1=xi1.numpy().reshape(-1), xi2=xi2.numpy().reshape(-1), F=F.numpy(), front=front,
        argmin_mu=int(np.argmin(mu.numpy().reshape(-1)[front])), argmax_sigma=int(np.argmax(var.numpy().reshape(-1)[front])),
        noise=float(f.noise), y_mean=f.y_mean, y_std=f.y_std, q=q,
        warp_a=(warp_a.numpy() if warp else np.zeros(0)), warp_b=(warp_b.numpy() if warp else np.zeros(0)),
        noise_diag=(nd.numpy() if hetero else np.zeros(0)))


def main():
    os.makedirs(OUT, exist_ok=True)
    gen_ref_mace()
    gen_ref_scalers()
    gen_ref_mace_seeded()
    gen_ref_psgld()
    gen_ref_kumar_warp()
    gen_ref_emb()
    gen_ref_design_space()
    gen_gp("c1_branin", "branin", 64, 2, 256, 1, "matern32", 1235)            # BASELINE config 1
    gen_gp("c2_ackley", "ackley", 160, 8, 384, 8, "matern52", 1236)           # config 2, reduced n/m
    gen_gp("c3_hartmann_warp", "hartmann6", 200, 32, 384, 8, "matern32", 1237, warp=True)   # config 3, reduced
    gen_gp("c4_hetero", "ackley", 130, 20, 256, 16, "matern32", 1238, hetero=True)          # config 4, reduced
    gen_gp("rbf", "ackley", 96, 4, 256, 4, "rbf", 1239)
    print("wrote", sorted(os.listdir(OUT)))


if __name__ == "__main__":
    main()
