"""Small end-to-end pass for compute-sanitizer (memcheck / racecheck / synccheck): numeric + mixed fit (tile-DAG Cholesky,
tcgen05 fit GEMMs, triangular inverse, gradient kernels, CUDA-graph epochs), refined inverse, tensor-path posterior with the
guard (vnorm_h16 + FP32 re-contraction), MACE, Pareto front, front pack / merge, device NSGA-II, and the multi-objective /
constrained path (GeneralAcq epilogue, K-objective constrained front, constrained K-objective survival).

    compute-sanitizer --tool memcheck  python tools/sanitize_run.py
    compute-sanitizer --tool racecheck python tools/sanitize_run.py
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hebo_b200                                                        # noqa: E402
from hebo_b200.evolution import DeviceNSGA2                              # noqa: E402
from hebo_b200.pareto import front_merge, front_pack, front_read, pareto_front, pareto_front_device   # noqa: E402

torch.manual_seed(0)
np.random.seed(0)
n, d, m = int(os.environ.get("SAN_N", 700)), 5, 1500
X = torch.rand(n, d) * 2 - 1
y = (torch.sin(3 * X[:, :1]) + 0.3 * X[:, 1:2] ** 2 + 0.05 * torch.randn(n, 1))
gp = hebo_b200.GP(d, 0, 1, lr=0.01, num_epochs=6, noise_lb=8e-4, pred_likeli=False, m_chunk=1024)
gp.fit(X, None, y)
Xs = torch.rand(m, d) * 2.4 - 1.2
Xs[:40] = X[:40]                                   # guarded rows
F, mu, var = gp.predict_mace(Xs, float(y.min()), 2.0, 1e-4, torch.randn(m, 1), torch.randn(m, 1), return_mu_var=True)
assert torch.isfinite(F).all()
idx = pareto_front(F.cuda())
i2, c2 = pareto_front_device(F.cuda())
buf = front_pack(F.cuda(), mu.cuda(), var.cuda(), i2, c2, 0, 64)
out = front_merge(torch.stack([buf, buf]).contiguous(), 2, 64)
front_read(out)
Fbig = torch.randn(20000, 3, device="cuda")            # sieve path (m > 4096): stratified sample front -> filter -> survivors
Fbig[:, 2] = 0.7 * Fbig[:, 0] + 0.3 * Fbig[:, 2]
Fbig[::997, 1] = float("nan")
ib = pareto_front(Fbig)
assert ib.numel() > 0 and not torch.isnan(Fbig[ib]).any()
bb = front_pack(Fbig, None, None, *pareto_front_device(Fbig), 5, 4096)
front_read(front_merge(torch.stack([bb, bb, bb]).contiguous(), 3, 4096))     # merge through the sieve (R = 12288)
xg = Xs[:50].clone().requires_grad_(True)
pm, pv = gp.predict(xg, None)
(pm.sum() + pv.sum()).backward()
gm = hebo_b200.GP(2, 1, 1, num_uniqs=[4], num_epochs=4, pred_likeli=False)
Xe = torch.randint(4, (300, 1))
gm.fit(X[:300, :2], Xe, y[:300] + 0.3 * Xe.float())
gm.predict(X[:64, :2], Xe[:64])
gm.evaluate_loss(return_grad=True)
evo = DeviceNSGA2(["real", "real", "choice"], [-1, -1, 0], [1, 1, 3], 2,
                  lambda xc, xe, g: gm.predict_mace(xc, 0.0, 2.0, 1e-4, seed=g, Xe=xe, device_out=True), pop=32, iters=4, seed=1)
evo.optimize()
gw = hebo_b200.GP(3, 0, 1, num_epochs=4, pred_likeli=False, warp=True)              # learned Kumaraswamy warp + sample_y
gw.fit(X[:200, :3], None, y[:200])
gw.predict(X[:64, :3], None)
gw.sample_y(X[:32, :3], None, 3)
mt = hebo_b200.MultiTaskModel(d, 0, 3, num_epochs=4, pred_likeli=False)           # GeneralAcq epilogue + constrained fronts
mt.fit(X[:300], None, torch.cat([y[:300], -y[:300], y[:300] - 0.2], 1))
gacq = hebo_b200.GeneralAcq(mt, 2, 1, kappa=2.0, c_kappa=0.5, use_noise=True)
gout, gcv = gacq.evaluate(Xs.cuda(), None, device_out=True, return_cv=True)
pareto_front(gout[:, :2], gcv)
Fk = torch.randn(20000, 5, device="cuda")
pareto_front(Fk, torch.rand(20000, device="cuda") + 0.1)                   # sieve path, nothing feasible
evo_k = DeviceNSGA2(["real", "real", "choice"], [-1, -1, 0], [1, 1, 3], 2,
                    lambda xc, xe, g: (torch.stack([xc[:, 0], -xc[:, 1]], 1), (xc[:, 0] + xc[:, 1]).clamp_min(0)), pop=32, iters=4,
                    seed=2, num_obj=2)
evo_k.optimize()
torch.cuda.synchronize()
print("sanitize_run ok", int(idx.numel()))
