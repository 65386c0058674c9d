"""Writes tests/golden/ref_general_acq.npz: outputs of the REFERENCE's own GeneralAcq.eval
(HEBO/hebo/acquisitions/acq.py:192-242, loaded by path with oracle.ref_loader) on a dummy multi-output model, for
(num_obj, num_constr) in {(1, 0), (2, 1), (3, 4)}, non-default and default kappa / c_kappa, use_noise on and off, and a few
ps2 = 1e-16 entries for the sigma clamp.  The N(0,1) draw xi is recorded by reseeding torch.  Only data is written.

    python -m oracle.make_golden_general
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import ref_loader

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def gen_ref_general_acq():
    ref = ref_loader.load_reference()
    acq_mod = ref_loader.sys.modules["_hebo_ref.acquisitions.acq"]

    class Dummy(ref.BaseModel):
        support_multi_output = True

        def __init__(self, mu, var, noise):
            super().__init__(1, 0, mu.shape[1])
            self.mu, self.var, self._n = mu, var, noise

        def fit(self, *a):
            pass

        def predict(self, x, xe):
            return self.mu.clone(), self.var.clone()

        @property
        def noise(self):
            return self._n

    cases = {}
    g = torch.Generator().manual_seed(20261017)
    ci = 0
    for no, nc in [(1, 0), (2, 1), (3, 4)]:
        O = no + nc
        for conf in [dict(kappa=2.7, c_kappa=1.3, use_noise=True), dict(use_noise=False), dict(), dict(kappa=0.4, c_kappa=-0.8, use_noise=False)]:
            m = 128
            mu = torch.randn(m, O, generator=g) * 1.5
            var = torch.rand(m, O, generator=g) ** 4 * 2 + 1e-8
            var[m // 2: m // 2 + 6] = 1e-16
            noise = torch.rand(O, generator=g) * 0.05 + 1e-4
            acq = acq_mod.GeneralAcq(Dummy(mu, var, noise), no, nc, **conf)
            torch.manual_seed(3000 + ci)
            out = acq.eval(torch.zeros(m, 1), None)
            torch.manual_seed(3000 + ci)
            xi = torch.randn(m, O)
            p = f"c{ci}_"
            cases.update({p + "mu": mu.numpy(), p + "var": var.numpy(), p + "noise": noise.numpy(), p + "xi": xi.numpy(),
                          p + "out": out.numpy(), p + "conf": np.array([no, nc, acq.kappa, acq.c_kappa, float(acq.use_noise)],
                                                                       dtype=np.float64)})
            ci += 1
    cases["n_cases"] = np.array(ci)
    np.savez_compressed(os.path.join(OUT, "ref_general_acq.npz"), **cases)


if __name__ == "__main__":
    gen_ref_general_acq()
    print("wrote", os.path.join(OUT, "ref_general_acq.npz"))
