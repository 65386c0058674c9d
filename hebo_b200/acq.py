"""Acquisitions behind HEBO's ``Acquisition`` plugin surface (HEBO/hebo/acquisitions/acq.py:17-39).

``MACE`` is the drop-in for the reference's MACE (acq.py:131-171): with a ``hebo_b200.GP`` model the
predict + (LCB, -logEI, -logPI) arithmetic is ONE fused C-ABI call (``GP.predict_mace``); with any other
``BaseModel`` that model's ``predict`` output is pushed through the same CUDA epilogue (``hb_mace_epilogue``), so the
class stays a valid general-purpose acquisition.  ``GeneralAcq`` (acq.py:192-242: LCB of every objective and constraint
output, the acquisition of ``GeneralBO``) follows the same pattern with ``hb_general_acq_epilogue``.  ``Mean`` / ``Sigma`` /
``LCB`` mirror acq.py:55-82.
"""
from __future__ import annotations

import numpy as np
import torch

from .base import Acquisition
from .gp import GP, MultiTaskModel


class SingleObjectiveAcq(Acquisition):
    def __init__(self, model, **conf):
        super().__init__(model, **conf)

    @property
    def num_obj(self):
        return 1

    @property
    def num_constr(self):
        return 0


class LCB(SingleObjectiveAcq):
    def __init__(self, model, **conf):
        super().__init__(model, **conf)
        self.kappa = conf.get("kappa", 3.0)
        assert model.num_out == 1

    def eval(self, x, xe):
        py, ps2 = self.model.predict(x, xe)
        return py - self.kappa * ps2.sqrt()


class Mean(SingleObjectiveAcq):
    def __init__(self, model, **conf):
        super().__init__(model, **conf)
        assert model.num_out == 1

    def eval(self, x, xe):
        py, _ = self.model.predict(x, xe)
        return py


class Sigma(SingleObjectiveAcq):
    def __init__(self, model, **conf):
        super().__init__(model, **conf)
        assert model.num_out == 1

    def eval(self, x, xe):
        _, ps2 = self.model.predict(x, xe)
        return -1 * ps2.sqrt()


class MACE(Acquisition):
    def __init__(self, model, best_y, **conf):
        super().__init__(model, **conf)
        self.kappa = conf.get("kappa", 2.0)
        self.eps = conf.get("eps", 1e-4)
        self.tau = best_y

    @property
    def num_constr(self):
        return 0

    @property
    def num_obj(self):
        return 3

    def eval(self, x, xe=None):
        """minimize (lcb, -log EI, -log PI) -- the column order of acq.py:166-170."""
        tau = float(np.asarray(self.tau).reshape(-1)[0])
        with torch.no_grad():
            if isinstance(self.model, GP):     # predict + MACE fused in ONE C-ABI call (a failed fit degrades inside it, gp.py:152-154)
                return self.model.predict_mace(x, tau, float(self.kappa), float(self.eps), Xe=xe)
            return self._eval_any_model(x, xe, tau)

    def _eval_any_model(self, x, xe, tau):
        """Any other BaseModel (e.g. the RF stand-in of HEBO/test/test_acq.py:18-21): its predict() output goes through the
        same CUDA epilogue (hb_mace_epilogue), with the two N(0,1) draws of acq.py:154-155 taken from torch's CPU generator
        in the reference's order."""
        from . import _lib
        py, ps2 = self.model.predict(x, xe)
        m = py.shape[0]
        xi1, xi2 = torch.randn(py.shape), torch.randn(py.shape)
        dev = torch.device("cuda")
        up = lambda t: t.reshape(-1).to(dev, torch.float32).contiguous()
        mu_d, var_d, z1, z2 = up(py), up(ps2), up(xi1), up(xi2)
        F = torch.empty(m, 3, dtype=torch.float32, device=dev)
        if m:
            with torch.cuda.device(dev):
                _lib.check(_lib.lib().hb_mace_epilogue(_lib.ptr(mu_d), _lib.ptr(var_d), m, float(self.model.noise.reshape(-1)[0]), tau,
                                                       float(self.kappa), float(self.eps), _lib.ptr(z1), _lib.ptr(z2), 0, _lib.ptr(F),
                                                       _lib.stream_ptr()), "hb_mace_epilogue")
        return F.cpu()


class GeneralAcq(Acquisition):
    """Constrained multi-objective LCB (acq.py:192-242): minimise (lcb_o1, ..., lcb_oK) subject to lcb_c1 < 0, ...

    out[:, :num_obj] = py - kappa ps and out[:, num_obj:] = py - c_kappa ps, with py += sqrt(noise) xi when use_noise.
    With a ``hebo_b200.MultiTaskModel`` (or a single-output ``GP`` when O = 1) the O per-output posteriors are enqueued back
    to back into one [O, m] device buffer and the CUDA epilogue follows, with no host synchronisation in between (each
    output's failed-fit degradation, gp.py:152-154, stays in its own posterior); with any other ``BaseModel`` its
    ``predict`` output goes through the same epilogue.  xi: one torch.randn(m, O) from torch's CPU generator after predict,
    like the reference, when the model's rng is 'host'; in-kernel Philox normals otherwise."""

    def __init__(self, model, num_obj, num_constr, **conf):
        super().__init__(model, **conf)
        self._num_obj = num_obj
        self._num_constr = num_constr
        self.kappa = conf.get("kappa", 2.0)
        self.c_kappa = conf.get("c_kappa", 0.)
        self.use_noise = conf.get("use_noise", True)
        assert self.model.num_out == self.num_obj + self.num_constr
        assert self.num_obj >= 1

    @property
    def num_obj(self) -> int:
        return self._num_obj

    @property
    def num_constr(self) -> int:
        return self._num_constr

    def eval(self, x, xe=None):
        return self.evaluate(x, xe)

    def _device_models(self):
        if isinstance(self.model, MultiTaskModel) and all(isinstance(g, GP) for g in self.model.models):
            return self.model.models
        if isinstance(self.model, GP) and self.model.num_out == 1:
            return [self.model]
        return None

    def evaluate(self, x, xe=None, device_out: bool = False, return_cv: bool = False, seed: int = 0):
        """out [m, O] (and cv [m] = sum_j max(0, out[:, num_obj + j]) with return_cv) on the input's device, or on the GPU
        with device_out=True.  seed keys the Philox draws of the 'device' rng."""
        from . import _lib
        O, K = self.num_obj + self.num_constr, self.num_obj
        gps = self._device_models()
        with torch.no_grad():
            if gps is not None:
                g0 = gps[0]
                dev = g0.device
                m = g0._rows(x, xe)
                on_cpu = not device_out and not any(torch.is_tensor(t) and t.is_cuda for t in (x, xe))
                mu = torch.empty(O, m, dtype=torch.float32, device=dev)
                var = torch.empty(O, m, dtype=torch.float32, device=dev)
                if m:
                    Xs, xe_dev = g0._to_dev(x), g0._xe_dev(xe, m)
                    for o, g in enumerate(gps):
                        g._posterior(Xs, False, Xe_dev=xe_dev, out_mu=mu[o], out_var=var[o])
                host_rng = g0.rng == "host"
            else:
                dev = torch.device("cuda")
                on_cpu = not device_out and not (torch.is_tensor(x) and x.is_cuda)
                py, ps2 = self.model.predict(x, xe)
                m = py.shape[0]
                mu = py.reshape(m, O).t().to(dev, torch.float32).contiguous()
                var = ps2.reshape(m, O).t().to(dev, torch.float32).contiguous()
                host_rng = True
            noise = torch.as_tensor(self.model.noise, dtype=torch.float32).reshape(-1).to(dev).contiguous() if self.use_noise else None
            xi = torch.randn(m, O).to(dev).contiguous() if (self.use_noise and host_rng) else None   # acq.py:238
            out = torch.empty(m, O, dtype=torch.float32, device=dev)
            cv = torch.empty(m, dtype=torch.float32, device=dev)
            if m:
                with torch.cuda.device(dev):
                    _lib.check(_lib.lib().hb_general_acq_epilogue(_lib.ptr(mu), _lib.ptr(var), m, K, O - K, _lib.ptr(noise), float(self.kappa),
                                                                  float(self.c_kappa), int(bool(self.use_noise)), _lib.ptr(xi), int(seed), 0,
                                                                  _lib.ptr(out), _lib.ptr(cv), _lib.stream_ptr()), "hb_general_acq_epilogue")
        if on_cpu:
            out, cv = out.cpu(), cv.cpu()
        return (out, cv) if return_cv else out


FusedMACE = MACE
