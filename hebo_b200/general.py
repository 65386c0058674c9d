"""GeneralBO: multi-objective and black-box-constrained BO on the B200 path (HEBO/hebo/optimizers/general.py:23-204).

Control flow of the reference: random start-up samples, one GP per output column (``MultiTaskModel``, no y power
transform), the kappa / c_kappa schedule, ``GeneralAcq`` (LCB of every objective and constraint), an acquisition optimiser
returning the constrained Pareto set, a random pick of q with the most uncertain candidate forced into slot 0.  The
reference optimises ``GeneralAcq`` with pymoo (NSGA-II with constraint handling, or its GA for one objective), which is not
installed here; its replacement runs on the device:

* ``acq_optimizer="sobol"`` (default, like ``suggest.HEBO``): one scrambled-Sobol mega-batch scored by ``GeneralAcq``
  (O posteriors + one epilogue), then the constrained front (``hb_pareto_front`` with cv).
* ``acq_optimizer="nsga2"``: the device NSGA-II (``DeviceNSGA2``, evo_pop x evo_iters) with K objectives and pymoo's
  filter_infeasible survival, returning the constrained front of the final population.

With ``num_obj == 1`` the result is the single best row (res.X of pymoo's GA: least acquisition among the feasible rows,
else least cv); the NSGA-II population still runs through the K = 1 survival, i.e. rank-and-crowding on one objective.

Deviations from the reference, on purpose: ``fix_input`` is honoured by the acquisition optimiser and by the random
top-up (the reference forgets both after the start-up phase); ``get_pf(..., return_optimal=True)`` / ``best_x`` index all
observations (the reference's mask covers the feasible rows only and cannot index ``self.X`` once a row is infeasible); with
no feasible observation ``best_y`` is empty.  The EHVI selection of ``ref_point`` (:124-158) needs pymoo's N-dimensional
hypervolume and is not implemented.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import pandas as pd
import torch

from .acq import GeneralAcq
from .evolution import dominance_matrix
from .gp import MultiTaskModel
from .pareto import pareto_front
from .suggest import HEBO

MODEL_NAMES = ("multi_task", "multi_task_b200", "gp", "gp_b200")


def general_kappa(n_paras: int, it: int, upsi: float = 0.1, delta: float = 0.01) -> float:
    """general.py:96-101: the kappa / c_kappa used when the constructor's value is None."""
    return float(np.sqrt(upsi * 2 * ((2.0 + n_paras / 2.0) * np.log(it) + np.log(3 * np.pi ** 2 / (3 * delta)))))


class GeneralBO(HEBO):
    support_parallel_opt = True

    def __init__(self, space, num_obj: int = 1, num_constr: int = 0, rand_sample: Optional[int] = None,
                 model_name: str = "multi_task", model_config: Optional[dict] = None, kappa: Optional[float] = 2.0,
                 c_kappa: Optional[float] = 0.0, use_noise: bool = False, evo_pop: int = 100, evo_iters: int = 200,
                 ref_point=None, acq_optimizer: str = "sobol", n_candidates: int = 10000, scramble_seed: Optional[int] = None,
                 device: str = "cuda"):
        if ref_point is not None:
            raise NotImplementedError("GeneralBO(ref_point=...): the EHVI selection needs an N-dimensional hypervolume "
                                      "(pymoo's HV in the reference) and is not implemented; leave ref_point=None")
        if model_name not in MODEL_NAMES:
            raise ValueError(f"GeneralBO fits one hebo_b200 GP per output; model_name must be one of {MODEL_NAMES}")
        assert 1 <= num_obj <= 8 and num_constr >= 0
        super().__init__(space, model_config=model_config, scramble_seed=scramble_seed, n_candidates=n_candidates, device=device,
                         acq_optimizer=acq_optimizer, evo_pop=evo_pop, evo_iters=evo_iters)
        self.num_obj, self.num_constr = int(num_obj), int(num_constr)
        self.rand_sample = 1 + self.space.num_paras if rand_sample is None else rand_sample      # general.py:44-46
        self.model_name = model_name
        self.kappa, self.c_kappa, self.use_noise = kappa, c_kappa, use_noise
        self.y = np.zeros((0, self.num_obj + self.num_constr))
        self.iter = 0
        self.model = None

    @property
    def model_config(self):
        cfg = dict(self._model_config or {})
        if self.e > 0:
            cfg["num_uniqs"] = self.space.num_uniqs                                    # general.py:74-78
        return cfg

    def _kappas(self):
        kappa = general_kappa(self.space.num_paras, self.iter) if self.kappa is None else self.kappa
        c_kappa = general_kappa(self.space.num_paras, self.iter) if self.c_kappa is None else self.c_kappa
        return kappa, c_kappa

    def _random(self, n: int, fix_input: Optional[dict]) -> pd.DataFrame:
        sample = self.space.sample(n)
        for k, v in (fix_input or {}).items():
            sample[k] = v
        return sample

    def suggest(self, n_suggestions: int = 1, fix_input: Optional[dict] = None):
        self.iter += 1
        if self.Xc.shape[0] < self.rand_sample:
            return self._random(n_suggestions, fix_input)                              # general.py:64-70
        O, K = self.num_obj + self.num_constr, self.num_obj
        model = MultiTaskModel(self.d, self.e, O, **dict({"device": self.device}, **self.model_config))
        model.fit(self.Xc if self.d else None, self.Xe if self.e else None, torch.FloatTensor(self.y))
        self.model = model
        kappa, c_kappa = self._kappas()
        acq = GeneralAcq(model, K, self.num_constr, kappa=kappa, c_kappa=c_kappa, use_noise=self.use_noise)

        def score(xc, xe, seed):
            out, cv = acq.evaluate(xc if self.d else None, xe if self.e else None, device_out=True, return_cv=True, seed=seed)
            return out[:, :K], (cv if self.num_constr else None)
        if self.acq_optimizer == "nsga2":
            from .evolution import DeviceNSGA2
            evo = DeviceNSGA2(self.space.var_kinds, self.lb.numpy(), self.ub.numpy(), self.d, score, pop=self.evo_pop,
                              iters=self.evo_iters, seed=int(np.random.randint(0, 2 ** 31 - 1)),
                              fixed=self._fixed_columns(fix_input), device=model.models[0].device, num_obj=K)
            rec_c, rec_e, _ = evo.optimize()
            rec_e = rec_e.long()
        else:
            rec_c, rec_e = self.quasi_sample(self.n_candidates, fix_input, self.cand_sobol, as_opt=True)
            dev = model.models[0].device
            rec_c, rec_e = rec_c.to(dev), rec_e.to(dev)
            F, cv = score(rec_c, rec_e, self.iter)
            idx = pareto_front(F, cv)
            rec_c, rec_e = rec_c[idx], rec_e[idx]
        if K == 1:
            rec_c, rec_e = rec_c[:1], rec_e[:1]                                        # res.X of the GA: one row
        rec_c, rec_e = rec_c.cpu(), rec_e.cpu()
        suggest = self._from_opt(rec_c, rec_e)
        if suggest.shape[0] < n_suggestions:                                           # general.py:112-115
            rand = self._random(n_suggestions - suggest.shape[0], fix_input)
            return pd.concat([suggest, rand], axis=0, ignore_index=True)
        _, ps2 = model.predict(rec_c if self.d else None, rec_e if self.e else None)  # general.py:117-123
        largest_uncert_id = int(np.argmax(np.log(ps2.double().numpy()).sum(axis=1)))
        select_id = np.random.choice(suggest.shape[0], n_suggestions, replace=False).tolist()
        if largest_uncert_id not in select_id:
            select_id[0] = largest_uncert_id
        return suggest.iloc[select_id]

    def observe(self, X, y):
        """general.py:163-180: rows with any non-finite output are dropped."""
        y = np.asarray(y, dtype=np.float64).reshape(-1, self.num_obj + self.num_constr)
        valid = np.isfinite(y).all(axis=1)
        Xc, Xe = self._to_opt(X)
        keep = torch.from_numpy(valid)
        self.Xc = torch.cat([self.Xc, Xc[keep]], 0)
        self.Xe = torch.cat([self.Xe, Xe[keep]], 0)
        self.y = np.vstack([self.y, y[valid]])

    observe_new_data = observe

    def get_pf(self, y: np.ndarray, return_optimal: bool = False):
        """general.py:182-195: the feasible (every constraint column <= 0), mutually non-dominated rows of y.
        return_optimal=True: a mask over ALL rows of y."""
        y = np.asarray(y, dtype=np.float64).reshape(-1, self.num_obj + self.num_constr)
        feasible = (y[:, self.num_obj:] <= 0).all(axis=1)
        optimal = np.zeros(y.shape[0], dtype=bool)
        fi = np.flatnonzero(feasible)
        if fi.size:
            optimal[fi[~dominance_matrix(y[fi, :self.num_obj]).any(0)]] = True
        return optimal if return_optimal else y[optimal].copy()

    @property
    def best_x(self) -> pd.DataFrame:
        optimal = torch.from_numpy(self.get_pf(self.y, return_optimal=True))
        return self._from_opt(self.Xc[optimal], self.Xe[optimal])

    @property
    def best_y(self) -> np.ndarray:
        return self.get_pf(self.y)
