"""B200-native exact-GP surrogate behind HEBO's ``BaseModel`` plugin surface.

Drop-in for ``hebo.models.gp.gp.GP`` (HEBO/hebo/models/gp/gp.py:35-184): same constructor keys, same
``fit / predict / noise / sample_y / sample_f`` contract, CPU tensors in and out, but the arithmetic
(Gram build, Cholesky, solves, log-det, MLL gradient, pSGLD loop, posterior, MACE) runs in the hand-written
sm_100a kernels of libhebo_b200.so through the C ABI -- no GPyTorch, no CPU fallback.

Extra conf keys (unknown keys are ignored by the reference's ``conf.get``, so they are safe to pass through
``HEBO(model_config=...)``):
    kernel      'matern32' (reference default, gp_util.py:46) | 'matern52' | 'rbf'  (numeric dims; the embedding dims of a
                mixed model always use Matern-3/2 with one lengthscale, gp_util.py:54-55)
    num_uniqs / emb_sizes   categorical columns (the reference's own keys: hebo.py:99-100, layers.py:17-19)
    noise_diag  optional per-row extra noise variance [n] in *standardised* y units (BASELINE config 4)
    warp        True: Kumaraswamy input warp of the numeric dims with exponents a, b LEARNED inside the MLL (BASELINE config 3;
                KumarWarp, nn/mono_layers/layers.py:85-117), initialised at the identity a = b = 1
    warp_a/warp_b  optional FIXED Kumaraswamy exponents [d] (same fused kernels, exponents never updated)
    device      CUDA device (default 'cuda')
    m_chunk     candidates per posterior chunk (workspace = m_chunk * NP * 4 bytes)
    rng         'host' (default: torch CPU generator, the reference's stream) | 'device' (Philox in-kernel)
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import numpy as np
import torch

from . import _lib
from .base import BaseModel
from .scalers import MinMaxScaler, StandardScaler, filter_nan, kumaraswamy_warp

EPS32 = float(torch.finfo(torch.float32).eps)


def _softplus_inv(v: torch.Tensor) -> torch.Tensor:
    return v + torch.log(-torch.expm1(-v))


class _PredictWithGrad(torch.autograd.Function):
    """GP.predict as an autograd node: forward and the input Jacobian-vector products come from ``hb_posterior_grad``."""

    @staticmethod
    def forward(ctx, Xin, gp, x_mul, x_add):
        mu, var, dmu, dvar = gp._posterior_grad(Xin, x_mul, x_add)
        ctx.save_for_backward(dmu, dvar)
        return mu, var

    @staticmethod
    def backward(ctx, gmu, gvar):
        dmu, dvar = ctx.saved_tensors
        return gmu.unsqueeze(1) * dmu + gvar.unsqueeze(1) * dvar, None, None, None


class GP(BaseModel):
    support_grad = True

    def __init__(self, num_cont, num_enum, num_out, **conf):
        super().__init__(num_cont, num_enum, num_out, **conf)
        # same keys and defaults as HEBO/hebo/models/gp/gp.py:37-49
        self.lr = conf.get("lr", 3e-2)
        self.num_epochs = conf.get("num_epochs", 100)
        self.verbose = conf.get("verbose", False)
        self.print_every = conf.get("print_every", 10)
        self.pred_likeli = conf.get("pred_likeli", True)
        self.noise_lb = conf.get("noise_lb", 1e-5)
        self.optimizer = conf.get("optimizer", "psgld")
        self.noise_guess = conf.get("noise_guess", 0.01)
        self.ard_kernel = conf.get("ard_kernel", True)
        self.xscaler = MinMaxScaler((-1, 1))
        self.yscaler = StandardScaler()
        # B200 extras
        self.kernel = self._resolve_kernel(conf)
        self.kern_id = _lib.KERNEL_IDS[self.kernel]
        self.device = torch.device(conf.get("device", "cuda"))
        self.m_chunk = int(conf.get("m_chunk", 32768))
        self.rng = conf.get("rng", "host")
        self.noise_diag = conf.get("noise_diag", None)
        self.warp_a = conf.get("warp_a", None)
        self.warp_b = conf.get("warp_b", None)
        self.langevin = conf.get("langevin", True)
        self.tensor_cores = conf.get("tensor_cores", True)   # posterior contraction on tcgen05 (fp16 two-level split / 3xTF32) vs FP32 SIMT
        # categorical columns: one learned embedding table per column (layers.py:14-34), product kernel (gp_util.py:54-57)
        self.num_uniqs = [int(v) for v in conf.get("num_uniqs", [])] if self.num_enum > 0 else []
        if self.num_enum > 0:
            assert len(self.num_uniqs) == self.num_enum, "num_uniqs must list the categories of every enum column"
            es = conf.get("emb_sizes", None)
            self.emb_sizes = [int(v) for v in es] if es is not None else [min(50, 1 + v // 2) for v in self.num_uniqs]   # layers.py:19
            if self.noise_diag is not None:
                raise NotImplementedError("noise_diag is only defined for numeric-only models")
        else:
            self.emb_sizes = []
        self.De = int(sum(self.emb_sizes))
        self.T = int(sum(u * e for u, e in zip(self.num_uniqs, self.emb_sizes)))
        if self.num_cont + self.De > 232:
            raise NotImplementedError("more than 232 feature dimensions exceed the shared-memory tiling of the kernels")
        # input warp: 0 none, 1 learned exponents, 2 fixed exponents (include/hebo_b200.h hb_model_spec_t.warp)
        self.warp_mode = 2 if self.warp_a is not None else (1 if conf.get("warp", False) and self.num_cont > 0 else 0)
        if self.warp_mode == 2:
            wa, wb = torch.as_tensor(self.warp_a, dtype=torch.float32), torch.as_tensor(self.warp_b, dtype=torch.float32)
            assert wa.numel() == self.num_cont == wb.numel() and bool(((wa > 0.01) & (wa < 10) & (wb > 0.01) & (wb < 10)).all()), \
                "fixed warp exponents must lie inside (0.01, 10)"
        self._general = self.num_enum > 0 or not self.ard_kernel or self.warp_mode > 0     # needs the `_ex` entry points
        self._c_uniqs = (C.c_int32 * max(1, self.num_enum))(*self.num_uniqs)
        self._c_embs = (C.c_int32 * max(1, self.num_enum))(*self.emb_sizes)
        self._spec = _lib.ModelSpec(int(bool(self.ard_kernel)), self.num_enum, self._c_uniqs, self._c_embs, self.warp_mode)
        self._spec_nowarp = _lib.ModelSpec(int(bool(self.ard_kernel)), self.num_enum, self._c_uniqs, self._c_embs, 0)
        # gp.py:96-101: 'lbfgs' -> torch LBFGS(max_iter=5, strong_wolfe), 'psgld' -> the fused device loop, anything else -> Adam
        self._fitted = False
        self._fit_failed = False
        self._post_ws = None

    @staticmethod
    def _resolve_kernel(conf) -> str:
        k = conf.get("kernel", None)
        if k is not None:
            if k not in _lib.KERNEL_IDS:
                raise ValueError(f"unknown kernel {k}")
            return k
        kern = conf.get("kern", None)      # the reference injects a gpytorch kernel object here (gp.py:201)
        if kern is not None:
            base = getattr(kern, "base_kernel", kern)
            nu = getattr(base, "nu", None)
            if nu is None:
                return "rbf"
            return {1.5: "matern32", 2.5: "matern52"}[float(nu)]
        return "matern32"

    # ------------------------------------------------------------------ scaling (gp.py:51-71)
    def fit_scaler(self, Xc, Xe, y):
        if Xc is not None and Xc.shape[1] > 0:
            self.xscaler.fit(Xc)
        self.yscaler.fit(y)

    def xtrans(self, Xc, Xe, y=None):
        """gp.py:56-71: MinMax on the numeric columns, categories as int64, y standardised."""
        if Xc is not None and Xc.shape[1] > 0:
            Xc_t = self.xscaler.transform(Xc)        # (an input warp is applied inside the kernels, after this scaling)
        else:
            Xc_t = torch.zeros(Xe.shape[0], 0)
        Xe_t = torch.zeros(Xc_t.shape[0], 0).long() if Xe is None else Xe.long()
        if y is not None:
            return Xc_t, Xe_t, self.yscaler.transform(y)
        return Xc_t, Xe_t

    def _spec_ptr(self):
        return C.byref(self._spec) if self._general else None

    # FIXED warp exponents (warp_a / warp_b) are not hyper-parameters: `raw`, `raw_init`, `init_raw`, `set_hypers` and the
    # Langevin draws use the vector WITHOUT them; the device vector carries them (frozen) between the tables and the mean.
    def _frozen_raw(self) -> torch.Tensor:
        wa, wb = torch.as_tensor(self.warp_a, dtype=torch.float32), torch.as_tensor(self.warp_b, dtype=torch.float32)
        return torch.cat([torch.logit((wa - 0.01) / 9.99), torch.logit((wb - 0.01) / 9.99)])

    def _expand_raw(self, raw: torch.Tensor) -> torch.Tensor:
        if self.warp_mode != 2:
            return raw
        lay = self._param_layout()
        if raw.shape[-1] == lay["P"]:
            return raw
        lead = raw.shape[:-1]
        fz = self._frozen_raw().to(raw.dtype).expand(*lead, -1) if lead else self._frozen_raw().to(raw.dtype)
        return torch.cat([raw[..., :lay["wa"]], fz, raw[..., lay["wa"]:]], -1)

    def _strip_raw(self, raw: torch.Tensor) -> torch.Tensor:
        if self.warp_mode != 2:
            return raw
        lay = self._param_layout()
        return torch.cat([raw[..., :lay["wa"]], raw[..., lay["wa"] + lay["n_w"]:]], -1)

    def _param_layout(self):
        """Index ranges of the raw vector (include/hebo_b200.h): noise, tables, mean, outputscale, numeric ls, emb ls."""
        d, T = self.num_cont, self.T
        n_ls = 0 if d == 0 else (d if self.ard_kernel else 1)
        W = 2 * d if self.warp_mode else 0
        return dict(noise=0, tab=1, wa=1 + T, wb=1 + T + d, n_w=W, mean=1 + T + W, os=2 + T + W, ls=3 + T + W, n_ls=n_ls,
                    le=3 + T + W + n_ls, P=3 + T + W + n_ls + (1 if self.num_enum > 0 else 0))

    # ------------------------------------------------------------------ initial hypers (gp.py:86-91, gp_util.py:39-59)
    def _init_raw(self, XtT: torch.Tensor, n: int, yt: torch.Tensor) -> torch.Tensor:
        lib = _lib.lib()
        d = self.num_cont
        lay = self._param_layout()
        raw = torch.zeros(lay["P"], dtype=torch.float32)
        # nn.Embedding weights ~ N(0,1) (layers.py:22-23), drawn when the model is built, i.e. before the kernel's
        # np.random.choice calls and before any Langevin draw
        o = lay["tab"]
        for u, e in zip(self.num_uniqs, self.emb_sizes):
            raw[o:o + u * e] = torch.empty(u, e).normal_().reshape(-1)
            o += u * e
        if self.warp_mode:
            # a, b = 0.01 + 9.99 sigmoid(raw) (layers.py:96-104).  Learned: start at the identity a = b = 1 (the reference
            # layer starts at raw = 0, i.e. a = b = 5.005, a strong distortion that no HEBO configuration uses for the GP)
            wa = torch.ones(d) if self.warp_mode == 1 else torch.as_tensor(self.warp_a, dtype=torch.float32)
            wb = torch.ones(d) if self.warp_mode == 1 else torch.as_tensor(self.warp_b, dtype=torch.float32)
            raw[lay["wa"]:lay["wa"] + d] = torch.logit((wa - 0.01) / 9.99)
            raw[lay["wb"]:lay["wb"] + d] = torch.logit((wb - 0.01) / 9.99)
            if self.warp_mode == 2:      # the median heuristic sees the inputs the kernel sees
                Xw = kumaraswamy_warp(XtT[:, :n].t(), wa.to(XtT.device), wb.to(XtT.device))
                XtT = XtT.clone()
                XtT[:, :n] = Xw.t()
        if d > 0 and self.ard_kernel:
            k = min(n, 1000)
            # gp_util.py:50 consumes numpy's global RNG once per dimension, for every n (and only changes the result
            # when n > 1000); the median itself is one CUDA kernel (hb_median_pdist)
            idx = np.stack([np.random.choice(n, k, replace=False) for _ in range(d)]).astype(np.int32)
            idx_dev = torch.from_numpy(idx).to(XtT.device) if n > 1000 else None
            ls_dev = torch.empty(d, dtype=torch.float32, device=XtT.device)
            with torch.cuda.device(XtT.device):
                _lib.check(lib.hb_median_pdist(_lib.ptr(XtT), n, d, _lib.ptr(idx_dev), k, 0.02, _lib.ptr(ls_dev),
                                               _lib.stream_ptr()), "hb_median_pdist")
            raw[lay["ls"]:lay["ls"] + d] = _softplus_inv(ls_dev.cpu())
        # (ard_kernel=False and the embedding kernel keep gpytorch's default raw_lengthscale = 0, gp_util.py:44-55)
        os_ = yt[torch.isfinite(yt)].var()
        noise = torch.tensor(max(1e-2, self.noise_lb), dtype=torch.float32)
        raw[lay["noise"]] = _softplus_inv((noise - self.noise_lb).clamp_min(1e-12))
        raw[lay["mean"]] = 0.0
        raw[lay["os"]] = _softplus_inv(os_.to(torch.float32).clamp_min(1e-12))
        return raw

    def _draw_langevin(self, P: int, d: int) -> Optional[torch.Tensor]:
        """The N(0,1) draws sgld.py:70 takes with torch.randn_like per parameter tensor in registration order
        (raw_noise [1], embedding tables [num_uniq, emb], mean constant [], raw_outputscale [], raw_lengthscale [1,d] or
        [1,1], embedding raw_lengthscale [1,1]) for every step after the pretrain phase -- taken from the same global CPU
        generator, in the same order and shapes."""
        if self.langevin is None or self.langevin is False:
            return None
        if torch.is_tensor(self.langevin) or isinstance(self.langevin, np.ndarray):
            lang = torch.as_tensor(self.langevin, dtype=torch.float32)     # caller-supplied draws [E, P]
            assert lang.shape == (self.num_epochs, P)
            return lang
        E = self.num_epochs
        lay = self._param_layout()
        out = torch.zeros(E, lay["P"], dtype=torch.float32)       # full device layout; frozen warp slots are stripped below
        pre = E // 10
        for ep in range(E):
            if ep + 1 > pre:
                out[ep, 0] = torch.randn(1)[0]
                o = lay["tab"]
                for u, e in zip(self.num_uniqs, self.emb_sizes):
                    out[ep, o:o + u * e] = torch.randn(u, e).reshape(-1)
                    o += u * e
                if self.warp_mode == 1:                             # KumarWarp._a, ._b: shape [d] each (layers.py:88-89)
                    out[ep, lay["wa"]:lay["wa"] + d] = torch.randn(d)
                    out[ep, lay["wb"]:lay["wb"] + d] = torch.randn(d)
                out[ep, lay["mean"]] = torch.randn(())
                out[ep, lay["os"]] = torch.randn(())
                if lay["n_ls"]:
                    out[ep, lay["ls"]:lay["ls"] + lay["n_ls"]] = torch.randn(1, lay["n_ls"])[0]
                if self.num_enum > 0:
                    out[ep, lay["le"]] = torch.randn(1, 1)[0, 0]
        return self._strip_raw(out)

    # ------------------------------------------------------------------ fit (gp.py:73-135)
    def _xe_dev(self, Xe, m: int) -> Optional[torch.Tensor]:
        """Categories as a contiguous int32 [m, e] device tensor (range-checked on the host when they arrive on the host)."""
        if self.num_enum == 0:
            return None
        assert Xe is not None and Xe.shape == (m, self.num_enum), "Xe must be [rows, num_enum]"
        if not Xe.is_cuda and m > 0:
            hi = torch.as_tensor(self.num_uniqs, dtype=torch.int64)
            if bool((Xe.long() < 0).any()) or bool((Xe.long() >= hi).any()):
                raise IndexError("categorical index out of range")     # nn.Embedding raises the same way
        return Xe.to(self.device, torch.int32, non_blocking=True).contiguous()

    def fit(self, Xc, Xe, y):
        lib = _lib.lib()
        Xc, Xe, y = filter_nan(Xc, Xe, y, "all")
        self.fit_scaler(Xc, Xe, y)
        Xt, Xe_t, yt = self.xtrans(Xc, Xe, y)
        assert Xt.shape[1] == self.num_cont
        assert Xe_t.shape[1] == self.num_enum
        assert y.shape[1] == self.num_out
        n, d = Xt.shape
        dev = self.device
        NP = int(lib.hb_padded_n(n))
        self.n, self.d, self.NP = n, d, NP
        XtT = torch.zeros(d, NP, dtype=torch.float32, device=dev)
        if d > 0:
            XtT[:, :n] = Xt.to(dev, torch.float32).t()
        Xe_dev = self._xe_dev(Xe_t, n)
        y_dev = yt.reshape(-1).to(dev, torch.float32).contiguous()
        raw0 = self.conf.get("init_raw", None)
        if raw0 is None:
            raw0 = self._init_raw(XtT, n, yt.reshape(-1).to(torch.float32))
        P = self._param_layout()["P"]
        raw_dev = self._expand_raw(torch.as_tensor(raw0, dtype=torch.float32)).to(dev).contiguous().clone()
        assert raw_dev.numel() == P == int(lib.hb_num_params(d, self._spec_ptr())), "raw hyper-parameter vector has the wrong length"
        self.raw_init = self._strip_raw(raw_dev.cpu().clone())
        nd_dev = None
        if self.noise_diag is not None:
            nd_dev = torch.as_tensor(self.noise_diag, dtype=torch.float32).to(dev).contiguous()
            assert nd_dev.numel() == n
        ws_bytes = int(lib.hb_fit_workspace_bytes_ex(n, d, self._spec_ptr()))
        self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        self._XtT, self._Xe_dev, self._y_dev, self._nd_dev = XtT, Xe_dev, y_dev, nd_dev
        if self.optimizer != "psgld":
            self._fit_torch_optimizer(raw_dev)
            self._fitted = True
            return
        lang = self._draw_langevin(P - (2 * d if self.warp_mode == 2 else 0), d)
        lang_dev = None if lang is None else self._expand_raw(lang).to(dev).contiguous()
        losses = (C.c_float * max(1, self.num_epochs))()
        with torch.cuda.device(dev):
            st = lib.hb_fit_ex(_lib.ptr(XtT) if d > 0 else None, _lib.ptr(Xe_dev), _lib.ptr(y_dev), n, d, self._spec_ptr(),
                               _lib.ptr(raw_dev), self.kern_id, _lib.ptr(nd_dev), float(self.noise_lb), float(self.noise_guess),
                               float(self.lr), int(self.num_epochs), _lib.ptr(lang_dev), losses, _lib.ptr(self._ws), ws_bytes,
                               _lib.stream_ptr())
        self.losses = np.array(losses[:self.num_epochs], dtype=np.float32)
        for ep in range(self.num_epochs):
            if not np.isfinite(self.losses[ep]):
                print("jitter is too large, give up fitting GP")
        self._fit_failed = False
        if st == _lib.HB_ERR_NOT_PD:
            self._fit_failed = True      # predict() falls back to N(0, I) like gp.py:152-154
        else:
            _lib.check(st, "hb_fit")
        self.raw = self._strip_raw(raw_dev.cpu())
        self._raw_dev = raw_dev
        self._bind_state()
        if self.verbose:
            for ep in range(self.num_epochs):
                if (ep + 1) % self.print_every == 0 or ep == 0:
                    # the reference re-evaluates the closure after the step; losses[ep+1] is that value
                    val = self.losses[ep + 1] if ep + 1 < self.num_epochs else self.evaluate_loss()
                    print("After %d epochs, loss = %g" % (ep + 1, val), flush=True)
        self._fitted = True

    def _fit_torch_optimizer(self, raw_dev: torch.Tensor) -> None:
        """optimizer='lbfgs' or anything that is not 'psgld' (-> Adam), gp.py:96-126.  As in the reference, torch's own
        optimizer objects hold the step rule and run on the host; every closure evaluation is ONE hb_mll_fwd_bwd (Gram,
        Cholesky, inverse, closed-form gradient: this library's kernels) on the raw vector, which lives on the device.
        Jitter ladder of gp.py:104-126: a step whose closure hits a non-PD matrix is retried with 10x the jitter."""
        lib = _lib.lib()
        n, d, dev = self.n, self.d, self.device
        lay = self._param_layout()
        p = torch.nn.Parameter(raw_dev, requires_grad=True)
        if str(self.optimizer).lower() == "lbfgs":
            opt = torch.optim.LBFGS([p], lr=self.lr, max_iter=5, line_search_fn="strong_wolfe")
        else:
            opt = torch.optim.Adam([p], lr=self.lr)
        grad = torch.empty_like(raw_dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        info = torch.zeros(1, dtype=torch.int32, device=dev)
        jitter = [0.0]

        def closure():
            with torch.cuda.device(dev):
                _lib.check(lib.hb_mll_fwd_bwd(_lib.ptr(self._XtT) if d > 0 else None, _lib.ptr(self._Xe_dev), _lib.ptr(self._y_dev),
                                              n, d, self._spec_ptr(), _lib.ptr(p.data), self.kern_id, _lib.ptr(self._nd_dev),
                                              float(self.noise_lb), float(self.noise_guess), float(jitter[0]), _lib.ptr(grad),
                                              _lib.ptr(loss), _lib.ptr(info), _lib.ptr(self._ws), self._ws.numel(),
                                              _lib.stream_ptr()), "hb_mll_fwd_bwd")
            if int(info.item()) != 0:
                raise _lib.NotPositiveDefinite(f"leading minor {int(info.item())} not positive definite")
            if self.warp_mode == 2:                       # fixed exponents are not parameters
                grad[lay["wa"]:lay["wa"] + lay["n_w"]] = 0.0
            p.grad = grad.clone()
            return loss[0].clone()

        self.losses = np.full(self.num_epochs, np.inf, dtype=np.float32)
        for ep in range(self.num_epochs):
            jitter[0] = 0.0
            while True:
                try:
                    first = []

                    def counted():
                        v = closure()
                        if not first:
                            first.append(float(v))
                        return v
                    opt.step(counted)
                    self.losses[ep] = first[0]
                    break
                except _lib.NotPositiveDefinite:
                    jitter[0] = 1e-6 if jitter[0] == 0.0 else jitter[0] * 10.0
                    if jitter[0] > 1e3:
                        print("jitter is too large, give up fitting GP")
                        break
                    print(f"jitter = {jitter[0] / 100:g}")
            if self.verbose and ((ep + 1) % self.print_every == 0 or ep == 0):
                print("After %d epochs, loss = %g" % (ep + 1, self.losses[ep]), flush=True)
        self.set_hypers(self._strip_raw(p.data.detach().cpu()))

    def set_hypers(self, raw: torch.Tensor):
        """Factorise at given raw hypers (parity tests / warm state); requires a previous fit() for the data."""
        lib = _lib.lib()
        self._raw_dev = self._expand_raw(torch.as_tensor(raw, dtype=torch.float32)).to(self.device).contiguous().clone()
        self.raw = self._strip_raw(self._raw_dev.cpu())
        jit = C.c_float(0.0)
        with torch.cuda.device(self.device):
            st = lib.hb_factorize_ex(_lib.ptr(self._XtT) if self.d > 0 else None, _lib.ptr(self._Xe_dev), _lib.ptr(self._y_dev),
                                     self.n, self.d, self._spec_ptr(), _lib.ptr(self._raw_dev), self.kern_id,
                                     _lib.ptr(self._nd_dev), float(self.noise_lb), C.byref(jit), _lib.ptr(self._ws),
                                     self._ws.numel(), _lib.stream_ptr())
        self.jitter_used = jit.value
        self._fit_failed = st == _lib.HB_ERR_NOT_PD
        if not self._fit_failed:
            _lib.check(st, "hb_factorize")
        self._bind_state()

    def _view(self, p: int, numel: int, dtype=torch.float32) -> torch.Tensor:
        off = p - self._ws.data_ptr()
        nbytes = numel * torch.empty((), dtype=dtype).element_size()
        return self._ws[off:off + nbytes].view(dtype)

    def _bind_state(self):
        lib = _lib.lib()
        fs = _lib.FitState()
        _lib.check(lib.hb_fit_state_ex(_lib.ptr(self._ws), self.n, self.d, self._spec_ptr(), C.byref(fs)), "hb_fit_state")
        NP, d = self.NP, self.d
        H = 3 + d + (1 if self.num_enum > 0 else 0) + (2 * d if self.warp_mode else 0)
        self._h_wa = 3 + d + (1 if self.num_enum > 0 else 0)
        self.hyp_dev = self._view(fs.hyp, H)
        self.L_dev = self._view(fs.L, NP * NP).view(NP, NP)
        self.Linv_dev = self._view(fs.Linv, NP * NP).view(NP, NP)
        self.alpha_dev = self._view(fs.alpha, NP)
        self.Zt_dev = self._view(fs.Zt, (d + self.De) * NP).view(d + self.De, NP)
        self.scal_dev = self._view(fs.scal, 2, torch.float64)
        self.Linv_hi_dev = self._view(fs.Linv_hi, NP * NP).view(NP, NP)
        self.Linv_lo_dev = self._view(fs.Linv_lo, NP * NP).view(NP, NP)
        self.tab_s_dev = self._view(fs.tab_s, max(1, self.T))
        self._emb_meta_dev = self._view(fs.emb_meta, 2 * self.De + 2 * self.num_enum + 3 * self.T + 1, torch.int32)
        self.hyp = self.hyp_dev.cpu()
        if d > 0:
            self._x_mul = self.xscaler.scale_.to(self.device, torch.float32).contiguous()
            self._x_add = self.xscaler.min_.to(self.device, torch.float32).contiguous()
        else:
            self._x_mul = self._x_add = None
        self._y_mean = float(self.yscaler.mean[0])
        self._y_std = float(self.yscaler.std[0])

    # ------------------------------------------------------------------ loss / gradient at the current hypers
    def evaluate_loss(self, return_grad: bool = False):
        """-mll/n (and its gradient w.r.t. the raw parameters) at the current hypers; used for verbose printing and the
        parity tests.  Numeric ARD models go through the individual C-ABI calls (gram, cholesky, ...), mixed / non-ARD
        models through the fused hb_mll_fwd_bwd on a scratch workspace (the prediction state is left untouched)."""
        lib = _lib.lib()
        n, d, NP, dev = self.n, self.d, self.NP, self.device
        st = _lib.stream_ptr()
        P = self._param_layout()["P"]
        info = torch.zeros(1, dtype=torch.int32, device=dev)
        grad = torch.empty(P, dtype=torch.float32, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        if self._general:
            scratch = torch.empty(self._ws.numel(), dtype=torch.uint8, device=dev)
            with torch.cuda.device(dev):
                _lib.check(lib.hb_mll_fwd_bwd(_lib.ptr(self._XtT) if d > 0 else None, _lib.ptr(self._Xe_dev), _lib.ptr(self._y_dev),
                                              n, d, self._spec_ptr(), _lib.ptr(self._raw_dev), self.kern_id, _lib.ptr(self._nd_dev),
                                              float(self.noise_lb), float(self.noise_guess), 0.0, _lib.ptr(grad), _lib.ptr(loss),
                                              _lib.ptr(info), _lib.ptr(scratch), scratch.numel(), st), "hb_mll_fwd_bwd")
            if int(info.item()) != 0:
                raise _lib.NotPositiveDefinite(f"leading minor {int(info.item())} not positive definite")
            return (float(loss.item()), self._strip_raw(grad.cpu())) if return_grad else float(loss.item())
        hyp = torch.empty(d + 3, dtype=torch.float32, device=dev)
        K = torch.empty(NP, NP, dtype=torch.float32, device=dev)
        Linv = torch.empty_like(K)
        tmp = torch.empty_like(K)
        cholws = torch.empty(128 * 128, dtype=torch.float32, device=dev)
        alpha = torch.empty(NP, dtype=torch.float32, device=dev)
        scal = torch.empty(2, dtype=torch.float64, device=dev)
        sws = torch.empty(NP * 8 * (1 + NP // 64) + 256, dtype=torch.uint8, device=dev)
        gws = torch.empty((NP // 128) * (NP // 128 + 1) // 2 * (d + 3) * 4 + 512, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.hb_transform_hypers(_lib.ptr(self._raw_dev), d, float(self.noise_lb), _lib.ptr(hyp), st), "transform")
            _lib.check(lib.hb_gram(_lib.ptr(self._XtT), n, d, _lib.ptr(hyp), self.kern_id, _lib.ptr(self._nd_dev), 0.0,
                                   _lib.ptr(K), st), "gram")
            _lib.check(lib.hb_cholesky(_lib.ptr(K), NP, _lib.ptr(cholws), _lib.ptr(info), st), "cholesky")
            _lib.check(lib.hb_tri_inverse(_lib.ptr(K), NP, _lib.ptr(Linv), _lib.ptr(tmp), st), "tri_inverse")
            _lib.check(lib.hb_solve_logdet(_lib.ptr(K), _lib.ptr(Linv), _lib.ptr(self._y_dev), n, NP, _lib.ptr(hyp),
                                           _lib.ptr(alpha), _lib.ptr(scal), _lib.ptr(sws), st), "solve_logdet")
            _lib.check(lib.hb_kinv(_lib.ptr(Linv), NP, _lib.ptr(tmp), st), "kinv")
            _lib.check(lib.hb_mll_grad(_lib.ptr(self._XtT), n, d, _lib.ptr(self._raw_dev), _lib.ptr(hyp), self.kern_id,
                                       _lib.ptr(tmp), _lib.ptr(alpha), _lib.ptr(scal), float(self.noise_guess),
                                       _lib.ptr(grad), _lib.ptr(loss), _lib.ptr(gws), st), "mll_grad")
        if int(info.item()) != 0:
            raise _lib.NotPositiveDefinite(f"leading minor {int(info.item())} not positive definite")
        if return_grad:
            return float(loss.item()), grad.cpu()
        return float(loss.item())

    # ------------------------------------------------------------------ posterior (gp.py:137-164) + MACE (acq.py:146-171)
    def _copy_stream(self):
        if getattr(self, "_side_stream", None) is None:
            self._side_stream = torch.cuda.Stream(self.device)
        return self._side_stream

    def _posterior(self, Xs_dev: Optional[torch.Tensor], want_F: bool, tau=0.0, kappa=0.0, eps=0.0, xi1=None, xi2=None,
                   seed: int = 0, want_mu_var: bool = True, Xe_dev: Optional[torch.Tensor] = None,
                   out_mu: Optional[torch.Tensor] = None, out_var: Optional[torch.Tensor] = None):
        """out_mu / out_var: optional contiguous fp32 device rows [m] to write the posterior into (GeneralAcq stacks the
        outputs of a MultiTaskModel into one [O, m] buffer this way)."""
        lib = _lib.lib()
        assert self._fitted or hasattr(self, "Linv_dev"), "fit() first"
        # a pinned host batch larger than one chunk is uploaded chunk by chunk under the scoring (same results)
        host_rows = None
        if (Xs_dev is not None and not Xs_dev.is_cuda and Xs_dev.is_pinned() and self.d > 0
                and Xs_dev.shape[0] > self.m_chunk and Xs_dev.dtype == torch.float32 and Xs_dev.is_contiguous()):
            host_rows = Xs_dev
        m = Xs_dev.shape[0] if Xs_dev is not None else Xe_dev.shape[0]
        dev = self.device
        if m == 0:      # empty batch: same (empty) shapes the reference would return
            e = torch.empty(0, dtype=torch.float32, device=dev)
            return (torch.empty(0, 3, dtype=torch.float32, device=dev) if want_F else None,
                    e if want_mu_var else None, e.clone() if want_mu_var else None)
        F = torch.empty(m, 3, dtype=torch.float32, device=dev) if want_F else None
        mu = (torch.empty(m, dtype=torch.float32, device=dev) if out_mu is None else out_mu) if want_mu_var else None
        var = (torch.empty(m, dtype=torch.float32, device=dev) if out_var is None else out_var) if want_mu_var else None
        if self._fit_failed:
            # gp.py:152-154: "jitter is too large, output random predictions" = N(0, I) in the standardised space, pushed
            # through the same un-scaling and (for F) the MACE epilogue kernel -- never the leftovers of a failed factorisation
            print("jitter is too large, output random predictions")
            mu_f = torch.full((m,), self._y_mean, dtype=torch.float32, device=dev) if out_mu is None else out_mu.fill_(self._y_mean)
            var_f = (torch.full((m,), max(self._y_std ** 2, EPS32), dtype=torch.float32, device=dev) if out_var is None
                     else out_var.fill_(max(self._y_std ** 2, EPS32)))
            if want_F:
                with torch.cuda.device(dev):
                    _lib.check(lib.hb_mace_epilogue(_lib.ptr(mu_f), _lib.ptr(var_f), m, float(self.noise[0]), float(tau), float(kappa),
                                                    float(eps), _lib.ptr(xi1), _lib.ptr(xi2), int(seed), _lib.ptr(F),
                                                    _lib.stream_ptr()), "hb_mace_epilogue")
            return F, (mu_f if want_mu_var else None), (var_f if want_mu_var else None)
        x_mul, x_add = self._x_mul, self._x_add      # (an input warp is applied inside the K* load stage)
        mc = min(self.m_chunk, max(128, -(-m // 128) * 128))
        need = int(lib.hb_posterior_workspace_bytes(self.n, self.d, mc))
        if self._post_ws is None or self._post_ws.numel() < need:
            self._post_ws = torch.empty(need, dtype=torch.uint8, device=dev)

        def call(xs, xe, rows, row0):
            off = lambda t, w=1: None if t is None else C.c_void_p(t.data_ptr() + row0 * w * 4)      # fp32 / int32 rows
            return lib.hb_posterior_mace_ex(off(xs, self.d) if self.d > 0 else None, off(xe, self.num_enum), rows, row0, self.n, self.d,
                                            self._spec_ptr(), _lib.ptr(self._emb_meta_dev) if self.num_enum else None,
                                            _lib.ptr(self.tab_s_dev) if self.num_enum else None, _lib.ptr(x_mul), _lib.ptr(x_add),
                                            _lib.ptr(self.Zt_dev), _lib.ptr(self.alpha_dev), _lib.ptr(self.Linv_dev),
                                            _lib.ptr(self.Linv_hi_dev if self.tensor_cores else None),
                                            _lib.ptr(self.Linv_lo_dev if self.tensor_cores else None),
                                            _lib.ptr(self.hyp_dev), self.kern_id, self._y_mean, self._y_std,
                                            int(bool(self.pred_likeli)), float(tau), float(kappa), float(eps),
                                            off(xi1), off(xi2), int(seed), off(F, 3), off(mu), off(var),
                                            _lib.ptr(self._post_ws), self._post_ws.numel(), mc, _lib.stream_ptr())
        with torch.cuda.device(dev):
            if host_rows is None:
                st = call(Xs_dev, Xe_dev, m, 0)
            else:
                # pinned HOST candidates: the copy of chunk i+1 runs on a side stream under the scoring of chunk i
                Xs_dev = torch.empty(m, self.d, dtype=torch.float32, device=dev)
                main, side = torch.cuda.current_stream(dev), self._copy_stream()
                side.wait_stream(main)
                events = []
                with torch.cuda.stream(side):
                    for c0 in range(0, m, mc):
                        Xs_dev[c0:c0 + mc].copy_(host_rows[c0:c0 + mc], non_blocking=True)
                        ev = torch.cuda.Event()
                        ev.record(side)
                        events.append(ev)
                st = _lib.HB_OK
                for ev, c0 in zip(events, range(0, m, mc)):
                    main.wait_event(ev)
                    st = call(Xs_dev, Xe_dev, min(mc, m - c0), c0)
                    if st != _lib.HB_OK:
                        break
                Xs_dev.record_stream(side)      # allocated on the main stream's pool, written on the copy stream
        _lib.check(st, "hb_posterior_mace")
        return F, mu, var

    def _to_dev(self, Xc, keep_pinned: bool = False) -> Optional[torch.Tensor]:
        if Xc is None or self.d == 0:
            return None
        Xc = torch.as_tensor(Xc)
        if (keep_pinned and not Xc.is_cuda and Xc.is_pinned() and Xc.dtype == torch.float32 and Xc.is_contiguous()
                and Xc.shape[0] > self.m_chunk and not self._fit_failed):
            return Xc            # _posterior pipelines the upload with the scoring
        return Xc.to(self.device, torch.float32, non_blocking=True).contiguous()

    def _rows(self, Xc, Xe) -> int:
        return (Xc if (Xc is not None and self.d > 0) else Xe).shape[0]

    def predict(self, Xc, Xe=None):
        if torch.is_tensor(Xc) and Xc.requires_grad and not self._fit_failed:
            return self._predict_autograd(Xc, Xe)
        probe = Xc if (Xc is not None and self.d > 0) else Xe
        on_cpu = not (torch.is_tensor(probe) and probe.is_cuda)
        m = self._rows(Xc, Xe)
        _, mu, var = self._posterior(self._to_dev(Xc), want_F=False, Xe_dev=self._xe_dev(Xe, m))
        mu, var = mu.view(-1, self.num_out), var.view(-1, self.num_out)
        if on_cpu:
            return mu.cpu(), var.cpu()
        return mu, var

    def predict_mace(self, Xc, tau: float, kappa: float, eps: float = 1e-4, xi1=None, xi2=None, seed: int = 0,
                     return_mu_var: bool = False, Xe=None, device_out: bool = False):
        """Fused GP.predict + MACE.eval: returns F [m,3] = (LCB, -logEI, -logPI) on the input's device (device_out=True:
        on the GPU even for host inputs -- a pinned host batch is then uploaded chunk by chunk under the scoring)."""
        probe = Xc if (Xc is not None and self.d > 0) else Xe
        on_cpu = not (torch.is_tensor(probe) and probe.is_cuda) and not device_out
        m = self._rows(Xc, Xe)
        Xs = self._to_dev(Xc, keep_pinned=True)
        if xi1 is None and self.rng == "host":
            xi1 = torch.randn(m, 1)      # acq.py:154 then :155 -- same generator, same order, same shapes
            xi2 = torch.randn(m, 1)
        if xi1 is not None:
            xi1 = torch.as_tensor(xi1).reshape(-1).to(self.device, torch.float32, non_blocking=True).contiguous()
            xi2 = torch.as_tensor(xi2).reshape(-1).to(self.device, torch.float32, non_blocking=True).contiguous()
        F, mu, var = self._posterior(Xs, True, tau, kappa, eps, xi1, xi2, seed, want_mu_var=return_mu_var,
                                     Xe_dev=self._xe_dev(Xe, m))
        if on_cpu:
            F = F.cpu()
            if return_mu_var:
                mu, var = mu.cpu(), var.cpu()
        return (F, mu, var) if return_mu_var else F

    def _predict_autograd(self, Xc, Xe=None):
        """Differentiable predict for the ``support_grad`` contract (test_base_model.py:94-108): value and closed-form
        input gradients from the CUDA kernels (``hb_posterior_grad``) behind a torch.autograd.Function; a Kumaraswamy
        warp stays in torch in front of it so autograd chains through it (SURVEY 8f-3)."""
        dev = self.device
        Xs = Xc.to(dev, torch.float32)
        self._grad_xe = self._xe_dev(Xe, Xs.shape[0])
        if self.warp_mode:
            wa, wb = self.hyp_dev[self._h_wa:self._h_wa + self.d], self.hyp_dev[self._h_wa + self.d:self._h_wa + 2 * self.d]
            Xin = kumaraswamy_warp(Xs * self._x_mul + self._x_add, wa, wb)
            x_mul, x_add = torch.ones_like(self._x_mul), torch.zeros_like(self._x_add)
        else:
            Xin, x_mul, x_add = Xs, self._x_mul, self._x_add
        mu, var = _PredictWithGrad.apply(Xin, self, x_mul, x_add)
        return mu.view(-1, 1).to(Xc.device), var.view(-1, 1).to(Xc.device)

    def _posterior_grad(self, Xin: torch.Tensor, x_mul, x_add):
        """(mu, var, dmu/dXin, dvar/dXin) on the device through the C ABI."""
        lib = _lib.lib()
        dev = self.device
        Xin = Xin.detach().contiguous()
        m = Xin.shape[0]
        mc = min(1024, max(128, -(-m // 128) * 128))
        need = int(lib.hb_posterior_workspace_bytes(self.n, self.d, mc))
        if self._post_ws is None or self._post_ws.numel() < need:
            self._post_ws = torch.empty(need, dtype=torch.uint8, device=dev)
        mu = torch.empty(m, dtype=torch.float32, device=dev)
        var = torch.empty(m, dtype=torch.float32, device=dev)
        dmu = torch.empty(m, self.d, dtype=torch.float32, device=dev)
        dvar = torch.empty(m, self.d, dtype=torch.float32, device=dev)
        if m == 0:
            return mu, var, dmu, dvar
        with torch.cuda.device(dev):
            # (a warp stays in torch in front of this call so that autograd chains through it: the kernels get warp = 0)
            st = lib.hb_posterior_grad_ex(_lib.ptr(Xin), _lib.ptr(self._grad_xe), m, self.n, self.d,
                                          C.byref(self._spec_nowarp) if self._general else None,
                                          _lib.ptr(self._emb_meta_dev) if self.num_enum else None,
                                          _lib.ptr(self.tab_s_dev) if self.num_enum else None, _lib.ptr(x_mul), _lib.ptr(x_add),
                                          _lib.ptr(self.Zt_dev), _lib.ptr(self.alpha_dev), _lib.ptr(self.Linv_dev),
                                          _lib.ptr(self.hyp_dev), self.kern_id, self._y_mean, self._y_std,
                                          int(bool(self.pred_likeli)), _lib.ptr(mu), _lib.ptr(var), _lib.ptr(dmu), _lib.ptr(dvar),
                                          _lib.ptr(self._post_ws), self._post_ws.numel(), mc, _lib.stream_ptr())
        _lib.check(st, "hb_posterior_grad")
        return mu, var, dmu, dvar

    def sample_y(self, Xc, Xe=None, n_samples=1):
        """Joint posterior samples (gp.py:166-177) through ``hb_sample_y``: K*, K**, the rank-n downdate and the Cholesky root
        of the m x m predictive covariance all run in this library's kernels; the N(0,1) draws come from torch's CPU
        generator."""
        lib = _lib.lib()
        dev = self.device
        m = self._rows(Xc, Xe)
        if self._fit_failed:          # gp.py:152-154 "output random predictions": N(y_mean, y_std^2) independent draws
            return torch.randn(n_samples, m, self.num_out) * self._y_std + self._y_mean
        with torch.no_grad():
            Xs, xe = self._to_dev(Xc), self._xe_dev(Xe, m)
            z = torch.randn(n_samples, m).to(dev).contiguous()
            out = torch.empty(n_samples, m, dtype=torch.float32, device=dev)
            need = int(lib.hb_sample_workspace_bytes(self.n, self.d, self._spec_ptr(), m))
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            hyp_host = self.hyp.contiguous()
            jit = C.c_float(0.0)
            with torch.cuda.device(dev):
                st = lib.hb_sample_y(_lib.ptr(Xs), _lib.ptr(xe), m, self.n, self.d, self._spec_ptr(),
                                     _lib.ptr(self._emb_meta_dev) if self.num_enum else None,
                                     _lib.ptr(self.tab_s_dev) if self.num_enum else None, _lib.ptr(self._x_mul), _lib.ptr(self._x_add),
                                     _lib.ptr(self.Zt_dev), _lib.ptr(self.alpha_dev), _lib.ptr(self.Linv_dev), _lib.ptr(self.hyp_dev),
                                     C.c_void_p(hyp_host.data_ptr()), self.kern_id, self._y_mean, self._y_std, int(bool(self.pred_likeli)),
                                     _lib.ptr(z), int(n_samples), _lib.ptr(out), C.byref(jit), _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
            _lib.check(st, "hb_sample_y")
            self.sample_jitter = jit.value
            return out.cpu().view(n_samples, m, self.num_out)

    def sample_f(self):
        raise NotImplementedError("Thompson sampling is not supported for GP, use `sample_y` instead")

    # ------------------------------------------------------------------ state replication (hebo_b200.dist)
    def export_meta(self) -> dict:
        return dict(n=self.n, d=self.d, NP=self.NP, kernel=self.kernel, noise_lb=self.noise_lb,
                    pred_likeli=self.pred_likeli, x_scale=self.xscaler.scale_, x_min=self.xscaler.min_,
                    y_mean=self.yscaler.mean.clone(), y_std=self.yscaler.std.clone(), warp_a=self.warp_a,
                    warp_b=self.warp_b, raw=self.raw.clone(), fit_failed=self._fit_failed)

    def allocate_from_meta(self, meta: dict) -> None:
        lib = _lib.lib()
        self.n, self.d, self.NP = meta["n"], meta["d"], meta["NP"]
        self.kernel, self.kern_id = meta["kernel"], _lib.KERNEL_IDS[meta["kernel"]]
        self.noise_lb, self.pred_likeli = meta["noise_lb"], meta["pred_likeli"]
        self.xscaler.scale_, self.xscaler.min_ = meta["x_scale"], meta["x_min"]
        self.yscaler.mean, self.yscaler.std = meta["y_mean"], meta["y_std"]
        self.warp_a, self.warp_b, self.raw = meta["warp_a"], meta["warp_b"], meta["raw"]
        self._fit_failed = meta["fit_failed"]
        ws_bytes = int(lib.hb_fit_workspace_bytes_ex(self.n, self.d, self._spec_ptr()))
        self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        self._bind_state()

    def state_tensors(self):
        """What candidate scoring reads (hebo_b200.dist.broadcast_state replicates exactly these): hypers, alpha, the
        scaled features, the fp16 operand split of L^-1 (half of each opaque buffer + the scale word), fp32 L^-1 for the
        guarded rows, and the categorical tables / layout of a mixed model."""
        half = self.NP * self.NP // 2
        ts = [self.hyp_dev, self.alpha_dev, self.Zt_dev, self.Linv_dev, self.Linv_hi_dev.view(-1)[:half],
              self.Linv_lo_dev.view(-1)[:half + 2]]
        if _lib.lib().hb_vnorm_operand_kind() != 0:       # 3xTF32 operands occupy the whole buffers
            ts[4:] = [self.Linv_hi_dev, self.Linv_lo_dev]
        if self.num_enum > 0:
            ts += [self.tab_s_dev, self._emb_meta_dev]
        return ts

    def finish_load(self) -> None:
        self.hyp = self.hyp_dev.cpu()
        self._fitted = True

    @property
    def noise(self):
        """gp.py:182-184: likelihood noise in original y units, shape [num_out], detached."""
        return (self.hyp[0] * self.yscaler.std ** 2).view(self.num_out).detach()


B200GP = GP


def register(name: str = "gp_b200", override_gp: bool = False) -> bool:
    """Register into a real HEBO install's model registry (model_factory.py:30-58).  Returns False when
    ``hebo`` is not importable."""
    try:
        from hebo.models import model_factory
    except Exception:
        return False
    model_factory.model_dict[name] = GP
    model_factory.model_dict["multi_task_b200"] = MultiTaskModel
    if override_gp:
        model_factory.model_dict["gp"] = GP
    model_factory.model_names = list(model_factory.model_dict.keys())
    return True


class MultiTaskModel(BaseModel):
    """Multi-output wrapper: one single-output model per column of y (HEBO/hebo/models/model_factory.py:60-92), the
    building block of the reference's multi-objective / constrained optimisers (GeneralBO)."""
    support_multi_output = True

    def __init__(self, num_cont, num_enum, num_out, **conf):
        super().__init__(num_cont, num_enum, num_out, **conf)
        self.model_conf = {k: v for k, v in conf.items() if k not in ("model_name", "base_model_name")}
        self.models = [GP(num_cont, num_enum, 1, **self.model_conf) for _ in range(num_out)]

    def fit(self, Xc, Xe, y):
        for i in range(self.num_out):
            self.models[i].fit(Xc, Xe, y[:, [i]])

    def predict(self, Xc, Xe=None):
        out = [m.predict(Xc, Xe) for m in self.models]
        return torch.cat([o[0] for o in out], dim=1), torch.cat([o[1] for o in out], dim=1)

    @property
    def noise(self):
        return torch.FloatTensor([float(m.noise) for m in self.models]).reshape(self.num_out)
