"""ctypes binding of libhebo_b200.so (the C ABI of include/hebo_b200.h).

The product path has no CPU / torch fallback: if the CUDA library is missing the import of the model
classes still works (so that host-only logic can be tested) but every compute call raises loudly.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libhebo_b200.so")

HB_OK, HB_ERR_INVALID, HB_ERR_NOT_PD, HB_ERR_CUDA = 0, 1, 2, 3
KERNEL_IDS = {"matern32": 0, "matern52": 1, "rbf": 2}


class HeboB200Error(RuntimeError):
    pass


class NotPositiveDefinite(HeboB200Error):
    pass


class FitState(C.Structure):      # hb_fit_state_t
    _fields_ = [("hyp", C.c_void_p), ("L", C.c_void_p), ("Linv", C.c_void_p), ("alpha", C.c_void_p),
                ("Zt", C.c_void_p), ("scal", C.c_void_p), ("Linv_hi", C.c_void_p), ("Linv_lo", C.c_void_p),
                ("tab_s", C.c_void_p), ("emb_meta", C.c_void_p), ("grad", C.c_void_p), ("loss", C.c_void_p)]


class ModelSpec(C.Structure):     # hb_model_spec_t
    _fields_ = [("ard_kernel", C.c_int32), ("num_enum", C.c_int32), ("num_uniqs", C.POINTER(C.c_int32)),
                ("emb_sizes", C.POINTER(C.c_int32)), ("warp", C.c_int32)]


_vp, _i64, _i32, _f32, _u64 = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_uint64
_sp = C.POINTER(ModelSpec)

# name -> (restype, argtypes); must list every function declared in include/hebo_b200.h
SIGNATURES = {
    "hb_version": (_i32, []),
    "hb_last_error": (C.c_char_p, []),
    "hb_padded_n": (_i64, [_i64]),
    "hb_launch_count": (_i64, [_i32]),
    "hb_profile_enable": (_i32, [_i32]),
    "hb_profile_collect": (_i32, [C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "hb_vnorm_operand_kind": (_i32, []),
    "hb_num_params": (_i64, [_i64, _sp]),
    "hb_guard_stats": (_i32, [C.POINTER(C.c_uint64), _i32]),
    "hb_fit_workspace_bytes": (_i64, [_i64, _i64]),
    "hb_fit_workspace_bytes_ex": (_i64, [_i64, _i64, _sp]),
    "hb_posterior_workspace_bytes": (_i64, [_i64, _i64, _i64]),
    "hb_pareto_workspace_bytes": (_i64, [_i64]),
    "hb_transform_hypers": (_i32, [_vp, _i64, _f32, _vp, _vp]),
    "hb_median_pdist": (_i32, [_vp, _i64, _i64, _vp, _i64, _f32, _vp, _vp]),
    "hb_gram": (_i32, [_vp, _i64, _i64, _vp, _i32, _vp, _f32, _vp, _vp]),
    "hb_cholesky": (_i32, [_vp, _i64, _vp, _vp, _vp]),
    "hb_tri_inverse": (_i32, [_vp, _i64, _vp, _vp, _vp]),
    "hb_kinv": (_i32, [_vp, _i64, _vp, _vp]),
    "hb_solve_logdet": (_i32, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "hb_mll_grad": (_i32, [_vp, _i64, _i64, _vp, _vp, _i32, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp]),
    "hb_psgld_step": (_i32, [_vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _vp, _vp]),
    "hb_fit": (_i32, [_vp, _vp, _i64, _i64, _vp, _i32, _vp, _f32, _f32, _f32, _i32, _vp,
                      C.POINTER(C.c_float), _vp, _i64, _vp]),
    "hb_factorize": (_i32, [_vp, _vp, _i64, _i64, _vp, _i32, _vp, _f32, C.POINTER(C.c_float), _vp, _i64, _vp]),
    "hb_fit_state": (_i32, [_vp, _i64, _i64, C.POINTER(FitState)]),
    "hb_fit_state_ex": (_i32, [_vp, _i64, _i64, _sp, C.POINTER(FitState)]),
    "hb_fit_ex": (_i32, [_vp, _vp, _vp, _i64, _i64, _sp, _vp, _i32, _vp, _f32, _f32, _f32, _i32, _vp,
                         C.POINTER(C.c_float), _vp, _i64, _vp]),
    "hb_factorize_ex": (_i32, [_vp, _vp, _vp, _i64, _i64, _sp, _vp, _i32, _vp, _f32, C.POINTER(C.c_float), _vp, _i64, _vp]),
    "hb_mll_fwd_bwd": (_i32, [_vp, _vp, _vp, _i64, _i64, _sp, _vp, _i32, _vp, _f32, _f32, _f32, _vp, _vp, _vp, _vp, _i64, _vp]),
    "hb_posterior_mace_ex": (_i32, [_vp, _vp, _i64, _i64, _i64, _i64, _sp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32,
                                    _f32, _f32, _i32, _f32, _f32, _f32, _vp, _vp, _u64, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "hb_posterior_grad_ex": (_i32, [_vp, _vp, _i64, _i64, _i64, _sp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _f32, _f32,
                                    _i32, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "hb_posterior_mace": (_i32, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _f32, _f32, _i32,
                                 _f32, _f32, _f32, _vp, _vp, _u64, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "hb_posterior_grad": (_i32, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _f32, _f32, _i32,
                                 _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "hb_sample_workspace_bytes": (_i64, [_i64, _i64, _sp, _i64]),
    "hb_sample_y": (_i32, [_vp, _vp, _i64, _i64, _i64, _sp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _f32, _f32, _i32, _vp, _i32,
                           _vp, C.POINTER(C.c_float), _vp, _i64, _vp]),
    "hb_mace_epilogue": (_i32, [_vp, _vp, _i64, _f32, _f32, _f32, _f32, _vp, _vp, _u64, _vp, _vp]),
    "hb_general_acq_epilogue": (_i32, [_vp, _vp, _i64, _i32, _i32, _vp, _f32, _f32, _i32, _vp, _u64, _i64, _vp, _vp, _vp]),
    "hb_pareto_front": (_i32, [_vp, _i64, _i32, _i64, _vp, _vp, _vp, _vp, _i64, _vp]),
    "hb_pareto_front3": (_i32, [_vp, _i64, _vp, _vp, _vp, _i64, _vp]),
    "hb_nsga2_init": (_i32, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _i64, _u64, _vp, _vp, _vp]),
    "hb_nsga2_mate": (_i32, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _u64, _i32, _vp, _vp, _vp, _vp]),
    "hb_nsga2_survive": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "hb_nsga2_survive_k": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hb_front_merge_workspace_bytes": (_i64, [_i64, _i64]),
    "hb_front_pack": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp]),
    "hb_front_merge": (_i32, [_vp, _i64, _i64, _vp, _vp, _i64, _vp]),
}

_lib = None


def available() -> bool:
    return os.path.isfile(LIB_PATH)


def lib():
    """Load (once) and return the bound library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not available():
            raise HeboB200Error(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  hebo_b200 has no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status: int, what: str) -> None:
    if status == HB_OK:
        return
    if status == HB_ERR_NOT_PD:
        raise NotPositiveDefinite(f"{what}: matrix not positive definite (jitter ladder exhausted)")
    if status == HB_ERR_CUDA:
        raise HeboB200Error(f"{what}: CUDA error: {lib().hb_last_error().decode()}")
    raise HeboB200Error(f"{what}: invalid argument (status {status})")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
