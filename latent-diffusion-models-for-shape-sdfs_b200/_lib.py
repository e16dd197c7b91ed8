"""ctypes binding of libsdfb200.so (the C ABI in include/sdfb200.h).

There is no fallback: if the shared library is missing or fails to load, importing the
product API raises.  The oracle under ``oracle/`` is never imported from here.
"""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB

PREC_FP32, PREC_BF16, PREC_FP16 = 0, 1, 2
PRECISIONS = {"fp32": PREC_FP32, "bf16": PREC_BF16, "fp16": PREC_FP16}

DECODER_PARAM_FLOATS = 1839358
DDPM_PARAM_FLOATS = 3936512

_vp, _i, _i64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/sdfb200.h declares
SIGNATURES = {
    "sdfb_version": (_i, []),
    "sdfb_last_error": (C.c_char_p, []),
    "sdfb_decoder_create": (_i, [_vp, _sz, _i, C.POINTER(_vp)]),
    "sdfb_decoder_destroy": (_i, [_vp]),
    "sdfb_decode_grid": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _vp]),
    "sdfb_decode_grid_bits": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "sdfb_decode_grid_batch": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp]),
    "sdfb_decode_points": (_i, [_vp, _vp, _vp, _i64, _vp, _i, _vp]),
    "sdfb_decoder_vjp_latent": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "sdfb_decoder_vjp_latent_tc": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _i, _vp]),
    "sdfb_decoder_fit_loss_grad": (_i, [_vp, _vp, _vp, _i64, _vp, C.c_float, _vp, _vp, _vp, _i, _vp]),
    "sdfb_mc_weld_workspace_bytes": (_i, [_i, C.POINTER(C.c_size_t)]),
    "sdfb_mc_weld_count": (_i, [_vp, _i64, _i, _vp, C.c_size_t, C.POINTER(C.c_int64), _vp]),
    "sdfb_mc_weld_fill": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    "sdfb_latent_adam_step": (_i, [_vp, _vp, _vp, _vp, _vp, _i, C.c_float, C.c_float, C.c_double, C.c_double, C.c_float, _i, _vp]),
    "sdfb_decoder_fit_loss_grad_batch": (_i, [_vp, _vp, _vp, _i, _i64, _vp, C.c_float, _vp, _vp, _i, _vp]),
    "sdfb_decode_grid_host": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i]),
    "sdfb_decode_points_host": (_i, [_vp, _vp, _vp, _i64, _vp, _i]),
    "sdfb_grid_points": (_i, [_i, _i, _i, _vp, _vp]),
    "sdfb_sign_change_mask": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "sdfb_mc_workspace_bytes": (_i, [_i, _i, _i, C.POINTER(_sz)]),
    "sdfb_mc_count": (_i, [_vp, _vp, _i, _i, _i, _vp, _sz, C.POINTER(_i64), _vp]),
    "sdfb_mc_generate": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "sdfb_decode_sparse_field": (_i, [_vp, _vp, _i, C.c_float, C.c_float, C.c_float, C.c_float, _vp, _vp, _i, _vp, _vp]),
    "sdfb_decode_debug_pass": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp]),
    "sdfb_decoder_last_kernel_ms": (_i, [_vp, C.POINTER(C.c_float)]),
    "sdfb_decoder_check": (_i, [_vp, _vp]),
    "sdfb_decoder_set_timeout_ns": (_i, [_vp, C.c_uint64]),
    "sdfb_ddpm_check": (_i, [_vp, _vp]),
    "sdfb_ddpm_set_timeout_ns": (_i, [_vp, C.c_uint64]),
    "sdfb_comm_unique_id": (_i, [_vp]),
    "sdfb_comm_create": (_i, [_vp, _i, _i, _i, C.POINTER(_vp)]),
    "sdfb_comm_wrap": (_i, [_vp, _i, _i, _i, C.POINTER(_vp)]),
    "sdfb_comm_destroy": (_i, [_vp]),
    "sdfb_comm_barrier": (_i, [_vp, _vp]),
    "sdfb_allgather_slabs": (_i, [_vp, _vp, _sz, _vp]),
    "sdfb_decode_grid_sharded": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_sz), _vp]),
    "sdfb_ddpm_create": (_i, [_vp, _sz, _i, C.POINTER(_vp)]),
    "sdfb_ddpm_destroy": (_i, [_vp]),
    "sdfb_ddpm_sample": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "sdfb_ddpm_denoise": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp]),
    "sdfb_ddpm_sample_host": (_i, [_vp, _vp, _vp, _i, _i, _i]),
    "sdfb_ddpm_last_kernel_ms": (_i, [_vp, C.POINTER(C.c_float)]),
    "sdfb_ddpm_sample_philox": (_i, [_vp, _vp, C.c_uint64, _i64, _i, _i, _i, _i, _vp]),
    "sdfb_ddpm_sample_philox_host": (_i, [_vp, _vp, C.c_uint64, _i64, _i, _i, _i, _i]),
    "sdfb_philox_normal": (_i, [C.c_uint64, _i64, _i, _i, _i, _vp, _vp]),
    "sdfb_ddim_schedule": (_i, [_i, C.c_float, _i, _vp, _vp]),
    "sdfb_ddpm_sample_ddim": (_i, [_vp, _vp, _vp, _i, _i, C.c_float, _i, _vp]),
    "sdfb_ddpm_sample_ddim_philox": (_i, [_vp, _vp, C.c_uint64, _i64, _i, _i, C.c_float, _i, _i, _vp]),
    "sdfb_ddpm_invert_ddim": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "sdfb_ddpm_trainer_create": (_i, [_vp, _sz, _i, _i, C.POINTER(_vp)]),
    "sdfb_ddpm_trainer_destroy": (_i, [_vp]),
    "sdfb_ddpm_trainer_step": (_i, [_vp, _vp, _vp, _vp, _i, C.c_float, C.c_float, C.c_float, C.c_float, _i, _vp, _vp, _vp]),
    "sdfb_ddpm_trainer_get_params": (_i, [_vp, _vp]),
    "sdfb_decoder_trainer_create": (_i, [_vp, _sz, _i, _i, C.POINTER(_vp)]),
    "sdfb_decoder_trainer_destroy": (_i, [_vp]),
    "sdfb_decoder_trainer_step": (_i, [_vp, _vp, _vp, _vp, _i, _i64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _i, _vp, _vp,
                                       _vp, _vp]),
    "sdfb_decoder_trainer_get_params": (_i, [_vp, _vp]),
    "sdfb_gemm_selftest": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "sdfb_umma_selftest": (_i, [_vp, _vp, _vp, _i, _vp]),
    "sdfb_umma_rate": (_i, [_i, _i, _i, _i, _i, _i, C.POINTER(C.c_double)]),
    "sdfb_tma_ingest_rate": (_i, [_i, _i, _i, _i, _i, _i, _i, _i, C.POINTER(C.c_double)]),
}

_lib = None


class SdfbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libsdfb200 error {code}: {msg}")
        self.code = code


def load() -> C.CDLL:
    """Load libsdfb200.so (must have been built: ``__graft_entry__.build()``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB):
        raise ImportError(f"{LIB} is missing - run __graft_entry__.build(); there is no CPU fallback")
    lib = C.CDLL(LIB)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise SdfbError(rc, load().sdfb_last_error().decode("utf-8", "replace"))
