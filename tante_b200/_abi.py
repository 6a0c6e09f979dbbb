"""ctypes binding of include/tante_b200.h (libtante_b200.so).

The library is the product's only compute path: if it is missing or fails to load the
import raises -- there is no PyTorch/CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtante_b200.so")

TANTE_MAX_ORDER = 8
TANTE_MAX_LAYERS = 32
PREC_FP32 = 0
PREC_BF16 = 1


class TanteConfig(C.Structure):
    """Mirror of `tante_config_t`."""
    _fields_ = [
        ("in_T", C.c_int32), ("n_fields", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("taylor_order", C.c_int32), ("n_head", C.c_int32), ("embed_dim", C.c_int32),
        ("patch_scale", C.c_int32), ("deg", C.c_int32), ("output_length", C.c_int32),
        ("frame_interval", C.c_float), ("precision", C.c_int32),
        ("n_layers", C.c_int32 * TANTE_MAX_ORDER),
        ("axes", (C.c_char * TANTE_MAX_LAYERS) * TANTE_MAX_ORDER),
        ("enc_dec_fno", C.c_int32), ("modes1", C.c_int32), ("modes2", C.c_int32),
        ("mlp_hidden", C.c_int32),
        ("expanded_channel", C.c_int32), ("mlp_hidden_c", C.c_int32),
        ("stride", C.c_int32 * 3),
    ]


class TanteError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libtante_b200 error {code}: {msg}")
        self.code = code
        self.msg = msg


# name -> (restype, argtypes); one entry per declaration in include/tante_b200.h
SIGNATURES = {
    "tante_last_error": (C.c_char_p, []),
    "tante_version": (C.c_int, []),
    "tante_create": (C.c_int, [C.POINTER(TanteConfig), C.c_int, C.POINTER(C.c_void_p)]),
    "tante_destroy": (C.c_int, [C.c_void_p]),
    "tante_reserve": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32]),
    "tante_workspace_bytes": (C.c_int64, [C.c_void_p]),
    "tante_param_count": (C.c_int32, [C.c_void_p]),
    "tante_param_name": (C.c_char_p, [C.c_void_p, C.c_int32]),
    "tante_param_numel": (C.c_int64, [C.c_void_p, C.c_int32]),
    "tante_bind_param": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "tante_pack_params": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tante_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_int32, C.c_int32,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]),
    "tante_rollout": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int32,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "tante_debug_stage": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.c_void_p]),
    "tante_launch_count": (C.c_int64, [C.c_void_p]),
    "tante_profile": (C.c_int, [C.c_void_p, C.c_int32]),
    "tante_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "tante_profile_read_class": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                           C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "tante_mse_cl": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int32,
                               C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tante_test_block_tail": (C.c_int, [C.c_void_p] * 12 + [C.c_int32, C.c_int32, C.c_void_p]),
    "tante_metric_moments": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "tante_test_gemm": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "tante_test_gemm_plan": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    "tante_comm_unique_id": (C.c_int, [C.c_void_p]),
    "tante_comm_init": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "tante_allreduce_grads": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tante_optimizer_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_float,
                                       C.c_float, C.c_float, C.c_int64, C.c_int32, C.c_float, C.c_float, C.c_void_p,
                                       C.c_void_p]),
    "tante_set_dropout": (C.c_int, [C.c_void_p, C.c_float, C.c_uint64]),
    "tante_grad_numel": (C.c_int64, [C.c_void_p]),
    "tante_param_grad_offset": (C.c_int64, [C.c_void_p, C.c_int32]),
    "tante_train_forward": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_float, C.c_int32,
                                      C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]),
    "tante_backward": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "tante_train_forward_hist": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32,
                                           C.c_float, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p]),
    "tante_backward_hist": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p]),
    "tante_test_wgrad": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                   C.c_int32, C.c_int32, C.c_void_p]),
    "tante_test_attention": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_uint64,
                                       C.c_uint32, C.POINTER(C.c_int32), C.c_void_p]),
    "tante_test_propagator": (C.c_int, [C.c_int32, C.c_int32] + [C.c_void_p] * 10 + [C.c_int32, C.c_int64, C.c_int64,
                                                                                    C.POINTER(C.c_int32), C.c_void_p]),
    "tante_bench_head": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                   C.POINTER(C.c_float), C.c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library (fails loudly; never falls back)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -m tante_b200.build` (nvcc, sm_100a). "
            "tante_b200 has no fallback path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code: int):
    if code != 0:
        raise TanteError(code, (load().tante_last_error() or b"").decode())
