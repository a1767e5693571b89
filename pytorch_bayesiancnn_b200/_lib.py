"""ctypes binding of libbbb_b200.so -- the C ABI declared in include/bbb_b200.h.

There is no CPU or PyTorch fallback: if the shared library is missing, or a call
returns an error code, this raises.  PyTorch is used by the callers only for
device memory, streams and autograd bookkeeping.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbbb_b200.so")

VARIANT_BBB, VARIANT_LRT = 0, 1
DTYPE_F32, DTYPE_BF16 = 0, 1
MATH_FP32, MATH_BF16_TC, MATH_AUTO, MATH_TF32_TC = 0, 1, 2, 3
KL_REFERENCE, KL_TEXTBOOK = 0, 1
ACT_NONE, ACT_SOFTPLUS, ACT_RELU = 0, 1, 2
LAYOUT_NCHW_F32, LAYOUT_PACKED_BF16, LAYOUT_ROWMAJOR_F32 = 0, 1, 2
FUSED_PREP_ONLY, FUSED_SKIP_PREP = 1, 2
E_UNSUPPORTED = -2              # BBB_E_UNSUPPORTED: a valid call whose shape / mode this path does not take

MATH_BY_NAME = {"fp32": MATH_FP32, "bf16": MATH_BF16_TC, "auto": MATH_AUTO, "tf32": MATH_TF32_TC}
KL_BY_NAME = {"reference": KL_REFERENCE, "textbook": KL_TEXTBOOK}
ACT_BY_NAME = {None: ACT_NONE, "none": ACT_NONE, "softplus": ACT_SOFTPLUS, "relu": ACT_RELU}

SYMBOLS = (
    "bbb_workspace_bytes", "bbb_conv2d_forward", "bbb_linear_forward", "bbb_layer_forward_fused", "bbb_fused_supported",
    "bbb_kl_forward",
    "bbb_kl_backward", "bbb_conv2d_backward", "bbb_linear_backward", "bbb_philox_normal_fill",
    "bbb_mc_combine", "bbb_noise_advance", "bbb_last_error", "bbb_abi_version", "bbb_launch_count",
    "bbb_mc_buffer_bytes", "bbb_mc_state_bytes", "bbb_mc_exchange",
    "bbb_comm_alloc", "bbb_comm_free", "bbb_comm_export", "bbb_comm_import", "bbb_comm_unimport", "bbb_set_wide_tiles",
)
MC_MOMENTS, MC_NORMALIZED = 1, 2


class LayerDesc(C.Structure):
    """struct bbb_layer_desc (include/bbb_b200.h)."""
    _fields_ = [(n, C.c_int32) for n in (
        "batch", "in_channels", "in_h", "in_w", "out_channels", "kernel_h", "kernel_w",
        "stride_h", "stride_w", "pad_h", "pad_w", "dil_h", "dil_w", "variant", "sample",
        "has_bias", "act_dtype", "math", "kl_convention", "epilogue_act", "pool_k", "pool_s")]
    _fields_ += [("reserved", C.c_int32 * 4), ("prior_mu", C.c_float), ("prior_sigma", C.c_float)]


class EngineError(RuntimeError):
    """``code``: the BBB_E_* status of the failed engine call (None for errors raised on the host side)."""

    def __init__(self, msg, code=None):
        super().__init__(msg)
        self.code = code


_lib = None
_lock = threading.Lock()


def _bind(lib):
    vp, fp, u64, i32, sz = C.c_void_p, C.c_void_p, C.c_uint64, C.c_int32, C.c_size_t
    dp = C.POINTER(LayerDesc)
    fwd = [dp, vp, fp, fp, fp, fp, vp, fp, fp, fp, fp, u64, u64, vp, vp, sz, vp]
    bwd = [dp, vp, vp, fp, fp, fp, fp, fp, fp, fp, u64, u64, vp, vp, fp, fp, fp, fp, vp, sz, vp]
    lib.bbb_workspace_bytes.argtypes = [dp]
    lib.bbb_workspace_bytes.restype = sz
    for name in ("bbb_conv2d_forward", "bbb_linear_forward"):
        getattr(lib, name).argtypes = fwd
        getattr(lib, name).restype = C.c_int
    for name in ("bbb_conv2d_backward", "bbb_linear_backward"):
        getattr(lib, name).argtypes = bwd
        getattr(lib, name).restype = C.c_int
    lib.bbb_layer_forward_fused.argtypes = [dp, vp, vp, i32, i32, i32, fp, fp, fp, fp, vp, vp, i32, i32, fp, fp, fp,
                                            u64, u64, vp, vp, sz, vp]
    lib.bbb_layer_forward_fused.restype = C.c_int
    lib.bbb_fused_supported.argtypes = [dp, i32, i32, i32, i32, i32]
    lib.bbb_fused_supported.restype = C.c_int
    lib.bbb_kl_forward.argtypes = [fp, fp, u64, fp, fp, u64, C.c_float, C.c_float, i32, fp, vp, sz, vp]
    lib.bbb_kl_forward.restype = C.c_int
    lib.bbb_kl_backward.argtypes = [fp, fp, u64, C.c_float, C.c_float, i32, fp, fp, fp, vp]
    lib.bbb_kl_backward.restype = C.c_int
    lib.bbb_philox_normal_fill.argtypes = [fp, u64, u64, u64, u64, vp]
    lib.bbb_philox_normal_fill.restype = C.c_int
    lib.bbb_mc_combine.argtypes = [fp, i32, i32, i32, fp, fp, vp]
    lib.bbb_mc_combine.restype = C.c_int
    lib.bbb_mc_buffer_bytes.argtypes = [i32, i32, i32, i32]
    lib.bbb_mc_buffer_bytes.restype = sz
    lib.bbb_mc_state_bytes.argtypes = []
    lib.bbb_mc_state_bytes.restype = sz
    lib.bbb_mc_exchange.argtypes = [fp, i32, i32, i32, i32, fp, i32, i32, vp, C.c_float, C.c_float, i32, i32,
                                    C.POINTER(C.c_void_p), vp, fp, fp, fp, fp, fp, fp, fp, vp, u64, vp]
    lib.bbb_mc_exchange.restype = C.c_int
    lib.bbb_comm_alloc.argtypes = [sz, C.POINTER(C.c_void_p)]
    lib.bbb_comm_export.argtypes = [vp, vp]
    lib.bbb_comm_import.argtypes = [vp, C.POINTER(C.c_void_p)]
    for name in ("bbb_comm_free", "bbb_comm_unimport"):
        getattr(lib, name).argtypes = [vp]
    for name in ("bbb_comm_alloc", "bbb_comm_free", "bbb_comm_export", "bbb_comm_import", "bbb_comm_unimport"):
        getattr(lib, name).restype = C.c_int
    lib.bbb_noise_advance.argtypes = [vp, u64, vp]
    lib.bbb_noise_advance.restype = C.c_int
    lib.bbb_last_error.argtypes = []
    lib.bbb_last_error.restype = C.c_char_p
    lib.bbb_abi_version.argtypes = []
    lib.bbb_abi_version.restype = i32
    lib.bbb_set_wide_tiles.argtypes = [C.c_int32]
    lib.bbb_set_wide_tiles.restype = C.c_int32
    lib.bbb_launch_count.argtypes = []
    lib.bbb_launch_count.restype = u64
    return lib


def lib():
    """The loaded library.  Raises EngineError (never falls back) if it is absent."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise EngineError(
                        f"{LIB_PATH} not found: the CUDA engine is not built. Run "
                        "`python -c 'import __graft_entry__ as g; g.build()'` at the repo root. "
                        "There is no CPU/PyTorch fallback for the Bayesian layer path.")
                _lib = _bind(C.CDLL(LIB_PATH))
                if _lib.bbb_abi_version() != 2:
                    raise EngineError("libbbb_b200.so ABI version mismatch")
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().bbb_last_error().decode("utf-8", "replace")
        raise EngineError(f"{what} failed (code {rc}): {msg}", rc)


def launch_count() -> int:
    return int(lib().bbb_launch_count())
