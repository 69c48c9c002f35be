"""ctypes binding of libavc_b200.so (the C ABI declared in include/avc_b200.h).

There is no CPU fallback: if the shared library is missing and cannot be built, importing
a symbol raises.  ``AVC_LIB`` can point at an explicit .so.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# engine.py: fused speaker dense stack / batched AdaIN affine layers (csrc/dense_fused.cu); ON since
# the B200 validation run (42 513 -> 45 462 seg/s); AVC_FUSED_DENSE=0 = one launch per nn.Linear
DEFAULT_FUSED_DENSE = True
# engine.py: conv weight gradients accumulated in place with vector atomics + ONE flush launch per
# backward pass (csrc/wgrad_tc.cu, ATOMIC).  ON since the round-2 B200 validation (tests green, 45 649 ->
# 49 658 seg/s); AVC_WGRAD_ACC=0 = per-slice partials + deterministic reduction
DEFAULT_WGRAD_ACC = True
# engine.py: reflect-padding / residual adjoint inside the data-gradient conv's epilogue (AVC_F_FOLD, 30
# avc_fold_add_fwd launches fewer per step).  ON since the round-2 validation (tests green, +0.5 %)
DEFAULT_FOLD_FUSED = True
# engine.py: the data-gradient conv of a block also runs the UPSTREAM block's InstanceNorm / AdaIN / ReLU backward in
# its epilogue (AVC_F_NORMBWD, persistent kernel): 27 avc_norm_bwd launches and their dy/dc round trips fewer per step.
# Validated on the B200 (tests/test_gpu_normbwd_fused.py, all model tests green) but SLOWER (47 853 vs 49 697 seg/s):
# the conv kernel is bound by its 8 epilogue warps, the stand-alone avc_norm_bwd runs at full occupancy -> opt-in
DEFAULT_NORM_BWD_FUSED = False
LIB_PATH = os.environ.get("AVC_LIB", os.path.join(_PKG, "libavc_b200.so"))

PAD_REFLECT, PAD_ZERO = 0, 1
RES_NONE, RES_SAME, RES_POOL, RES_UP = 0, 1, 2, 3
PACK_FWD, PACK_DGRAD = 0, 1
F_ROUND_OUT, F_IN_TF32, F_FOLD, F_NORMBWD = 1, 2, 4, 8
OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA = 0, -1, -2, -3

_fp = C.c_void_p  # device pointers travel as integers


class ConvDesc(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32), ("K", C.c_int32),
        ("stride", C.c_int32), ("pad_left", C.c_int32), ("pad_mode", C.c_int32), ("in_ups", C.c_int32),
        ("Tin", C.c_int32), ("Tout", C.c_int32),
        ("in_", _fp), ("in_bstride", C.c_int64),
        ("w_packed", _fp), ("w_ld", C.c_int32),
        ("bias", _fp),
        ("out", _fp), ("out_bstride", C.c_int64),
        ("shuffle", C.c_int32), ("norm", C.c_int32), ("eps", C.c_float), ("relu", C.c_int32),
        ("cond", _fp), ("cond_bstride", C.c_int64),
        ("res", _fp), ("res_bstride", C.c_int64), ("res_mode", C.c_int32), ("res_T", C.c_int32),
        ("mask", _fp), ("mask_bstride", C.c_int64),
        ("save_c", _fp), ("stats", _fp),
        ("dy", _fp), ("dy_bstride", C.c_int64),
        ("dc", _fp), ("dcond", _fp), ("dcond_bstride", C.c_int64), ("dbias", _fp),
        ("w_tc", _fp), ("flags", C.c_int32), ("out_tstride", C.c_int32), ("out_toff", C.c_int32), ("out_T", C.c_int32),
    ]


class WgradDesc(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32), ("K", C.c_int32),
        ("stride", C.c_int32), ("pad_left", C.c_int32), ("Tin", C.c_int32), ("Tout", C.c_int32),
        ("x", _fp), ("x_bstride", C.c_int64),
        ("dc", _fp), ("dc_bstride", C.c_int64),
        ("dw", _fp),
    ]


class FoldDesc(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("C", C.c_int32), ("Tin", C.c_int32), ("pad_left", C.c_int32), ("pad_right", C.c_int32),
        ("dxp", _fp), ("dres", _fp), ("dres_bstride", C.c_int64),
        ("res_mode", C.c_int32), ("res_T", C.c_int32),
        ("dx", _fp), ("dx_bstride", C.c_int64),
    ]


class PackItem(C.Structure):
    _fields_ = [("w", _fp), ("simt_fwd", _fp), ("simt_dgrad", _fp), ("tc_fwd", _fp), ("tc_dgrad", _fp),
                ("tc_dgrad_even", _fp), ("tc_dgrad_odd", _fp),
                ("Cout", C.c_int32), ("Cin", C.c_int32), ("K", C.c_int32), ("reserved", C.c_int32)]


class LinearDesc(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("relu", C.c_int32),
        ("x", _fp), ("x_bstride", C.c_int64),
        ("w", _fp), ("bias", _fp), ("res", _fp), ("y_act", _fp),
        ("out", _fp), ("out_bstride", C.c_int64),
        ("dy", _fp), ("dy_bstride", C.c_int64),
        ("dx_add", _fp), ("dx", _fp), ("dw", _fp), ("db", _fp),
    ]


class WgradAccItem(C.Structure):
    _fields_ = [("acc", _fp), ("dw", _fp), ("Cout", C.c_int32), ("Cin", C.c_int32), ("K", C.c_int32), ("reserved", C.c_int32)]


class DenseStackDesc(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("C", C.c_int32), ("c_out", C.c_int32), ("n_blocks", C.c_int32),
        ("params", _fp), ("x", _fp), ("save", _fp), ("out", _fp), ("dout", _fp), ("gsave", _fp), ("dx", _fp),
    ]


class SnItem(C.Structure):
    _fields_ = [("w_orig", _fp), ("w_sn", _fp), ("u", _fp), ("v", _fp), ("sigma", _fp), ("grad", _fp),
                ("rows", C.c_int32), ("cols", C.c_int32)]


LINEAR_BATCH_MAX = 16


class LinearBatchDesc(C.Structure):
    _fields_ = [
        ("L", C.c_int32), ("B", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
        ("params", _fp), ("grads", _fp),
        ("x", _fp), ("x_off", C.c_int64 * LINEAR_BATCH_MAX), ("x_bstride", C.c_int64),
        ("y", _fp), ("out", _fp), ("y_off", C.c_int64 * LINEAR_BATCH_MAX), ("y_bstride", C.c_int64),
        ("part", _fp), ("dx_add", _fp), ("dx", _fp),
    ]


# name -> (restype, argtypes); the single source of truth for tests/test_cabi_symbols.py
_i, _i64, _p = C.c_int, C.c_int64, C.c_void_p
PROTOTYPES = {
    "avc_conv_block_fwd": (_i, [C.POINTER(ConvDesc), _p]),
    "avc_conv_block_tc": (_i, [C.POINTER(ConvDesc), _p, _p]),
    "avc_pack_conv_weight_tc": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "avc_tc_packed_floats": (_i64, [_i, _i, _i]),
    "avc_tc_set_debug": (None, [_p]),
    "avc_tc2_set_debug": (None, [_p]),
    "avc_tc2_set_variant": (None, [_i]),
    "avc_wgrad_tc_set_debug": (None, [_p]),
    "avc_set_option": (_i, [C.c_char_p, _i]),
    "avc_get_option": (_i, [C.c_char_p]),
    "avc_pack_conv_weights_batch": (_i, [_p, _i, _i64, _p]),
    "avc_norm_apply_fwd": (_i, [C.POINTER(ConvDesc), _p]),
    "avc_norm_bwd": (_i, [C.POINTER(ConvDesc), _p]),
    "avc_conv_wgrad": (_i, [C.POINTER(WgradDesc), _p]),
    "avc_wgrad_tc_scratch_floats": (_i64, [C.POINTER(WgradDesc)]),
    "avc_conv_wgrad_tc": (_i, [C.POINTER(WgradDesc), _p, _p, _p]),
    "avc_wgrad_acc_floats": (_i64, [_i, _i, _i]),
    "avc_conv_wgrad_tc_acc": (_i, [C.POINTER(WgradDesc), _p, _p, _p]),
    "avc_wgrad_acc_flush": (_i, [_p, _i, _i64, _p]),
    "avc_fold_add_fwd": (_i, [C.POINTER(FoldDesc), _p]),
    "avc_pack_conv_weight": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "avc_pack_a4": (_i, [_p, _p, _i64, _i, _i, _i, _i, _p]),
    "avc_unpack_a4": (_i, [_p, _i64, _p, _i, _i, _i, _p]),
    "avc_bias_grad": (_i, [_p, _i64, _p, _i, _i, _i, _p]),
    "avc_bias_grad_groups": (_i, [_p, _i64, _p, _i, _i, _i, _i, _p]),
    "avc_time_mean_fwd": (_i, [_p, _i64, _p, _i, _i, _i, _p]),
    "avc_time_mean_bwd": (_i, [_p, _p, _i64, _i, _i, _i, _p]),
    "avc_linear_fwd": (_i, [C.POINTER(LinearDesc), _p]),
    "avc_linear_bwd": (_i, [C.POINTER(LinearDesc), _p]),
    "avc_dense_stack_fwd": (_i, [C.POINTER(DenseStackDesc), _p]),
    "avc_dense_stack_bwd": (_i, [C.POINTER(DenseStackDesc), _p]),
    "avc_linear_batch_fwd": (_i, [C.POINTER(LinearBatchDesc), _p]),
    "avc_linear_batch_dx": (_i, [C.POINTER(LinearBatchDesc), _p]),
    "avc_linear_batch_dw": (_i, [C.POINTER(LinearBatchDesc), _p]),
    "avc_reparam_fwd": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "avc_reparam_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "avc_vae_loss": (_i, [_p, _p, _i64, _p, _p, _i64, _p, _p, _p, _p, _p, _p]),
    "avc_sqnorm": (_i, [_p, _i64, _p, _p, _p]),
    "avc_adam_step": (_i, [_p, _p, _p, _p, _p, _i64, _p, _p, _p, _p]),
    "avc_fill_zero": (_i, [_p, _i64, _p]),
    "avc_spectral_norm_fwd": (_i, [_p, _i, _i, _p]),
    "avc_spectral_norm_bwd": (_i, [_p, _i, _p]),
    "avc_tc_probe_gemm": (_i, [_p, _i, _p, _i, C.POINTER(C.c_uint32), _i, _i, _i, _i, _i, _p, _p, _p]),
    "avc_tc_probe_set_ld_shift": (None, [_i]),
    "avc_probe_store": (_i, [_p, C.c_longlong, _i, _i, _p, _p]),
    "avc_last_error": (C.c_char_p, []),
    "avc_build_info": (C.c_char_p, []),
    "avc_launch_count": (_i64, []),
}

_lib = None


class AvcError(RuntimeError):
    pass


def load(build_if_missing: bool = True):
    """Load (building first if necessary) the shared library; raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if "AVC_LIB" not in os.environ:
        # stamp-checked: a no-op when libavc_b200.so matches the sources, a rebuild when a
        # .cu/.cuh/.h changed, an error when it is stale and nvcc is unavailable
        from . import build as _build
        if build_if_missing or os.path.exists(LIB_PATH):
            _build.build(allow_build=build_if_missing)
    if not os.path.exists(LIB_PATH):
        raise AvcError(f"{LIB_PATH} is missing (run `python -m adaptive_voice_conversion_b200.build`); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().avc_last_error().decode()


def check(rc: int, what: str = ""):
    if rc != OK:
        raise AvcError(f"{what}: rc={rc}: {last_error()}")


def launch_count() -> int:
    return int(load().avc_launch_count())


def set_option(name: str, value: bool):
    """Process-wide runtime option of the library (include/avc_b200.h: avc_set_option)."""
    check(load().avc_set_option(name.encode(), int(bool(value))), f"set_option[{name}]")


def get_option(name: str) -> int:
    return int(load().avc_get_option(name.encode()))
