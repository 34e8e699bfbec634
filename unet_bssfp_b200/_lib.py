"""ctypes binding of ``libubssfp.so`` (C ABI declared in ``include/ub_api.h``).

The library is the product: there is no Python/CPU fallback. ``load()`` raises if the shared object
has not been built (``python -c 'import __graft_entry__ as g; g.build()'``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# UB_LIB_PATH: load another build of the same ABI (A/B timing of kernel changes); default = the in-tree build
LIB_PATH = os.environ.get("UB_LIB_PATH") or os.path.join(_HERE, "libubssfp.so")

UB_CONV_K3S1P1, UB_CONV_K1, UB_CONV_K4S2P1, UB_DECONV_K2S2, UB_CONV_K4S2P1_S2D = 0, 1, 2, 3, 4
UB_NORM_INSTANCE, UB_NORM_BATCH_TRAIN, UB_NORM_BATCH_EVAL, UB_NORM_NONE = 0, 1, 2, 3
UB_PACK_F16_SRC0 = 2


class NormBwdFuse(C.Structure):
    """Mirror of ``ub_norm_bwd_fuse`` (include/ub_api.h)."""
    _fields_ = [("y", C.c_void_p), ("scale", C.c_void_p), ("shift", C.c_void_p), ("mean", C.c_void_p),
                ("rstd", C.c_void_p), ("slope", C.c_float), ("drop_p", C.c_float), ("drop_seed", C.c_uint32),
                ("partial", C.c_void_p)]


class DeferredAct(C.Structure):
    """Mirror of ``ub_deferred_act`` (include/ub_api.h)."""
    _fields_ = [("scale", C.c_void_p), ("shift", C.c_void_p), ("slope", C.c_float), ("drop_p", C.c_float),
                ("drop_seed", C.c_uint32), ("f16_operand", C.c_int)]


class AdamWTensor(C.Structure):
    """Mirror of ``ub_adamw_tensor`` (include/ub_api.h)."""
    _fields_ = [("p", C.c_void_p), ("g", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p), ("numel", C.c_longlong)]


class F32ConvDesc(C.Structure):
    """Mirror of ``ub_f32_conv_desc`` (include/ub_api.h)."""
    _fields_ = [(k, C.c_int) for k in ("n", "c0", "c1", "co", "d", "h", "w", "k", "stride", "pad")]


class ConvDesc(C.Structure):
    """Mirror of ``ub_conv_desc`` (include/ub_api.h)."""
    _fields_ = [(k, C.c_int) for k in ("kind", "n", "d", "h", "w", "c0", "c0p", "c1", "c1p", "co", "cop")]


class WeightPackItem(C.Structure):
    """Mirror of ``ub_weight_pack_item`` (include/ub_api.h)."""
    _fields_ = [("desc", ConvDesc), ("dir", C.c_int), ("w", C.c_void_p), ("packed", C.c_void_p)]


_P = C.c_void_p
_F = C.c_float
_I = C.c_int
_LL = C.c_longlong
_U32 = C.c_uint32
_D = C.c_double
_DP = C.POINTER(ConvDesc)
_AP = C.POINTER(DeferredAct)

# name -> (restype, argtypes); every symbol of include/ub_api.h
SIGNATURES = {
    "ub_version": (_I, []),
    "ub_last_error": (C.c_char_p, []),
    "ub_launch_count": (_LL, []),
    "ub_packed_weight_elems": (_LL, [_DP, _I]),
    "ub_pack_conv_weights": (_I, [_DP, _I, _P, _P, _P]),
    "ub_pack_conv_weights_multi": (_I, [C.POINTER(WeightPackItem), _I, _P]),
    "ub_conv_num_tiles": (_I, [_DP]),
    "ub_conv_deferred_src0_ok": (_I, [_DP]),
    "ub_conv_fwd": (_I, [_DP, _P, _P, _P, _P, _I, _F, _P, _P, _AP, _I, _P]),
    "ub_conv_dgrad": (_I, [_DP, _P, _P, _P, _P, _P]),
    "ub_conv_dgrad_fuse_records": (_I, [_DP]),
    "ub_conv_dgrad_fused": (_I, [_DP, _P, _P, _P, _P, C.POINTER(NormBwdFuse), _P]),
    "ub_conv_kernel_class": (_I, [_DP, _I]),
    "ub_conv_wgrad_workspace_bytes": (_LL, [_DP]),
    "ub_conv_wgrad": (_I, [_DP, _P, _P, _P, _P, _P, _AP, _P]),
    "ub_pack_ncdhw": (_I, [_P, _I, _I, _P, _I, _I, _LL, _I, _P, _P]),
    "ub_pack_ncdhw_s2d": (_I, [_P, _I, _I, _P, _I, _I, _I, _I, _I, _I, _P, _P]),
    "ub_pack_patches": (_I, [_P, _I, _I, C.POINTER(C.c_longlong), _I, _I, _I, _LL, _LL, _LL, _I, _P, _P]),
    "ub_unpack_patch": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _P, _LL, _LL, _LL, _LL, _P]),
    "ub_paste_patch": (_I, [_P, _I, _I, _I, _I, _P, _LL, _LL, _LL, _LL, _P]),
    "ub_blend_patches": (_I, [_P, _I, _I, _I, _I, _I, C.POINTER(C.c_int), C.POINTER(C.c_int), _I, _P, _P, _P, _I, _I,
                              _I, _P]),
    "ub_blend_finish": (_I, [_P, _P, _I, _LL, _P]),
    "ub_unpack_ncdhw": (_I, [_P, _I, _I, _I, _I, _LL, _P, _P]),
    "ub_conv1x1_workspace_bytes": (_LL, []),
    "ub_conv1x1_to_ncdhw": (_I, [_P, _I, _P, _I, _P, _I, _I, _LL, _P, _P, _AP, _P]),
    "ub_conv1x1_from_ncdhw_bwd": (_I, [_P, _I, _P, _I, _P, _I, _I, _LL, _P, _P, _P, _P, _AP, _P]),
    "ub_norm_finalize": (_I, [_P, _I, _I, _I, _I, _D, _P, _P, _F, _I, _F, _P, _P, _P, _P, _P, _P, _P]),
    "ub_bn_running_update": (_I, [_P, _P, _I, _D, _F, _F, _P, _P, _P]),
    "ub_norm_act_fwd": (_I, [_P, _P, _P, _F, _F, _U32, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "ub_norm_act_bwd_workspace_bytes": (_LL, [_I, _I]),
    "ub_norm_act_bwd": (_I, [_P, _P, _P, _I, _P, _P, _P, _P, _F, _F, _U32, _I, _LL, _I, _I, _P, _P, _P, _P, _P, _P, _I,
                             _P]),
    "ub_maxpool_bwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _AP, _P]),
    "ub_head_bwd_fused_workspace_bytes": (_LL, [_I]),
    "ub_head_bwd_fused": (_I, [_P, _I, _P, _I, _I, _LL, C.POINTER(NormBwdFuse), _I, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ub_to_s2d": (_I, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "ub_maxpool_bwd_fuse_records": (_I, [_I, _I, _I, _I, _I]),
    "ub_maxpool_bwd_fused": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, C.POINTER(NormBwdFuse), _P]),
    "ub_colsum_workspace_bytes": (_LL, [_I]),
    "ub_colsum": (_I, [_P, _LL, _I, _I, _P, _P, _P]),
    "ub_l1_workspace_bytes": (_LL, []),
    "ub_l1_fwd": (_I, [_P, _P, _LL, _P, _P, _P]),
    "ub_l1_bwd": (_I, [_P, _P, _P, _LL, _P, _P]),
    "ub_bce_logits": (_I, [_P, _P, _F, _I, _P, _P, _P]),
    "ub_scale": (_I, [_P, _P, _LL, _P, _P]),
    "ub_dti_scalar_maps": (_I, [_P, _LL, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ub_relerr_map_reduce": (_I, [_P, _P, _P, _P, _I, _I, _LL, _I, _P, _P, _P, _P]),
    "ub_adamw_step": (_I, [C.POINTER(AdamWTensor), _I, _D, _D, _D, _D, _D, _LL, _F, _P]),
    "ub_denorm_to_nifti": (_I, [_P, _I, _I, _I, _I, _D, _D, _P, _P]),
    "ub_f32_conv_fwd": (_I, [C.POINTER(F32ConvDesc), _P, _P, _P, _P, _P, _P]),
    "ub_f32_conv_dgrad": (_I, [C.POINTER(F32ConvDesc), _P, _P, _P, _P, _P]),
    "ub_f32_conv_wgrad": (_I, [C.POINTER(F32ConvDesc), _P, _P, _P, _P, _P, _P]),
    "ub_f32_deconv2_fwd": (_I, [_I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "ub_f32_deconv2_dgrad": (_I, [_I, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "ub_f32_deconv2_wgrad": (_I, [_I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "ub_f32_norm_stats": (_I, [_P, _I, _I, _LL, _I, _P, _P, _F, _F, _P, _P, _P, _P, _P, _P, _P]),
    "ub_f32_norm_act_fwd": (_I, [_P, _P, _P, _F, _F, _U32, _I, _I, _I, _I, _I, _P, _P, _P]),
    "ub_f32_norm_act_bwd": (_I, [_P, _P, _P, _P, _I, _P, _P, _P, _P, _F, _F, _U32, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
}

_lib = None


def load():
    """Load the shared library and bind every entry point; raise loudly when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built and there is no fallback. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'` at the repo root.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().ub_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libubssfp {what} failed (rc={rc}): {msg}")
