"""ctypes binding of libgdl_b200.so (the C-ABI declared in include/gdl_b200.h).

The product path has NO fallback: if the shared library is missing, or a call returns a
negative status, a GdlError is raised.  Nothing here imports the oracle.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgdl_b200.so")

GDL_OK, GDL_EINVAL, GDL_EARCH, GDL_ECUDA, GDL_ENOMEM = 0, -1, -2, -3, -4


class GdlError(RuntimeError):
    pass


class PackEntry(C.Structure):  # mirrors gdl_pack_entry
    _fields_ = [("w", C.c_void_p), ("wp", C.c_void_p), ("wT", C.c_void_p), ("Co", C.c_int32), ("Ci", C.c_int32),
                ("ci_real", C.c_int32), ("R", C.c_int32), ("S", C.c_int32), ("Kp", C.c_int32), ("start", C.c_int64),
                ("scale", C.c_void_p)]


class ConvDesc(C.Structure):
    """Mirror of gdl_conv_desc."""
    _fields_ = [(n, C.c_int32) for n in
                ("N", "Hi", "Wi", "Ci", "Ho", "Wo", "Co", "R", "S", "stride", "pad")]


_p = C.c_void_p
_i = C.c_int
_l = C.c_int64
_f = C.c_float
_d = C.c_double
_dp = C.POINTER(ConvDesc)

# name -> (restype, argtypes); every symbol of include/gdl_b200.h
SIGNATURES = {
    "gdl_version": (_i, []),
    "gdl_last_error_string": (C.c_char_p, []),
    "gdl_init": (_i, [_i]),
    "gdl_conv_packed_k": (_l, [_dp]),
    "gdl_conv_wgrad_workspace_bytes": (_l, [_dp]),
    "gdl_conv_pack_weights": (_i, [_dp, _i, _p, _p, _p, _p]),
    "gdl_conv_fwd": (_i, [_dp, _p, _p, _p, _p]),
    "gdl_conv_fwd_bias_act": (_i, [_dp, _p, _p, _p, _p, _i, _p, _p]),
    "gdl_stem_pack_weights_scaled": (_i, [_p, _p, _p, _i, _p]),
    "gdl_conv_dgrad": (_i, [_dp, _p, _p, _p, _p, _i, _p]),
    "gdl_conv_wgrad": (_i, [_dp, _i, _p, _p, _p, _p, _l, _p]),
    "gdl_stem_geometry": (_i, [_i, _i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "gdl_stem_layout": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "gdl_stem_pack_weights": (_i, [_p, _p, _i, _p]),
    "gdl_stem_fwd": (_i, [_p, _p, _p, _i, _i, _i, _p]),
    "gdl_stem_fwd_stats": (_i, [_p, _p, _p, _i, _i, _i, _p, _p, _p]),
    "gdl_stem_wgrad_workspace_bytes": (_l, [_i, _i, _i]),
    "gdl_stem_wgrad": (_i, [_p, _p, _p, _i, _i, _i, _i, _p, _l, _p]),
    "gdl_layout_ncthw_to_nhwc8": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "gdl_bn_partial_floats": (_l, [_l, _i]),
    "gdl_bn_stats": (_i, [_p, _l, _i, _p, _p, _p, _f, _f, _p, _p, _p, _p, _p, _p, _p]),
    "gdl_conv_pack_weights_multi": (_i, [_p, _i, _l, _p]),
    "gdl_conv_pack_weights_tiled": (_i, [_p, _i, _i, _i, _p]),
    "gdl_set_fused_stats_min_k": (_i, [_i]),
    "gdl_set_sweep": (_i, [_i]),
    "gdl_conv_fwd_stats": (_i, [_p, _p, _p, _p, _p, _p, _p]),
    "gdl_bn_stats_finalize": (_i, [_p, _i, _l, _i, _p, _p, _f, _f, _p, _p, _p, _p, _p, _p, _p]),
    "gdl_bn_eval_affine": (_i, [_p, _p, _p, _p, _f, _p, _p, _i, _p]),
    "gdl_bn_apply": (_i, [_p, _p, _p, _l, _i, _p, _p, _i, _p]),
    "gdl_bn_bwd": (_i, [_p, _p, _p, _p, _p, _l, _i, _p, _p, _p, _p, _p, _p, _i, _p]),
    "gdl_bn_bwd_nores": (_i, [_p, _p, _p, _l, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "gdl_bn_relu_maxpool_fwd": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p]),
    "gdl_bn_relu_maxpool_bwd": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "gdl_gemm_nt_bf16": (_i, [_p, _l, _p, _p, _l, _i, _i, _p]),
    "gdl_gemm_tn_workspace_bytes": (_l, [_i, _i, _l]),
    "gdl_gemm_tn_f32": (_i, [_p, _p, _p, _p, _i, _i, _l, _p, _l, _p]),
    "gdl_gemm_tn_f32_acc": (_i, [_p, _p, _p, _i, _i, _l, _p, _l, _p]),
    "gdl_film_scratch_floats": (_l, [_i, _i]),
    "gdl_film_outer": (_i, [_p, _p, _p, _i, _i, _i, _i, _p, _p]),
    "gdl_film_outer_chunk": (_i, [_p, _p, _p, _i, _i, _i, _i, _p, _l, _l, _p]),
    "gdl_cast_pad_bf16": (_i, [_p, _i, _p, _i, _i, _i, _i, _p, _i, _i, _p]),
    "gdl_film_contract": (_i, [_p, _i, _i, _p, _p, _p, _p, _i, _i, _i, _p, _p]),
    "gdl_film_contract_chunk": (_i, [_p, _i, _i, _p, _p, _p, _p, _i, _i, _i, _p, _i, _i, _i, _i, _p]),
    "gdl_transpose_f32_to_bf16": (_i, [_p, _p, _i, _l, _p]),
    "gdl_transpose_bf16_to_f32": (_i, [_p, _p, _i, _l, _p]),
    "gdl_transpose_bf16_to_f32_window": (_i, [_p, _p, _i, _l, _l, _l, _p]),
    "gdl_maxpool_fwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _p]),
    "gdl_maxpool_bwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _p]),
    "gdl_gap_fwd": (_i, [_p, _p, _i, _i, _i, _p]),
    "gdl_gap_bwd": (_i, [_p, _p, _i, _i, _i, _p]),
    "gdl_linear_fwd": (_i, [_p, _p, _i, _p, _p, _i, _i, _i, _p]),
    "gdl_linear_bwd": (_i, [_p, _p, _p, _i, _p, _p, _i, _p, _i, _i, _i, _i, _p]),
    "gdl_head_scratch_floats": (_l, [_i, _i]),
    "gdl_dgl_head_linear": (_i, [_i, _p, _p, _p, _p, _i, _p, _p, _p, _f, _f, _p, _p, _p, _p, _p,
                                 _p, _i, _p, _p, _p, _i, _i, _i, _p]),
    "gdl_gated_head_scratch_floats": (_l, [_i, _i]),
    "gdl_dgl_head_gated": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _f, _f, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "gdl_softmax_ce": (_i, [_p, _p, _f, _f, _p, _p, _p, _i, _i, _p]),
    "gdl_eval_head": (_i, [_i, _p, _i, _p, _i, _p, _p, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _i, _i, _p]),
    "gdl_eval_count": (_i, [_p, _p, _p, _i, _i, _p]),
    "gdl_gated_fwd": (_i, [_p, _p, _p, _p, _p, _l, _p]),
    "gdl_gated_bwd": (_i, [_p, _p, _p, _p, _p, _p, _l, _p]),
    "gdl_optim_scratch_floats": (_l, [_l, _i]),
    "gdl_grad_stats": (_i, [_p, _l, _p, _p, _p, _i, _f, _p, _p, _p]),
    "gdl_sgd_momentum": (_i, [_p, _p, _p, _l, _f, _f, _f, _i, _p, _p]),
    "gdl_adam": (_i, [_p, _p, _p, _p, _p, _l, _d, _d, _d, _d, _d, _p, _p]),
    "gdl_adagrad": (_i, [_p, _p, _p, _p, _l, _d, _d, _d, _d, _p, _p]),
    "gdl_grad_accumulate": (_i, [_p, _p, _l, _i, _p]),
    "gdl_check_conv_fwd": (_i, [_dp, _i, _p, _p, _p, _p]),
    "gdl_check_conv_dgrad": (_i, [_dp, _i, _p, _p, _p, _p, _p]),
    "gdl_check_conv_wgrad": (_i, [_dp, _i, _p, _p, _p, _p]),
    "gdl_check_bn_fwd": (_i, [_p, _p, _p, _i, _i, _i, _p, _p, _f, _f, _p, _p, _p, _p, _i, _i, _p]),
    "gdl_check_bn_bwd": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _p, _p, _p, _p, _p, _i, _p]),
    "gdl_check_maxpool_fwd": (_i, [_p, _p, _p, _l, _i, _i, _i, _i, _p]),
    "gdl_check_maxpool_bwd": (_i, [_p, _p, _p, _l, _i, _i, _i, _i, _p]),
    "gdl_check_gap_fwd": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "gdl_check_gap_bwd": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "gdl_check_fold_frames": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "gdl_log_stft": (_i, [_p, _l, _p, _p, _i, _i, _i, _i, _i, _p, _p]),
    "gdl_crop_table_ints": (_l, [_i, _i]),
    "gdl_crop_resize_normalize": (_i, [_p, _l, _i, _i, _p, _i, _i, _i, _p, _p, _p, _p, _p]),
}

_lib = None


def load():
    """dlopen the extension once; raise loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GdlError(
            "libgdl_b200.so not found at %s — build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` or `make -C iccv2025-gdl_b200/csrc`. There is no CPU/PyTorch fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, what):
    if status != GDL_OK:
        msg = load().gdl_last_error_string()
        raise GdlError("%s failed with status %d: %s" % (what, status, (msg or b"").decode()))
