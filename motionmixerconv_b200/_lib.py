"""ctypes binding of libmmx.so (the C ABI declared in include/mmx.h).

There is exactly one implementation behind these entry points: the sm_100a CUDA kernels in
``csrc/``.  If the shared library is missing or cannot be loaded this module raises — there is
no CPU or PyTorch fallback anywhere in the product package.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmmx.so")

MMX_ACT = {"gelu": 0, "mish": 1}
MMX_PREC = {"fp32": 0, "tf32": 1}

c_float_p = C.POINTER(C.c_float)


class MmxDropout(C.Structure):
    _fields_ = [("p", C.c_float), ("seed", C.c_ulonglong), ("step", C.c_uint), ("step_dev", C.c_void_p)]


class MmxMlpBlockParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "ln1_w", "ln1_b", "tok_w1", "tok_b1", "tok_w2", "tok_b2", "ln2_w", "ln2_b",
        "ch_w1", "ch_b1", "ch_w2", "ch_b2", "se_w1", "se_w2")]


class MmxMlpBlockDesc(C.Structure):
    _fields_ = [("B", C.c_int), ("T", C.c_int), ("H", C.c_int), ("tok", C.c_int), ("ch", C.c_int),
                ("se_hidden", C.c_int), ("act", C.c_int), ("use_se", C.c_int), ("use_max_pooling", C.c_int),
                ("training", C.c_int), ("block_index", C.c_int), ("dropout", MmxDropout), ("precision", C.c_int)]


class MmxMlpHeadParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("ln_w", "ln_b", "wt", "bt", "wf", "bf")]


class MmxMlpHeadDesc(C.Structure):
    _fields_ = [("B", C.c_int), ("T", C.c_int), ("To", C.c_int), ("H", C.c_int), ("D", C.c_int)]


class MmxConvHalfParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("ln_w", "ln_b", "conv_w", "conv_b", "se_w1", "se_w2", "bn_aff")]


class MmxConvHalfDesc(C.Structure):
    _fields_ = [("B", C.c_int), ("C", C.c_int), ("T", C.c_int), ("E", C.c_int),
                ("kt", C.c_int), ("kp", C.c_int), ("pad_t", C.c_int), ("pad_p", C.c_int),
                ("se_hidden", C.c_int), ("act", C.c_int), ("use_se", C.c_int), ("use_max_pooling", C.c_int),
                ("training", C.c_int), ("site", C.c_int), ("dropout", MmxDropout)]


class MmxEncoderParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("freq", "w", "b", "wc", "bc")]


class MmxEncoderDesc(C.Structure):
    _fields_ = [("B", C.c_int), ("T", C.c_int), ("D", C.c_int), ("E", C.c_int), ("C", C.c_int), ("n_harmonic", C.c_int)]


class MmxConvHeadParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("ln_w", "ln_b", "wt", "bt", "wp", "bp", "wf", "bf")]


class MmxConvHeadDesc(C.Structure):
    _fields_ = [("B", C.c_int), ("C", C.c_int), ("T", C.c_int), ("To", C.c_int), ("E", C.c_int), ("D", C.c_int)]


# name -> (restype, argtypes).  Everything declared in include/mmx.h must appear here
# (tests/test_abi.py checks the two lists against each other and against the built library).
SIGNATURES = {
    "mmx_version": (C.c_int, []),
    "mmx_last_error": (C.c_char_p, []),
    "mmx_mlp_block_fwd": (C.c_int, [C.POINTER(MmxMlpBlockDesc), C.POINTER(MmxMlpBlockParams), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_mlp_block_bwd": (C.c_int, [C.POINTER(MmxMlpBlockDesc), C.POINTER(MmxMlpBlockParams), C.POINTER(MmxMlpBlockParams),
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_tc5_abort_count": (C.c_int, []),
    "mmx_mlp_token_half_fwd": (C.c_int, [C.POINTER(MmxMlpBlockDesc), C.POINTER(MmxMlpBlockParams)] + [C.c_void_p] * 4),
    "mmx_mlp_token_half_bwd": (C.c_int, [C.POINTER(MmxMlpBlockDesc), C.POINTER(MmxMlpBlockParams), C.POINTER(MmxMlpBlockParams)] + [C.c_void_p] * 6),
    "mmx_mlp_channel_half_fwd": (C.c_int, [C.POINTER(MmxMlpBlockDesc), C.POINTER(MmxMlpBlockParams)] + [C.c_void_p] * 3),
    "mmx_mlp_channel_half_bwd": (C.c_int, [C.POINTER(MmxMlpBlockDesc), C.POINTER(MmxMlpBlockParams), C.POINTER(MmxMlpBlockParams)] + [C.c_void_p] * 4),
    "mmx_tc5_dropout_mask": (C.c_int, [C.POINTER(MmxDropout), C.c_uint, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]),
    "mmx_mlp_block_saves": (C.c_int, [C.POINTER(MmxMlpBlockDesc)]),
    "mmx_mlp_block_fwd_save": (C.c_int, [C.POINTER(MmxMlpBlockDesc), C.POINTER(MmxMlpBlockParams)] + [C.c_void_p] * 5),
    "mmx_mlp_block_bwd_saved": (C.c_int, [C.POINTER(MmxMlpBlockDesc), C.POINTER(MmxMlpBlockParams), C.POINTER(MmxMlpBlockParams)] + [C.c_void_p] * 6),
    "mmx_linear_fwd": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_linear_bwd": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "mmx_linear_fwd_prec": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "mmx_linear_bwd_prec": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int, C.c_void_p]),
    "mmx_mlp_head_fwd_prec": (C.c_int, [C.POINTER(MmxMlpHeadDesc), C.POINTER(MmxMlpHeadParams), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "mmx_mlp_head_bwd_prec": (C.c_int, [C.POINTER(MmxMlpHeadDesc), C.POINTER(MmxMlpHeadParams), C.POINTER(MmxMlpHeadParams),
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "mmx_mlp_head_fwd": (C.c_int, [C.POINTER(MmxMlpHeadDesc), C.POINTER(MmxMlpHeadParams), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_mlp_head_bwd": (C.c_int, [C.POINTER(MmxMlpHeadDesc), C.POINTER(MmxMlpHeadParams), C.POINTER(MmxMlpHeadParams),
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_conv_half_fwd": (C.c_int, [C.POINTER(MmxConvHalfDesc), C.POINTER(MmxConvHalfParams), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_conv_half_bwd": (C.c_int, [C.POINTER(MmxConvHalfDesc), C.POINTER(MmxConvHalfParams), C.POINTER(MmxConvHalfParams),
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_conv_half_plan": (C.c_int, [C.POINTER(MmxConvHalfDesc), C.c_int, C.c_void_p, C.c_void_p]),
    "mmx_conv2d_large_fwd": (C.c_int, [C.POINTER(MmxConvHalfDesc), C.c_int] + [C.c_void_p] * 5),
    "mmx_conv2d_large_wgrad": (C.c_int, [C.POINTER(MmxConvHalfDesc)] + [C.c_void_p] * 5),
    "mmx_conv2d_large_fwd_prec": (C.c_int, [C.POINTER(MmxConvHalfDesc), C.c_int] + [C.c_void_p] * 4 + [C.c_int, C.c_void_p]),
    "mmx_conv2d_large_wgrad_prec": (C.c_int, [C.POINTER(MmxConvHalfDesc)] + [C.c_void_p] * 4 + [C.c_int, C.c_void_p]),
    "mmx_conv2d_tc5_serves": (C.c_int, [C.POINTER(MmxConvHalfDesc)]),
    "mmx_conv_tail_fwd": (C.c_int, [C.POINTER(MmxConvHalfDesc)] + [C.c_void_p] * 7),
    "mmx_conv_tail_bwd1": (C.c_int, [C.POINTER(MmxConvHalfDesc)] + [C.c_void_p] * 10),
    "mmx_conv_tail_bwd2": (C.c_int, [C.POINTER(MmxConvHalfDesc)] + [C.c_void_p] * 7),
    "mmx_conv_half_bn_stats": (C.c_int, [C.POINTER(MmxConvHalfDesc), C.POINTER(MmxConvHalfParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_conv_half_bn_apply": (C.c_int, [C.POINTER(MmxConvHalfDesc), C.POINTER(MmxConvHalfParams)] + [C.c_void_p] * 5),
    "mmx_conv_half_bn_bwd1": (C.c_int, [C.POINTER(MmxConvHalfDesc), C.POINTER(MmxConvHalfParams), C.POINTER(MmxConvHalfParams)] + [C.c_void_p] * 6),
    "mmx_conv_half_bn_bwd2": (C.c_int, [C.POINTER(MmxConvHalfDesc), C.POINTER(MmxConvHalfParams), C.POINTER(MmxConvHalfParams)] + [C.c_void_p] * 8),
    "mmx_bn_finalize": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_float, C.c_float, C.c_void_p, C.c_void_p]),
    "mmx_bn_coef": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_ln_fwd": (C.c_int, [C.c_longlong, C.c_int, C.c_int] + [C.c_void_p] * 6),
    "mmx_ln_bwd": (C.c_int, [C.c_longlong, C.c_int, C.c_int] + [C.c_void_p] * 9),
    "mmx_bn1d_stats": (C.c_int, [C.c_longlong, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 3),
    "mmx_bn1d_apply": (C.c_int, [C.c_longlong, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 4),
    "mmx_bn1d_bwd_reduce": (C.c_int, [C.c_longlong, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 5),
    "mmx_bn1d_bwd_apply": (C.c_int, [C.c_longlong, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 6),
    "mmx_se_res_fwd": (C.c_int, [C.c_int] * 7 + [C.c_void_p] * 7),
    "mmx_se_res_bwd": (C.c_int, [C.c_int] * 7 + [C.c_void_p] * 9),
    "mmx_se_tail_fwd": (C.c_int, [C.c_int] * 7 + [C.c_void_p] * 5),
    "mmx_se_tail_bwd": (C.c_int, [C.c_int] * 7 + [C.c_void_p] * 8),
    "mmx_pose_encoder_fwd": (C.c_int, [C.POINTER(MmxEncoderDesc), C.POINTER(MmxEncoderParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_pose_encoder_bwd": (C.c_int, [C.POINTER(MmxEncoderDesc), C.POINTER(MmxEncoderParams), C.POINTER(MmxEncoderParams),
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_conv_head_fwd": (C.c_int, [C.POINTER(MmxConvHeadDesc), C.POINTER(MmxConvHeadParams), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_conv_head_bwd": (C.c_int, [C.POINTER(MmxConvHeadDesc), C.POINTER(MmxConvHeadParams), C.POINTER(MmxConvHeadParams),
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_window_split": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_pck_hist": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "mmx_mpjpe_fwd_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_float, C.c_void_p]),
    "mmx_l1_fwd_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_float, C.c_void_p]),
    "mmx_adam_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]),
    "mmx_peer_flag_bytes": (C.c_int, [C.c_int]),
    "mmx_peer_alloc": (C.c_int, [C.c_longlong, C.POINTER(C.c_void_p)]),
    "mmx_peer_free": (C.c_int, [C.c_void_p]),
    "mmx_ipc_export": (C.c_int, [C.c_void_p, C.c_char_p]),
    "mmx_ipc_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "mmx_ipc_close": (C.c_int, [C.c_void_p]),
    "mmx_adam_step_peer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong,
                                     C.c_void_p, C.c_void_p, C.c_void_p]),
    "mmx_adam_advance": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
}


class MmxError(RuntimeError):
    pass


def bind(cdll):
    """Attach restype/argtypes for every entry point; raises AttributeError on a missing symbol."""
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(cdll, name)
        fn.restype = res
        fn.argtypes = args
    return cdll


_lib = None


def load():
    """Load libmmx.so (built by ``python -m motionmixerconv_b200.build`` / ``__graft_entry__.build()``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MmxError(
                "motionmixerconv_b200: %s not found — the CUDA extension is not built. Run "
                "`python -m motionmixerconv_b200.build` (needs nvcc). There is no CPU fallback." % LIB_PATH)
        _lib = bind(C.CDLL(LIB_PATH))
    return _lib


def check(lib, rc, what):
    if rc != 0:
        msg = lib.mmx_last_error()
        text = msg.decode() if msg else "?"
        if rc == -1:
            raise ValueError("%s: %s" % (what, text))
        raise MmxError("%s failed (%d): %s" % (what, rc, text))
