"""ctypes binding of libltb200 (include/ltb200.h).  Fails loudly when the CUDA library is missing —
there is deliberately no CPU fallback behind this module."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libltb200.so")

LTB_SESSION_KEEP_LAYERS = 1
LTB_SESSION_NO_GRAPH = 2
LTB_SESSION_NO_HALO = 4
LTB_SESSION_NO_PDL = 8
LTB_SESSION_SLOTS = 16
LTB_SESSION_MEL_ONLY = 32


class LtbError(RuntimeError):
    pass


class ConvOp(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in ("in_", "w", "w_tap", "bias", "res", "out")] +
                [(n, C.c_int) for n in ("N", "IH", "IW", "ICtot", "ic_off", "Cin", "OH", "OW", "Cout", "OCtot", "oc_off", "RCtot",
                                        "rc_off", "KH", "KW", "sy", "sx", "pad_t", "pad_l", "Ktot", "w_koff", "relu", "no_halo",
                                        "zbatch", "zdiv")] +
                [(n, C.c_longlong) for n in ("in_zo", "in_zi", "w_zo", "w_zi", "out_zo", "out_zi")] +
                [("gn_stats", C.c_void_p), ("gn_groups", C.c_int), ("gn_hw", C.c_int), ("upsample2x", C.c_int)])


class MtPasteOp(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in ("frames", "coords", "crop", "masks", "mask_off", "pred", "out")] +
                [(n, C.c_int) for n in ("nf", "H", "W", "index", "explicit_idx", "slot0", "count", "pred_hw")] +
                [("body", C.c_void_p), ("region_h", C.c_int), ("region_w", C.c_int)])


class W2LSlot(C.Structure):
    _fields_ = [("avatar", C.c_void_p), ("idx", C.c_int), ("mel", C.c_void_p)]


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in
                ("N", "IH", "IW", "Cin", "Cout", "KH", "KW", "sy", "sx", "pad", "transposed", "relu", "has_res",
                 "force_path")]


_SIGS = {
    "ltb_version": (C.c_int, []),
    "ltb_last_error": (C.c_char_p, []),
    "ltb_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "ltb_set_device": (C.c_int, [C.c_int]),
    "ltb_w2l_model_create": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "ltb_w2l_model_create_from_device": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "ltb_w2l_model_destroy": (C.c_int, [C.c_void_p]),
    "ltb_w2l_avatar_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.POINTER(C.c_void_p)]),
    "ltb_w2l_avatar_destroy": (C.c_int, [C.c_void_p]),
    "ltb_w2l_avatar_region_max": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ltb_mem_get_info": (C.c_int, [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "ltb_w2l_session_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.POINTER(C.c_void_p)]),
    "ltb_w2l_session_destroy": (C.c_int, [C.c_void_p]),
    "ltb_w2l_mel_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "ltb_w2l_set_pcm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "ltb_w2l_infer": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "ltb_w2l_paste": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "ltb_w2l_paste_pred": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "ltb_w2l_paste_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "ltb_w2l_infer_paste": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "ltb_w2l_infer_slots": (C.c_int, [C.c_void_p, C.POINTER(W2LSlot), C.c_int, C.c_void_p]),
    "ltb_w2l_infer_paste_region": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "ltb_w2l_infer_slots_region": (C.c_int, [C.c_void_p, C.POINTER(W2LSlot), C.c_int, C.c_void_p]),
    "ltb_w2l_paste_pred_region": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "ltb_w2l_mel_resident": (C.c_int, [C.c_void_p]),
    "ltb_w2l_step_async": (C.c_int, [C.c_void_p, C.c_int]),
    "ltb_w2l_forward_async": (C.c_int, [C.c_void_p, C.c_int]),
    "ltb_w2l_profile_ops": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_void_p, C.c_void_p, C.c_void_p]),
    "ltb_w2l_step_e2e_async": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "ltb_w2l_e2e_acquire": (C.c_int, [C.c_void_p]),
    "ltb_w2l_sync": (C.c_int, [C.c_void_p]),
    "ltb_w2l_stream": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "ltb_w2l_launch_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_longlong)]),
    "ltb_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "ltb_host_free": (C.c_int, [C.c_void_p]),
    "ltb_w2l_num_layers": (C.c_int, []),
    "ltb_w2l_layer_shape": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ltb_w2l_layer_read": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    "ltb_ctx_create": (C.c_int, [C.POINTER(C.c_void_p)]),
    "ltb_ctx_destroy": (C.c_int, [C.c_void_p]),
    "ltb_ctx_stream": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "ltb_ctx_sync": (C.c_int, [C.c_void_p]),
    "ltb_ctx_launch_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_longlong)]),
    "ltb_dev_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]),
    "ltb_dev_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ltb_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]),
    "ltb_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]),
    "ltb_set_i32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "ltb_capture_begin": (C.c_int, [C.c_void_p]),
    "ltb_capture_end": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "ltb_graph_launch": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ltb_graph_destroy": (C.c_int, [C.c_void_p]),
    "ltb_op_conv2d": (C.c_int, [C.c_void_p, C.POINTER(ConvOp)]),
    "ltb_op_w_tap_major": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "ltb_op_groupnorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                   C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "ltb_op_groupnorm_apply": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "ltb_op_layernorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ltb_op_softmax": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "ltb_op_geglu": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    "ltb_op_eltwise": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p]),
    "ltb_op_upsample2x": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "ltb_op_copy_channels": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "ltb_op_transpose_heads": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_void_p]),
    "ltb_op_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_int]),
    "ltb_op_dwconv3x3": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                   C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "ltb_op_upsample_bilinear2x": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                             C.c_int]),
    "ltb_op_ul_prep": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "ltb_op_head_sigmoid255": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "ltb_op_ul_paste": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_int, C.c_int, C.c_int]),
    "ltb_op_ul_paste_region": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_int, C.c_int, C.c_int]),
    "ltb_op_hubert_conv0": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "ltb_op_hubert_pos_conv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ltb_op_hubert_slice": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int,
                                      C.c_void_p, C.c_void_p]),
    "ltb_op_vae_post": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    "ltb_op_bgr_to_i420": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "ltb_op_stamp_pixels": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "ltb_op_vae_pre": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "ltb_op_gather_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_longlong, C.c_void_p]),
    "ltb_op_whisper_logmel": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ltb_op_whisper_slice": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p,
                                       C.c_int]),
    "ltb_op_mt_paste": (C.c_int, [C.c_void_p, C.POINTER(MtPasteOp)]),
    "ltb_conv2d_f16": (C.c_int, [C.POINTER(ConvDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ltb_conv2d_f16_timed": (C.c_int, [C.POINTER(ConvDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                       C.POINTER(C.c_float)]),
}

# hardware probes: only in lib/libltb200_diag.so (include/ltb200_diag.h)
DIAG_SIGS = {
    "ltb_umma_probe": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "ltb_umma_probe_noswz": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGS)

_lib = None


def lib() -> C.CDLL:
    """Load libltb200.so (once).  Raises LtbError if it has not been built — no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LtbError(f"{LIB_PATH} not found: build it with `python -m livetalking_b200.build` "
                           "(sm_100a CUDA library; there is no CPU fallback)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        for name, (res, args) in DIAG_SIGS.items():      # present in the diagnostic build only
            fn = getattr(l, name, None)
            if fn is not None:
                fn.restype = res
                fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().ltb_last_error()
        raise LtbError(msg.decode("utf-8", "replace") if msg else f"libltb200 error {rc}")
