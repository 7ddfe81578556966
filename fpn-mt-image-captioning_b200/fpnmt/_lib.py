"""ctypes binding of libfpnmt.so (C ABI declared in include/fpnmt.h).

The library is built in-tree by `build.py` (nvcc, sm_100a).  There is no fallback: if the shared object is
missing or cannot be loaded this module raises, and every product entry point fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "libfpnmt.so")

OK, ERR_INVALID, ERR_STATE, ERR_CUDA, ERR_MISSING = 0, 1, 2, 3, 4
BACKBONE_IDS = {"mobilenet224_1.0": 0, "mobilenetv2": 0, "resnet50": 1, "densenet121": 2}
PREC_IDS = {"bf16": 0, "bf16x3": 1}
SCORE_IDS = {"log": 0, "prob": 1}
CACHE_IDS = {"ancestry": 0, "physical": 1}
DECODE_IDS = {"auto": 0, "chain": 1, "fused": 2}
# fpnmt_config.kernel_opts bits (include/fpnmt.h FPNMT_OPT_*): each switches one fused kernel back to its unfused equivalent
OPT_BITS = {"no_xattn": 1, "no_stem": 2, "no_tgemm": 4, "enc_att_simt": 8, "no_pdl": 32, "dstep_taps": 128, "dec_att_simt": 256, "tgemm_wide": 512, "no_tgemm_wide": 1024, "no_kv_share": 2048, "no_vstats": 4096, "no_dense_1x1": 8192, "no_tma_store": 16384, "no_b_stationary": 32768}


class FpnmtConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "backbone", "image_size", "batch", "beam", "vocab", "max_len", "num_layers", "d_model", "num_heads", "dff",
        "precision", "score_mode", "start_id", "end_id", "true_beam", "use_graphs", "kernel_opts", "cache_mode",
        "decode_path")] + [("length_penalty", C.c_float), ("finished_beams", C.c_int32), ("dec_groups", C.c_int32),
                           ("lanes", C.c_int32), ("reserved", C.c_int32 * 1)]


class FpnmtSampling(C.Structure):
    """fpnmt_sampling (include/fpnmt.h): temperature, top-k, top-p and seed of a sampled decode."""
    _fields_ = [("temperature", C.c_float), ("top_k", C.c_int32), ("top_p", C.c_float), ("seed", C.c_uint64),
                ("reserved", C.c_int32 * 4)]


class FpnmtConstraints(C.Structure):
    """fpnmt_constraints (include/fpnmt.h): no-repeat n-gram size, minimum length and banned token ids (host array)."""
    _fields_ = [("no_repeat_ngram", C.c_int32), ("min_len", C.c_int32), ("banned", C.POINTER(C.c_int32)),
                ("n_banned", C.c_int32), ("reserved", C.c_int32 * 4)]


class FpnmtError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("fpnmt error %d: %s" % (code, msg))
        self.code = code


# every symbol include/fpnmt.h declares: name -> (restype, argtypes)
_vp, _i, _f = C.c_void_p, C.c_int, C.c_void_p
SIGNATURES = {
    "fpnmt_version": (C.c_char_p, []),
    "fpnmt_last_error": (C.c_char_p, []),
    "fpnmt_create": (_i, [C.POINTER(FpnmtConfig), _i, C.POINTER(_vp)]),
    "fpnmt_destroy": (_i, [_vp]),
    "fpnmt_set_weight": (_i, [_vp, C.c_char_p, _vp, C.POINTER(C.c_int64), _i]),
    "fpnmt_finalize_weights": (_i, [_vp]),
    "fpnmt_encode": (_i, [_vp, _vp, _i, _vp, _vp]),
    "fpnmt_features": (_i, [_vp, _vp, _i, C.POINTER(_vp), _vp]),
    "fpnmt_get_tap": (_i, [_vp, C.c_char_p, _vp, C.c_size_t, C.POINTER(C.c_size_t), _vp]),
    "fpnmt_decode_logits": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "fpnmt_beam_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "fpnmt_beam_step_vstats": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "fpnmt_generate": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i, _vp, _vp]),
    "fpnmt_stage_images": (_i, [_vp, _vp, _i]),
    "fpnmt_generate_staged": (_i, [_vp, _i, _vp, _vp, _i, _i, _vp, _vp]),
    "fpnmt_decode": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp]),
    "fpnmt_profile": (_i, [_vp, _i, C.c_char_p, C.c_size_t]),
    "fpnmt_launch_count": (C.c_int64, [_vp]),
    "fpnmt_lanes": (_i, [_vp]),
    "fpnmt_submit": (_i, [_vp, _i, _vp, _i, _i, _vp]),
    "fpnmt_collect": (_i, [_vp, _i, _vp, _vp, _i, _vp]),
    "fpnmt_op_conv2d": (_i, [_i, _i, _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _vp]),
    "fpnmt_op_preprocess": (_i, [_i, _vp, _i, _i, _i, _i, _vp, _vp]),
    "fpnmt_op_decode_jpeg": (_i, [_i, C.POINTER(_vp), C.POINTER(C.c_size_t), _i, _i, _vp, _vp, _vp]),
    "fpnmt_op_dense": (_i, [_i, _i, _vp, _i, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, C.c_float, _vp, _i, _vp]),
    "fpnmt_op_vocab_stats": (_i, [_i, _i, _vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "fpnmt_op_vocab_stats_target": (_i, [_i, _i, _vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "fpnmt_op_depthwise3x3": (_i, [_i, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "fpnmt_op_pool": (_i, [_i, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "fpnmt_op_scale_shift_relu": (_i, [_i, _i, _vp, C.c_int64, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "fpnmt_op_score_conv": (_i, [_i, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "fpnmt_op_coattention": (_i, [_i, _i, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "fpnmt_op_tokens_ln_pos": (_i, [_i, _i, _vp, _i, _i, _vp, _vp, C.c_float, _vp, _vp, _vp]),
    "fpnmt_op_enc_attention": (_i, [_i, _i, _vp, C.POINTER(_vp), C.POINTER(_i), _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "fpnmt_op_dec_self_attention": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "fpnmt_op_dec_cross_attention": (_i, [_i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "fpnmt_op_xattn": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp,
                            _vp]),
    "fpnmt_op_kv_reorder": (_i, [_i, _i, _vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp]),
    "fpnmt_op_embed_pos": (_i, [_i, _i, _vp, _i, _vp, _i, _vp, _i, _i, _i, _vp, _vp]),
    "fpnmt_op_layernorm_rows": (_i, [_i, _i, _vp, _i, _vp, _vp, C.c_float, _vp, _vp]),
    "fpnmt_sample": (_i, [_vp, _vp, _i, C.POINTER(FpnmtSampling), _vp, _vp, _vp, _i, _i, _vp]),
    "fpnmt_op_sample_step": (_i, [_i, _vp, _i, _i, _i, _i, C.POINTER(FpnmtSampling), _vp, _vp, _vp, _vp]),
    "fpnmt_score": (_i, [_vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp]),
    "fpnmt_beam_search": (_i, [_vp, _vp, _i, C.c_float, _vp, _vp, _vp, _i, _i, _vp]),
    "fpnmt_beam_search_diverse": (_i, [_vp, _vp, _i, _i, C.c_float, C.c_float, _vp, _vp, _vp, _i, _i, _vp]),
    "fpnmt_sample_prefix": (_i, [_vp, _vp, _i, _vp, _vp, _i, C.POINTER(FpnmtSampling), _vp, _vp, _vp, _i, _i, _vp]),
    "fpnmt_beam_search_prefix": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i, C.c_float, C.c_float, _vp, _vp, _vp, _i, _i, _vp]),
    "fpnmt_sample_constrained": (_i, [_vp, _vp, _i, _vp, _vp, _i, C.POINTER(FpnmtSampling), C.POINTER(FpnmtConstraints), _vp, _vp,
                                      _vp, _i, _i, _vp]),
    "fpnmt_beam_search_constrained": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i, C.c_float, C.c_float, C.POINTER(FpnmtConstraints),
                                           _vp, _vp, _vp, _i, _i, _vp]),
    "fpnmt_op_vocab_stats_mask": (_i, [_i, _i, _vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "fpnmt_op_ban_mask": (_i, [_i, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp]),
}



# ---- DLPack (include/fpnmt_dlpack.h): the `_dl` entry points take `const DLTensor*` --------------------------------------
class DLDevice(C.Structure):
    _fields_ = [("device_type", C.c_int32), ("device_id", C.c_int32)]


class DLDataType(C.Structure):
    _fields_ = [("code", C.c_uint8), ("bits", C.c_uint8), ("lanes", C.c_uint16)]


class DLTensor(C.Structure):
    _fields_ = [("data", C.c_void_p), ("device", DLDevice), ("ndim", C.c_int32), ("dtype", DLDataType),
                ("shape", C.POINTER(C.c_int64)), ("strides", C.POINTER(C.c_int64)), ("byte_offset", C.c_uint64)]


_dlp = C.POINTER(DLTensor)
SIGNATURES.update({
    "fpnmt_decode_hidden": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "fpnmt_decode_attention": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "fpnmt_set_weight_dl": (_i, [_vp, C.c_char_p, _dlp]),
    "fpnmt_encode_dl": (_i, [_vp, _dlp, _dlp, _vp]),
    "fpnmt_features_dl": (_i, [_vp, _dlp, C.POINTER(_dlp), _vp]),
    "fpnmt_decode_logits_dl": (_i, [_vp, _dlp, _dlp, _dlp, _vp]),
    "fpnmt_decode_hidden_dl": (_i, [_vp, _dlp, _dlp, _dlp, _vp]),
    "fpnmt_decode_attention_dl": (_i, [_vp, _dlp, _dlp, _dlp, _dlp, _vp]),
    "fpnmt_generate_dl": (_i, [_vp, _dlp, _dlp, _dlp, _i, _dlp, _vp]),
    "fpnmt_sample_dl": (_i, [_vp, _dlp, C.POINTER(FpnmtSampling), _dlp, _dlp, _dlp, _i, _vp]),
    "fpnmt_score_dl": (_i, [_vp, _dlp, _dlp, _dlp, _dlp, _dlp, _vp]),
    "fpnmt_beam_search_dl": (_i, [_vp, _dlp, C.c_float, _dlp, _dlp, _dlp, _i, _vp]),
    "fpnmt_beam_search_diverse_dl": (_i, [_vp, _dlp, _i, C.c_float, C.c_float, _dlp, _dlp, _dlp, _i, _vp]),
    "fpnmt_sample_prefix_dl": (_i, [_vp, _dlp, _dlp, _dlp, C.POINTER(FpnmtSampling), _dlp, _dlp, _dlp, _i, _vp]),
    "fpnmt_beam_search_prefix_dl": (_i, [_vp, _dlp, _dlp, _dlp, _i, C.c_float, C.c_float, _dlp, _dlp, _dlp, _i, _vp]),
    "fpnmt_sample_constrained_dl": (_i, [_vp, _dlp, _dlp, _dlp, C.POINTER(FpnmtSampling), C.POINTER(FpnmtConstraints), _dlp, _dlp,
                                         _dlp, _i, _vp]),
    "fpnmt_beam_search_constrained_dl": (_i, [_vp, _dlp, _dlp, _dlp, _i, C.c_float, C.c_float, C.POINTER(FpnmtConstraints),
                                              _dlp, _dlp, _dlp, _i, _vp]),
    "fpnmt_comm_unique_id": (_i, [_vp]),
    "fpnmt_comm_create": (_i, [_i, _i, _vp, _i, C.POINTER(_vp)]),
    "fpnmt_comm_destroy": (_i, [_vp]),
    "fpnmt_allgather_ids": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "fpnmt_allgather_ids_dl": (_i, [_vp, _dlp, _dlp, _dlp, _dlp, _vp]),
})


def dl_tensor(obj):
    """(pointer to the DLTensor inside the DLPack capsule of `obj`, keep-alive).  `obj` is anything with `__dlpack__`
    (torch / numpy >= 1.23 / cupy ...): the pointer is the `dl_tensor` member that starts the capsule's DLManagedTensor."""
    if obj is None:
        return None, None
    try:
        cap = obj.__dlpack__()
    except TypeError:
        cap = obj.__dlpack__(stream=None)
    get = C.pythonapi.PyCapsule_GetPointer
    get.restype, get.argtypes = C.c_void_p, [C.py_object, C.c_char_p]
    ptr = get(cap, b"dltensor")
    return C.cast(ptr, _dlp), (cap, obj)


_lib = None


def load() -> C.CDLL:
    """Load libfpnmt.so (once) and attach the prototypes.  Raises if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libfpnmt.so not found at %s — build it with `python fpn-mt-image-captioning_b200/build.py` "
            "(or __graft_entry__.build()); there is no CPU / PyTorch fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here == header and library out of sync
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def sampling(temperature: float = 1.0, top_k: int = 0, top_p: float = 1.0, seed: int = 0) -> FpnmtSampling:
    """An fpnmt_sampling with the reserved words zero."""
    sp = FpnmtSampling()
    sp.temperature, sp.top_k, sp.top_p, sp.seed = float(temperature), int(top_k), float(top_p), int(seed) & 0xFFFFFFFFFFFFFFFF
    return sp


def constraints(no_repeat_ngram: int = 0, min_len: int = 0, banned=None) -> FpnmtConstraints:
    """An fpnmt_constraints with the reserved words zero.  `banned` (token ids) is copied into an int32 array the struct
    keeps alive."""
    c = FpnmtConstraints()
    c.no_repeat_ngram, c.min_len = int(no_repeat_ngram), int(min_len)
    ids = [int(v) for v in (banned if banned is not None else [])]
    if ids:
        c._banned = (C.c_int32 * len(ids))(*ids)
        c.banned = C.cast(c._banned, C.POINTER(C.c_int32))
    c.n_banned = len(ids)
    return c


def check(rc: int) -> None:
    if rc != 0:
        raise FpnmtError(rc, load().fpnmt_last_error().decode("utf-8", "replace"))
