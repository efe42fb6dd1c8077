"""ctypes binding of libnttt_b200.so (C-ABI declared in include/nttt_b200.h).

The library is the product: if it is missing or a call fails this module raises — there is no CPU or
torch fallback for the matching stage.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_size_t, c_void_p

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libnttt_b200.so")

NTTT_OK = 0


class NtttError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str = ""):
        self.code = code
        super().__init__(f"{where} failed with code {code}" + (f": {detail}" if detail else ""))


class MatchArgs(ctypes.Structure):
    """Mirror of `nttt_match_args` (include/nttt_b200.h)."""
    _fields_ = [
        ("logits", c_void_p), ("pred_ious", c_void_p), ("tar_feat", c_void_p), ("proto", c_void_p),
        ("n", c_int32), ("lr_h", c_int32), ("lr_w", c_int32), ("eh", c_int32), ("ew", c_int32), ("c", c_int32),
        ("n_cls", c_int32), ("ori_h", c_int32), ("ori_w", c_int32),
        ("nms_thr", c_float),
        ("num_out_instance", c_int32), ("max_sel", c_int32),
        ("out_masks", c_void_p), ("out_boxes", c_void_p), ("out_scores", c_void_p), ("out_labels", c_void_p),
        ("out_index", c_void_p), ("counts", c_void_p),
        ("sim", c_void_p), ("obj_feats", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
        ("proto_neg", c_void_p), ("l_neg", c_int32), ("sigma", c_float),
        ("iou_thr", c_float), ("filter_iou", c_int32),
        ("out_prev_rect", c_void_p),
        ("multi_ious", c_void_p), ("n_multi", c_int32), ("multi_first", c_int32),
        ("logits_chunks_host", POINTER(c_void_p)), ("n_chunks", c_int32), ("chunk_prompts", c_int32),
        ("rle_counts", c_void_p), ("rle_n_counts", c_void_p), ("rle_chars", c_void_p), ("rle_n_chars", c_void_p),
        ("rle_cap_counts", c_int32), ("rle_cap_chars", c_int32),
        ("low_latency", c_int32),
        ("sel", c_void_p), ("ios", c_void_p), ("ios_inter", c_void_p),
    ]


class MatchSizeRange(ctypes.Structure):
    """Mirror of `nttt_match_size_range` (include/nttt_b200.h)."""
    _fields_ = [("ori_hw_dev", c_void_p), ("min_h", c_int32), ("min_w", c_int32)]


MAX_CHUNKS = 64  # NTTT_MAX_CHUNKS
MAX_CANDIDATES = 16384  # NTTT_MAX_CANDIDATES: candidate masks per image (points_per_side up to 128)


class MatchInputs(ctypes.Structure):
    """Mirror of `nttt_match_inputs` (include/nttt_b200.h): the input addresses a bound stage reads on the device."""
    _fields_ = [("logits", c_void_p), ("pred_ious", c_void_p), ("multi_ious", c_void_p), ("tar_feat", c_void_p),
                ("chunks", c_void_p * MAX_CHUNKS), ("ori_hw", c_int32 * 2)]


class MatchBank(ctypes.Structure):
    """Mirror of `nttt_match_bank` (include/nttt_b200.h): the prototype table a banked stage reads on the device."""
    _fields_ = [("proto", c_void_p), ("proto_neg", c_void_p), ("n_cls", c_int32), ("l_neg", c_int32)]


# name -> (restype, argtypes); every symbol include/nttt_b200.h declares
_P = c_void_p
SIGNATURES = {
    "nttt_version": (c_int, []),
    "nttt_build_is_ablation": (c_int, []),
    "nttt_error_string": (c_char_p, [c_int]),
    "nttt_last_cuda_error": (c_char_p, []),
    "nttt_ctx_create": (c_int, [POINTER(c_void_p), c_int]),
    "nttt_ctx_destroy": (None, [c_void_p]),
    "nttt_ctx_tune": (c_int, [c_void_p, c_int, ctypes.c_longlong]),
    "nttt_threshold_pack": (c_int, [_P, c_int, c_int, c_int, c_float, c_float, _P, _P, _P, _P, _P, _P]),
    "nttt_threshold_pack_stability": (c_int, [_P, c_int, c_int, c_int, c_float, c_float, _P, _P, _P, _P, _P, _P, _P]),
    "nttt_select_multimask": (c_int, [_P, c_int, c_int, c_int, POINTER(c_void_p), c_int, c_int, c_int, c_int, _P, _P, _P]),
    "nttt_threshold_pack_ptrs": (c_int, [_P, _P, c_float, c_int, c_int, c_int, c_float, c_float, _P, _P, _P, _P, _P, _P]),
    "nttt_upsample_threshold_pack_ptrs": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, _P, _P, c_int, c_int, c_int, _P, _P,
                                                  _P, _P, _P]),
    "nttt_project_masks": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "nttt_pool_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "nttt_pool_normalize": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, _P, _P, c_size_t, _P]),
    "nttt_proto_prepare": (c_int, [_P, c_int, c_int, c_int, _P, _P]),
    "nttt_similarity_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "nttt_similarity_top1": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P, _P, _P, _P, c_size_t, _P]),
    "nttt_nms_workspace_bytes": (c_size_t, [c_int]),
    "nttt_box_nms": (c_int, [_P, _P, _P, _P, c_int, c_float, c_int, _P, _P, _P, _P, _P, c_size_t, _P]),
    "nttt_upsample_threshold_pack": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, _P, _P, c_int, c_int, c_int, _P, _P,
                                             _P, _P, _P]),
    "nttt_mask_ios_workspace_bytes": (c_size_t, [c_int]),
    "nttt_mask_ios": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, _P, _P, c_int, _P, _P, _P, c_size_t, _P]),
    "nttt_decay_topk": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, _P, _P, _P, c_int, c_int, _P, _P, _P, _P, _P, _P,
                                _P, _P]),
    "nttt_unpack_masks": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P, _P]),
    "nttt_rle_encode": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "nttt_rle_compact": (c_int, [_P, _P, c_int, c_int, _P, ctypes.c_int64, _P]),
    "nttt_fill_pool_accumulate": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "nttt_fill_pool_batch": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "nttt_fill_scatter": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, _P, _P, _P, _P]),
    "nttt_fill_finalize": (c_int, [_P, _P, c_int, c_int, c_int, _P, _P, _P]),
    "nttt_match_workspace_bytes": (c_size_t, [c_int] * 10),
    "nttt_match_workspace_bytes_neg": (c_size_t, [c_int] * 11),
    "nttt_similarity_neg_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "nttt_similarity_neg_top1": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_float, _P, _P, _P, _P, c_size_t,
                                          _P]),
    "nttt_match_image": (c_int, [_P, POINTER(MatchArgs), _P]),
    "nttt_sizeof_match_args": (c_size_t, []),
    "nttt_match_workspace_bytes_sized": (c_size_t, [c_int] * 13),
    "nttt_match_image_sized": (c_int, [_P, POINTER(MatchArgs), POINTER(MatchSizeRange), _P]),
    "nttt_ctx_atlas_stats": (c_int, [_P, POINTER(c_size_t), POINTER(ctypes.c_double)]),
    "nttt_sizeof_match_inputs": (c_size_t, []),
    "nttt_match_bind": (c_int, [_P, POINTER(MatchInputs), POINTER(MatchArgs), _P]),
    "nttt_match_image_bound": (c_int, [_P, POINTER(MatchArgs), POINTER(MatchSizeRange), _P, _P]),
    "nttt_sizeof_match_bank": (c_size_t, []),
    "nttt_match_bank_bind": (c_int, [_P, POINTER(MatchBank), POINTER(MatchArgs), _P]),
    "nttt_match_image_banked": (c_int, [_P, POINTER(MatchArgs), POINTER(MatchSizeRange), _P, _P, _P]),
    "nttt_match_count_bind": (c_int, [_P, ctypes.c_int32, POINTER(MatchArgs), _P]),
    "nttt_match_image_counted": (c_int, [_P, POINTER(MatchArgs), POINTER(MatchSizeRange), _P, _P, _P, _P]),
    "nttt_launch_count": (ctypes.c_ulonglong, []),
    "nttt_profile_num_stages": (c_int, []),
    "nttt_profile_stage_name": (c_char_p, [c_int]),
    "nttt_ctx_profile": (c_int, [_P, c_int]),
    "nttt_ctx_profile_read": (c_int, [_P, POINTER(c_float), c_int]),
}

_lib = None


def load() -> ctypes.CDLL:
    """dlopen the in-tree library and type every entry point.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python no-time-to-train_b200/build.py` "
            "(or __graft_entry__.build()).  There is no fallback path for the matching stage.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code: int, where: str) -> None:
    if code != NTTT_OK:
        lib = load()
        detail = lib.nttt_error_string(code).decode()
        cuda = lib.nttt_last_cuda_error().decode()
        raise NtttError(code, where, detail + (f" [{cuda}]" if cuda else ""))
