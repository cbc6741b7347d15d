"""ctypes binding of the C ABI declared in include/fpm_b200.h.

The product path has no CPU fallback: if the CUDA library is missing this module raises, and
`fpm_create` failing (no GPU) raises `FpmError` from the matcher.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libfpm_b200.so")


class fpm_result(C.Structure):
    """POD mirror of s_SingleTargetMatch (/root/reference/include/DataStructures.h:97-115)."""
    _fields_ = [(n, C.c_double) for n in
                ("score", "angle", "cx", "cy", "ltx", "lty", "rtx", "rty", "rbx", "rby", "lbx", "lby")]


PARAM_MAX_POSITIONS, PARAM_MAX_OVERLAP, PARAM_SCORE, PARAM_TOLERANCE_ANGLE, PARAM_MIN_REDUCE_AREA, \
    PARAM_USE_SIMD, PARAM_SUBPIXEL, PARAM_TRACE, PARAM_WORKSPACE_MB, PARAM_PROFILE, PARAM_H2D_CHUNK, PARAM_TENSOR_CORES, PARAM_MFC_COMPAT, PARAM_STOP_LAYER1, PARAM_BITWISE_NOT, PARAM_TOLERANCE_RANGE, \
    PARAM_TOLERANCE1, PARAM_TOLERANCE2, PARAM_TOLERANCE3, PARAM_TOLERANCE4, PARAM_SPLIT_BATCH, PARAM_SHARD_UPLOAD, PARAM_ASYNC_DESCENT, \
    PARAM_JPEG_DEVICE_HUFFMAN, PARAM_JPEG_PASSES, PARAM_SCALE_MIN, PARAM_SCALE_MAX = range(27)

_vp, _i, _d, _sz = C.c_void_p, C.c_int, C.c_double, C.c_size_t
_pi, _pd = C.POINTER(C.c_int), C.POINTER(C.c_double)

# name -> (restype, argtypes); must list every symbol of include/fpm_b200.h
SIGNATURES = {
    "fpm_create": (_vp, [_i]),
    "fpm_destroy": (None, [_vp]),
    "fpm_last_error": (C.c_char_p, [_vp]),
    "fpm_version": (C.c_char_p, []),
    "fpm_set_param": (_i, [_vp, _i, _d]),
    "fpm_get_param": (_d, [_vp, _i]),
    "fpm_learn": (_i, [_vp, _vp, _i, _i, _i]),
    "fpm_learn_set": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "fpm_learn_masked": (_i, [_vp, _vp, _i, _i, _i, _vp, _i]),
    "fpm_learn_set_masked": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "fpm_set_size": (_i, [_vp]),
    "fpm_match_set_batch": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _sz, _vp, _i, _vp]),
    "fpm_match_ingested_set_batch": (_i, [_vp, _vp, _i, _vp]),
    "fpm_match_set_batch_merged": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _sz, _d, _vp, _vp, _i, _vp, _vp]),
    "fpm_match_ingested_set_batch_merged": (_i, [_vp, _d, _vp, _vp, _i, _vp, _vp]),
    "fpm_match_set_scaled": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _sz, _vp, _vp, _i, _vp]),
    "fpm_match_ingested_set_scaled": (_i, [_vp, _vp, _vp, _i, _vp]),
    "fpm_match_set_scaled_merged": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _sz, _d, _vp, _vp, _vp, _i, _vp, _vp]),
    "fpm_match_ingested_set_scaled_merged": (_i, [_vp, _d, _vp, _vp, _vp, _i, _vp, _vp]),
    "fpm_is_learned": (_i, [_vp]),
    "fpm_clear": (None, [_vp]),
    "fpm_match": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _pi]),
    "fpm_match_batch": (_i, [_vp, _vp, _i, _i, _i, _i, _sz, _vp, _i, _vp]),
    "fpm_match_multi": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _i, _vp]),
    "fpm_ocr_assemble": (_i, [_vp, _vp, _vp, _i, _d, _vp, _i]),
    "fpm_ingest_bmp": (_i, [_vp, _vp, _sz, _pi, _pi]),
    "fpm_ingest_rgb32": (_i, [_vp, _vp, _i, _i, _i]),
    "fpm_ingest_jpeg": (_i, [_vp, _vp, _sz, _pi, _pi]),
    "fpm_ingest_image": (_i, [_vp, _vp, _sz, _pi, _pi]),
    "fpm_dbg_jpeg_luma": (_i, [_vp, _sz, _pi, _pi, _pi, _pi, _vp, _vp, _sz, _vp, _i]),
    "fpm_dbg_jpeg_luma_parallel": (_i, [_vp, _sz, _vp, _sz, _pi, _vp, _i]),
    "fpm_ingested_pixels": (_i, [_vp, _vp]),
    "fpm_match_ingested": (_i, [_vp, _vp, _i, _pi]),
    "fpm_learn_ingested": (_i, [_vp]),
    "fpm_ingest_jpeg_batch": (_i, [_vp, _vp, _vp, _i, _pi, _pi]),
    "fpm_ingested_count": (_i, [_vp]),
    "fpm_ingested_frame_pixels": (_i, [_vp, _i, _vp]),
    "fpm_match_ingested_batch": (_i, [_vp, _vp, _i, _vp]),
    "fpm_match_scaled": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _sz, _vp, _vp, _i, _vp]),
    "fpm_match_ingested_scaled": (_i, [_vp, _vp, _vp, _i, _vp]),
    "fpm_dbg_jpeg_luma_parallel_batch": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i]),
    "fpm_dbg_jpeg_unstuff": (_i, [_vp, _sz, _i, _vp, _sz, _vp, _i, _vp, _pi, _pi]),
    "fpm_match_batch_device": (_i, [_vp, _vp, _i, _i, _i, _i, _sz, _vp, _i, _vp]),
    "fpm_last_time_ms": (_d, [_vp]),
    "fpm_set_user_rect": (None, [_vp, _i, _i, _i, _i]),
    "fpm_get_user_rect": (_i, [_vp, _pi, _pi, _pi, _pi]),
    "fpm_launch_count": (C.c_longlong, [_vp]),
    "fpm_timer_record": (_i, [_vp, _i]),
    "fpm_timer_elapsed_ms": (_d, [_vp]),
    "fpm_profile_num_kernels": (_i, []),
    "fpm_profile_name": (C.c_char_p, [_i]),
    "fpm_profile_get": (_i, [_vp, _i, _pd, C.POINTER(C.c_longlong), _pd]),
    "fpm_profile_reset": (None, [_vp]),
    "fpm_tpl_levels": (_i, [_vp]),
    "fpm_tpl_level_info": (_i, [_vp, _i, _pi, _pi, _pd, _pd, _pd, _pi]),
    "fpm_tpl_level_pixels": (_i, [_vp, _i, _vp]),
    "fpm_tpl_level_mask": (_i, [_vp, _i, _vp]),
    "fpm_tpl_border_color": (_i, [_vp]),
    "fpm_stage_num_angles": (_i, [_vp, _i, _i]),
    "fpm_stage_top": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _pi]),
    "fpm_stage_sort_candidates": (_i, [_vp, _vp, _i, _vp]),
    "fpm_stage_refine": (_i, [_vp, _vp, _i, _vp, _i, _pi]),
    "fpm_stage_final": (_i, [_vp, _vp, _i, _vp, _i, _pi]),
    "fpm_comm_available": (_i, []),
    "fpm_comm_get_unique_id": (_i, [_vp]),
    "fpm_comm_init": (_i, [_vp, _i, _i, _vp]),
    "fpm_comm_attach": (_i, [_vp, _vp, _i, _i]),
    "fpm_comm_destroy": (None, [_vp]),
    "fpm_match_sharded": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _pi]),
    "fpm_match_sharded_virtual": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _i, _vp]),
    "fpm_match_set_sharded": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _vp]),
    "fpm_match_set_sharded_merged": (_i, [_vp, _vp, _i, _i, _i, _i, _d, _vp, _vp, _i, _vp, _vp]),
    "fpm_match_set_sharded_virtual": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _i, _vp]),
    "fpm_match_set_sharded_merged_virtual": (_i, [_vp, _i, _vp, _i, _i, _i, _d, _vp, _vp, _i, _vp, _vp]),
    "fpm_match_set_sharded_scaled": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _i, _vp]),
    "fpm_match_set_sharded_scaled_merged": (_i, [_vp, _vp, _i, _i, _i, _i, _d, _vp, _vp, _vp, _i, _vp, _vp]),
    "fpm_match_set_sharded_scaled_virtual": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _vp, _i, _vp]),
    "fpm_match_set_sharded_scaled_merged_virtual": (_i, [_vp, _i, _vp, _i, _i, _i, _d, _vp, _vp, _vp, _i, _vp, _vp]),
    "fpm_shard_angle_range": (_i, [_i, _i, _i, _pi, _pi]),
    "fpm_collective_count": (C.c_longlong, [_vp]),
    "fpm_dbg_pyrdown": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "fpm_dbg_pyrdown2": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "fpm_dbg_warp_affine": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _i, _i, _vp]),
    "fpm_dbg_corr_rows": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "fpm_dbg_corr_rows_mma": (_i, [_vp, _vp, _i, _vp, _i, _i, _vp, _vp, _vp]),
    "fpm_dbg_corr_fused": (_i, [_vp, _vp, _i, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "fpm_dbg_top_score": (_i, [_vp, _vp, _i, _i, _vp]),
    "fpm_dbg_top_score_production": (_i, [_vp, _vp, _i, _i, _vp, C.POINTER(C.c_float)]),
    "fpm_dbg_peaks": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _d, _d, _i, _vp, _pi]),
    "fpm_dbg_rrect_overlap": (_i, [_vp, _vp, _d, _pi, _pd]),
    "fpm_dbg_rrect_from3": (_i, [_vp, _vp]),
    "fpm_trace_num_candidates": (_i, [_vp]),
    "fpm_trace_candidates": (_i, [_vp, _vp]),
    "fpm_trace_num_evals": (_i, [_vp, _i]),
    "fpm_trace_evals": (_i, [_vp, _i, _vp]),
    "fpm_trace_level": (_i, [_vp, _i, _vp, _pi, _pi]),
    "fpm_trace_eval_scores": (_i, [_vp, _i, _vp]),
    "fpm_trace_eval_rois": (_i, [_vp, _i, _vp, _pi, _pi, _pi]),
}

_lib = None


def load():
    """Load libfpm_b200.so; raises (loudly) when the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m fastest_image_pattern_matching_b200._build` "
            "(or __graft_entry__.build()).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
