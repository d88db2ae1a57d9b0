"""ctypes binding of ``libzoe_cuda.so`` -- the same symbols a Rust ``-sys`` crate would bind
(include/zoe_cuda.h).  Loading fails loudly when the CUDA extension has not been built."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ZOE_CUDA_LIB") or os.path.join(HERE, "libzoe_cuda.so")  # env: another build (A/B timing)

SOME, OVERFLOWED, UNMAPPED = 0, 1, 2
E_EMPTY_SEQUENCE, E_GAP_OPEN_RANGE, E_GAP_EXTEND_RANGE, E_BAD_GAP_WEIGHTS = -1, -2, -3, -4
E_BAD_ARG, E_CIGAR_CAP, E_CUDA, E_STATE, E_UNSUPPORTED = -5, -6, -7, -8, -9

#: every symbol include/zoe_cuda.h declares (checked by tests/test_abi.py)
SYMBOLS = [
    "zoe_cuda_create", "zoe_cuda_destroy", "zoe_cuda_last_error", "zoe_cuda_set_scoring", "zoe_cuda_set_lanes",
    "zoe_cuda_set_profiled", "zoe_cuda_sw_score_batch", "zoe_cuda_sw_align_batch", "zoe_cuda_stage_streamed",
    "zoe_cuda_run_score_staged", "zoe_cuda_run_align_staged", "zoe_cuda_fetch_scores", "zoe_cuda_last_timing",
    "zoe_cuda_last_stats", "zoe_cuda_dpx_peak", "zoe_cuda_stream", "zoe_cuda_set_align_options", "zoe_cuda_set_width_policy",
    "zoe_cuda_sw_score_ranges_batch", "zoe_cuda_run_ranges_staged", "zoe_cuda_sw_align_3pass_batch",
    "zoe_cuda_run_3pass_staged", "zoe_cuda_sneaky_snake_batch", "zoe_cuda_set_memory_budget",
    "zoe_cuda_sw_score_both_strands_batch", "zoe_cuda_sw_score_ranges_both_strands_batch",
    "zoe_cuda_sw_align_both_strands_batch", "zoe_cuda_sw_align_3pass_both_strands_batch",
    "zoe_cuda_sw_score_best_hit_batch", "zoe_cuda_sw_align_best_hit_batch",
    "zoe_cuda_sw_score_paired_best_hit_batch", "zoe_cuda_sw_align_paired_best_hit_batch",
]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in
                ("pairs", "cells", "tier8", "tier16", "tier32", "overflowed", "unmapped", "rerun_wide", "hazard",
                 "window_fallback", "window_pinned", "tp_nogaps", "tp_banded", "tp_scalar", "tp_band_attempts")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


_lib = None


def load() -> C.CDLL:
    """Load the CUDA library; raises if it is missing (there is no fallback implementation)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m zoe_b200.build` (nvcc, sm_100a). "
            "zoe_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    p, u8p, u32p, u64p = C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)
    lib.zoe_cuda_create.argtypes = [C.POINTER(p), C.POINTER(C.c_int), C.c_int]
    lib.zoe_cuda_destroy.argtypes = [p]
    lib.zoe_cuda_destroy.restype = None
    lib.zoe_cuda_last_error.argtypes = [p]
    lib.zoe_cuda_last_error.restype = C.c_char_p
    lib.zoe_cuda_set_scoring.argtypes = [p, C.POINTER(C.c_int8), C.c_int, u8p, C.c_int8, C.c_int8, C.c_int]
    lib.zoe_cuda_set_lanes.argtypes = [p, C.c_int, C.c_int, C.c_int]
    lib.zoe_cuda_set_align_options.argtypes = [p, C.c_int, C.c_int, C.c_int]
    lib.zoe_cuda_set_width_policy.argtypes = [p, C.c_int, C.c_int, C.c_int]
    lib.zoe_cuda_set_memory_budget.argtypes = [p, C.c_uint64]
    lib.zoe_cuda_set_profiled.argtypes = [p, u8p, u64p, C.c_uint32]
    lib.zoe_cuda_sw_score_batch.argtypes = [p, u8p, u64p, C.c_uint64, u32p, u8p, u8p]
    lib.zoe_cuda_sw_align_batch.argtypes = [p, u8p, u64p, C.c_uint64, u32p, u8p, u8p, u32p, u32p, u32p, u32p, u32p,
                                            u64p, C.c_uint64, u8p]
    lib.zoe_cuda_sw_score_ranges_batch.argtypes = [p, u8p, u64p, C.c_uint64, u32p, u8p, u8p, u32p, u32p, u32p, u32p]
    lib.zoe_cuda_run_ranges_staged.argtypes = [p]
    lib.zoe_cuda_sw_align_3pass_batch.argtypes = [p, u8p, u64p, C.c_uint64, u32p, u8p, u8p, u32p, u32p, u32p, u32p, u32p,
                                                  u64p, C.c_uint64]
    lib.zoe_cuda_run_3pass_staged.argtypes = [p]
    lib.zoe_cuda_sw_score_both_strands_batch.argtypes = lib.zoe_cuda_sw_score_batch.argtypes + [u8p]
    lib.zoe_cuda_sw_score_ranges_both_strands_batch.argtypes = lib.zoe_cuda_sw_score_ranges_batch.argtypes + [u8p]
    lib.zoe_cuda_sw_align_both_strands_batch.argtypes = lib.zoe_cuda_sw_align_batch.argtypes + [u8p]
    lib.zoe_cuda_sw_align_3pass_both_strands_batch.argtypes = lib.zoe_cuda_sw_align_3pass_batch.argtypes + [u8p]
    lib.zoe_cuda_sw_score_best_hit_batch.argtypes = [p, u8p, u64p, C.c_uint64, C.c_int, u32p, u8p, u32p, u8p, u8p, u32p]
    lib.zoe_cuda_sw_align_best_hit_batch.argtypes = [p, u8p, u64p, C.c_uint64, C.c_int, C.c_int, u32p, u8p, u32p, u8p, u8p,
                                                     u32p, u32p, u32p, u32p, u32p, u32p, u64p, C.c_uint64, u8p]
    lib.zoe_cuda_sw_score_paired_best_hit_batch.argtypes = [p, u8p, u64p, u8p, u64p, C.c_uint64, u32p, u8p, u32p, u8p,
                                                            u8p, u32p]
    lib.zoe_cuda_sw_align_paired_best_hit_batch.argtypes = [p, u8p, u64p, u8p, u64p, C.c_uint64, C.c_int, C.c_uint32,
                                                            C.c_uint32, u32p, u8p, C.POINTER(C.c_int32), u8p, u32p, u8p,
                                                            u8p, u32p, u32p, u32p, u32p, u32p, u32p, u64p, C.c_uint64, u8p]
    lib.zoe_cuda_sneaky_snake_batch.argtypes = [p, u8p, u64p, u8p, u64p, C.c_uint64, C.c_float, u8p]
    lib.zoe_cuda_stage_streamed.argtypes = [p, u8p, u64p, C.c_uint64]
    lib.zoe_cuda_run_score_staged.argtypes = [p]
    lib.zoe_cuda_run_align_staged.argtypes = [p]
    lib.zoe_cuda_fetch_scores.argtypes = [p, u32p, u8p, u8p]
    lib.zoe_cuda_last_timing.argtypes = [p, C.POINTER(C.c_float), C.POINTER(C.c_float), u32p]
    lib.zoe_cuda_last_stats.argtypes = [p, C.POINTER(Stats)]
    lib.zoe_cuda_dpx_peak.argtypes = [p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_float)]
    lib.zoe_cuda_stream.argtypes = [p, C.c_int]
    lib.zoe_cuda_stream.restype = C.c_void_p
    _lib = lib
    return lib
