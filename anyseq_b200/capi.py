"""ctypes binding of libanyseq_b200.so -- the C ABI declared in include/anyseq.h.

This is the host-side mirror of the reference's operator surface for the hot
path: the six legacy entry points of src/import.h:14-41 plus the parametrised
scheme surface (alignment scheme x scoring scheme, src/align.impala:96-166).
There is no CPU fallback: without the CUDA library / a GPU every call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ANYSEQ_LIB") or os.path.join(_HERE, "_build", "libanyseq_b200.so")   # ANYSEQ_LIB: kernel-variant experiments

GLOBAL, SEMIGLOBAL, LOCAL = 0, 1, 2
MODES = {"global": GLOBAL, "semiglobal": SEMIGLOBAL, "local": LOCAL}

# every symbol include/anyseq.h declares (checked by tests/test_abi.py)
EXPORTED_SYMBOLS = [
    "global_alignment_score", "semiglobal_alignment_score", "local_alignment_score",
    "construct_global_alignment", "construct_semiglobal_alignment", "construct_local_alignment",
    "construct_global_alignment_fulltb", "construct_semiglobal_alignment_fulltb", "construct_local_alignment_fulltb",
    "anyseq_align_full", "anyseq_align_sharded", "anyseq_align_batch", "anyseq_align_batch_device",
    "anyseq_ctx_create", "anyseq_ctx_destroy", "anyseq_last_error", "anyseq_ctx_tune", "anyseq_ctx_set_option",
    "anyseq_score", "anyseq_score_device", "anyseq_align", "anyseq_last_splits", "anyseq_last_split_types", "anyseq_cigar",
    "anyseq_score_batch", "anyseq_score_batch_device", "anyseq_score_batch_ends", "anyseq_score_batch_ends_device",
    "anyseq_score_batch_packed2", "anyseq_score_batch_packed2_device", "anyseq_pack2",
    "anyseq_score_batch_packed2_ends", "anyseq_score_batch_packed2_ends_device",
    "anyseq_batch_stream_open", "anyseq_batch_stream_open_ends", "anyseq_batch_stream_chunk_ends",
    "anyseq_batch_stream_acquire", "anyseq_batch_stream_submit", "anyseq_batch_stream_finish",
    "anyseq_batch_stream_collect", "anyseq_batch_stream_release", "anyseq_batch_stream_stats", "anyseq_batch_stream_close",
    "anyseq_strip_inbox_create", "anyseq_strip_inbox_open", "anyseq_strip_inbox_reset",
    "anyseq_strip_inbox_destroy", "anyseq_score_strip_device", "anyseq_score_strip", "anyseq_score_strip_device_multi", "anyseq_strip_combine",
    "anyseq_measure_int_peak", "anyseq_device_info", "anyseq_plan_launch", "anyseq_plan_launch_scheme",
]


class Scoring(C.Structure):
    _fields_ = [("mode", C.c_int32), ("same", C.c_int32), ("diff", C.c_int32),
                ("gap_init", C.c_int32), ("gap_extend", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("score", C.c_int64), ("end_i", C.c_int32), ("end_j", C.c_int32),
                ("kernel_ms", C.c_float), ("kernel_launches", C.c_int32)]


class LaunchPlan(C.Structure):
    _fields_ = [("cols_per_lane", C.c_int32), ("rows_per_step", C.c_int32), ("cell_form", C.c_int32), ("strips", C.c_int32),
                ("warps_per_scheduler", C.c_int32), ("bands", C.c_int32), ("band_rows", C.c_int32), ("grid", C.c_int32),
                ("warps_per_cta", C.c_int32), ("first_items", C.c_int64), ("packed_cells", C.c_int32)]


class StripPartial(C.Structure):
    _fields_ = [("row_best", C.c_int32), ("row_best_j", C.c_int32),
                ("col_best", C.c_int32), ("col_best_i", C.c_int32),
                ("local_best", C.c_int32), ("corner", C.c_int32),
                ("kernel_ms", C.c_float), ("kernel_launches", C.c_int32),
                ("lenq", C.c_int32), ("lens_total", C.c_int32)]


class PackedBatch(C.Structure):
    """anyseq_packed_batch: 2-bit packed DNA batch (host or device pointers as plain addresses)"""
    _fields_ = [("q2", C.c_void_p), ("s2", C.c_void_p), ("q_boff", C.c_void_p), ("s_boff", C.c_void_p),
                ("q_len", C.c_void_p), ("s_len", C.c_void_p),
                ("q_len_uniform", C.c_int32), ("s_len_uniform", C.c_int32),
                ("q_stride", C.c_int64), ("s_stride", C.c_int64), ("npairs", C.c_int64)]


class BatchChunk(C.Structure):
    _fields_ = [("queries", C.c_void_p), ("q_off", C.POINTER(C.c_int64)),
                ("subjects", C.c_void_p), ("s_off", C.POINTER(C.c_int64)),
                ("cap_pairs", C.c_int64), ("cap_query_bytes", C.c_int64), ("cap_subject_bytes", C.c_int64),
                ("npairs", C.c_int64), ("scores", C.POINTER(C.c_int32)),
                ("kernel_ms", C.c_float), ("slot", C.c_int32)]


# anyseq_bcast_fn: int (*)(void* user, void* d_buffer, int64_t nbytes, int src_rank)
BCAST_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int)


class AnyseqError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"anyseq_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load_library(path: str | None = None):
    """dlopen the CUDA library; raises if it has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise FileNotFoundError(
            f"{p} is missing: build it with `python -m anyseq_b200.build` (nvcc, sm_100a). "
            "anyseq_b200 has no CPU fallback.")
    L = C.CDLL(p)
    cp, vp, i64p = C.c_char_p, C.c_void_p, C.POINTER(C.c_int64)
    for name in ("global_alignment_score", "semiglobal_alignment_score", "local_alignment_score"):
        f = getattr(L, name)
        f.restype = C.c_int64
        f.argtypes = [vp, C.c_int, vp, C.c_int]
    for name in ("construct_global_alignment", "construct_semiglobal_alignment", "construct_local_alignment",
                 "construct_global_alignment_fulltb", "construct_semiglobal_alignment_fulltb",
                 "construct_local_alignment_fulltb"):
        f = getattr(L, name)
        f.restype = C.c_int64
        f.argtypes = [vp, C.c_int, vp, C.c_int, vp, vp]
    L.anyseq_ctx_create.restype = C.c_int
    L.anyseq_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.anyseq_ctx_destroy.restype = None
    L.anyseq_ctx_destroy.argtypes = [vp]
    L.anyseq_last_error.restype = cp
    L.anyseq_last_error.argtypes = []
    L.anyseq_ctx_tune.restype = C.c_int
    L.anyseq_ctx_tune.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int]
    L.anyseq_ctx_set_option.restype = C.c_int
    L.anyseq_ctx_set_option.argtypes = [vp, cp, C.c_int]
    L.anyseq_score.restype = C.c_int
    L.anyseq_score.argtypes = [vp, C.POINTER(Scoring), vp, C.c_int, vp, C.c_int, C.POINTER(Result)]
    L.anyseq_score_device.restype = C.c_int
    L.anyseq_score_device.argtypes = [vp, C.POINTER(Scoring), vp, C.c_int, vp, C.c_int, C.POINTER(Result)]
    L.anyseq_align.restype = C.c_int
    L.anyseq_align.argtypes = [vp, C.POINTER(Scoring), vp, C.c_int, vp, C.c_int, vp, vp, C.POINTER(Result)]
    L.anyseq_align_full.restype = C.c_int
    L.anyseq_align_full.argtypes = [vp, C.POINTER(Scoring), vp, C.c_int, vp, C.c_int, vp, vp, C.POINTER(Result),
                                    C.POINTER(C.c_int32)]
    L.anyseq_align_batch.restype = C.c_int
    L.anyseq_align_batch.argtypes = [vp, C.POINTER(Scoring), vp, i64p, vp, i64p, C.c_int64, vp, vp, vp, vp, vp,
                                     C.POINTER(Result)]
    L.anyseq_align_batch_device.restype = C.c_int
    L.anyseq_align_batch_device.argtypes = [vp, C.POINTER(Scoring), vp, vp, vp, vp, C.c_int64, vp, vp, vp, vp, vp,
                                            C.POINTER(Result)]
    L.anyseq_last_splits.restype = C.c_int
    L.anyseq_last_splits.argtypes = [vp, C.POINTER(C.c_int32), C.c_int]
    L.anyseq_last_split_types.restype = C.c_int
    L.anyseq_last_split_types.argtypes = [vp, C.POINTER(C.c_int32), C.c_int]
    L.anyseq_cigar.restype = C.c_int64
    L.anyseq_cigar.argtypes = [vp, vp, C.c_int64, vp, C.c_int64]
    L.anyseq_score_batch.restype = C.c_int
    L.anyseq_score_batch.argtypes = [vp, C.POINTER(Scoring), vp, i64p, vp, i64p, C.c_int64,
                                     C.POINTER(C.c_int32), C.POINTER(Result)]
    L.anyseq_score_batch_device.restype = C.c_int
    L.anyseq_score_batch_device.argtypes = [vp, C.POINTER(Scoring), vp, vp, vp, vp, C.c_int64, vp, C.POINTER(Result)]
    L.anyseq_score_batch_ends.restype = C.c_int
    L.anyseq_score_batch_ends.argtypes = [vp, C.POINTER(Scoring), vp, i64p, vp, i64p, C.c_int64,
                                          C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(Result)]
    L.anyseq_score_batch_ends_device.restype = C.c_int
    L.anyseq_score_batch_ends_device.argtypes = [vp, C.POINTER(Scoring), vp, vp, vp, vp, C.c_int64, vp, vp,
                                                 C.POINTER(Result)]
    L.anyseq_score_batch_packed2_ends.restype = C.c_int
    L.anyseq_score_batch_packed2_ends.argtypes = [vp, C.POINTER(Scoring), C.POINTER(PackedBatch), vp, vp, C.POINTER(Result)]
    L.anyseq_score_batch_packed2_ends_device.restype = C.c_int
    L.anyseq_score_batch_packed2_ends_device.argtypes = [vp, C.POINTER(Scoring), C.POINTER(PackedBatch), vp, vp,
                                                         C.POINTER(Result)]
    L.anyseq_score_batch_packed2.restype = C.c_int
    L.anyseq_score_batch_packed2.argtypes = [vp, C.POINTER(Scoring), C.POINTER(PackedBatch), vp, C.POINTER(Result)]
    L.anyseq_score_batch_packed2_device.restype = C.c_int
    L.anyseq_score_batch_packed2_device.argtypes = [vp, C.POINTER(Scoring), C.POINTER(PackedBatch), vp, C.POINTER(Result)]
    L.anyseq_pack2.restype = C.c_int64
    L.anyseq_pack2.argtypes = [vp, C.c_int64, vp]
    L.anyseq_batch_stream_open.restype = C.c_int
    L.anyseq_batch_stream_open.argtypes = [vp, C.POINTER(Scoring), C.c_int64, C.c_int64, C.c_int64, C.c_int, C.POINTER(vp)]
    L.anyseq_batch_stream_open_ends.restype = C.c_int
    L.anyseq_batch_stream_open_ends.argtypes = [vp, C.POINTER(Scoring), C.c_int64, C.c_int64, C.c_int64, C.c_int, C.POINTER(vp)]
    L.anyseq_batch_stream_chunk_ends.restype = C.POINTER(C.c_int32)
    L.anyseq_batch_stream_chunk_ends.argtypes = [vp, C.POINTER(BatchChunk)]
    for name in ("acquire", "submit", "collect", "release"):
        f = getattr(L, "anyseq_batch_stream_" + name)
        f.restype = C.c_int
        f.argtypes = [vp, C.POINTER(BatchChunk)]
    L.anyseq_batch_stream_finish.restype = C.c_int
    L.anyseq_batch_stream_finish.argtypes = [vp]
    L.anyseq_batch_stream_stats.restype = C.c_int
    L.anyseq_batch_stream_stats.argtypes = [vp, C.POINTER(Result), i64p, i64p]
    L.anyseq_batch_stream_close.restype = None
    L.anyseq_batch_stream_close.argtypes = [vp]
    L.anyseq_strip_inbox_create.restype = C.c_int
    L.anyseq_strip_inbox_create.argtypes = [vp, C.c_int, C.POINTER(vp), vp]
    L.anyseq_strip_inbox_open.restype = C.c_int
    L.anyseq_strip_inbox_open.argtypes = [vp, vp, C.c_int, C.POINTER(vp)]
    L.anyseq_strip_inbox_reset.restype = C.c_int
    L.anyseq_strip_inbox_reset.argtypes = [vp, vp]
    L.anyseq_strip_inbox_destroy.restype = None
    L.anyseq_strip_inbox_destroy.argtypes = [vp, vp]
    L.anyseq_score_strip_device.restype = C.c_int
    L.anyseq_score_strip_device.argtypes = [vp, C.POINTER(Scoring), vp, C.c_int, vp, C.c_int, C.c_int, C.c_int,
                                            vp, vp, C.POINTER(StripPartial)]
    L.anyseq_score_strip.restype = C.c_int
    L.anyseq_score_strip.argtypes = [vp, C.POINTER(Scoring), vp, C.c_int, vp, C.c_int, C.c_int, C.c_int,
                                     vp, vp, C.POINTER(StripPartial)]
    L.anyseq_score_strip_device_multi.restype = C.c_int
    L.anyseq_score_strip_device_multi.argtypes = [vp, C.POINTER(Scoring), C.c_int, C.POINTER(vp), C.c_int, C.POINTER(vp),
                                                  C.c_int, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(vp),
                                                  C.POINTER(StripPartial)]
    L.anyseq_strip_combine.restype = C.c_int
    L.anyseq_strip_combine.argtypes = [C.POINTER(Scoring), C.POINTER(StripPartial), C.c_int, C.POINTER(Result)]
    L.anyseq_align_sharded.restype = C.c_int
    L.anyseq_align_sharded.argtypes = [vp, C.POINTER(Scoring), vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, BCAST_FN, vp,
                                       vp, vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(Result)]
    L.anyseq_measure_int_peak.restype = C.c_int
    L.anyseq_measure_int_peak.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_float)]
    L.anyseq_device_info.restype = C.c_int
    L.anyseq_device_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), vp]
    L.anyseq_plan_launch.restype = C.c_int
    L.anyseq_plan_launch.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(LaunchPlan)]
    L.anyseq_plan_launch_scheme.restype = C.c_int
    L.anyseq_plan_launch_scheme.argtypes = [C.c_int, C.POINTER(Scoring), C.c_int, C.c_int, C.c_int, C.POINTER(LaunchPlan)]
    if path is None:
        _lib = L
    return L


def as_u8(a) -> np.ndarray:
    """bytes / str / ndarray -> contiguous uint8 array (raw bytes, no case folding:
    the reference compares symbols as bytes, src/align.impala:132)."""
    if isinstance(a, str):
        a = a.encode("latin-1")
    if isinstance(a, (bytes, bytearray, memoryview)):
        a = np.frombuffer(bytes(a), dtype=np.uint8)
    return np.ascontiguousarray(a, dtype=np.uint8)


def _ptr(a: np.ndarray):
    return C.c_void_p(a.ctypes.data if a.size else 0)


def make_scoring(mode, same=2, diff=-1, gap_init=0, gap_extend=-1) -> Scoring:
    """the C struct of a scheme; ctypes would silently wrap values outside int32 (2**32 + 5 stored as 5)"""
    m = MODES[mode] if isinstance(mode, str) else int(mode)
    vals = [int(v) for v in (same, diff, gap_init, gap_extend)]
    for name, v in zip(("same", "diff", "gap_init", "gap_extend"), vals):
        if not -2**31 <= v < 2**31:
            raise ValueError(f"scoring scheme: {name} = {v} is outside int32")
    return Scoring(m, *vals)
