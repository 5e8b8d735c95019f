"""Host-side mirror of the reference's operator surface for the DP hot path.

Names follow the reference: alignment schemes ``global`` / ``semiglobal`` /
``local`` (src/align.impala:96-124), scoring schemes ``linear_scoring_scheme`` /
``affine_scoring_scheme`` (src/align.impala:144-166), operators ``score`` and
``traceback_lintime`` (src/align.impala:218-271) and the six exported entry
points of src/export.impala.  Everything executes in libanyseq_b200.so (CUDA,
sm_100a) through the C ABI of include/anyseq.h; nothing here computes a DP cell.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import capi
from .capi import AnyseqError, Result, Scoring, StripPartial, as_u8, make_scoring


@dataclass(frozen=True)
class ScoringScheme:
    same: int = 2
    diff: int = -1
    gap_init: int = 0       # 0 => linear gaps
    gap_extend: int = -1

    @property
    def affine(self) -> bool:
        return self.gap_init != 0


def linear_scoring_scheme(same: int = 2, diff: int = -1, gap: int = -1) -> ScoringScheme:
    """linear_scoring_scheme(same, diff, gap): src/align.impala:144-150."""
    return ScoringScheme(same, diff, 0, gap)


def affine_scoring_scheme(same: int = 2, diff: int = -1, gap_init: int = -2, gap_extend: int = -1) -> ScoringScheme:
    """affine_scoring_scheme(same, diff, gapInit, gapExtend): src/align.impala:153-166
    (parameter names only -- Gotoh as defined in DESIGN.md)."""
    return ScoringScheme(same, diff, gap_init, gap_extend)


REFERENCE_SCORING = linear_scoring_scheme(2, -1, -1)   # src/export.impala:14


@dataclass
class AlignmentResult:
    score: int
    end_i: int
    end_j: int
    kernel_ms: float
    kernel_launches: int
    aligned_query: bytes | None = None
    aligned_subject: bytes | None = None
    start: tuple | None = None       # full-matrix traceback: get_alignment_start()

    def cigar(self) -> str:
        if self.aligned_query is None:
            raise ValueError("no traceback in this result")
        return cigar(self.aligned_query, self.aligned_subject)


def cigar(aligned_query: bytes, aligned_subject: bytes) -> str:
    L = capi.load_library()
    a, b = as_u8(aligned_query), as_u8(aligned_subject)
    need = -L.anyseq_cigar(capi._ptr(a), capi._ptr(b), len(a), None, 0)
    buf = C.create_string_buffer(int(need))
    n = L.anyseq_cigar(capi._ptr(a), capi._ptr(b), len(a), buf, need)
    return buf.raw[:n].decode("ascii")


@dataclass
class BatchAlignment:
    """Full-matrix tracebacks of a batch (``Aligner.align_batch``): per pair p the score, end cell
    (get_score_pos()), start cell (get_alignment_start()) and aligned rows anyseq_align_full gives for it."""
    scores: np.ndarray              # (npairs,) int32
    ends: np.ndarray                # (npairs, 2) int32
    starts: np.ndarray              # (npairs, 2) int32
    aligned_query: np.ndarray       # uint8, pair p at offsets[p] .. offsets[p] + lq + ls
    aligned_subject: np.ndarray
    offsets: np.ndarray             # (npairs + 1,) int64: (q_off[p] - q_off[0]) + (s_off[p] - s_off[0])
    kernel_ms: float = 0.0
    kernel_launches: int = 0

    def alignment(self, p: int):
        """(aligned_query, aligned_subject) of pair p as bytes"""
        a, b = int(self.offsets[p]), int(self.offsets[p + 1])
        return self.aligned_query[a:b].tobytes(), self.aligned_subject[a:b].tobytes()

    def cigar(self, p: int) -> str:
        return cigar(*self.alignment(p))


class Aligner:
    """One engine per (process, GPU): wraps an ``anyseq_ctx``."""

    def __init__(self, device: int = -1):
        self._lib = capi.load_library()
        self._ctx = C.c_void_p()
        rc = self._lib.anyseq_ctx_create(device, C.byref(self._ctx))
        if rc != 0:
            raise AnyseqError(rc, self._err())

    def _err(self) -> str:
        m = self._lib.anyseq_last_error()
        return m.decode() if m else ""

    def _check(self, rc: int):
        if rc != 0:
            raise AnyseqError(rc, self._err())

    def close(self):
        if self._ctx:
            self._lib.anyseq_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._ctx

    def tune(self, cols_per_lane: int = 0, band_rows: int = 0, blocks_per_sm: int = 0, watchdog_ms: int = 0):
        self._check(self._lib.anyseq_ctx_tune(self._ctx, cols_per_lane, band_rows, blocks_per_sm, watchdog_ms))

    def set_option(self, name: str, value: int):
        self._check(self._lib.anyseq_ctx_set_option(self._ctx, name.encode(), int(value)))

    def device_info(self):
        sm, rw = C.c_int(), C.c_int()
        name = C.create_string_buffer(64)
        self._check(self._lib.anyseq_device_info(self._ctx, C.byref(sm), C.byref(rw), name))
        return {"sm_count": sm.value, "resident_warps": rw.value, "name": name.value.decode()}

    # -- score(): src/align.impala:218-235 ---------------------------------
    def score(self, mode, query, subject, scoring: ScoringScheme = REFERENCE_SCORING) -> AlignmentResult:
        q, s = as_u8(query), as_u8(subject)
        sc = make_scoring(mode, scoring.same, scoring.diff, scoring.gap_init, scoring.gap_extend)
        res = Result()
        self._check(self._lib.anyseq_score(self._ctx, C.byref(sc), capi._ptr(q), len(q), capi._ptr(s), len(s),
                                           C.byref(res)))
        return AlignmentResult(res.score, res.end_i, res.end_j, res.kernel_ms, res.kernel_launches)

    def score_device(self, mode, d_query: int, lenq: int, d_subject: int, lens: int,
                     scoring: ScoringScheme = REFERENCE_SCORING) -> AlignmentResult:
        """Sequences already resident in HBM (raw device pointers, e.g. tensor.data_ptr())."""
        sc = make_scoring(mode, scoring.same, scoring.diff, scoring.gap_init, scoring.gap_extend)
        res = Result()
        self._check(self._lib.anyseq_score_device(self._ctx, C.byref(sc), C.c_void_p(d_query), lenq,
                                                  C.c_void_p(d_subject), lens, C.byref(res)))
        return AlignmentResult(res.score, res.end_i, res.end_j, res.kernel_ms, res.kernel_launches)

    # -- traceback_lintime(): src/align.impala:237-271 ---------------------
    def align(self, mode, query, subject, scoring: ScoringScheme = REFERENCE_SCORING) -> AlignmentResult:
        q, s = as_u8(query), as_u8(subject)
        sc = make_scoring(mode, scoring.same, scoring.diff, scoring.gap_init, scoring.gap_extend)
        res = Result()
        n = len(q) + len(s)
        oq = np.zeros(max(n, 1), dtype=np.uint8)
        os_ = np.zeros(max(n, 1), dtype=np.uint8)
        self._check(self._lib.anyseq_align(self._ctx, C.byref(sc), capi._ptr(q), len(q), capi._ptr(s), len(s),
                                           capi._ptr(oq), capi._ptr(os_), C.byref(res)))
        return AlignmentResult(res.score, res.end_i, res.end_j, res.kernel_ms, res.kernel_launches,
                               oq[:n].tobytes(), os_[:n].tobytes())

    # -- traceback_full(): src/align.impala:190-216 ------------------------
    def align_full(self, mode, query, subject, scoring: ScoringScheme = REFERENCE_SCORING) -> AlignmentResult:
        """full predecessor matrix + one walk from get_score_pos(): exact semiglobal / local alignments;
        m*n/2 bytes of HBM (AnyseqError ANYSEQ_ERR_UNSUPPORTED when that does not fit)"""
        q, s = as_u8(query), as_u8(subject)
        sc = make_scoring(mode, scoring.same, scoring.diff, scoring.gap_init, scoring.gap_extend)
        res = Result()
        n = len(q) + len(s)
        oq = np.zeros(max(n, 1), dtype=np.uint8)
        os_ = np.zeros(max(n, 1), dtype=np.uint8)
        start = (C.c_int32 * 2)()
        self._check(self._lib.anyseq_align_full(self._ctx, C.byref(sc), capi._ptr(q), len(q), capi._ptr(s), len(s),
                                                capi._ptr(oq), capi._ptr(os_), C.byref(res), start))
        return AlignmentResult(res.score, res.end_i, res.end_j, res.kernel_ms, res.kernel_launches,
                               oq[:n].tobytes(), os_[:n].tobytes(), (int(start[0]), int(start[1])))

    def last_splits(self):
        """split rows of the last align() (slot -1 first), src/traceback_lintime.impala:9-42"""
        n = self._lib.anyseq_last_splits(self._ctx, None, 0)
        buf = (C.c_int32 * max(n, 1))()
        self._lib.anyseq_last_splits(self._ctx, buf, n)
        return list(buf[:n])

    def last_split_types(self):
        """Gotoh traceback: vertex type per split row (0 = H, 1 = E); empty for linear gaps"""
        n = self._lib.anyseq_last_split_types(self._ctx, None, 0)
        buf = (C.c_int32 * max(n, 1))()
        self._lib.anyseq_last_split_types(self._ctx, buf, n)
        return list(buf[:n])

    # -- batches of independent pairs --------------------------------------
    def score_batch(self, mode, queries, q_off, subjects, s_off, scoring: ScoringScheme = REFERENCE_SCORING):
        q, s = as_u8(queries), as_u8(subjects)
        qo = np.ascontiguousarray(q_off, dtype=np.int64)
        so = np.ascontiguousarray(s_off, dtype=np.int64)
        npairs = len(qo) - 1
        scores = np.zeros(max(npairs, 1), dtype=np.int32)
        sc = make_scoring(mode, scoring.same, scoring.diff, scoring.gap_init, scoring.gap_extend)
        res = Result()
        i64p = C.POINTER(C.c_int64)
        self._check(self._lib.anyseq_score_batch(self._ctx, C.byref(sc), capi._ptr(q), qo.ctypes.data_as(i64p),
                                                 capi._ptr(s), so.ctypes.data_as(i64p), npairs,
                                                 scores.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(res)))
        return scores[:npairs], AlignmentResult(res.score, -1, -1, res.kernel_ms, res.kernel_launches)

    def score_batch_device(self, mode, d_queries: int, d_q_off: int, d_subjects: int, d_s_off: int, npairs: int,
                           d_scores: int, scoring: ScoringScheme = REFERENCE_SCORING) -> AlignmentResult:
        sc = make_scoring(mode, scoring.same, scoring.diff, scoring.gap_init, scoring.gap_extend)
        res = Result()
        self._check(self._lib.anyseq_score_batch_device(self._ctx, C.byref(sc), C.c_void_p(d_queries),
                                                        C.c_void_p(d_q_off), C.c_void_p(d_subjects),
                                                        C.c_void_p(d_s_off), npairs, C.c_void_p(d_scores),
                                                        C.byref(res)))
        return AlignmentResult(res.score, -1, -1, res.kernel_ms, res.kernel_launches)

    # -- full-matrix tracebacks of batches (anyseq_align_batch) --------------
    def align_batch(self, mode, queries, q_off, subjects, s_off, scoring: ScoringScheme = REFERENCE_SCORING) -> BatchAlignment:
        """traceback_full of every pair (as align_full) in one launch; every subject <= 1024 symbols"""
        q, s = as_u8(queries), as_u8(subjects)
        qo = np.ascontiguousarray(q_off, dtype=np.int64)
        so = np.ascontiguousarray(s_off, dtype=np.int64)
        npairs = len(qo) - 1
        offsets = (qo - qo[0]) + (so - so[0])
        total = int(offsets[-1])
        scores = np.zeros(max(npairs, 1), dtype=np.int32)
        ends = np.zeros((max(npairs, 1), 2), dtype=np.int32)
        starts = np.zeros((max(npairs, 1), 2), dtype=np.int32)
        oq = np.zeros(max(total, 1), dtype=np.uint8)
        os_ = np.zeros(max(total, 1), dtype=np.uint8)
        sc = make_scoring(mode, scoring.same, scoring.diff, scoring.gap_init, scoring.gap_extend)
        res = Result()
        i64p = C.POINTER(C.c_int64)
        self._check(self._lib.anyseq_align_batch(self._ctx, C.byref(sc), capi._ptr(q), qo.ctypes.data_as(i64p),
                                                 capi._ptr(s), so.ctypes.data_as(i64p), npairs, capi._ptr(scores),
                                                 capi._ptr(ends), capi._ptr(starts), capi._ptr(oq), capi._ptr(os_),
                                                 C.byref(res)))
        return BatchAlignment(scores[:npairs], ends[:npairs], starts[:npairs], oq[:total], os_[:total], offsets,
                              res.kernel_ms, res.kernel_launches)

    def align_batch_device(self, mode, d_queries: int, d_q_off: int, d_subjects: int, d_s_off: int, npairs: int,
                           d_scores: int, d_ends: int, d_starts: int, d_aligned_query: int, d_aligned_subject: int,
                           scoring: ScoringScheme = REFERENCE_SCORING) -> AlignmentResult:
        """align_batch on device memory (raw pointers; d_ends / d_starts may be 0): the aligned rows of pair p start at
        (q_off[p] - q_off[0]) + (s_off[p] - s_off[0])"""
        sc = make_scoring(mode, scoring.same, scoring.diff, scoring.gap_init, scoring.gap_extend)
        res = Result()
        vp = C.c_void_p
        self._check(self._lib.anyseq_align_batch_device(self._ctx, C.byref(sc), vp(d_queries), vp(d_q_off),
                                                        vp(d_subjects), vp(d_s_off), npairs, vp(d_scores),
                                                        vp(d_ends or None), vp(d_starts or None), vp(d_aligned_query),
                                                        vp(d_aligned_subject), C.byref(res)))
        return AlignmentResult(res.score, -1, -1, res.kernel_ms, res.kernel_launches)

    # -- 2-bit packed DNA batches (anyseq_score_batch_packed2) -----------------
    def score_batch_packed2(self, mode, batch: "capi.PackedBatch", scores, scoring: ScoringScheme = REFERENCE_SCORING,
                            device: bool = False) -> AlignmentResult:
        """batch: capi.PackedBatch with host addresses (device=False: chunks are copied from the caller's memory under
        the kernels; pin the arrays for full H2D speed) or device addresses (device=True); scores: address of npairs
        int32 (host resp. device)"""
        sc = make_scoring(mode, scoring.same, scoring.diff, scoring.gap_init, scoring.gap_extend)
        res = Result()
        fn = self._lib.anyseq_score_batch_packed2_device if device else self._lib.anyseq_score_batch_packed2
        self._check(fn(self._ctx, C.byref(sc), C.byref(batch), C.c_void_p(int(scores)), C.byref(res)))
        return AlignmentResult(res.score, -1, -1, res.kernel_ms, res.kernel_launches)

    def batch_stream(self, mode, scoring: ScoringScheme = REFERENCE_SCORING, cap_pairs: int = 1 << 17,
                     cap_query_bytes: int = 32 << 20, cap_subject_bytes: int = 32 << 20, slots: int = 3) -> "BatchStream":
        return BatchStream(self, mode, scoring, cap_pairs, cap_query_bytes, cap_subject_bytes, slots)

    # -- roofline denominator ----------------------------------------------
    def measure_int_peak(self, kind: int = 0):
        ops, mhz = C.c_double(), C.c_float()
        self._check(self._lib.anyseq_measure_int_peak(self._ctx, kind, C.byref(ops), C.byref(mhz)))
        return ops.value, mhz.value


def plan_launch(mode, lenq: int, lens: int, affine: bool = False, sm_count: int = 148, chained: bool = False,
                scheme=None) -> dict:
    """The launch the engine makes for one lenq x lens score-only problem (``anyseq_plan_launch``): strip width, tile
    height, cell form, bands, grid, packed cells.  Host logic only -- works without a GPU.  ``scheme`` = (same, diff,
    gap_init, gap_extend) (``anyseq_plan_launch_scheme``; it decides packed_cells, and gap_init != 0 means affine);
    default: (2, -1, -2, -1), or (2, -1, 0, -1) with affine=False."""
    L = capi.load_library()
    plan = capi.LaunchPlan()
    m = capi.MODES[mode] if isinstance(mode, str) else int(mode)
    if scheme is None:
        rc = L.anyseq_plan_launch(int(sm_count), m, int(bool(affine)), int(lenq), int(lens), int(bool(chained)), C.byref(plan))
    else:
        same, diff, gap_init, gap_extend = (int(v) for v in scheme)
        sc = capi.Scoring(m, same, diff, gap_init, gap_extend)
        rc = L.anyseq_plan_launch_scheme(int(sm_count), C.byref(sc), int(lenq), int(lens), int(bool(chained)), C.byref(plan))
    if rc != 0:
        raise AnyseqError(rc, L.anyseq_last_error().decode())
    return {name: int(getattr(plan, name)) for name, _ in capi.LaunchPlan._fields_}


def pack2(seqs: np.ndarray) -> np.ndarray:
    """(npairs, L) uint8 array of A/C/G/T (either case) -> (npairs, ceil(L/4)) packed bytes: four symbols per byte, least
    significant bits first, every row starting on a byte boundary (the layout anyseq_score_batch_packed2 reads with
    stride = ceil(L/4)).  Vectorised equivalent of the C helper anyseq_pack2."""
    a = np.ascontiguousarray(seqs, dtype=np.uint8)
    if a.ndim == 1:
        a = a[None, :]
    lut = np.full(256, 255, dtype=np.uint8)
    for k, ch in enumerate(b"ACGT"):
        lut[ch] = k
        lut[ch + 32] = k
    codes = lut[a]
    if (codes == 255).any():
        raise ValueError("pack2: only A/C/G/T can be packed")
    L = a.shape[1]
    pad = (-L) % 4
    if pad:
        codes = np.concatenate([codes, np.zeros((a.shape[0], pad), dtype=np.uint8)], axis=1)
    c = codes.reshape(a.shape[0], -1, 4)
    return np.ascontiguousarray(c[:, :, 0] | (c[:, :, 1] << 2) | (c[:, :, 2] << 4) | (c[:, :, 3] << 6))


class BatchStream:
    """anyseq_batch_stream_*: one producer thread (acquire -> fill -> submit, finally finish) and one
    consumer thread (collect -> release) run concurrently; the ctypes calls drop the GIL.  Chunk buffers
    are pinned host memory owned by the stream, exposed as numpy views."""

    def __init__(self, aligner: Aligner, mode, scoring: ScoringScheme, cap_pairs: int, cap_query_bytes: int,
                 cap_subject_bytes: int, slots: int = 3):
        self._al, self._lib = aligner, aligner._lib
        sc = make_scoring(mode, scoring.same, scoring.diff, scoring.gap_init, scoring.gap_extend)
        self._h = C.c_void_p()
        aligner._check(self._lib.anyseq_batch_stream_open(aligner.handle, C.byref(sc), cap_pairs, cap_query_bytes,
                                                          cap_subject_bytes, slots, C.byref(self._h)))

    @staticmethod
    def _view(addr, n, dtype):
        if not addr or n <= 0:
            return np.zeros(0, dtype=dtype)
        buf = (C.c_char * (n * np.dtype(dtype).itemsize)).from_address(addr)
        return np.frombuffer(buf, dtype=dtype, count=n)

    def acquire(self):
        """-> (chunk, queries u8 view, q_off i64 view, subjects u8 view, s_off i64 view)"""
        c = capi.BatchChunk()
        self._al._check(self._lib.anyseq_batch_stream_acquire(self._h, C.byref(c)))
        return (c, self._view(c.queries, c.cap_query_bytes, np.uint8),
                self._view(C.cast(c.q_off, C.c_void_p).value, c.cap_pairs + 1, np.int64),
                self._view(c.subjects, c.cap_subject_bytes, np.uint8),
                self._view(C.cast(c.s_off, C.c_void_p).value, c.cap_pairs + 1, np.int64))

    def submit(self, chunk, npairs: int):
        chunk.npairs = npairs
        self._al._check(self._lib.anyseq_batch_stream_submit(self._h, C.byref(chunk)))

    def finish(self):
        self._al._check(self._lib.anyseq_batch_stream_finish(self._h))

    def collect(self):
        """-> (chunk, scores view valid until release) or None when every chunk has been collected"""
        c = capi.BatchChunk()
        rc = self._lib.anyseq_batch_stream_collect(self._h, C.byref(c))
        if rc == 1:
            return None
        self._al._check(rc)
        return c, self._view(C.cast(c.scores, C.c_void_p).value, c.npairs, np.int32)

    def release(self, chunk):
        self._al._check(self._lib.anyseq_batch_stream_release(self._h, C.byref(chunk)))

    def stats(self):
        res = Result()
        h2d, d2h = C.c_int64(), C.c_int64()
        self._al._check(self._lib.anyseq_batch_stream_stats(self._h, C.byref(res), C.byref(h2d), C.byref(d2h)))
        return {"kernel_ms": res.kernel_ms, "kernel_launches": res.kernel_launches, "h2d_bytes": h2d.value,
                "d2h_bytes": d2h.value}

    def close(self):
        if self._h:
            self._lib.anyseq_batch_stream_close(self._h)
            self._h = C.c_void_p()


_default: Aligner | None = None


def default_aligner() -> Aligner:
    global _default
    if _default is None:
        _default = Aligner(-1)
    return _default


# The six exported entry points (src/export.impala:5-147 / src/import.h:14-41),
# called through the very symbols a C host would link against.
def _legacy_score(name: str, query, subject) -> int:
    L = capi.load_library()
    q, s = as_u8(query), as_u8(subject)
    return int(getattr(L, name)(capi._ptr(q), len(q), capi._ptr(s), len(s)))


def _legacy_construct(name: str, query, subject):
    L = capi.load_library()
    q, s = as_u8(query), as_u8(subject)
    n = len(q) + len(s)
    oq = np.full(max(n, 1), ord(" "), dtype=np.uint8)
    os_ = np.full(max(n, 1), ord(" "), dtype=np.uint8)
    r = int(getattr(L, name)(capi._ptr(q), len(q), capi._ptr(s), len(s), capi._ptr(oq), capi._ptr(os_)))
    return r, oq[:n].tobytes(), os_[:n].tobytes()


def global_alignment_score(query, subject) -> int:
    return _legacy_score("global_alignment_score", query, subject)


def semiglobal_alignment_score(query, subject) -> int:
    return _legacy_score("semiglobal_alignment_score", query, subject)


def local_alignment_score(query, subject) -> int:
    return _legacy_score("local_alignment_score", query, subject)


def construct_global_alignment(query, subject):
    return _legacy_construct("construct_global_alignment", query, subject)


def construct_semiglobal_alignment(query, subject):
    return _legacy_construct("construct_semiglobal_alignment", query, subject)


def construct_local_alignment(query, subject):
    return _legacy_construct("construct_local_alignment", query, subject)
