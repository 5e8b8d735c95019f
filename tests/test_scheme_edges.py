"""Scoring schemes at the edges of their domain, on every kernel path.

The C ABI takes any scheme with gap_init <= 0 and gap_extend <= 0: nothing requires same >= diff, same > 0 or
diff < 0.  Each fast path decides from bounds derived for the scheme whether it may run (16-bit batch kernels:
bias and eligibility in batch.cu launch_batch; packed strip cells: engine.cu packed_fits), so these tests run
schemes on both sides of those decisions -- diff > same, same == diff, same <= 0, positive mismatches, zero-cost
gaps, gap costs next to the 16-bit constant bound, and scores next to the top of a 16-bit half -- against the CPU
oracle (itself checked here against a plain Python DP) or against closed-form answers where the oracle is too slow.
"""
import itertools
import zlib

import numpy as np
import pytest

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
MODES = ("global", "semiglobal", "local")
NEG_INF = -(1 << 30)

# (same, diff, gap_init, gap_extend); gap_init == 0 means linear gaps of gap_extend
EDGE_SCHEMES = {
    "diff_gt_same_gotoh": (1, 3, -2, -1),
    "diff_gt_same_linear": (1, 3, 0, -1),
    "same_eq_diff": (2, 2, -1, -1),
    "same_zero": (0, -1, 0, -1),
    "same_negative": (-1, -3, -2, -1),
    "diff_positive_below_same": (3, 1, 0, -2),
    "zero_cost_gaps": (2, -1, 0, 0),
    "go_1999": (2, -1, -1000, -999),
    "go_2000": (2, -1, -1000, -1000),
}
SCHEME_IDS = list(EDGE_SCHEMES)


def _rand(rng, n, alphabet=ACGT):
    return alphabet[rng.integers(0, len(alphabet), n)]


def _related(rng, q, n, sub=0.05):
    s = np.resize(q, n).copy()
    k = max(1, n // int(1 / sub))
    s[rng.integers(0, n, k)] = _rand(rng, k)
    return s


def _scheme(sch):
    import anyseq_b200 as A
    return A.ScoringScheme(*sch)


def _local_refused(mode, sch):
    """the batch kernels refuse local alignment with positive mismatches (padding columns would outscore)"""
    return mode == "local" and sch[1] > 0


# --------------------------------------------------------------------------- plain reference
def py_dp(mode, q, s, same, diff, gi, ge):
    """Gotoh in Python ints, the recurrences and result extraction of the textbook oracle (gi = 0: linear gaps)"""
    m, n = len(q), len(s)
    glob, loc = mode == "global", mode == "local"
    H = [0] + [gi + j * ge if glob else 0 for j in range(1, n + 1)]
    F = [NEG_INF] * (n + 1)
    best_local, best_lastcol = -2147483647, H[n]
    for i in range(1, m + 1):
        cur = [gi + i * ge if glob else 0] + [0] * n
        E = NEG_INF
        for j in range(1, n + 1):
            E = max(E + ge, cur[j - 1] + gi + ge)
            F[j] = max(F[j] + ge, H[j] + gi + ge)
            v = max(H[j - 1] + (same if q[i - 1] == s[j - 1] else diff), E, F[j])
            if loc:
                v = max(v, 0)
            cur[j] = v
            best_local = max(best_local, v)
        best_lastcol = max(best_lastcol, cur[n])
        H = cur
    if glob:
        return H[n]
    if loc:
        return best_local
    return max([best_lastcol] + H)


def _oracle_score(oracle, mode, q, s, sch):
    """(score, end_i, end_j) of the restated reference"""
    same, diff, gi, ge = sch
    if gi == 0:
        return tuple(oracle.score_linear(mode, q, s, same, diff, ge, threads=8))
    return tuple(oracle.score_affine(mode, q, s, same, diff, gi, ge, threads=8))


def _textbook(oracle, mode, q, s, sch):
    same, diff, gi, ge = sch
    if gi == 0:
        return oracle.textbook_linear(mode, q, s, same, diff, ge)
    return oracle.textbook_affine(mode, q, s, same, diff, gi, ge)


def _column_score(oracle, aq, as_, sch):
    same, diff, gi, ge = sch
    return oracle.column_score(aq, as_, same, diff, ge) if gi == 0 else oracle.column_score_affine(aq, as_, same, diff, gi, ge)


def _small_pairs(rng):
    """every pair over {A, C} of up to 4 symbols, and random ACGT pairs of 0 - 12 symbols"""
    pairs = []
    words = [bytes(w) for L in range(5) for w in itertools.product(b"AC", repeat=L)]
    pairs += [(a, b) for a in words for b in words]
    for _ in range(300):
        pairs.append((bytes(_rand(rng, int(rng.integers(0, 13)))), bytes(_rand(rng, int(rng.integers(0, 13))))))
    return pairs


@pytest.mark.parametrize("name", SCHEME_IDS)
def test_oracle_equals_python_dp(oracle, name):
    """the oracle's scores (textbook and restated reference) on this scheme equal a plain Python DP; the global end
    cell is the last cell"""
    sch = EDGE_SCHEMES[name]
    rng = np.random.default_rng(sum(map(abs, sch)) + 1)
    for q, s in _small_pairs(rng):
        for mode in MODES:
            want = py_dp(mode, q, s, *sch)
            assert _textbook(oracle, mode, q, s, sch) == want, (mode, q, s)
            if q and s:
                got = _oracle_score(oracle, mode, q, s, sch)
                assert got[0] == want, (mode, q, s, got)
                if mode == "global":
                    assert got[1:] == (len(q) - 1, len(s) - 1)


@pytest.mark.parametrize("name", SCHEME_IDS)
def test_oracle_tracebacks_score_the_optimum(oracle, name):
    """the columns traceback_full emits score exactly the optimum in every mode; the linear-space tracebacks do so
    for global alignment (subjects longer than 64 symbols, below which the reference emits its quirk Q4 output)"""
    sch = EDGE_SCHEMES[name]
    same, diff, gi, ge = sch
    rng = np.random.default_rng(sum(map(abs, sch)) + 2)
    pairs = [(bytes(_rand(rng, int(rng.integers(1, 13)))), bytes(_rand(rng, int(rng.integers(1, 13))))) for _ in range(60)]
    for q, s in pairs:
        for mode in MODES:
            sc, aq, as_, st = oracle.traceback_full(mode, q, s, same, diff, gi, ge)
            assert sc == py_dp(mode, q, s, *sch)
            a = np.frombuffer(aq, np.uint8); b = np.frombuffer(as_, np.uint8)
            nonblank = int(((a != 32) | (b != 32)).sum())
            assert _column_score(oracle, aq, as_, sch) == sc or (nonblank == 0 and sc <= 0), (mode, q, s)
    for _ in range(6):
        q = _rand(rng, int(rng.integers(65, 140)))
        s = _related(rng, q, int(rng.integers(65, 160)), sub=0.2) if rng.random() < 0.5 else _rand(rng, int(rng.integers(65, 160)))
        opt = py_dp("global", bytes(q), bytes(s), *sch)
        if gi == 0:
            ret, aq, as_, _ = oracle.traceback_lintime("global", q, s, same, diff, ge)
        else:
            ret, aq, as_, _, _ = oracle.traceback_lintime_affine("global", q, s, same, diff, gi, ge)
        assert _column_score(oracle, aq, as_, sch) == opt


def test_closed_forms_equal_python_dp():
    """the closed forms the 600 kbp tests use: identical sequences score same * n; A^m vs A^n scores
    same * min(m, n) + gi + |m - n| * ge globally (gi = gap_init) and same * min(m, n) semiglobally"""
    for (same, diff, gi, ge) in ((9, -1, -2, -1), (19, -1, -2, -1)):
        for m, n in ((1, 1), (5, 5), (3, 11), (12, 4), (9, 10), (7, 1)):
            k = min(m, n)
            tail = gi + abs(m - n) * ge if m != n else 0
            assert py_dp("global", b"A" * m, b"A" * n, same, diff, gi, ge) == same * k + tail
            assert py_dp("semiglobal", b"A" * m, b"A" * n, same, diff, gi, ge) == same * k
            w = bytes(ACGT[np.random.default_rng(m * 13 + n).integers(0, 4, n)])
            assert py_dp("global", w, w, same, diff, gi, ge) == py_dp("semiglobal", w, w, same, diff, gi, ge) == same * n


# --------------------------------------------------------------------------- restated host decisions
def x2_bias(sch, max_long, max_short, large_alphabet=False):
    """batch.cu launch_batch: the bias of the 16-bit batch kernels for pairs of at most (max_long, max_short)
    symbols, or None when they are not eligible.  The largest cell is max(same, diff, 0) * min(rows, cols)."""
    same, diff, gi, ge = sch
    limit = 512 if large_alphabet else 1024
    if max_long <= limit:
        ncols, rows = max_long, max_short
    elif max_short <= limit:
        ncols, rows = max_short, max_long
    else:
        return None
    K = 4
    while 32 * K < ncols:
        K *= 2
    cols_pad = 32 * K
    go = gi + ge if gi != 0 else 0
    lowest = 2 * gi + (rows + cols_pad + 2) * ge + go + min(0, same, diff)
    hmax = max(same, diff, 0) * min(rows, cols_pad)
    b = -lowest + 8
    small = max(abs(same), abs(diff), abs(go), abs(ge))
    return b if b + hmax + 2 * small < 32000 and small < 2000 else None


def packed_fits(sch, K):
    """engine.cu packed_fits: the live window of a warp fits 16-bit halves around the centre"""
    same, diff, gi, ge = sch
    go = gi + ge
    if K not in (16, 32) or same < diff:
        return False
    D = max(same - go, -go)
    return D * (128 + 32 + 32 * K) + 4 * (abs(same) + abs(diff) + abs(go)) <= 0x3C00


def test_x2_bound_holds_for_positive_mismatches():
    """the 150 x 500 all-mismatch pair under (2, 300, 0, -1) scores 150 * 300 - 350 = 44650 globally, which no 16-bit
    half holds: the restated eligibility must refuse it, and for every scheme it accepts the largest cell it
    allows (bias + largest score) stays below 0x7fff"""
    assert py_dp("global", b"A" * 15, b"C" * 50, 2, 300, 0, -1) == 15 * 300 - 35
    assert x2_bias((2, 300, 0, -1), 500, 150) is None
    assert x2_bias((2, -1, -2, -1), 500, 150) is not None          # the reads workload keeps the 16-bit kernels
    for sch in EDGE_SCHEMES.values():
        for shape in ((500, 150), (1024, 1000), (128, 100)):
            b = x2_bias(sch, *shape)
            if b is not None:
                assert b + max(sch[0], sch[1], 0) * min(shape) < 0x7FFF


def test_packed_cells_bound_matches_the_planner():
    """the restated packed_fits and the launch planner put the bound at the same scheme: K = 32 strips (1024
    columns) take (9, -1, -2, -1) (D = 12) but not (10, -1, -2, -1); K = 16 strips take (19, -1, -2, -1) (D = 22)
    but not (20, -1, -2, -1); a scheme with diff > same never runs packed"""
    import anyseq_b200 as A
    for K, (lenq, lens), S in ((32, (4641652, 4600000), 9), (16, (1000000, 1000000), 19)):
        for mode in ("global", "semiglobal"):
            for same, fits in ((S, True), (S + 1, False)):
                sch = (same, -1, -2, -1)
                assert packed_fits(sch, K) is fits
                p = A.plan_launch(mode, lenq, lens, scheme=sch)
                assert p["cols_per_lane"] == K and p["packed_cells"] == int(fits), (K, mode, sch, p)
            for sch in EDGE_SCHEMES.values():
                if sch[2] != 0:
                    p = A.plan_launch(mode, lenq, lens, scheme=sch)
                    assert p["packed_cells"] == int(packed_fits(sch, p["cols_per_lane"])), (mode, sch, p)


# --------------------------------------------------------------------------- single-pair paths (GPU)
SCORE_SHAPES = [(1, 1), (7, 1), (2, 129), (33, 31), (100, 128), (100, 129), (300, 1025), (1000, 513), (129, 4096),
                (1500, 3000)]
# path -> (cols_per_lane, band_rows, options)
SCORE_PATHS = {
    "mask_k4": (4, 96, {}),
    "mask_k8": (8, 64, {}),
    "mask_k16": (16, 32, {}),
    "mask_k32": (32, 160, {}),
    "generic": (16, 0, {"force_generic": 1}),
    "mixed_cells": (16, 64, {"cell_form": 2}),
    "packed_cells_k16": (16, 0, {"packed_cells": 1}),
    "packed_cells_k32": (32, 64, {"packed_cells": 1}),
    "local_end_cell": (8, 0, {"local_end_cell": 1}),
}
OPTION_DEFAULTS = {"force_generic": 0, "cell_form": -1, "packed_cells": -1, "local_end_cell": 0,
                   "batch_packed": 1, "batch_quad": 1}


def _inputs(rng, m, n):
    q = _rand(rng, m)
    if min(m, n) > 50:
        return [(q, _related(rng, q, n)), (np.full(m, ord("A"), np.uint8), np.full(n, ord("C"), np.uint8))]
    return [(q, _rand(rng, n))]


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(SCORE_PATHS))
@pytest.mark.parametrize("name", SCHEME_IDS)
def test_score_paths(aligner, oracle, name, path):
    """score and end cell of every single-pair score path against the oracle (local: score, and the end cell with
    option local_end_cell)"""
    sch = EDGE_SCHEMES[name]
    K, band, opts = SCORE_PATHS[path]
    rng = np.random.default_rng(zlib.crc32(f"{name} {path}".encode()))
    aligner.tune(cols_per_lane=K, band_rows=band, watchdog_ms=10000)
    for k, v in opts.items():
        aligner.set_option(k, v)
    try:
        for (m, n) in SCORE_SHAPES:
            for q, s in _inputs(rng, m, n):
                for mode in MODES:
                    r = aligner.score(mode, q, s, _scheme(sch))
                    ref = _oracle_score(oracle, mode, q, s, sch)
                    if mode != "local" or path == "local_end_cell":
                        assert (r.score, r.end_i, r.end_j) == ref, (m, n, mode)
                    else:
                        assert r.score == ref[0], (m, n, mode)
    finally:
        aligner.tune(0, 0, 0, 10000)
        for k in opts:
            aligner.set_option(k, OPTION_DEFAULTS[k])


@pytest.mark.gpu
@pytest.mark.parametrize("name", SCHEME_IDS)
def test_align_linear_space(aligner, oracle, name):
    """linear-space traceback (linear and Gotoh gaps): strings, split rows and split types equal the oracle's"""
    same, diff, gi, ge = sch = EDGE_SCHEMES[name]
    rng = np.random.default_rng(11 + sum(map(abs, sch)))
    for (m, n) in [(300, 70), (1, 200), (200, 129), (1500, 2600)]:
        for q, s in _inputs(rng, m, n):
            for mode in MODES:
                r = aligner.align(mode, q, s, _scheme(sch))
                if gi == 0:
                    ret, aq, as_, sp = oracle.traceback_lintime(mode, q, s, same, diff, ge, threads=8)
                    ty = []
                else:
                    ret, aq, as_, sp, ty = oracle.traceback_lintime_affine(mode, q, s, same, diff, gi, ge, threads=8)
                    ty = ty.tolist()
                assert aligner.last_splits() == sp.tolist(), (m, n, mode)
                assert aligner.last_split_types() == ty, (m, n, mode)
                assert (r.aligned_query, r.aligned_subject) == (aq, as_), (m, n, mode)
                assert r.score == _oracle_score(oracle, mode, q, s, sch)[0], (m, n, mode)


@pytest.mark.gpu
@pytest.mark.parametrize("name", SCHEME_IDS)
def test_align_full(aligner, oracle, name):
    """full-matrix traceback: score, start cell and strings equal the oracle's"""
    same, diff, gi, ge = sch = EDGE_SCHEMES[name]
    rng = np.random.default_rng(13 + sum(map(abs, sch)))
    for (m, n) in [(1, 1), (1, 300), (300, 1), (127, 128), (200, 129), (129, 1100), (900, 700)]:
        for q, s in _inputs(rng, m, n):
            for mode in MODES:
                r = aligner.align_full(mode, q, s, _scheme(sch))
                sc, aq, as_, st = oracle.traceback_full(mode, q, s, same, diff, gi, ge)
                assert (r.score, r.start) == (sc, st), (m, n, mode)
                assert (r.aligned_query, r.aligned_subject) == (aq, as_), (m, n, mode)


def _pack(seqs):
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(x) for x in seqs])
    data = np.concatenate([np.asarray(x, dtype=np.uint8) for x in seqs]) if off[-1] else np.zeros(0, np.uint8)
    return data, off


@pytest.mark.gpu
@pytest.mark.parametrize("name", SCHEME_IDS)
def test_align_batch(aligner, oracle, name):
    """full-matrix tracebacks of a batch: score, end cell, start cell and strings of every pair equal the oracle's"""
    same, diff, gi, ge = sch = EDGE_SCHEMES[name]
    rng = np.random.default_rng(17 + sum(map(abs, sch)))
    pairs = []
    for (m, n) in [(0, 5), (1, 1), (150, 500), (33, 31), (100, 128), (700, 1024), (2, 513)]:
        pairs += _inputs(rng, m, n)
    qd, qo = _pack([p[0] for p in pairs]); sd, so = _pack([p[1] for p in pairs])
    for mode in MODES:
        b = aligner.align_batch(mode, qd, qo, sd, so, _scheme(sch))
        for p, (q, s) in enumerate(pairs):
            if len(q) == 0 or len(s) == 0:
                continue
            sc, aq, as_, st = oracle.traceback_full(mode, q, s, same, diff, gi, ge)
            ends = _oracle_score(oracle, mode, q, s, sch)[1:]
            got = (int(b.scores[p]), tuple(int(x) for x in b.ends[p]), tuple(int(x) for x in b.starts[p]), *b.alignment(p))
            assert got == (sc, ends, st, aq, as_), (mode, p, len(q), len(s))


# --------------------------------------------------------------------------- batch paths (GPU)
def _batch(rng, shape):
    """pairs of one shape (or a ragged mix): identical / prefix pairs and all-mismatch pairs reach the largest and
    the smallest cells, random and related pairs the rest; an odd count leaves a half-filled last item"""
    pairs = []
    if shape == "ragged":
        for p in range(61):
            lq, ls = int(rng.integers(0, 201)), int(rng.integers(0, 513))
            if p % 7 == 0:
                lq, ls = ls, lq
            pairs.append((lq, ls))
    else:
        pairs = [shape] * 23
    out = []
    for p, (lq, ls) in enumerate(pairs):
        kind = p % 4
        if kind == 0:                                   # the shorter one is a prefix of the longer one
            w = _rand(rng, max(lq, ls))
            q, s = w[:lq].copy(), w[:ls].copy()
        elif kind == 1:                                 # all mismatch
            q, s = np.full(lq, ord("A"), np.uint8), np.full(ls, ord("C"), np.uint8)
        elif kind == 2:
            q, s = _rand(rng, lq), _rand(rng, ls)
        else:
            q = _rand(rng, lq)
            s = _related(rng, q, ls, sub=0.1) if lq and ls else _rand(rng, ls)
        out.append((np.ascontiguousarray(q), np.ascontiguousarray(s)))
    return out


BATCH_SHAPES = {"150x500": (150, 500), "1000x1024": (1000, 1024), "100x128": (100, 128), "ragged": "ragged"}


def _packed2(pairs):
    """the arrays of an anyseq_packed_batch with explicit byte offsets and lengths, in field order (q2, s2, q_boff,
    s_boff, q_len, s_len)"""
    import anyseq_b200 as A
    qp = [A.pack2(p[0]).reshape(-1) if len(p[0]) else np.zeros(0, np.uint8) for p in pairs]
    sp = [A.pack2(p[1]).reshape(-1) if len(p[1]) else np.zeros(0, np.uint8) for p in pairs]
    q2 = np.concatenate(qp + [np.zeros(8, np.uint8)]); s2 = np.concatenate(sp + [np.zeros(8, np.uint8)])
    qb = np.concatenate([[0], np.cumsum([len(x) for x in qp])[:-1]]).astype(np.int64)
    sb = np.concatenate([[0], np.cumsum([len(x) for x in sp])[:-1]]).astype(np.int64)
    ql = np.array([len(p[0]) for p in pairs], np.int32); sl = np.array([len(p[1]) for p in pairs], np.int32)
    return q2, s2, qb, sb, ql, sl


def _packed_batch(addrs, npairs):
    from anyseq_b200 import capi
    return capi.PackedBatch(*addrs, 0, 0, 0, 0, npairs)


def _run_batch_paths(aligner, mode, pairs, sch):
    """scores of every batch path: {path: scores}"""
    import torch
    qd, qo = _pack([p[0] for p in pairs]); sd, so = _pack([p[1] for p in pairs])
    arrays = _packed2(pairs)
    dev = [torch.from_numpy(x).cuda() for x in arrays]
    got = {}
    try:
        for packed, quad in ((1, 1), (1, 0), (0, 1), (0, 0)):
            aligner.set_option("batch_packed", packed)
            aligner.set_option("batch_quad", quad)
            tag = f"packed={packed} quad={quad}"
            got["score_batch " + tag] = aligner.score_batch(mode, qd, qo, sd, so, _scheme(sch))[0].copy()
            out = np.full(len(pairs), -12345, np.int32)
            aligner.score_batch_packed2(mode, _packed_batch([a.ctypes.data for a in arrays], len(pairs)), out.ctypes.data,
                                        _scheme(sch))
            got["packed2 host " + tag] = out
            dsc = torch.full((len(pairs),), -12345, dtype=torch.int32, device="cuda")
            aligner.score_batch_packed2(mode, _packed_batch([t.data_ptr() for t in dev], len(pairs)), dsc.data_ptr(),
                                        _scheme(sch), device=True)
            got["packed2 device " + tag] = dsc.cpu().numpy()
    finally:
        aligner.set_option("batch_packed", 1)
        aligner.set_option("batch_quad", 1)
    return got


def _assert_batch_refused(aligner, mode, pairs, sch):
    import anyseq_b200 as A
    qd, qo = _pack([p[0] for p in pairs]); sd, so = _pack([p[1] for p in pairs])
    with pytest.raises(A.AnyseqError) as e:
        aligner.score_batch(mode, qd, qo, sd, so, _scheme(sch))
    assert e.value.code == -4 and "diff" in str(e.value)          # ANYSEQ_ERR_UNSUPPORTED, with the reason
    arrays = _packed2(pairs)
    out = np.zeros(len(pairs), np.int32)
    with pytest.raises(A.AnyseqError) as e:
        aligner.score_batch_packed2(mode, _packed_batch([a.ctypes.data for a in arrays], len(pairs)), out.ctypes.data,
                                    _scheme(sch))
    assert e.value.code == -4 and "diff" in str(e.value)


def _check_batch(aligner, oracle, mode, pairs, sch, tag):
    qd, qo = _pack([p[0] for p in pairs]); sd, so = _pack([p[1] for p in pairs])
    want = oracle.score_batch(mode, qd, qo, sd, so, *sch, threads=8)
    for path, got in _run_batch_paths(aligner, mode, pairs, sch).items():
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, (tag, mode, sch, path, [(int(p), len(pairs[p][0]), len(pairs[p][1]), int(got[p]),
                                                       int(want[p])) for p in bad[:3]])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(BATCH_SHAPES))
@pytest.mark.parametrize("name", SCHEME_IDS)
def test_batch_paths(aligner, oracle, name, shape):
    """score_batch (16-bit four and two pairs per warp, 32-bit) and score_batch_packed2 (host and device entry) against
    the oracle on every pair; local alignment with diff > 0 is refused with ANYSEQ_ERR_UNSUPPORTED"""
    sch = EDGE_SCHEMES[name]
    rng = np.random.default_rng(zlib.crc32(f"{name} {shape}".encode()))
    pairs = _batch(rng, BATCH_SHAPES[shape])
    for mode in MODES:
        if _local_refused(mode, sch):
            _assert_batch_refused(aligner, mode, pairs, sch)
        else:
            _check_batch(aligner, oracle, mode, pairs, sch, shape)


def _largest_eligible(make, max_long, max_short, lo=1, hi=40000):
    """the largest v in [lo, hi) with make(v) eligible for the 16-bit kernels (eligibility is monotone in v)"""
    assert x2_bias(make(lo), max_long, max_short) is not None
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if x2_bias(make(mid), max_long, max_short) is not None:
            lo = mid
        else:
            hi = mid
    return lo


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(150, 500), (1000, 1024), (100, 128)])
def test_batch_top_of_16_bit_range(aligner, oracle, shape):
    """on both sides of the eligibility bound of the 16-bit batch kernels: the largest `same` they take and one more
    and twice it (identical pairs: the largest cell is same * rows), the largest positive `diff` they take, one
    more and twice it (all-mismatch pairs: the largest cell is diff * rows); every path equals the oracle"""
    lq, ls = shape
    if shape == (1000, 1024):
        assert _largest_eligible(lambda v: (v, -1, -2, -1), ls, lq) == 29
    rng = np.random.default_rng(lq + ls)
    w = _rand(rng, ls)
    ident = [(w[:lq].copy(), w.copy()) for _ in range(5)] + [(_rand(rng, lq), _rand(rng, ls)) for _ in range(2)]
    mism = [(np.full(lq, ord("A"), np.uint8), np.full(ls, ord("C"), np.uint8)) for _ in range(5)] + ident[5:]
    for make, pairs, modes in ((lambda v: (v, -1, -2, -1), ident, MODES),
                               (lambda v: (v, -1, 0, -1), ident, MODES),
                               (lambda v: (1, v, -2, -1), mism, ("global", "semiglobal")),
                               (lambda v: (1, v, 0, -1), mism, ("global", "semiglobal"))):
        top = _largest_eligible(make, ls, lq)
        for v in (top, top + 1, 2 * top):
            sch = make(v)
            assert (x2_bias(sch, ls, lq) is None) == (v != top)
            for mode in modes:
                _check_batch(aligner, oracle, mode, pairs, sch, (shape, v))


@pytest.mark.gpu
def test_batch_positive_mismatches_beyond_16_bits(aligner, oracle):
    """(2, 300, 0, -1), 150 x 500 all-mismatch pairs: every mismatch scores 300, so the global score is
    150 * 300 - 350 = 44650, beyond any 16-bit half; the batch paths must not pick the 16-bit kernels for it"""
    sch = (2, 300, 0, -1)
    rng = np.random.default_rng(44650)
    pairs = [(np.full(150, ord("A"), np.uint8), np.full(500, ord("C"), np.uint8)) for _ in range(6)]
    pairs += [(_rand(rng, 150), _rand(rng, 500)) for _ in range(3)]
    assert _oracle_score(oracle, "global", pairs[0][0], pairs[0][1], sch)[0] == 44650
    for mode in ("global", "semiglobal"):
        _check_batch(aligner, oracle, mode, pairs, sch, "44650")


# --------------------------------------------------------------------------- packed strip cells at their bound (GPU)
def _stretch_inputs(rng, m, n):
    """inputs that stretch a warp's live window the most"""
    L = max(m, n)
    w = _rand(rng, L)
    return {
        "homopolymers": (np.full(m, ord("A"), np.uint8), np.full(n, ord("A"), np.uint8)),
        "identical": (w[:n].copy(), w[:n].copy()),
        "cliff": (w.copy(), np.concatenate([w[: L // 2], w[L // 2 + 3000:]])),     # 3 kbp deleted in the middle
        "mismatch": (np.full(m, ord("A"), np.uint8), np.full(n, ord("C"), np.uint8)),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("K", [16, 32])
def test_packed_cells_at_their_bound(aligner, oracle, K):
    """packed strip cells with the largest `same` that fits (and one more, which runs the 32-bit cells): homopolymers of
    different lengths, identical sequences, a 3 kbp deletion and all-mismatch pairs, global and semiglobal, ragged
    last strips, several bands, 1 - 3 warps per scheduler; equal to packed_cells = 0 and to the oracle"""
    S = 9 if K == 32 else 19
    rng = np.random.default_rng(K)
    SW = 32 * K
    sizes = [(5000, 6 * SW + SW // 3), (20011, 22 * SW + 3 * SW // 4 + 1)]
    try:
        for same in (S, S + 1):
            sch = (same, -1, -2, -1)
            assert packed_fits(sch, K) is (same == S)
            for (m, n) in sizes:
                for kind, (q, s) in _stretch_inputs(rng, m, n).items():
                    for mode in ("global", "semiglobal"):
                        ref = _oracle_score(oracle, mode, q, s, sch) if m < 10000 or same == S else None
                        for bps, band in ((1, 0), (2, 256), (3, 0)):
                            aligner.tune(cols_per_lane=K, band_rows=band, blocks_per_sm=bps, watchdog_ms=10000)
                            got = []
                            for packed in (1, 0):
                                aligner.set_option("packed_cells", packed)
                                r = aligner.score(mode, q, s, _scheme(sch))
                                got.append((r.score, r.end_i, r.end_j))
                            assert got[0] == got[1], (K, same, m, n, kind, mode, bps, band, got)
                            if ref is not None:
                                assert got[0] == ref, (K, same, m, n, kind, mode, bps, band, got, ref)
    finally:
        aligner.set_option("packed_cells", -1)
        aligner.tune(0, 0, 0, 10000)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [16, 32])
def test_packed_cells_large_closed_form(aligner, K):
    """600 kbp at the fitting edge scheme: identical sequences score same * n, A^m vs A^n scores
    same * min(m, n) + gi + |m - n| * ge globally and same * min(m, n) semiglobally; packed_cells = 0 gives the same
    score and end cell"""
    S = 9 if K == 32 else 19
    sch = (S, -1, -2, -1)
    rng = np.random.default_rng(600 + K)
    n = 600_000
    w = _rand(rng, n)
    m2 = n - 12_345
    cases = [("identical", w, w, S * n, S * n),
             ("homopolymers", np.full(m2, ord("A"), np.uint8), np.full(n, ord("A"), np.uint8),
              S * m2 + sch[2] + (n - m2) * sch[3], S * m2)]
    aligner.tune(cols_per_lane=K, watchdog_ms=10000)
    try:
        for kind, q, s, want_global, want_semi in cases:
            for mode, want in (("global", want_global), ("semiglobal", want_semi)):
                got = []
                for packed in (1, 0):
                    aligner.set_option("packed_cells", packed)
                    r = aligner.score(mode, q, s, _scheme(sch))
                    got.append((r.score, r.end_i, r.end_j))
                assert got[0][0] == want, (K, kind, mode, got, want)
                assert got[0] == got[1], (K, kind, mode, got)
                if mode == "global":
                    assert got[0][1:] == (len(q) - 1, len(s) - 1)
    finally:
        aligner.set_option("packed_cells", -1)
        aligner.tune(0, 0, 0, 10000)
