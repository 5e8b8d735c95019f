"""Scores at the edge of the 32-bit cell range, on every entry point.

Cells are 32-bit and "minus infinity" is -2^30 (csrc/common.cuh), in the kernels and in the CPU oracle alike, so a
problem whose scores leave that range would agree with the oracle and still be wrong.  The reference here is an exact
int64 DP (checked against a Python-int DP without any sentinel).  Every entry point refuses a problem outside the range
check_score_range (csrc/engine.cu) defines -- restated once below as in_range -- and scores exactly at its edge: for
each direction the largest accepted parameter v is found by bisection; at v results equal the exact reference, v + 1
is refused with ANYSEQ_ERR_UNSUPPORTED, and the exact DP confirms that v sits at the edge.
"""
import zlib

import numpy as np
import pytest

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
MODES = ("global", "semiglobal", "local")
NEG = -(1 << 62)
HI_CELL, LO_CELL = 2**31 - 1, -2**30
WHOLE_GENOME = (4641652, 4600000)


# --------------------------------------------------------------------------- the rule (csrc/engine.cu check_score_range)
def in_range(mode, sch, m, n):
    """True when every H, E, F of an m x n problem under sch = (same, diff, gap_init, gap_extend) stays inside the
    32-bit cells: lo and hi bound every H, 4 P covers the additions a cell makes on top of them"""
    same, diff, gi, ge = sch
    P = max(abs(same), abs(diff), abs(gi), abs(ge))
    if P > 2**24:
        return False
    k, sigma = min(m, n), min(0, same, diff)
    hi = max(same, diff, 0) * k
    lo = {"global": max(2 * gi + (m + n) * ge, sigma * k + gi + (max(m, n) - 1) * ge),
          "semiglobal": max(sigma * k, gi + k * ge),
          "local": 0}[mode]
    return hi <= HI_CELL - 4 * P and lo >= LO_CELL + 4 * P


def largest(make, mode, m, n, lo=1, hi=2**31):
    """the largest v in [lo, hi) with make(v) in range (the rule is monotone in v)"""
    assert in_range(mode, make(lo), m, n) and not in_range(mode, make(hi), m, n)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if in_range(mode, make(mid), m, n):
            lo = mid
        else:
            hi = mid
    return lo


def at_the_edge(sch, exact):
    """the exact score or an extreme H is within 1 % of the limit the rule puts on it"""
    P = max(map(abs, sch))
    _, hmin, hmax = exact
    return hmax >= 0.99 * (HI_CELL - 4 * P) or hmin <= 0.99 * (LO_CELL + 4 * P)


# --------------------------------------------------------------------------- exact references
def py_exact(mode, q, s, same, diff, gi, ge):
    """Gotoh in Python ints with no sentinel (None = no gap open yet); gi = 0: linear gaps.  -> (score, min H, max H)
    over the cells of the matrix"""
    m, n = len(q), len(s)
    glob, loc = mode == "global", mode == "local"
    H = [0] + [gi + j * ge if glob else 0 for j in range(1, n + 1)]
    F = [None] * (n + 1)
    cells = []
    best_lastcol = H[n]
    for i in range(1, m + 1):
        cur = [gi + i * ge if glob else 0] + [0] * n
        E = None
        for j in range(1, n + 1):
            E = max(x for x in (None if E is None else E + ge, cur[j - 1] + gi + ge) if x is not None)
            F[j] = max(x for x in (None if F[j] is None else F[j] + ge, H[j] + gi + ge) if x is not None)
            v = max(H[j - 1] + (same if q[i - 1] == s[j - 1] else diff), E, F[j])
            cur[j] = max(v, 0) if loc else v
            cells.append(cur[j])
        best_lastcol = max(best_lastcol, cur[n])
        H = cur
    score = H[n] if glob else max(cells) if loc else max([best_lastcol] + H)
    return score, min(cells), max(cells)


def exact_dp(mode, q, s, same, diff, gi, ge):
    """py_exact in int64, one numpy pass per row.  gi <= 0, so opening a gap from an H that came from E never beats
    extending E: a row's E is a running maximum over Hd[k] + go + (j - 1 - k) ge, Hd = max(diagonal, F) (local: and 0)"""
    q, s = np.asarray(bytearray(bytes(q)), np.uint8), np.asarray(bytearray(bytes(s)), np.uint8)
    m, n = len(q), len(s)
    glob, loc = mode == "global", mode == "local"
    go = gi + ge
    kge = np.arange(n + 1, dtype=np.int64) * ge
    H = gi + kge if glob else np.zeros(n + 1, np.int64)
    H[0] = 0
    F = np.full(n + 1, NEG, np.int64)
    best_lastcol, best, hmin, hmax = int(H[n]), NEG, None, None
    for i in range(1, m + 1):
        sig = np.where(s == q[i - 1], same, diff).astype(np.int64)
        F[1:] = np.maximum(F[1:] + ge, H[1:] + go)
        Hd = np.empty(n + 1, np.int64)
        Hd[0] = gi + i * ge if glob else 0
        Hd[1:] = np.maximum(H[:-1] + sig, F[1:])
        if loc:
            Hd[1:] = np.maximum(Hd[1:], 0)
        E = np.maximum.accumulate(Hd[:-1] - kge[:-1]) + (go - ge) + kge[1:]
        H = Hd
        H[1:] = np.maximum(Hd[1:], E)
        lo_, hi_ = int(H[1:].min()), int(H[1:].max())
        hmin = lo_ if hmin is None else min(hmin, lo_)
        hmax = hi_ if hmax is None else max(hmax, hi_)
        best_lastcol, best = max(best_lastcol, int(H[n])), max(best, hi_)
    score = int(H[n]) if glob else best if loc else max(best_lastcol, int(H.max()))
    return score, hmin, hmax


def column_score(aq, as_, sch):
    """score of aligned rows in Python ints ('_' gap, ' ' blank column; a gap run costs gi + L ge)"""
    same, diff, gi, ge = sch
    t, run = 0, 0
    for a, b in zip(aq, as_):
        if a == 32 and b == 32:
            continue
        if a == 95:
            t += ge + (0 if run == 1 else gi); run = 1
        elif b == 95:
            t += ge + (0 if run == 2 else gi); run = 2
        else:
            t += same if a == b else diff; run = 0
    return t


# --------------------------------------------------------------------------- directions towards the edge
def _rand(rng, n):
    return ACGT[rng.integers(0, 4, n)]


def _pair(kind, rng, m, n):
    if kind == "identical":                        # the shorter one is a prefix of the longer one
        w = _rand(rng, max(m, n))
        return w[:m].copy(), w[:n].copy()
    return np.full(m, ord("A"), np.uint8), np.full(n, ord("C"), np.uint8)


def _gap_extend_max(gi, m, n):
    return largest(lambda v: (2, -1, gi, -v), "global", m, n)


# name -> (make(v, gi), pair kind, modes, single-pair shapes); gi is gap_init (0: linear gaps)
DIRECTIONS = {
    "same_up": (lambda v, gi, m, n: (v, -1, gi, -1), "identical", MODES, [(200, 300), (1000, 513), (1500, 3000)]),
    "diff_up": (lambda v, gi, m, n: (1, v, gi, -1), "mismatch", MODES, [(200, 300), (1000, 513), (1500, 3000)]),
    "gap_extend_down": (lambda v, gi, m, n: (2, -1, gi, -v), "mismatch", ("global",),
                        [(300, 2), (1000, 3), (3000, 70)]),
    "gap_init_down": (lambda v, gi, m, n: (2, -1, -v, -_gap_extend_max(-2, m, n)), "mismatch", ("global",),
                      [(300, 2), (1000, 3), (3000, 70)]),
    "semiglobal_sigma": (lambda v, gi, m, n: (2, -v, gi, -v), "mismatch", ("semiglobal",), [(200, 300), (1000, 513)]),
}
CASES = [(d, g) for d in DIRECTIONS for g in ("linear", "gotoh") if not (d == "gap_init_down" and g == "linear")]
CASE_IDS = [f"{d}-{g}" for d, g in CASES]


def _edge(direction, gaps, mode, m, n):
    """(scheme at v, scheme at v + 1)"""
    make = DIRECTIONS[direction][0]
    gi = 0 if gaps == "linear" else -2
    v = largest(lambda x: make(x, gi, m, n), mode, m, n, lo=2)
    return make(v, gi, m, n), make(v + 1, gi, m, n)


def _oracle_score(oracle, mode, q, s, sch):
    same, diff, gi, ge = sch
    if gi == 0:
        return tuple(oracle.score_linear(mode, q, s, same, diff, ge, threads=8))
    return tuple(oracle.score_affine(mode, q, s, same, diff, gi, ge, threads=8))


# --------------------------------------------------------------------------- CPU tests
EXTREME_SCHEMES = [(2, -1, -2, -1), (1, 3, -2, -1), (0, 0, 0, 0), (-5, -3, 0, -2), (2**29, -1, -2, -1),
                   (3, -2**28, -2**28, -2**28), (2, -1, -2, -4_000_000), (2**31 - 1, -2**31, -2**31, -2**31),
                   (-2**31, 2**31 - 1, 0, -1)]


def test_numpy_reference_equals_python_dp():
    """score, smallest and largest H of the row-vectorised int64 DP equal the plain Python-int DP on every pair over
    {A, C} up to 3 symbols and random pairs, under ordinary and extreme schemes"""
    import itertools
    rng = np.random.default_rng(7)
    words = [bytes(w) for L in range(1, 4) for w in itertools.product(b"AC", repeat=L)]
    pairs = [(a, b) for a in words for b in words]
    pairs += [(bytes(_rand(rng, int(rng.integers(1, 15)))), bytes(_rand(rng, int(rng.integers(1, 15))))) for _ in range(40)]
    pairs += [(b"A" * 30, b"C" * 2), (b"ACGT" * 3, b"A")]
    for sch in EXTREME_SCHEMES:
        for q, s in pairs:
            for mode in MODES:
                assert exact_dp(mode, q, s, *sch) == py_exact(mode, q, s, *sch), (sch, mode, q, s)


def test_exact_reference_sees_what_the_sentinel_hides():
    """the three cases the 32-bit sentinel gets wrong: A^300 vs C^2 scores -1 192 000 004 globally under
    (2, -1, -2, -4 000 000), below -2^30 without any overflow; and the rule refuses all three"""
    assert exact_dp("global", b"A" * 300, b"C" * 2, 2, -1, -2, -4_000_000)[0] == -1_192_000_004
    assert exact_dp("global", b"ACGT" * 3, b"A", 2, -1, -2, -2**28)[0] == -2_952_790_016
    for mode in MODES:
        assert exact_dp(mode, b"A" * 5, b"A" * 5, 2**29, -1, -2, -1)[0] == 5 * 2**29
    assert not in_range("global", (2, -1, -2, -4_000_000), 300, 2)
    assert not in_range("global", (2, -1, -2, -2**28), 12, 1)
    assert not any(in_range(mode, (2**29, -1, -2, -1), 5, 5) for mode in MODES)


@pytest.mark.parametrize("case", CASE_IDS)
def test_oracle_is_exact_inside_the_rule(oracle, case):
    """at the largest accepted parameter of each direction the CPU oracle (32-bit cells, -2^30 sentinel) still equals
    the exact reference, so its end cells and strings remain a valid reference up to the edge"""
    direction, gaps = CASES[CASE_IDS.index(case)]
    _, kind, modes, shapes = DIRECTIONS[direction]
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    for (m, n) in shapes:
        q, s = _pair(kind, rng, m, n)
        for mode in modes:
            sch, _ = _edge(direction, gaps, mode, m, n)
            ex = exact_dp(mode, q, s, *sch)
            assert at_the_edge(sch, ex), (mode, m, n, sch, ex)
            assert _oracle_score(oracle, mode, q, s, sch)[0] == ex[0], (mode, m, n, sch)


def _plan_accepts(mode, m, n, sch):
    import anyseq_b200 as A
    try:
        A.plan_launch(mode, m, n, scheme=sch)
    except A.AnyseqError as e:
        assert e.code == -4 and "32-bit cell range" in str(e), str(e)
        return False
    return True


def test_planner_applies_the_rule():
    """anyseq_plan_launch_scheme accepts and refuses exactly what the restated rule does, on both sides of every limit:
    P = 2^24 / 2^24 + 1, the hi limit (same, positive diff), the lo limit (gap_extend, gap_init, sigma * k), at small
    and whole-genome shapes"""
    probes = []
    for mode in MODES:
        for sch in ((2**24, -1, -2, -1), (2**24 + 1, -1, -2, -1), (2, -1, -2**24, -1), (2, -1, -2**24 - 1, -1),
                    (2, -2**24, 0, -2**24), (2, -2**24 - 1, 0, -1)):
            probes.append((mode, 1, 1, sch))
    shapes = [(300, 2), (200, 300), (1000, 513), (1500, 3000), WHOLE_GENOME, (1 << 21, 1 << 21)]
    for (m, n) in shapes:
        for mode in MODES:
            for gi in (0, -2):
                for make in (lambda v: (v, -1, gi, -1), lambda v: (1, v, gi, -1)):
                    v = largest(make, mode, m, n)
                    probes += [(mode, m, n, make(v)), (mode, m, n, make(v + 1))]
            if mode != "local":
                for gi in (0, -2):
                    for make in (lambda v: (2, -1, gi, -v), lambda v: (2, -v, gi, -v)):
                        v = largest(make, mode, m, n)
                        probes += [(mode, m, n, make(v)), (mode, m, n, make(v + 1))]
                ge = largest(lambda v: (2, -1, -2, -v), mode, m, n)
                v = largest(lambda v: (2, -1, -v, -ge), mode, m, n)
                probes += [(mode, m, n, (2, -1, -v, -ge)), (mode, m, n, (2, -1, -v - 1, -ge))]
    for mode, m, n, sch in probes:
        assert _plan_accepts(mode, m, n, sch) == in_range(mode, sch, m, n), (mode, m, n, sch)
    # the whole-genome figures: semiglobal / local take same <= 466, global |gap_extend| <= 230 under (2, -1, -2, ge)
    for mode in ("semiglobal", "local"):
        assert largest(lambda v: (v, -1, -2, -1), mode, *WHOLE_GENOME) == 466
    assert largest(lambda v: (2, -1, -2, -v), "global", *WHOLE_GENOME) == 230
    # the benchmark's scheme is far inside
    assert all(_plan_accepts(mode, *WHOLE_GENOME, (2, -1, -2, -1)) for mode in MODES)


def test_scheme_values_outside_int32_are_refused():
    """a scheme value outside int32 raises instead of being wrapped by ctypes (2^32 + 5 would be scored as 5)"""
    import anyseq_b200 as A
    from anyseq_b200 import capi
    for bad in ((2**31, -1, -2, -1), (2**32 + 5, -1, -2, -1), (2, -2**31 - 1, -2, -1), (2, -1, -2**32, -1),
                (2, -1, -2, -2**32 - 1)):
        with pytest.raises(ValueError, match="int32"):
            capi.make_scoring("global", *bad)
        with pytest.raises(ValueError, match="int32"):
            A.plan_launch("global", 10, 10, scheme=bad)
    sc = capi.make_scoring("local", 2**31 - 1, -2**31, -2**31, -2**31)
    assert (sc.same, sc.diff, sc.gap_init, sc.gap_extend) == (2**31 - 1, -2**31, -2**31, -2**31)


# --------------------------------------------------------------------------- GPU: single-pair score paths
# path -> (cols_per_lane, band_rows, options), as tests/test_scheme_edges.py runs them
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
OPTION_DEFAULTS = {"force_generic": 0, "cell_form": -1, "packed_cells": -1, "local_end_cell": 0}


def _scheme(sch):
    import anyseq_b200 as A
    return A.ScoringScheme(*sch)


def _assert_refused(fn):
    import anyseq_b200 as A
    with pytest.raises(A.AnyseqError) as e:
        fn()
    assert e.value.code == -4 and "32-bit cell range" in str(e.value), str(e.value)


def _edge_cases(case):
    """(mode, m, n, q, s, scheme at v, scheme at v + 1, exact at v) of every shape and mode of a direction"""
    direction, gaps = CASES[CASE_IDS.index(case)]
    _, kind, modes, shapes = DIRECTIONS[direction]
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    out = []
    for (m, n) in shapes:
        q, s = _pair(kind, rng, m, n)
        for mode in modes:
            sch, over = _edge(direction, gaps, mode, m, n)
            ex = exact_dp(mode, q, s, *sch)
            assert at_the_edge(sch, ex), (mode, m, n, sch, ex)
            out.append((mode, m, n, q, s, sch, over, ex))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASE_IDS)
def test_score_paths_at_the_edge(aligner, oracle, case):
    """every single-pair score path at v: the exact score, the oracle's end cell (local: with local_end_cell); at
    v + 1 every path refuses"""
    cases = _edge_cases(case)
    for path, (K, band, opts) in SCORE_PATHS.items():
        aligner.tune(cols_per_lane=K, band_rows=band, watchdog_ms=10000)
        for k, v in opts.items():
            aligner.set_option(k, v)
        try:
            for mode, m, n, q, s, sch, over, ex in cases:
                r = aligner.score(mode, q, s, _scheme(sch))
                assert r.score == ex[0], (path, mode, m, n, sch, r.score, ex)
                if mode != "local" or path == "local_end_cell":
                    assert (r.end_i, r.end_j) == _oracle_score(oracle, mode, q, s, sch)[1:], (path, mode, m, n)
                _assert_refused(lambda: aligner.score(mode, q, s, _scheme(over)))
        finally:
            aligner.tune(0, 0, 0, 10000)
            for k in opts:
                aligner.set_option(k, OPTION_DEFAULTS[k])


# --------------------------------------------------------------------------- GPU: tracebacks
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASE_IDS)
def test_tracebacks_at_the_edge(aligner, oracle, case):
    """align (linear space), align_full and align_batch at v: aligned rows equal the oracle's and score exactly the
    optimum in Python ints (align: global with subjects over 64 symbols; its score in every mode); v + 1 is refused by
    all three"""
    for mode, m, n, q, s, sch, over, ex in _edge_cases(case):
        same, diff, gi, ge = sch
        tag = (mode, m, n, sch)
        r = aligner.align(mode, q, s, _scheme(sch))
        if gi == 0:
            _, aq, as_, _ = oracle.traceback_lintime(mode, q, s, same, diff, ge, threads=8)
        else:
            _, aq, as_, _, _ = oracle.traceback_lintime_affine(mode, q, s, same, diff, gi, ge, threads=8)
        assert (r.aligned_query, r.aligned_subject) == (aq, as_), tag
        assert r.score == ex[0], tag
        if mode == "global" and n > 64:           # shorter subjects get the reference's quirk Q4 rows
            assert column_score(aq, as_, sch) == ex[0], tag
        r = aligner.align_full(mode, q, s, _scheme(sch))
        sc, aq, as_, st = oracle.traceback_full(mode, q, s, same, diff, gi, ge)
        assert (r.score, r.start, r.aligned_query, r.aligned_subject) == (ex[0], st, aq, as_), tag
        assert column_score(aq, as_, sch) == ex[0], tag
        if n <= 1024:
            qd, qo = _pack([q, q]); sd, so = _pack([s, s])
            b = aligner.align_batch(mode, qd, qo, sd, so, _scheme(sch))
            for p in range(2):
                assert (int(b.scores[p]), tuple(int(x) for x in b.starts[p]), *b.alignment(p)) == (ex[0], st, aq, as_), tag
            _assert_refused(lambda: aligner.align_batch(mode, qd, qo, sd, so, _scheme(over)))
        _assert_refused(lambda: aligner.align(mode, q, s, _scheme(over)))
        _assert_refused(lambda: aligner.align_full(mode, q, s, _scheme(over)))


# --------------------------------------------------------------------------- GPU: batch paths
def _pack(seqs):
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(x) for x in seqs])
    return np.concatenate([np.asarray(x, dtype=np.uint8) for x in seqs]), off


def _packed2(pairs):
    """the arrays of an anyseq_packed_batch with explicit byte offsets and lengths, in field order"""
    import anyseq_b200 as A
    qp = [A.pack2(p[0]).reshape(-1) for p in pairs]
    sp = [A.pack2(p[1]).reshape(-1) for p in pairs]
    q2 = np.concatenate(qp + [np.zeros(8, np.uint8)]); s2 = np.concatenate(sp + [np.zeros(8, np.uint8)])
    qb = np.concatenate([[0], np.cumsum([len(x) for x in qp])[:-1]]).astype(np.int64)
    sb = np.concatenate([[0], np.cumsum([len(x) for x in sp])[:-1]]).astype(np.int64)
    ql = np.array([len(p[0]) for p in pairs], np.int32); sl = np.array([len(p[1]) for p in pairs], np.int32)
    return q2, s2, qb, sb, ql, sl


def _batch_calls(aligner, mode, pairs, sch):
    """{path: call returning the scores} of score_batch (four batch_packed / batch_quad settings) and
    score_batch_packed2 (host and device entry)"""
    import torch
    from anyseq_b200 import capi
    qd, qo = _pack([p[0] for p in pairs]); sd, so = _pack([p[1] for p in pairs])
    arrays = _packed2(pairs)
    dev = [torch.from_numpy(x).cuda() for x in arrays]

    def batch(packed, quad):
        aligner.set_option("batch_packed", packed)
        aligner.set_option("batch_quad", quad)
        try:
            return aligner.score_batch(mode, qd, qo, sd, so, _scheme(sch))[0].copy()
        finally:
            aligner.set_option("batch_packed", 1)
            aligner.set_option("batch_quad", 1)

    def packed2_host():
        out = np.full(len(pairs), -12345, np.int32)
        aligner.score_batch_packed2(mode, capi.PackedBatch(*[a.ctypes.data for a in arrays], 0, 0, 0, 0, len(pairs)),
                                    out.ctypes.data, _scheme(sch))
        return out

    def packed2_device():
        out = torch.full((len(pairs),), -12345, dtype=torch.int32, device="cuda")
        aligner.score_batch_packed2(mode, capi.PackedBatch(*[t.data_ptr() for t in dev], 0, 0, 0, 0, len(pairs)),
                                    out.data_ptr(), _scheme(sch), device=True)
        return out.cpu().numpy()

    calls = {f"score_batch packed={p} quad={qd_}": (lambda p=p, qd_=qd_: batch(p, qd_)) for p in (1, 0) for qd_ in (1, 0)}
    calls["packed2 host"] = packed2_host
    calls["packed2 device"] = packed2_device
    return calls


def _chunk(aligner, mode, pairs, sch):
    """one chunk through a batch stream -> its scores"""
    bs = aligner.batch_stream(mode, _scheme(sch), cap_pairs=64, cap_query_bytes=1 << 16, cap_subject_bytes=1 << 16)
    try:
        c, qv, qo, sv, so = bs.acquire()
        qd, qoff = _pack([p[0] for p in pairs]); sd, soff = _pack([p[1] for p in pairs])
        qv[:len(qd)] = qd; sv[:len(sd)] = sd
        qo[:len(qoff)] = qoff; so[:len(soff)] = soff
        bs.submit(c, len(pairs))
        bs.finish()
        chunk, scores = bs.collect()
        out = scores.copy()
        bs.release(chunk)
        assert bs.collect() is None
        return out
    finally:
        bs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASE_IDS)
def test_batch_paths_at_the_edge(aligner, case):
    """score_batch under every batch_packed / batch_quad setting, score_batch_packed2 host and device, and one
    batch-stream chunk at v: every pair exact (the edge pair and random pairs of the same shape); at v + 1 each is
    refused -- the stream at collect, where the chunk's lengths are known.  Local alignment with diff > 0 is refused
    by the batch paths whatever the range, so it is not run here."""
    rng = np.random.default_rng(zlib.crc32(case.encode()) + 1)
    for mode, m, n, q, s, sch, over, ex in _edge_cases(case):
        if min(m, n) > 1024 or (mode == "local" and sch[1] > 0):
            continue
        pairs = [(q, s)] * 3 + [(_rand(rng, m), _rand(rng, n)) for _ in range(2)]
        want = np.array([ex[0]] * 3 + [exact_dp(mode, a, b, *sch)[0] for a, b in pairs[3:]], np.int64)
        for path, call in _batch_calls(aligner, mode, pairs, sch).items():
            got = call()
            assert got.tolist() == want.tolist(), (path, mode, m, n, sch)
        for path, call in _batch_calls(aligner, mode, pairs, over).items():
            _assert_refused(call)
        assert _chunk(aligner, mode, pairs, sch).tolist() == want.tolist(), (mode, m, n, sch)
        _assert_refused(lambda: _chunk(aligner, mode, pairs, over))


# --------------------------------------------------------------------------- GPU: slices of an out-of-range problem
@pytest.mark.gpu
def test_slices_of_an_out_of_range_problem_are_refused(aligner):
    """a narrow column slice can be in range while the whole problem is not: score_strip (one GPU) and align_sharded
    (world 1) judge the whole problem"""
    import anyseq_b200 as A
    from anyseq_b200.multigpu import ShardedTraceback, StripWavefront
    m, n_total, w = 300, 3000, 64
    v = largest(lambda x: (x, -1, -2, -1), "semiglobal", m, n_total)
    sch = (v + 1, -1, -2, -1)
    assert in_range("semiglobal", sch, m, w) and not in_range("semiglobal", sch, m, n_total)
    rng = np.random.default_rng(3000)
    q, s = _rand(rng, m), _rand(rng, n_total)
    wf = StripWavefront(aligner, 0, 1, rows=m)
    try:
        for col_begin in (0, 1024):
            _assert_refused(lambda: wf.run_host("semiglobal", A.ScoringScheme(*sch), q, s[col_begin:col_begin + w],
                                                col_begin, col_begin + w, n_total))
        wf.run_host("semiglobal", A.ScoringScheme(v, -1, -2, -1), q, s[:w], 0, w, n_total)
    finally:
        wf.close()
    over = _edge("gap_extend_down", "gotoh", "global", 300, 2)[1]
    tb = ShardedTraceback(aligner, 0, 1)
    _assert_refused(lambda: tb.align("global", b"A" * 300, b"C" * 2, A.ScoringScheme(*over)))
    _assert_refused(lambda: tb.align("semiglobal", q, s, A.ScoringScheme(*sch)))


# --------------------------------------------------------------------------- GPU: the default launch near INT_MAX
@pytest.mark.gpu
def test_large_closed_form_near_int_max(aligner):
    """2^21 identical symbols under (1023, -1, -2, -1) score 1023 * 2^21 = 2 145 386 496 globally and semiglobally
    through the planner's default launch (K = 32, several bands); same = 1024 is refused.  Global A^(n - d) vs A^n with
    the largest accepted |gap_extend| scores same * (n - d) + gi + d * ge exactly; one more is refused."""
    import anyseq_b200 as A
    n = 1 << 21
    sch = (1023, -1, -2, -1)
    w = _rand(np.random.default_rng(21), n)
    for mode in ("global", "semiglobal"):
        plan = A.plan_launch(mode, n, n, scheme=sch)
        assert plan["cols_per_lane"] == 32 and plan["bands"] > 1, plan
        r = aligner.score(mode, w, w, _scheme(sch))
        assert (r.score, r.end_i, r.end_j) == (2_145_386_496, n - 1, n - 1), (mode, r)
        assert not in_range(mode, (1024, -1, -2, -1), n, n)
        _assert_refused(lambda: aligner.score(mode, w, w, _scheme((1024, -1, -2, -1))))
    d = 12_345
    ge = largest(lambda v: (1023, -1, -2, -v), "global", n - d, n)
    sch = (1023, -1, -2, -ge)
    q, s = np.full(n - d, ord("A"), np.uint8), np.full(n, ord("A"), np.uint8)
    r = aligner.score("global", q, s, _scheme(sch))
    assert r.score == 1023 * (n - d) - 2 - d * ge, (ge, r)
    _assert_refused(lambda: aligner.score("global", q, s, _scheme((1023, -1, -2, -ge - 1))))
