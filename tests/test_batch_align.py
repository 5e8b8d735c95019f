"""Full-matrix tracebacks of batches (anyseq_align_batch): every pair must give exactly what anyseq_align_full and
oracle.traceback_full give for it alone -- score, end cell, start cell and both aligned rows."""
import ctypes as C
import hashlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
MODES = ("global", "semiglobal", "local")
SCHEMES = ((2, -1, 0, -1), (2, -1, -2, -1), (3, -2, 0, -4), (5, -4, -10, -1), (1, -1, -1, 0))
SUBJECT_LENS = (0, 1, 31, 32, 33, 127, 128, 129, 255, 256, 257, 511, 512, 513, 1023, 1024)
QUERY_LENS = (0, 1, 2, 33, 150, 700, 2100)


def _scheme(t):
    import anyseq_b200 as A
    return A.ScoringScheme(*t)


def _rand(rng, n, alphabet=ACGT):
    return alphabet[rng.integers(0, len(alphabet), n)]


def _pair(rng, kind, m, n, alphabet=ACGT):
    q = _rand(rng, m, alphabet)
    if kind == 0 or m == 0:                                     # random
        s = _rand(rng, n, alphabet)
    elif kind == 1:                                             # related: a mutated copy
        s = np.resize(q, n).copy()
        k = max(1, n // 20)
        s[rng.integers(0, max(n, 1), k)[: n]] = _rand(rng, min(k, n), alphabet)
    elif kind == 2:                                             # all mismatch
        q = np.full(m, alphabet[0], np.uint8)
        s = np.full(n, alphabet[1], np.uint8)
    else:                                                       # planted overlap: the query's prefix ends the subject
        h = min(m, n) // 2
        s = np.concatenate([_rand(rng, n - h, alphabet), q[:h]])
    return np.ascontiguousarray(q, np.uint8), np.ascontiguousarray(s[:n], np.uint8)


def _pack(pairs, pad_q=0, pad_s=0):
    """queries / subjects back to back after pad_q / pad_s unused bytes (offsets then start there)"""
    qs = [np.full(pad_q, 7, np.uint8)] + [p[0] for p in pairs]
    ss = [np.full(pad_s, 9, np.uint8)] + [p[1] for p in pairs]
    qo = np.cumsum([0, pad_q] + [len(p[0]) for p in pairs])[1:].astype(np.int64)
    so = np.cumsum([0, pad_s] + [len(p[1]) for p in pairs])[1:].astype(np.int64)
    return np.concatenate(qs), qo, np.concatenate(ss), so


def _oracle(oracle, mode, q, s, sch):
    same, diff, gi, ge = sch
    sc, aq, as_, st = oracle.traceback_full(mode, q, s, same, diff, gi, ge)
    if gi == 0:
        _, ei, ej = oracle.score_linear(mode, q, s, same, diff, ge)
    else:
        _, ei, ej = oracle.score_affine(mode, q, s, same, diff, gi, ge)
    return sc, (ei, ej), st, aq, as_


def _got(b, p):
    aq, as_ = b.alignment(p)
    return int(b.scores[p]), tuple(int(x) for x in b.ends[p]), tuple(int(x) for x in b.starts[p]), aq, as_


def _full(aligner, mode, q, s, sch):
    r = aligner.align_full(mode, q, s, sch)
    return r.score, (r.end_i, r.end_j), r.start, r.aligned_query, r.aligned_subject


def _sha(aq, as_):
    return hashlib.sha256(aq + b"\n" + as_).hexdigest()[:16]


# --------------------------------------------------------------------------- 1. oracle parity, every K
@pytest.mark.parametrize("sch", SCHEMES)
def test_batch_align_vs_oracle(aligner, oracle, sch):
    """ragged pairs over every subject length boundary of K = 4, 8, 16, 32 (32K - 1, 32K, 32K + 1) and queries of 0, 1,
    2, 33 (past the 32-row lane skew), 150, 700 and 2100 rows; one batch per K (longest subject <= 32 K)"""
    rng = np.random.default_rng(sum(abs(x) for x in sch))
    pairs = []
    for a, n in enumerate(SUBJECT_LENS):
        for b, m in enumerate(QUERY_LENS):
            pairs.append(_pair(rng, (a + b) % 4, m, n))
    ref = {}
    for mode in MODES:
        for K in (4, 8, 16, 32):
            idx = [k for k, (q, s) in enumerate(pairs) if len(s) <= 32 * K]
            sub = [pairs[k] for k in idx]
            b = aligner.align_batch(mode, *_pack(sub), _scheme(sch))
            for p, k in enumerate(idx):
                q, s = pairs[k]
                if len(q) == 0 or len(s) == 0:               # degenerate results are anyseq_align_full's
                    want = _full(aligner, mode, q, s, _scheme(sch))
                else:
                    if (mode, k) not in ref:
                        ref[(mode, k)] = _oracle(oracle, mode, q, s, sch)
                    want = ref[(mode, k)]
                assert _got(b, p) == want, (mode, sch, K, len(q), len(s), k % 4)


# --------------------------------------------------------------------------- 2. equality with align_full
@pytest.mark.parametrize("alphabet", ["bytes256", "alpha24_31", "local_diff_positive"])
def test_batch_align_equals_align_full(aligner, oracle, alphabet):
    rng = np.random.default_rng(len(alphabet))
    if alphabet == "bytes256":
        alpha = np.arange(256, dtype=np.uint8)
        schemes, modes = ((2, -1, 0, -1), (2, -1, -2, -1)), MODES
    elif alphabet == "alpha24_31":
        alpha = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWYBZX*_#@", dtype=np.uint8)[: int(rng.integers(24, 32))]
        schemes, modes = ((5, -4, -10, -1), (3, -2, 0, -4)), MODES
    else:
        alpha = ACGT
        schemes, modes = ((2, 1, 0, -1), (3, 1, -2, -1)), ("local",)
    pairs = [_pair(rng, k % 4, int(rng.integers(0, 400)), int(rng.integers(0, 1025)), alpha) for k in range(40)]
    pairs += [_pair(rng, 1, 1024, 1024, alpha), _pair(rng, 3, 1, 700, alpha), _pair(rng, 0, 33, 1, alpha)]
    for mode in modes:
        for sch in schemes:
            b = aligner.align_batch(mode, *_pack(pairs), _scheme(sch))
            for p, (q, s) in enumerate(pairs):
                got = _got(b, p)
                assert got == _full(aligner, mode, q, s, _scheme(sch)), (alphabet, mode, sch, p)
                if alphabet == "local_diff_positive" and len(q) and len(s):
                    assert got == _oracle(oracle, mode, q, s, sch), (mode, sch, p)


# --------------------------------------------------------------------------- 3. frozen fixtures
def test_batch_align_golden_fixtures(aligner, golden):
    cases = [c for c in golden["cases"] if len(c["s"].encode("latin-1")) <= 1024]
    assert len(cases) == 11 and any(c["name"] == "bytes" for c in cases)
    pairs = [(np.frombuffer(c["q"].encode("latin-1"), np.uint8), np.frombuffer(c["s"].encode("latin-1"), np.uint8))
             for c in cases]
    for mode in MODES:
        for sch, key in (((2, -1, 0, -1), None), ((2, -1, -2, -1), "affine")):
            b = aligner.align_batch(mode, *_pack(pairs), _scheme(sch))
            for p, c in enumerate(cases):
                t = c["traceback_full"][mode]
                t = t[key] if key else t
                aq, as_ = b.alignment(p)
                assert (int(b.scores[p]), [int(x) for x in b.starts[p]], _sha(aq, as_)) == \
                    (t["score"], t["start"], t["sha"]), (c["name"], mode, key)


# --------------------------------------------------------------------------- 4. planted ties
def test_batch_align_planted_ties(aligner, oracle):
    """local: equal maxima in two rows and two columns (one of them in row >= 1024) -- the first in row-major order
    wins; semiglobal: equal maxima on the last row and on the last column"""
    rng = np.random.default_rng(11)
    X = _rand(rng, 20)
    N = lambda k: np.full(k, ord("N"), np.uint8)           # noqa: E731  (matches nothing in X or M)
    M = lambda k: np.full(k, ord("M"), np.uint8)           # noqa: E731
    cat = lambda *a: np.ascontiguousarray(np.concatenate(a), np.uint8)   # noqa: E731
    local = [
        (cat(X, N(1100), X), cat(X, M(200), X)),            # rows 19 / 1139, columns 19 / 239
        (cat(N(1030), X, N(40), X), cat(M(100), X, M(300), X)),   # both rows >= 1024
        (cat(N(1030), X), cat(X, M(10), X)),                # one row >= 1024, two columns
        (cat(N(5), X, N(1040), X), cat(X, M(3))),           # two rows, one column, the second >= 1024
    ]
    semi = [
        (X.copy(), cat(X, M(50), X, M(20))),                # last row: two equal maxima
        (cat(X, N(50), X, N(10)), X.copy()),                # last column: two equal maxima
        (cat(X, N(30)), cat(M(30), X)),                     # last row vs last column
        (cat(N(3), X), cat(X, M(3))),
    ]
    for mode, pairs in (("local", local), ("semiglobal", semi)):
        for sch in ((2, -1, 0, -1), (2, -1, -2, -1), (1, -1, -1, 0)):
            b = aligner.align_batch(mode, *_pack(pairs), _scheme(sch))
            for p, (q, s) in enumerate(pairs):
                want = _oracle(oracle, mode, q, s, sch)
                assert _got(b, p) == want, (mode, sch, p)
                assert _got(b, p) == _full(aligner, mode, q, s, _scheme(sch)), (mode, sch, p)


# --------------------------------------------------------------------------- 5. scale
@pytest.mark.parametrize("mode,sch", [("semiglobal", (2, -1, -2, -1)), ("local", (2, -1, 0, -1))])
def test_batch_align_reads_vs_windows_at_scale(aligner, oracle, mode, sch):
    import torch
    from anyseq_b200 import workloads as W
    npairs, lq, ls = 100_000, 150, 500
    qd, qo, sd, so = W.read_batch(npairs, lq, ls, seed=5)
    b = aligner.align_batch(mode, qd, qo, sd, so, _scheme(sch))
    dq, dqo, ds, dso = (torch.from_numpy(x).cuda() for x in (qd, qo, sd, so))
    out = torch.zeros(npairs, dtype=torch.int32, device="cuda")
    aligner.score_batch_device(mode, dq.data_ptr(), dqo.data_ptr(), ds.data_ptr(), dso.data_ptr(), npairs,
                               out.data_ptr(), _scheme(sch))
    assert np.array_equal(b.scores, out.cpu().numpy())

    # every alignment: column score == score, de-gapped rows are the sequences from the start cell to the end cell
    same, diff, gi, ge = sch
    L = lq + ls
    aq = b.aligned_query.reshape(npairs, L)
    as_ = b.aligned_subject.reshape(npairs, L)
    blank = (aq == 32) & (as_ == 32)
    assert not ((aq == 32) ^ (as_ == 32)).any()
    gq, gs = aq == 95, as_ == 95
    sub = np.where(aq == as_, same, diff) * ~(gq | gs | blank)
    runs = (gq[:, 1:] & ~gq[:, :-1]).sum(1) + gq[:, 0] + (gs[:, 1:] & ~gs[:, :-1]).sum(1) + gs[:, 0]
    col = sub.sum(1) + ge * (gq.sum(1) + gs.sum(1)) + gi * runs
    assert np.array_equal(col, b.scores)
    for rows, gaps, seqs, k, n in ((aq, gq, qd.reshape(npairs, lq), 0, lq), (as_, gs, sd.reshape(npairs, ls), 1, ls)):
        sym = ~gaps & ~blank
        cnt = sym.sum(1)
        assert np.array_equal(b.starts[:, k] + cnt, b.ends[:, k] + 1)
        idx = np.clip(b.starts[:, k:k + 1] + np.cumsum(sym, 1) - 1, 0, n - 1)
        want = np.take_along_axis(seqs, idx, 1)
        assert (np.where(sym, rows, 0) == np.where(sym, want, 0)).all()
    qs, ss = qd.reshape(npairs, lq), sd.reshape(npairs, ls)
    for p in np.random.default_rng(1).choice(npairs, 2000, replace=False):
        assert _got(b, int(p)) == _oracle(oracle, mode, qs[p], ss[p], sch), (mode, int(p))


# --------------------------------------------------------------------------- 6. host == device variant
def test_batch_align_host_equals_device(aligner):
    import torch
    import anyseq_b200 as A
    rng = np.random.default_rng(6)
    pairs = [_pair(rng, k % 4, int(rng.integers(0, 300)), int(rng.integers(0, 600))) for k in range(300)]
    pairs[7] = (pairs[7][0][:0], pairs[7][1])
    pairs[8] = (pairs[8][0], pairs[8][1][:0])
    qd, qo, sd, so = _pack(pairs, pad_q=13, pad_s=5)           # q_off[0] = 13, s_off[0] = 5
    sch = _scheme((2, -1, -2, -1))
    for mode in MODES:
        b = aligner.align_batch(mode, qd, qo, sd, so, sch)
        total = int(b.offsets[-1])
        dq, dqo, ds, dso = (torch.from_numpy(x).cuda() for x in (qd, qo, sd, so))
        sc = torch.zeros(len(pairs), dtype=torch.int32, device="cuda")
        en = torch.zeros(2 * len(pairs), dtype=torch.int32, device="cuda")
        st = torch.zeros(2 * len(pairs), dtype=torch.int32, device="cuda")
        oq = torch.zeros(total, dtype=torch.uint8, device="cuda")
        os_ = torch.zeros(total, dtype=torch.uint8, device="cuda")
        aligner.align_batch_device(mode, dq.data_ptr(), dqo.data_ptr(), ds.data_ptr(), dso.data_ptr(), len(pairs),
                                   sc.data_ptr(), en.data_ptr(), st.data_ptr(), oq.data_ptr(), os_.data_ptr(), sch)
        assert np.array_equal(sc.cpu().numpy(), b.scores)
        assert np.array_equal(en.cpu().numpy().reshape(-1, 2), b.ends)
        assert np.array_equal(st.cpu().numpy().reshape(-1, 2), b.starts)
        assert np.array_equal(oq.cpu().numpy(), b.aligned_query)
        assert np.array_equal(os_.cpu().numpy(), b.aligned_subject)
        for p in (0, 7, 8, 299):
            assert _got(b, p) == _full(aligner, mode, *pairs[p], sch), (mode, p)
        # NULL ends / starts: the same scores and rows
        sc.zero_(); oq.zero_(); os_.zero_()
        aligner.align_batch_device(mode, dq.data_ptr(), dqo.data_ptr(), ds.data_ptr(), dso.data_ptr(), len(pairs),
                                   sc.data_ptr(), 0, 0, oq.data_ptr(), os_.data_ptr(), sch)
        assert np.array_equal(sc.cpu().numpy(), b.scores)
        assert np.array_equal(oq.cpu().numpy(), b.aligned_query)
        assert np.array_equal(os_.cpu().numpy(), b.aligned_subject)
        # host entry with NULL ends / starts
        L = A.capi.load_library()
        scores = np.zeros(len(pairs), np.int32)
        hq = np.zeros(total, np.uint8); hs = np.zeros(total, np.uint8)
        i64p = C.POINTER(C.c_int64)
        res = A.capi.Result()
        rc = L.anyseq_align_batch(aligner.handle, C.byref(A.capi.make_scoring(mode, 2, -1, -2, -1)), A.capi._ptr(qd),
                                  qo.ctypes.data_as(i64p), A.capi._ptr(sd), so.ctypes.data_as(i64p), len(pairs),
                                  A.capi._ptr(scores), None, None, A.capi._ptr(hq), A.capi._ptr(hs), C.byref(res))
        assert rc == 0 and np.array_equal(scores, b.scores)
        assert np.array_equal(hq, b.aligned_query) and np.array_equal(hs, b.aligned_subject)
    # an empty batch, host and device
    e = aligner.align_batch("local", b"", np.zeros(1, np.int64), b"", np.zeros(1, np.int64), sch)
    assert len(e.scores) == 0 and len(e.aligned_query) == 0
    aligner.align_batch_device("local", 0, dqo.data_ptr(), 0, dso.data_ptr(), 0, 0, 0, 0, 0, 0, sch)


# --------------------------------------------------------------------------- 7. refusals
def test_batch_align_refusals(aligner):
    import anyseq_b200 as A
    q = np.frombuffer(b"ACGT" * 10, np.uint8)
    s = np.frombuffer(b"ACGT" * 300, np.uint8)[:1025]
    with pytest.raises(A.AnyseqError) as e:
        aligner.align_batch("global", q, np.array([0, 40], np.int64), s, np.array([0, 1025], np.int64))
    assert e.value.code == -4 and "anyseq_align_full" in str(e.value)
    with pytest.raises(A.AnyseqError) as e:                    # decreasing offsets
        aligner.align_batch("global", q, np.array([0, 30, 20], np.int64), s, np.array([0, 10, 20], np.int64))
    assert e.value.code == -2
    L = A.capi.load_library()
    sc = A.capi.make_scoring("global")
    i64p = C.POINTER(C.c_int64)
    qo, so = np.array([0, 40], np.int64), np.array([0, 100], np.int64)
    out = np.zeros(140, np.uint8)
    scores = np.zeros(1, np.int32)
    res = A.capi.Result()
    args = dict(q=A.capi._ptr(q), qo=qo.ctypes.data_as(i64p), s=A.capi._ptr(s), so=so.ctypes.data_as(i64p),
                sc=A.capi._ptr(scores), aq=A.capi._ptr(out), as_=A.capi._ptr(out))
    for missing in ("q", "qo", "s", "so", "sc", "aq", "as_"):
        a = dict(args, **{missing: None})
        rc = L.anyseq_align_batch(aligner.handle, C.byref(sc), a["q"], a["qo"], a["s"], a["so"], 1, a["sc"], None, None,
                                  a["aq"], a["as_"], C.byref(res))
        assert rc == -2, missing
    rc = L.anyseq_align_batch(aligner.handle, C.byref(sc), args["q"], args["qo"], args["s"], args["so"], -1, args["sc"],
                              None, None, args["aq"], args["as_"], C.byref(res))
    assert rc == -2
