"""Batch scores with end cells (anyseq_score_batch_ends and its packed, device and streaming variants): every pair must
give the score anyseq_score_batch gives and the end cell anyseq_score reports for it alone (local alignment with the
option local_end_cell), i.e. oracle.score_linear / score_affine's (score, pos_i, pos_j)."""
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
MODES = ("global", "semiglobal", "local")
SCHEMES = ((2, -1, 0, -1), (2, -1, -2, -1), (3, -2, 0, -4), (5, -4, -10, -1), (1, -1, -1, 0))
SUBJECT_LENS = (0, 1, 31, 32, 33, 127, 128, 129, 255, 256, 257, 511, 512, 513, 1023, 1024)
QUERY_LENS = (0, 1, 2, 33, 150, 700, 2100)
# kernel families: (option, value) pairs set for the run -- x4 (default for DNA), x2, 32-bit mask kernels
FAMILIES = {"x4": (), "x2": (("batch_quad", 0),), "mask32": (("batch_packed", 0),)}
_ORACLE = {}     # (mode, scheme, query bytes, subject bytes) -> oracle result, shared by the tests of this module


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


def _pack(pairs):
    qo = np.cumsum([0] + [len(p[0]) for p in pairs]).astype(np.int64)
    so = np.cumsum([0] + [len(p[1]) for p in pairs]).astype(np.int64)
    cat = lambda xs: np.concatenate(xs) if xs else np.zeros(0, np.uint8)    # noqa: E731
    return cat([p[0] for p in pairs]), qo, cat([p[1] for p in pairs]), so


def _oracle(oracle, mode, q, s, sch):
    same, diff, gi, ge = sch
    if len(q) == 0 or len(s) == 0:      # empty_result: (lq - 1, ls - 1)
        return None, (len(q) - 1, len(s) - 1)
    if gi == 0:
        sc, ei, ej = oracle.score_linear(mode, q, s, same, diff, ge)
    else:
        sc, ei, ej = oracle.score_affine(mode, q, s, same, diff, gi, ge)
    return sc, (ei, ej)


class _options:
    """set engine options for a block and put the defaults back afterwards"""
    DEFAULTS = {"batch_quad": 1, "batch_packed": 1, "force_generic": 0, "local_end_cell": 0, "batch_chunk_pairs": 1 << 18}

    def __init__(self, aligner, opts):
        self.al, self.opts = aligner, opts

    def __enter__(self):
        for k, v in self.opts:
            self.al.set_option(k, v)

    def __exit__(self, *exc):
        for k, _ in self.opts:
            self.al.set_option(k, self.DEFAULTS[k])


def _check(aligner, oracle, mode, pairs, sch, tag, cache=_ORACLE):
    """score_batch_ends of `pairs` against the oracle and score_batch, pair by pair"""
    packed = _pack(pairs)
    scores, ends, _ = aligner.score_batch_ends(mode, *packed, _scheme(sch))
    ref_scores, _ = aligner.score_batch(mode, *packed, _scheme(sch))
    assert np.array_equal(scores, ref_scores), tag
    for p, (q, s) in enumerate(pairs):
        key = (mode, sch, q.tobytes(), s.tobytes())
        if key not in cache:
            cache[key] = _oracle(oracle, mode, q, s, sch)
        want_sc, want_end = cache[key]
        if want_sc is not None:
            assert int(scores[p]) == want_sc, (tag, mode, sch, p, len(q), len(s))
        assert (int(ends[p, 0]), int(ends[p, 1])) == want_end, (tag, mode, sch, p, len(q), len(s))
    return scores, ends


# --------------------------------------------------------------------------- 1. oracle parity, every K and family
@pytest.mark.parametrize("family", sorted(FAMILIES) + ["generic"])
@pytest.mark.parametrize("sch", SCHEMES)
def test_ends_vs_oracle(aligner, oracle, sch, family):
    """ragged pairs over every subject length boundary of K = 4..32 (32K - 1, 32K, 32K + 1) and queries of 0, 1, 2, 33,
    150, 700 and 2100 rows (queries longer than subjects run transposed for global / semiglobal); one batch per K;
    then a batch whose longest sequence exceeds 1024 (columns are the shorter sequences)"""
    rng = np.random.default_rng(sum(abs(x) for x in sch))
    if family == "generic":
        alpha, opts, Ks = np.arange(256, dtype=np.uint8), (("force_generic", 1),), (4, 8, 16)
    else:
        alpha, opts, Ks = ACGT, FAMILIES[family], (4, 8, 16, 32)
    pairs = [_pair(rng, (a + b) % 4, m, n, alpha) for a, n in enumerate(SUBJECT_LENS) for b, m in enumerate(QUERY_LENS)]
    with _options(aligner, opts):
        for mode in MODES:
            if mode == "local" and sch[1] > 0:
                continue
            for K in Ks:
                sub = [(q, s) for q, s in pairs if len(s) <= 32 * K]
                _check(aligner, oracle, mode, sub, sch, (family, K))
            if mode != "local":                      # columns = the shorter sequence of every pair
                long_pairs = [_pair(rng, 1, 2100, 700, alpha), _pair(rng, 3, 150, 1500, alpha), _pair(rng, 0, 1100, 33, alpha)]
                if family == "generic":
                    long_pairs = [_pair(rng, 1, 2100, 500, alpha), _pair(rng, 3, 150, 1500, alpha)]
                _check(aligner, oracle, mode, long_pairs, sch, (family, "long"))


@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_ends_protein_alphabet(aligner, oracle, family):
    """a 20-symbol alphabet (21 mask codes): the column masks of the 16-bit kernels plus the local row store need more
    than the default 48 KiB of shared memory a block; subjects up to 512 (x4) and 513..1024 (x2 / 32-bit)"""
    rng = np.random.default_rng(20)
    alpha = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWY", dtype=np.uint8)
    short = [_pair(rng, k % 4, int(rng.integers(1, 300)), int(rng.integers(1, 513)), alpha) for k in range(40)]
    wide = [_pair(rng, k % 4, int(rng.integers(1, 300)), int(rng.integers(513, 1025)), alpha) for k in range(24)]
    with _options(aligner, FAMILIES[family]):
        for mode in MODES:
            for sch in ((2, -1, -2, -1), (5, -4, 0, -1)):
                _check(aligner, oracle, mode, short, sch, (family, "protein <= 512"))
                _check(aligner, oracle, mode, wide, sch, (family, "protein 513..1024"))


def test_score_batch_after_ends_is_unchanged(aligner):
    """a host ends call leaves the engine's cached pipeline behind; later score-only calls must still run the score
    kernels: local pairs whose subject is too wide for subject columns run transposed, as before"""
    import anyseq_b200 as A
    rng = np.random.default_rng(12)
    sch = _scheme((2, -1, 0, -1))
    small = [(_rand(rng, 50), _rand(rng, 80)) for _ in range(8)]
    aligner.score_batch_ends("local", *_pack(small), sch)
    alpha = np.arange(256, dtype=np.uint8)
    for pairs in ([(_rand(rng, 100), _rand(rng, 1025))], [(_rand(rng, 100, alpha), _rand(rng, 600, alpha))]):
        got, _ = aligner.score_batch("local", *_pack(pairs), sch)
        q, s = pairs[0]
        assert int(got[0]) == aligner.score("local", q, s, sch).score
        with pytest.raises(A.AnyseqError):
            aligner.score_batch_ends("local", *_pack(pairs), sch)
        got2, _ = aligner.score_batch("local", *_pack(pairs), sch)
        assert np.array_equal(got, got2)


# --------------------------------------------------------------------------- 2. planted ties
def _tie_pairs():
    rng = np.random.default_rng(11)
    X = _rand(rng, 20)
    Y = _rand(rng, 20)
    N = lambda k: np.full(k, ord("N"), np.uint8)           # noqa: E731  (matches nothing in X or M)
    M = lambda k: np.full(k, ord("M"), np.uint8)           # noqa: E731
    cat = lambda *a: np.ascontiguousarray(np.concatenate(a), np.uint8)   # noqa: E731
    local = [
        (cat(X, N(1100), X), cat(X, M(200), X)),            # rows 19 / 1139, columns 19 / 239
        (cat(N(1030), X, N(40), X), cat(M(100), X, M(300), X)),   # both rows >= 1024
        (cat(N(1030), X), cat(X, M(10), X)),                # one row >= 1024, two columns
        (cat(N(5), X, N(1040), X), cat(X, M(3))),           # two rows, one column, the second >= 1024
        (cat(X, N(10)), cat(X, M(30), X)),                  # x2 / x4 item: A and B of one shape,
        (cat(N(10), X), cat(X, M(30), X)),                  # ties in different rows and columns
        (N(40), M(300)),                                    # no positive cell: (0, 0)
    ]
    semi = [
        (X.copy(), cat(X, M(50), X, M(20))),                # last row: two equal maxima
        (cat(X, N(50), X, N(10)), X.copy()),                # last column: two equal maxima
        (cat(X, N(30)), cat(M(30), X)),                     # last row vs last column
        (cat(N(3), X), cat(X, M(3))),
        (cat(X, Y), cat(Y, M(10), X)),                      # x2 / x4 item: A and B of one shape,
        (cat(Y, X), cat(X, M(10), Y)),                      # ties in different places
        (N(30), M(90)),                                     # all negative: the j = -1 candidate (value 0)
        (N(90), M(30)),
    ]
    # both orientations: the score path transposes pairs whose query is the longer sequence
    semi += [(s, q) for q, s in semi]
    return local, semi


@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_ends_planted_ties(aligner, oracle, family):
    local, semi = _tie_pairs()
    with _options(aligner, FAMILIES[family]):
        for mode, pairs in (("local", local), ("semiglobal", semi)):
            for sch in ((2, -1, 0, -1), (2, -1, -2, -1), (1, -1, -1, 0)):
                _check(aligner, oracle, mode, pairs, sch, family)
                # A and B of a packed item differ in where they tie: every pair twice, with its neighbour swapped
                _check(aligner, oracle, mode, [pairs[k ^ 1] for k in range(len(pairs) - len(pairs) % 2)], sch,
                       (family, "swapped"))


# --------------------------------------------------------------------------- 3. cross-entry equality
def _reads(npairs, seed, lq=150, ls=500):
    from anyseq_b200 import workloads as W
    return W.read_batch(npairs, lq, ls, seed=seed)


@pytest.mark.parametrize("mode", MODES)
def test_ends_cross_entries(aligner, oracle, mode):
    """host == device == chunked host == packed2 (host and device) == stream; ends == align_batch's; == anyseq_score"""
    import torch
    import anyseq_b200 as A
    from anyseq_b200 import capi
    sch = _scheme((2, -1, -2, -1))
    npairs = 5000
    qd, qo, sd, so = _reads(npairs, 3)
    rng = np.random.default_rng(4)
    scores, ends, _ = aligner.score_batch_ends(mode, qd, qo, sd, so, sch)
    ref, _ = aligner.score_batch(mode, qd, qo, sd, so, sch)
    assert np.array_equal(scores, ref)
    b = aligner.align_batch(mode, qd, qo, sd, so, sch)
    assert np.array_equal(b.scores, scores) and np.array_equal(b.ends, ends)
    # device
    dq, dqo, ds, dso = (torch.from_numpy(x).cuda() for x in (qd, qo, sd, so))
    dsc = torch.zeros(npairs, dtype=torch.int32, device="cuda")
    den = torch.zeros(2 * npairs, dtype=torch.int32, device="cuda")
    aligner.score_batch_ends_device(mode, dq.data_ptr(), dqo.data_ptr(), ds.data_ptr(), dso.data_ptr(), npairs,
                                    dsc.data_ptr(), den.data_ptr(), sch)
    assert np.array_equal(dsc.cpu().numpy(), scores) and np.array_equal(den.cpu().numpy().reshape(-1, 2), ends)
    # host, chunked into many tiny chunks
    with _options(aligner, (("batch_chunk_pairs", 333),)):
        s2, e2, _ = aligner.score_batch_ends(mode, qd, qo, sd, so, sch)
    assert np.array_equal(s2, scores) and np.array_equal(e2, ends)
    # packed2, host and device (uniform lengths, strided)
    q2 = A.pack2(qd.reshape(npairs, 150))
    s2p = A.pack2(sd.reshape(npairs, 500))
    got_s = np.zeros(npairs, np.int32)
    got_e = np.zeros((npairs, 2), np.int32)
    pb = capi.PackedBatch(q2.ctypes.data, s2p.ctypes.data, None, None, None, None, 150, 500, q2.shape[1], s2p.shape[1],
                          npairs)
    aligner.score_batch_packed2(mode, pb, got_s.ctypes.data, sch, ends=got_e.ctypes.data)
    assert np.array_equal(got_s, scores) and np.array_equal(got_e, ends)
    dq2, ds2 = torch.from_numpy(q2).cuda(), torch.from_numpy(s2p).cuda()
    pbd = capi.PackedBatch(dq2.data_ptr(), ds2.data_ptr(), None, None, None, None, 150, 500, q2.shape[1], s2p.shape[1],
                           npairs)
    den.zero_()
    aligner.score_batch_packed2(mode, pbd, dsc.data_ptr(), sch, device=True, ends=den.data_ptr())
    assert np.array_equal(dsc.cpu().numpy(), scores) and np.array_equal(den.cpu().numpy().reshape(-1, 2), ends)
    # anyseq_score on a sample (local: with local_end_cell)
    with _options(aligner, (("local_end_cell", 1),)):
        for p in rng.choice(npairs, 40, replace=False):
            r = aligner.score(mode, qd[qo[p]:qo[p + 1]], sd[so[p]:so[p + 1]], sch)
            assert (r.score, r.end_i, r.end_j) == (scores[p], ends[p, 0], ends[p, 1]), p


def test_ends_stream_producer_consumer(aligner):
    import threading
    sch = _scheme((2, -1, 0, -1))
    npairs = 3000
    qd, qo, sd, so = _reads(npairs, 9)
    scores, ends, _ = aligner.score_batch_ends("local", qd, qo, sd, so, sch)
    st = aligner.batch_stream("local", sch, cap_pairs=256, cap_query_bytes=1 << 16, cap_subject_bytes=1 << 18, ends=True)
    got_s, got_e = [], []

    def produce():
        p = 0
        while p < npairs:
            c, q, qv, s, sv = st.acquire()
            n = min(256, npairs - p)
            qv[: n + 1] = qo[p:p + n + 1] - qo[p]
            sv[: n + 1] = so[p:p + n + 1] - so[p]
            q[: qo[p + n] - qo[p]] = qd[qo[p]:qo[p + n]]
            s[: so[p + n] - so[p]] = sd[so[p]:so[p + n]]
            st.submit(c, n)
            p += n
        st.finish()

    th = threading.Thread(target=produce)
    th.start()
    while True:
        r = st.collect()
        if r is None:
            break
        c, sc = r
        got_s.append(sc.copy())
        got_e.append(st.chunk_ends(c).copy())
        st.release(c)
    th.join()
    st.close()
    assert np.array_equal(np.concatenate(got_s), scores) and np.array_equal(np.concatenate(got_e), ends)
    plain = aligner.batch_stream("local", sch, cap_pairs=16, cap_query_bytes=1 << 12, cap_subject_bytes=1 << 12)
    c, q, qv, s, sv = plain.acquire()
    qv[:2] = [0, 3]
    sv[:2] = [0, 3]
    q[:3] = np.frombuffer(b"ACG", np.uint8)
    s[:3] = np.frombuffer(b"ACG", np.uint8)
    plain.submit(c, 1)
    plain.finish()
    c, sc = plain.collect()
    assert plain.chunk_ends(c) is None and int(sc[0]) == 6
    plain.release(c)
    plain.close()


def test_cli_batch_ends(oracle, tmp_path):
    """align --batch --ends: FASTQ reads x FASTA windows; without --ends the output is the score-only format"""
    from anyseq_b200 import build
    build.build()
    rng = np.random.default_rng(8)
    qs = [_rand(rng, int(rng.integers(1, 200))) for _ in range(157)]
    ss = [np.concatenate([_rand(rng, 40), q[: len(q) // 2], _rand(rng, 30)]) for q in qs]
    fq, fa = tmp_path / "reads.fq", tmp_path / "windows.fa"
    with open(fq, "w") as f:
        for k, q in enumerate(qs):
            f.write(f"@r{k}\n{bytes(q).decode()}\n+\n{'I' * len(q)}\n")
    with open(fa, "w") as f:
        for k, s in enumerate(ss):
            t = bytes(s).decode()
            f.write(f">w{k}\n" + "\n".join(t[i:i + 60] for i in range(0, len(t), 60)) + "\n")
    for mode in ("semiglobal", "local"):
        args = [build.CLI, "--mode", mode, "--gap-init", "-2", "-b", str(fq), str(fa)]
        r = subprocess.run(args[:1] + ["--ends"] + args[1:], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        plain = subprocess.run(args, capture_output=True, text=True, timeout=300)
        assert plain.returncode == 0, plain.stderr
        lines, plain_lines = r.stdout.strip().splitlines(), plain.stdout.strip().splitlines()
        assert len(lines) == len(plain_lines) == 157
        for k in range(157):
            idx, sc, ei, ej = (int(x) for x in lines[k].split("\t"))
            assert plain_lines[k] == f"{idx}\t{sc}"
            want = oracle.score_affine(mode, qs[k], ss[k], 2, -1, -2, -1)
            assert idx == k + 1 and (sc, ei, ej) == tuple(want), (mode, k)


# --------------------------------------------------------------------------- 4. refusals
def test_ends_refusals(aligner):
    import anyseq_b200 as A
    from anyseq_b200 import capi
    sch = _scheme((2, -1, 0, -1))
    rng = np.random.default_rng(2)
    pairs = [(_rand(rng, 100), _rand(rng, 1025)), (_rand(rng, 10), _rand(rng, 10))]
    with pytest.raises(A.AnyseqError) as e:
        aligner.score_batch_ends("local", *_pack(pairs), sch)
    assert e.value.code == -4                                          # ANYSEQ_ERR_UNSUPPORTED
    assert "anyseq_score" in str(e.value) and "local_end_cell" in str(e.value)
    aligner.score_batch_ends("semiglobal", *_pack(pairs), sch)          # other modes transpose such pairs
    # the generic kernels take 512 columns: 512 runs, 513 is refused
    with _options(aligner, (("force_generic", 1),)):
        aligner.score_batch_ends("local", *_pack([(_rand(rng, 30), _rand(rng, 512))]), sch)
        with pytest.raises(A.AnyseqError) as e:
            aligner.score_batch_ends("local", *_pack([(_rand(rng, 30), _rand(rng, 513))]), sch)
        assert e.value.code == -4
    # local with diff > 0, as score_batch
    with pytest.raises(A.AnyseqError):
        aligner.score_batch_ends("local", *_pack(pairs[1:]), _scheme((2, 1, 0, -1)))
    # NULL ends
    q, qo, s, so = _pack(pairs[1:])
    sc = capi.make_scoring("global", 2, -1, 0, -1)
    res = capi.Result()
    out = np.zeros(1, np.int32)
    i64p, i32p = capi.C.POINTER(capi.C.c_int64), capi.C.POINTER(capi.C.c_int32)
    rc = aligner._lib.anyseq_score_batch_ends(aligner.handle, capi.C.byref(sc), capi._ptr(q), qo.ctypes.data_as(i64p),
                                              capi._ptr(s), so.ctypes.data_as(i64p), 1, out.ctypes.data_as(i32p), None,
                                              capi.C.byref(res))
    assert rc == -2                                                    # ANYSEQ_ERR_BAD_ARG
    # the 32-bit score range (include/anyseq.h): local, same = 2^24 takes min(m, n) <= 123; one more is refused by
    # both entries alike
    big = _scheme((1 << 24, -1, 0, -1))
    inside = [(_rand(rng, 123), _rand(rng, 400)), (np.full(123, 65, np.uint8), np.full(123, 65, np.uint8))]
    sc_in, e_in, _ = aligner.score_batch_ends("local", *_pack(inside), big)
    assert np.array_equal(sc_in, aligner.score_batch("local", *_pack(inside), big)[0])
    assert int(sc_in[1]) == 123 << 24 and tuple(e_in[1]) == (122, 122)
    past = [(np.full(124, 65, np.uint8), np.full(124, 65, np.uint8))]
    for fn in (aligner.score_batch, aligner.score_batch_ends):
        with pytest.raises(A.AnyseqError) as e:
            fn("local", *_pack(past), big)
        assert e.value.code == -4


# --------------------------------------------------------------------------- 5. scale
@pytest.mark.parametrize("mode,sch", [("semiglobal", (2, -1, -2, -1)), ("local", (2, -1, 0, -1))])
def test_ends_reads_vs_windows_at_scale(aligner, oracle, mode, sch):
    npairs, lq, ls = 100_000, 150, 500
    qd, qo, sd, so = _reads(npairs, 5, lq, ls)
    scores, ends, _ = aligner.score_batch_ends(mode, qd, qo, sd, so, _scheme(sch))
    ref, _ = aligner.score_batch(mode, qd, qo, sd, so, _scheme(sch))
    assert np.array_equal(scores, ref)
    rng = np.random.default_rng(1)
    for p in rng.choice(npairs, 2000, replace=False):
        q, s = qd[qo[p]:qo[p + 1]], sd[so[p]:so[p + 1]]
        assert _oracle(oracle, mode, q, s, sch) == (scores[p], (ends[p, 0], ends[p, 1])), p
    ei, ej = ends[:, 0], ends[:, 1]
    if mode == "semiglobal":
        on_row = ei == lq - 1
        assert np.all(on_row | (ej == ls - 1))
        assert np.all((ej >= 0) | (scores == 0))
    else:
        assert np.all((ei >= 0) & (ei < lq) & (ej >= 0) & (ej < ls))
        for p in rng.choice(npairs, 300, replace=False):
            q, s = qd[qo[p]:qo[p] + ei[p] + 1], sd[so[p]:so[p] + ej[p] + 1]
            assert oracle.score_linear("local", q, s, *sch[:2], sch[3])[0] == scores[p], p
