"""Parity tests proper (need a B200): the CUDA path, called through the C ABI, against
the CPU oracle on the same inputs, against the frozen golden fixtures, and -- at sizes the
oracle cannot finish -- through size-independent properties."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
MODES = ("global", "semiglobal", "local")


def _rand(rng, n, alphabet=ACGT):
    return alphabet[rng.integers(0, len(alphabet), n)]


def _related(rng, q, n, sub=0.05):
    s = q[: min(len(q), n)].copy()
    if len(s) < n:
        s = np.concatenate([s, _rand(rng, n - len(s))])
    k = max(1, int(n * sub))
    s[rng.integers(0, n, k)] = _rand(rng, k)
    # a few indels
    for _ in range(max(1, n // 400)):
        p = int(rng.integers(0, n))
        s = np.concatenate([s[:p], s[p + 1:], _rand(rng, 1)]) if rng.random() < 0.5 else np.concatenate([s[:p], _rand(rng, 1), s[p:-1]])
    return np.ascontiguousarray(s[:n])


def _sha(aq, as_):
    return hashlib.sha256(aq + b"\n" + as_).hexdigest()[:16]


# --------------------------------------------------------------------------- scores
def test_native_library_is_the_one_running(aligner):
    info = aligner.device_info()
    assert info["sm_count"] > 0 and "B200" in info["name"] or info["sm_count"] > 0
    maps = open("/proc/self/maps").read()
    assert "libanyseq_b200.so" in maps


def test_legacy_symbols_appendix_c(oracle, golden):
    """the six entry points of src/import.h on the reference CLI's own inputs"""
    import anyseq_b200 as A
    for (lo, hi), key in (((256, 1024), "align -r"), ((10000, 1024), "align -r 10000"), ((10000, 10000), "align -r 10000 10000")):
        q, s = oracle.reference_random_pair(lo, hi)
        got = [A.global_alignment_score(q, s), A.semiglobal_alignment_score(q, s), A.local_alignment_score(q, s)]
        assert got == golden["appendix_c"][key]["scores"]
    g = golden["appendix_c"]["align -r"]
    q, s = oracle.reference_random_pair(256, 1024)
    for k, (mode, fn) in enumerate(zip(MODES, (A.construct_global_alignment, A.construct_semiglobal_alignment,
                                               A.construct_local_alignment))):
        ret, aq, as_ = fn(q, s)
        assert ret == g["legacy_return"][k]                      # quirk Q1 reproduced by the legacy symbols
        assert _sha(aq, as_) == g["sha"][mode]
        o = oracle.traceback_lintime(mode, q, s)
        assert (aq, as_) == (o[1], o[2])


@pytest.mark.parametrize("K,band,generic", [(4, 0, 0), (8, 64, 0), (16, 32, 0), (32, 0, 0), (4, 96, 1), (32, 160, 0),
                                            (16, 0, 1), (8, 160, 1), (32, 64, 1)])
def test_score_sweep_vs_oracle(aligner, oracle, K, band, generic):
    """all schemes x linear/affine x ragged shapes, every columns-per-lane variant, multi-band;
    generic = byte-register kernels instead of the column-mask kernels"""
    import anyseq_b200 as A
    rng = np.random.default_rng(100 + K + band)
    aligner.tune(cols_per_lane=K, band_rows=band, watchdog_ms=10000)
    aligner.set_option("force_generic", generic)
    schemes = [A.linear_scoring_scheme(2, -1, -1), A.affine_scoring_scheme(2, -1, -2, -1),
               A.linear_scoring_scheme(3, -2, -4), A.affine_scoring_scheme(5, -4, -10, -1),
               A.affine_scoring_scheme(1, -1, -1, 0)]
    shapes = [(1, 1), (1, 7), (7, 1), (2, 129), (31, 33), (33, 31), (64, 128), (100, 127), (100, 128), (100, 129),
              (257, 255), (300, 1024), (300, 1025), (1000, 513), (700, 2048), (129, 4096), (1500, 3000), (4097, 1000)]
    try:
        for (m, n) in shapes:
            q = _rand(rng, m)
            s = _related(rng, q, n) if min(m, n) > 50 else _rand(rng, n)
            for mode in MODES:
                for sch in schemes:
                    r = aligner.score(mode, q, s, sch)
                    if sch.affine:
                        ref = oracle.score_affine(mode, q, s, sch.same, sch.diff, sch.gap_init, sch.gap_extend)
                    else:
                        ref = oracle.score_linear(mode, q, s, sch.same, sch.diff, sch.gap_extend)
                    assert r.score == ref[0], (m, n, mode, sch)
                    if mode != "local":      # end cell as the reference's get_score_pos (src/scoring.impala:34,46-64)
                        assert (r.end_i, r.end_j) == ref[1:], (m, n, mode, sch)
    finally:
        aligner.tune(0, 0, 0, 10000)
        aligner.set_option("force_generic", 0)


@pytest.mark.parametrize("K,band,generic", [(0, 0, 0), (4, 96, 0), (8, 0, 1), (16, 160, 0), (32, 0, 0), (16, 64, 1)])
def test_local_end_cell_vs_oracle(aligner, oracle, K, band, generic):
    """option local_end_cell: the cell get_score_pos() reports for the local scheme (src/scoring.impala:103-110),
    i.e. the slot order of the 1024 x 1024 block wavefront (src/scoring_cpu.impala:48-73) -- checked on inputs
    whose maximum occurs in several blocks (planted repeats) and on low-complexity sequences full of ties"""
    import anyseq_b200 as A
    rng = np.random.default_rng(7 + K + band)
    aligner.tune(cols_per_lane=K, band_rows=band, watchdog_ms=10000)
    aligner.set_option("force_generic", generic)
    aligner.set_option("local_end_cell", 1)
    pairs = []
    for (m, n) in [(1, 1), (40, 300), (300, 200), (1024, 1024), (1025, 1030), (2100, 3100), (3100, 2100), (5000, 1500),
                   (1, 5000), (4200, 4300)]:
        pairs.append((_rand(rng, m), _rand(rng, n)))
        pairs.append((_rand(rng, m, ACGT[:2]), _rand(rng, n, ACGT[:2])))          # ties everywhere
    unit = _rand(rng, 150)

    def planted(total, offsets):
        a = _rand(rng, total, ACGT[2:] if total % 2 else ACGT[:2])
        for o in offsets:
            a[o:o + len(unit)] = unit
        return a
    pairs.append((planted(3500, [100, 1500, 2900]), planted(4101, [700, 2300, 3900])))
    pairs.append((planted(4101, [30, 1100, 2200, 3300]), planted(3500, [3000, 1900, 60])))
    pairs.append((planted(2301, [1000]), planted(5000, [10, 1034, 2058, 3082, 4106])))
    schemes = [A.linear_scoring_scheme(2, -1, -1), A.affine_scoring_scheme(2, -1, -2, -1)]
    try:
        for (q, s) in pairs:
            for sch in schemes:
                r = aligner.score("local", q, s, sch)
                if sch.affine:
                    ref = oracle.score_affine("local", q, s, sch.same, sch.diff, sch.gap_init, sch.gap_extend)
                else:
                    ref = oracle.score_linear("local", q, s, sch.same, sch.diff, sch.gap_extend)
                assert (r.score, r.end_i, r.end_j) == tuple(ref), (len(q), len(s), sch)
    finally:
        aligner.tune(0, 0, 0, 10000)
        aligner.set_option("force_generic", 0)
        aligner.set_option("local_end_cell", 0)


def test_score_golden_fixtures(aligner, golden):
    import anyseq_b200 as A
    for c in golden["cases"]:
        q, s = c["q"].encode("latin-1"), c["s"].encode("latin-1")
        for mode in MODES:
            for key, exp in c["linear"][mode].items():
                sa, di, ga = map(int, key.split(","))
                r = aligner.score(mode, q, s, A.linear_scoring_scheme(sa, di, ga))
                assert r.score == exp[0], (c["name"], mode, key)
                if mode != "local":
                    assert [r.end_i, r.end_j] == exp[1:]
            for key, exp in c["affine"][mode].items():
                sa, di, gi, ge = map(int, key.split(","))
                assert aligner.score(mode, q, s, A.affine_scoring_scheme(sa, di, gi, ge)).score == exp


def test_empty_inputs(aligner):
    """quirk Q12: global = all-gap score of the non-empty side; semiglobal 0; local SCORE_MIN"""
    import anyseq_b200 as A
    assert aligner.score("global", b"", b"ACGT").score == -4
    assert aligner.score("global", b"ACG", b"").score == -3
    assert aligner.score("global", b"", b"").score == 0
    assert aligner.score("global", b"", b"ACGT", A.affine_scoring_scheme(2, -1, -2, -1)).score == -6
    assert aligner.score("semiglobal", b"", b"ACGT").score == 0
    assert aligner.score("local", b"", b"ACGT").score == -2147483647


def test_raw_byte_symbols(aligner, oracle):
    """symbols are compared as raw bytes: no case folding, N and CR are ordinary symbols (quirk Q8)"""
    rng = np.random.default_rng(5)
    alpha = np.frombuffer(b"ACGTacgtNn\r-*", dtype=np.uint8)
    q, s = _rand(rng, 900, alpha), _rand(rng, 1100, alpha)
    allb = np.arange(256, dtype=np.uint8)
    q2, s2 = _rand(rng, 600, allb), _rand(rng, 700, allb)
    import anyseq_b200 as A
    for mode in MODES:
        assert aligner.score(mode, q, s).score == oracle.score_linear(mode, q, s)[0]
        assert aligner.score(mode, q2, s2, A.affine_scoring_scheme()).score == oracle.score_affine(mode, q2, s2)[0]


def test_medium_vs_oracle(aligner, oracle):
    """sizes where the oracle still finishes in seconds; default tuning (auto K / band)"""
    import anyseq_b200 as A
    rng = np.random.default_rng(77)
    q = _rand(rng, 20011)
    s = _related(rng, q, 23456, sub=0.1)
    for mode in MODES:
        assert aligner.score(mode, q, s).score == oracle.score_linear(mode, q, s, threads=8)[0]
        assert aligner.score(mode, q, s, A.affine_scoring_scheme()).score == oracle.score_affine(mode, q, s, threads=8)[0]


def test_large_properties(aligner):
    """sizes the oracle cannot reach: size-independent properties"""
    import anyseq_b200 as A
    rng = np.random.default_rng(42)
    n = 600_000
    q = _rand(rng, n)
    lin, aff = A.linear_scoring_scheme(2, -1, -1), A.affine_scoring_scheme(2, -1, -2, -1)
    # identity: every scheme scores 2 per symbol on identical sequences
    for sch in (lin, aff):
        for mode in MODES:
            assert aligner.score(mode, q, q, sch).score == 2 * n
    # containment: q inside flanks -> semiglobal and local find it exactly
    s = np.concatenate([_rand(rng, 70_001), q, _rand(rng, 33_333)])
    for sch in (lin, aff):
        assert aligner.score("semiglobal", q, s, sch).score == 2 * n
        assert aligner.score("local", q, s, sch).score >= 2 * n
    # symmetry under transposition + monotonicity local >= semiglobal >= global
    t = _related(rng, q, n - 12_345, sub=0.03)
    for sch in (lin, aff):
        g = aligner.score("global", q, t, sch).score
        sg = aligner.score("semiglobal", q, t, sch).score
        lo = aligner.score("local", q, t, sch).score
        assert lo >= sg >= g
        assert aligner.score("global", t, q, sch).score == g
        assert aligner.score("semiglobal", t, q, sch).score == sg
        assert aligner.score("local", t, q, sch).score == lo
    # gi = 0 Gotoh == linear (SURVEY.md A.7), via two different kernels: force_affine runs the Gotoh cells with go == ge
    for mode in MODES:
        want = aligner.score(mode, q, t, lin)
        aligner.set_option("force_affine", 1)
        try:
            got = aligner.score(mode, q, t, A.affine_scoring_scheme(2, -1, 0, -1))
        finally:
            aligner.set_option("force_affine", 0)
        assert (got.score, got.end_i, got.end_j) == (want.score, want.end_i, want.end_j), mode


def test_large_mismatch_rich_all_strip_widths(aligner):
    """600 kbp, mismatch- and indel-rich (scores far from the identity line, E/F alive everywhere): every strip width,
    the generic (byte-compare) kernels and several CTA counts must give the same score and end cell -- an inter-strip
    race or a lost border record would show up as a difference between decompositions"""
    import anyseq_b200 as A
    rng = np.random.default_rng(4242)
    n = 600_000
    q = _rand(rng, n)
    t = _related(rng, q, n - 7_777, sub=0.25)
    sch = A.affine_scoring_scheme(2, -1, -2, -1)
    for mode in MODES:
        ref = None
        for (K, bps, generic) in ((8, 0, 0), (16, 0, 0), (32, 0, 0), (16, 1, 0), (32, 1, 0), (16, 0, 1), (4, 0, 0)):
            aligner.tune(cols_per_lane=K, blocks_per_sm=bps)
            aligner.set_option("force_generic", generic)
            try:
                r = aligner.score(mode, q, t, sch)
            finally:
                aligner.set_option("force_generic", 0)
                aligner.tune()
            got = (r.score, r.end_i, r.end_j)
            if ref is None:
                ref = got
            assert got == ref, (mode, K, bps, generic, got, ref)


def test_full_size_c2_against_cpu(aligner):
    """BASELINE.json configs[1] at its stated size against the frozen CPU result (tests/golden/fullsize.json, produced by
    tools/freeze_fullsize.py with oracle/fullsize_check.c): score AND end cell of the 4.64 Mbp x 4.6 Mbp semiglobal Gotoh run"""
    import json
    import anyseq_b200 as A
    from anyseq_b200 import workloads as W
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fullsize.json")
    gold = json.load(open(path)).get("c2_semiglobal_affine")
    if gold is None:
        pytest.skip("tests/golden/fullsize.json has no full-size C2 entry yet")
    q, s, _ = W.whole_genome_pair(1.0)
    assert (len(q), len(s)) == (gold["m"], gold["n"])
    r = aligner.score("semiglobal", q, s, A.affine_scoring_scheme(*gold["scheme"]))
    assert (r.score, r.end_i, r.end_j) == (gold["score"], gold["end_i"], gold["end_j"])


def test_full_size_identity(aligner):
    """BASELINE.json full size (4.64 Mbp): semiglobal affine of the genome against itself"""
    import anyseq_b200 as A
    from anyseq_b200 import workloads as W
    q, s, _ = W.whole_genome_pair(1.0)
    r = aligner.score("semiglobal", q, q, A.affine_scoring_scheme(2, -1, -2, -1))
    assert r.score == 2 * len(q) and (r.end_i, r.end_j) == (len(q) - 1, len(q) - 1)


def test_split_ranks_equal_single_run(aligner, oracle):
    """the multi-GPU strip path, emulated sequentially on one GPU: rank 0 streams its right
    edge into an inbox, rank 1 then consumes it; combined result == single run == oracle"""
    import anyseq_b200 as A
    from anyseq_b200 import capi
    from anyseq_b200.capi import Result, StripPartial, make_scoring
    import torch
    L = capi.load_library()
    rng = np.random.default_rng(8)
    q = _rand(rng, 5000)
    s = _related(rng, q, 7000, sub=0.08)
    dq = torch.from_numpy(q).cuda(); ds = torch.from_numpy(s).cuda()
    for sch in (A.linear_scoring_scheme(), A.affine_scoring_scheme()):
        for mode in MODES:
            for cut in (1024, 3000, 4096):
                sc = make_scoring(mode, sch.same, sch.diff, sch.gap_init, sch.gap_extend)
                box = C.c_void_p()
                assert L.anyseq_strip_inbox_create(aligner.handle, len(q), C.byref(box), None) == 0
                parts = (StripPartial * 2)()
                rc = L.anyseq_score_strip_device(aligner.handle, C.byref(sc), C.c_void_p(dq.data_ptr()), len(q),
                                                 C.c_void_p(ds.data_ptr()), 0, cut, len(s), None, box, C.byref(parts[0]))
                assert rc == 0, L.anyseq_last_error()
                rc = L.anyseq_score_strip_device(aligner.handle, C.byref(sc), C.c_void_p(dq.data_ptr()), len(q),
                                                 C.c_void_p(ds.data_ptr() + cut), cut, len(s), len(s), box, None,
                                                 C.byref(parts[1]))
                assert rc == 0, L.anyseq_last_error()
                res = Result()
                assert L.anyseq_strip_combine(C.byref(sc), parts, 2, C.byref(res)) == 0
                L.anyseq_strip_inbox_destroy(aligner.handle, box)
                ref = (oracle.score_affine(mode, q, s, sch.same, sch.diff, sch.gap_init, sch.gap_extend) if sch.affine
                       else oracle.score_linear(mode, q, s, sch.same, sch.diff, sch.gap_extend))
                one = aligner.score(mode, q, s, sch)
                assert res.score == ref[0] == one.score, (mode, sch, cut)
                # end cells of the combined ranks == single-GPU run (== get_score_pos of the restated reference)
                assert (res.end_i, res.end_j) == (one.end_i, one.end_j), (mode, sch, cut)
                if mode != "local":
                    assert (res.end_i, res.end_j) == ref[1:], (mode, sch, cut)


def test_inbox_shorter_than_the_query_is_refused(aligner):
    """an inbox holds one border record per query row; a longer query would make the last strip write past the end of
    the NEXT rank's (peer) memory -- the call must fail with ANYSEQ_ERR_BAD_ARG instead"""
    from anyseq_b200 import capi
    from anyseq_b200.capi import StripPartial, make_scoring
    import torch
    L = capi.load_library()
    rng = np.random.default_rng(3)
    q = _rand(rng, 3000); s = _rand(rng, 4000)
    dq = torch.from_numpy(q).cuda(); ds = torch.from_numpy(s).cuda()
    sc = make_scoring("semiglobal", 2, -1, -2, -1)
    box = C.c_void_p()
    assert L.anyseq_strip_inbox_create(aligner.handle, 2999, C.byref(box), None) == 0
    part = StripPartial()
    vp = C.c_void_p
    rc = L.anyseq_score_strip_device(aligner.handle, C.byref(sc), vp(dq.data_ptr()), len(q), vp(ds.data_ptr()), 0, 2048,
                                     len(s), None, box, C.byref(part))
    assert rc == -2 and b"inbox" in L.anyseq_last_error()
    rc = L.anyseq_score_strip_device(aligner.handle, C.byref(sc), vp(dq.data_ptr()), len(q), vp(ds.data_ptr() + 2048), 2048,
                                     len(s), len(s), box, None, C.byref(part))
    assert rc == -2
    qp = (vp * 2)(dq.data_ptr(), dq.data_ptr()); sp = (vp * 2)(ds.data_ptr(), ds.data_ptr())
    boxes = (vp * 2)(box, box)
    parts = (StripPartial * 2)()
    rc = L.anyseq_score_strip_device_multi(aligner.handle, C.byref(sc), 2, qp, len(q), sp, 0, 2048, len(s), None, boxes, parts)
    assert rc == -2
    L.anyseq_strip_inbox_destroy(aligner.handle, box)


def test_multi_pair_launch_equals_single_runs(aligner, oracle):
    """anyseq_score_strip_device_multi: several DIFFERENT pairs of one shape in a single launch (items interleaved band by
    band), alone and as the two emulated ranks of a wavefront with one inbox per pair; every pair must get exactly the
    result of its own single run"""
    import anyseq_b200 as A
    from anyseq_b200 import capi
    from anyseq_b200.capi import Result, StripPartial, make_scoring
    import torch
    L = capi.load_library()
    vp = C.c_void_p
    rng = np.random.default_rng(12)
    m, n, cut, P = 6000, 9000, 4096, 3
    qs = [_rand(rng, m) for _ in range(P)]
    ss = [_related(rng, q, n, sub=0.05 + 0.03 * i) for i, q in enumerate(qs)]
    dq = [torch.from_numpy(x).cuda() for x in qs]
    ds = [torch.from_numpy(x).cuda() for x in ss]
    aligner.tune(band_rows=1024, watchdog_ms=10000)          # several bands, so the interleaved order matters
    try:
        for sch in (A.affine_scoring_scheme(), A.linear_scoring_scheme(3, -2, -4)):
            for mode in MODES:
                sc = make_scoring(mode, sch.same, sch.diff, sch.gap_init, sch.gap_extend)
                want = [aligner.score(mode, q, s, sch).score for q, s in zip(qs, ss)]
                # (a) whole width, no inbox
                parts = (StripPartial * P)()
                rc = L.anyseq_score_strip_device_multi(aligner.handle, C.byref(sc), P, (vp * P)(*[vp(t.data_ptr()) for t in dq]), m,
                                                       (vp * P)(*[vp(t.data_ptr()) for t in ds]), 0, n, n, None, None, parts)
                assert rc == 0, L.anyseq_last_error()
                for p in range(P):
                    res = Result()
                    assert L.anyseq_strip_combine(C.byref(sc), C.byref(parts[p]), 1, C.byref(res)) == 0
                    assert res.score == want[p], (mode, sch, p)
                # (b) two emulated ranks, one inbox per pair
                boxes = [vp() for _ in range(P)]
                for b in boxes:
                    assert L.anyseq_strip_inbox_create(aligner.handle, m, C.byref(b), None) == 0
                left = (StripPartial * P)()
                right = (StripPartial * P)()
                rc = L.anyseq_score_strip_device_multi(aligner.handle, C.byref(sc), P, (vp * P)(*[vp(t.data_ptr()) for t in dq]), m,
                                                       (vp * P)(*[vp(t.data_ptr()) for t in ds]), 0, cut, n, None, (vp * P)(*boxes), left)
                assert rc == 0, L.anyseq_last_error()
                rc = L.anyseq_score_strip_device_multi(aligner.handle, C.byref(sc), P, (vp * P)(*[vp(t.data_ptr()) for t in dq]), m,
                                                       (vp * P)(*[vp(t.data_ptr() + cut) for t in ds]), cut, n, n, (vp * P)(*boxes), None,
                                                       right)
                assert rc == 0, L.anyseq_last_error()
                for p in range(P):
                    both = (StripPartial * 2)(left[p], right[p])
                    res = Result()
                    assert L.anyseq_strip_combine(C.byref(sc), both, 2, C.byref(res)) == 0
                    assert res.score == want[p], (mode, sch, p, "chained")
                for b in boxes:
                    L.anyseq_strip_inbox_destroy(aligner.handle, b)
        ref = oracle.score_affine("semiglobal", qs[1], ss[1])[0]
        assert aligner.score("semiglobal", qs[1], ss[1], A.affine_scoring_scheme()).score == ref
    finally:
        aligner.tune(0, 0, 0, 10000)


# --------------------------------------------------------------------------- tracebacks
def test_traceback_golden_fixtures(aligner, golden):
    import anyseq_b200 as A
    for c in golden["cases"]:
        q, s = c["q"].encode("latin-1"), c["s"].encode("latin-1")
        for mode in MODES:
            t = c["traceback"][mode]
            r = aligner.align(mode, q, s)
            assert aligner.last_splits() == t["splits"], (c["name"], mode)
            assert _sha(r.aligned_query, r.aligned_subject) == t["sha"], (c["name"], mode)
            if t["aq"] is not None:
                assert r.aligned_query == t["aq"].encode("latin-1") and r.aligned_subject == t["as"].encode("latin-1")
            ta = c["traceback_affine"][mode]            # build-defined Gotoh traceback, frozen
            r = aligner.align(mode, q, s, A.affine_scoring_scheme(2, -1, -2, -1))
            assert aligner.last_splits() == ta["splits"] and aligner.last_split_types() == ta["types"], (c["name"], mode)
            assert _sha(r.aligned_query, r.aligned_subject) == ta["sha"], (c["name"], mode, "affine")


@pytest.mark.parametrize("m,n", [(300, 70), (1, 200), (200, 129), (5000, 9000), (9000, 5000), (2500, 16385),
                                 (20000, 30000), (40000, 1100)])
def test_traceback_vs_oracle(aligner, oracle, m, n):
    """bit-exact alignment strings and split rows vs the restated reference CPU path
    (CPU hb_sum candidate order, BLOCK_WIDTH = 1024: parts wider than 1024 take the strided scan)"""
    rng = np.random.default_rng(m * 7 + n)
    q = _rand(rng, m)
    s = _related(rng, q, n, sub=0.07) if min(m, n) > 100 else _rand(rng, n)
    for mode in MODES:
        r = aligner.align(mode, q, s)
        ret, aq, as_, sp = oracle.traceback_lintime(mode, q, s, threads=8)
        assert aligner.last_splits() == sp.tolist(), mode
        assert r.aligned_query == aq and r.aligned_subject == as_, mode
        assert r.score == oracle.score_linear(mode, q, s, threads=8)[0]


def test_traceback_other_scoring(aligner, oracle):
    import anyseq_b200 as A
    rng = np.random.default_rng(21)
    q = _rand(rng, 3000); s = _related(rng, q, 3500, sub=0.15)
    for mode in MODES:
        r = aligner.align(mode, q, s, A.linear_scoring_scheme(3, -2, -4))
        ret, aq, as_, sp = oracle.traceback_lintime(mode, q, s, 3, -2, -4)
        assert (r.aligned_query, r.aligned_subject) == (aq, as_)


def test_traceback_large_structure(aligner):
    """300 kbp: de-gapped rows reproduce the inputs and the column score is the optimal global score"""
    rng = np.random.default_rng(31)
    n = 300_000
    q = _rand(rng, n); s = _related(rng, q, n + 777, sub=0.04)
    r = aligner.align("global", q, s)
    aq, as_ = np.frombuffer(r.aligned_query, np.uint8), np.frombuffer(r.aligned_subject, np.uint8)
    assert bytes(aq[(aq != 32) & (aq != 95)]) == bytes(q) and bytes(as_[(as_ != 32) & (as_ != 95)]) == bytes(s)
    keep = ~((aq == 32) & (as_ == 32))
    a, b = aq[keep], as_[keep]
    gaps = (a == 95) | (b == 95)
    col = int((-1 * gaps).sum() + (2 * ((a == b) & ~gaps)).sum() + (-1 * ((a != b) & ~gaps)).sum())
    assert col == r.score == aligner.score("global", q, s).score
    cg = r.cigar()
    assert cg and cg[-1] in "=XID"


# --------------------------------------------------------------------------- CLI
def test_cli_report_format():
    """`align -r`: the report of src/main.cpp (lengths 861 x 914 for the default seed)"""
    from anyseq_b200 import build
    build.build()
    r = subprocess.run([build.CLI, "-r"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.strip().splitlines()
    assert lines[0] == "random strings with length from [256,1024]"
    assert lines[1] == "sequence lengths: 861, 914"
    names = ["global score", "semiglobal score", "local score", "global alignment", "semiglobal alignment", "local alignment"]
    for ln, nm in zip(lines[2:8], names):
        assert ln.startswith("testing " + nm + " ") and ln.endswith(" ms")
    r = subprocess.run([build.CLI, "-r", "10000"], capture_output=True, text=True, timeout=300)
    assert "sequence lengths: 8087, 9011" in r.stdout       # quirk Q7


def test_reference_host_program_runs_on_the_library():
    """the reference's unmodified main.cpp, linked against libanyseq_b200.so (oracle/Makefile ref_host), runs its
    benchmark of all six entry points on the GPU: the drop-in boundary exercised by the reference's own caller"""
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "align_reference_host")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/align_reference_host was not built (needs /root/reference at build time)")
    r = subprocess.run([exe, "-r"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.strip().splitlines()
    assert lines[0] == "random strings with length from [256,1024]" and lines[1] == "sequence lengths: 861, 914"
    names = ["global score", "semiglobal score", "local score", "global alignment", "semiglobal alignment", "local alignment"]
    assert [ln.split(" ")[1:-2] for ln in lines[2:8]] == [nm.split(" ") for nm in names]
    r = subprocess.run([exe, "-r", "10000"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "sequence lengths: 8087, 9011" in r.stdout


# --------------------------------------------------------------------------- batches
def _pack(seqs):
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(x) for x in seqs])
    data = np.concatenate([np.asarray(x, dtype=np.uint8) for x in seqs]) if off[-1] else np.zeros(0, np.uint8)
    return data, off


@pytest.mark.parametrize("alphabet", ["dna", "bytes"])
def test_batch_vs_oracle(aligner, oracle, alphabet):
    """ragged batch (empty, 1-symbol, up to 1024 symbols), every scheme, linear + Gotoh, vs the oracle per pair"""
    import anyseq_b200 as A
    rng = np.random.default_rng(99)
    alpha = ACGT if alphabet == "dna" else np.arange(256, dtype=np.uint8)
    lim = 1024 if alphabet == "dna" else 512
    qs, ss = [], []
    for p in range(160):
        lq = int(rng.integers(0, 200)) if p % 7 else int(rng.integers(0, 3))
        ls = int(rng.integers(1, lim + 1)) if p % 5 else int(rng.integers(0, 40))
        q = _rand(rng, lq, alpha)
        s = _rand(rng, ls, alpha)
        if lq and ls > lq and p % 3 == 0:          # implant a mutated copy of the read
            o = int(rng.integers(0, ls - lq + 1)); s[o:o + lq] = q; s[o + lq // 2] = alpha[0]
        if p % 11 == 0:
            q, s = s, q                            # long query, short subject
        qs.append(q); ss.append(s)
    qd, qo = _pack(qs); sd, so = _pack(ss)
    for sch in (A.linear_scoring_scheme(2, -1, -1), A.affine_scoring_scheme(2, -1, -2, -1), A.affine_scoring_scheme(5, -4, -10, -1)):
        for mode in MODES:
            got, info = aligner.score_batch(mode, qd, qo, sd, so, sch)
            for p, (q, s) in enumerate(zip(qs, ss)):
                if len(q) == 0 or len(s) == 0:
                    ref = aligner.score(mode, q, s, sch).score       # quirk Q12 values, same as the single-pair path
                elif sch.affine:
                    ref = oracle.textbook_affine(mode, q, s, sch.same, sch.diff, sch.gap_init, sch.gap_extend)
                else:
                    ref = oracle.textbook_linear(mode, q, s, sch.same, sch.diff, sch.gap_extend)
                assert got[p] == ref, (alphabet, mode, sch, p, len(q), len(s))


def test_batch_reads_vs_windows(aligner, oracle):
    """BASELINE.json configs[3] shape (150 bp reads vs 500 bp windows), 20k pairs: sample vs oracle, all vs the
    single-pair strip engine through a 64-bit checksum"""
    import anyseq_b200 as A
    from anyseq_b200 import workloads as W
    npairs = 20000
    qd, qo, sd, so = W.read_batch(npairs)
    sch = A.affine_scoring_scheme(2, -1, -2, -1)
    for mode in ("global", "semiglobal"):
        got, info = aligner.score_batch(mode, qd, qo, sd, so, sch)
        for p in range(0, npairs, 97):
            q, s = qd[qo[p]:qo[p + 1]], sd[so[p]:so[p + 1]]
            assert got[p] == oracle.textbook_affine(mode, q, s, 2, -1, -2, -1), (mode, p)
        for p in range(0, 64):
            q, s = qd[qo[p]:qo[p + 1]], sd[so[p]:so[p + 1]]
            assert got[p] == aligner.score(mode, q, s, sch).score
        assert info.kernel_ms > 0


# --------------------------------------------------------------------------- Gotoh traceback (build-defined)
@pytest.mark.parametrize("m,n", [(300, 70), (1, 200), (200, 129), (700, 1500), (5000, 9000), (9000, 5000), (2500, 16385),
                                 (20000, 30000)])
def test_affine_traceback_vs_oracle(aligner, oracle, m, n):
    """Gotoh linear-space traceback: bit-exact strings, split rows and vertex types vs the CPU restatement;
    for the global scheme the emitted alignment is optimal (affine column score == textbook optimum)"""
    import anyseq_b200 as A
    rng = np.random.default_rng(m * 13 + n)
    q = _rand(rng, m)
    if min(m, n) > 100:
        # mutated copy with block indels so that gaps cross 128-column boundaries
        parts, p = [], 0
        while p < m:
            L = int(rng.integers(40, 300)); parts.append(q[p:p + L]); p += L
            if rng.random() < 0.6:
                parts.append(_rand(rng, int(rng.integers(1, 50))))
            else:
                p += int(rng.integers(1, 50))
        s = np.concatenate(parts)
        s = np.concatenate([s, _rand(rng, max(0, n - len(s)))])[:n]
        s[rng.integers(0, n, max(1, n // 20))] = ord("A")
    else:
        s = _rand(rng, n)
    for (sa, di, gi, ge) in ((2, -1, -2, -1), (5, -4, -10, -1)):
        sch = A.affine_scoring_scheme(sa, di, gi, ge)
        for mode in MODES:
            r = aligner.align(mode, q, s, sch)
            ret, aq, as_, sp, ty = oracle.traceback_lintime_affine(mode, q, s, sa, di, gi, ge, threads=8)
            assert aligner.last_splits() == sp.tolist(), (mode, sch)
            assert aligner.last_split_types() == ty.tolist(), (mode, sch)
            assert r.aligned_query == aq and r.aligned_subject == as_, (mode, sch)
            if mode == "global":
                opt = oracle.textbook_affine("global", q, s, sa, di, gi, ge)
                assert oracle.column_score_affine(r.aligned_query, r.aligned_subject, sa, di, gi, ge) == opt == r.score


# --------------------------------------------------------------------------- streaming batches (SURVEY 8f.2)
def _read_pairs(rng, npairs):
    qs, ss = [], []
    for p in range(npairs):
        q = _rand(rng, int(rng.integers(20, 160)))
        s = _rand(rng, int(rng.integers(100, 520)))
        if len(s) > len(q):
            o = int(rng.integers(0, len(s) - len(q) + 1)); s[o:o + len(q)] = q; s[o + len(q) // 3] = ACGT[p % 4]
        qs.append(q); ss.append(s)
    return qs, ss


def test_host_batch_is_chunked_and_exact(aligner, oracle):
    """anyseq_score_batch with host buffers runs as a pipeline of pinned chunks; tiny chunk limits force many
    chunks (and ragged chunk boundaries) -- scores must not depend on the chunking"""
    import anyseq_b200 as A
    rng = np.random.default_rng(5)
    qs, ss = _read_pairs(rng, 3000)
    qd, qo = _pack(qs); sd, so = _pack(ss)
    sch = A.affine_scoring_scheme(2, -1, -2, -1)
    want, _ = aligner.score_batch("semiglobal", qd, qo, sd, so, sch)
    for p in range(0, 3000, 97):
        assert want[p] == oracle.score_affine("semiglobal", qs[p], ss[p], 2, -1, -2, -1)[0]
    try:
        for pairs, nbytes in [(7, 1 << 16), (1000, 1 << 16), (64, 1 << 20)]:
            aligner.set_option("batch_chunk_pairs", pairs)
            aligner.set_option("batch_chunk_bytes", nbytes)
            got, res = aligner.score_batch("semiglobal", qd, qo, sd, so, sch)
            assert (got == want).all()
            assert res.kernel_launches >= 3000 // max(pairs, 1)       # several chunks really ran
    finally:
        aligner.set_option("batch_chunk_pairs", 1 << 18)
        aligner.set_option("batch_chunk_bytes", 64 << 20)


def test_batch_stream_producer_consumer(aligner, oracle):
    """the stream ABI itself: a producer thread fills pinned chunks while this thread collects"""
    import threading
    import anyseq_b200 as A
    rng = np.random.default_rng(6)
    qs, ss = _read_pairs(rng, 1200)
    sch = A.linear_scoring_scheme(2, -1, -1)
    st = aligner.batch_stream("global", sch, cap_pairs=100, cap_query_bytes=1 << 15, cap_subject_bytes=1 << 16, slots=2)
    errors = []

    def produce():
        try:
            p = 0
            while p < len(qs):
                c, q, qo, s, so = st.acquire()
                k = nq = ns = 0
                qo[0] = so[0] = 0
                while p < len(qs) and k < c.cap_pairs and nq + len(qs[p]) <= c.cap_query_bytes and \
                        ns + len(ss[p]) <= c.cap_subject_bytes:
                    q[nq:nq + len(qs[p])] = qs[p]; s[ns:ns + len(ss[p])] = ss[p]
                    nq += len(qs[p]); ns += len(ss[p]); k += 1; p += 1
                    qo[k] = nq; so[k] = ns
                st.submit(c, k)
        except Exception as e:     # noqa: BLE001
            errors.append(e)
        st.finish()

    t = threading.Thread(target=produce)
    t.start()
    got = []
    while True:
        r = st.collect()
        if r is None:
            break
        c, scores = r
        got.extend(int(x) for x in scores)
        st.release(c)
    t.join()
    info = st.stats()
    st.close()
    assert not errors, errors
    assert len(got) == 1200 and info["h2d_bytes"] > sum(map(len, qs)) and info["d2h_bytes"] == 4 * 1200
    for p in range(0, 1200, 13):
        assert got[p] == oracle.score_linear("global", qs[p], ss[p])[0], p


def test_cli_batch_mode(oracle, tmp_path):
    """align --batch: FASTQ reads x multi-line FASTA windows, streamed through the batch path"""
    from anyseq_b200 import build
    build.build()
    rng = np.random.default_rng(8)
    qs, ss = _read_pairs(rng, 257)
    fq, fa, out = tmp_path / "reads.fq", tmp_path / "windows.fa", tmp_path / "scores.tsv"
    with open(fq, "w") as f:
        for k, q in enumerate(qs):
            f.write(f"@r{k}\n{bytes(q).decode()}\n+\n{'I' * len(q)}\n")
    with open(fa, "w") as f:
        for k, s in enumerate(ss):
            t = bytes(s).decode()
            f.write(f">w{k}\n" + "\n".join(t[i:i + 60] for i in range(0, len(t), 60)) + "\n")
    r = subprocess.run([build.CLI, "-o", str(out), "--mode", "semiglobal", "--gap-init", "-2", "-b", str(fq), str(fa)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    lines = open(out).read().strip().splitlines()
    assert len(lines) == 257
    for k in range(0, 257, 8):
        idx, sc = lines[k].split("\t")
        assert int(idx) == k + 1 and int(sc) == oracle.score_affine("semiglobal", qs[k], ss[k], 2, -1, -2, -1)[0]


# --------------------------------------------------------------------------- full-matrix traceback (SURVEY 8f.4)
def test_traceback_full_golden_and_legacy_symbols(aligner, golden):
    import anyseq_b200 as A
    L = A.capi.load_library()
    for c in golden["cases"]:
        q, s = c["q"].encode("latin-1"), c["s"].encode("latin-1")
        for mode in MODES:
            t = c["traceback_full"][mode]
            r = aligner.align_full(mode, q, s)
            assert (r.score, list(r.start), _sha(r.aligned_query, r.aligned_subject)) == (t["score"], t["start"], t["sha"]), \
                (c["name"], mode)
            r = aligner.align_full(mode, q, s, A.affine_scoring_scheme(2, -1, -2, -1))
            ta = t["affine"]
            assert (r.score, list(r.start), _sha(r.aligned_query, r.aligned_subject)) == (ta["score"], ta["start"], ta["sha"]), \
                (c["name"], mode, "affine")
            # construct_*_alignment_fulltb (src/export.impala:38,94,151): same bytes, real score
            qa, sa = A.capi.as_u8(q), A.capi.as_u8(s)
            oq = np.zeros(len(qa) + len(sa), np.uint8); os_ = np.zeros(len(qa) + len(sa), np.uint8)
            ret = getattr(L, f"construct_{mode}_alignment_fulltb")(A.capi._ptr(qa), len(qa), A.capi._ptr(sa), len(sa),
                                                                   A.capi._ptr(oq), A.capi._ptr(os_))
            assert ret == t["score"] and _sha(oq.tobytes(), os_.tobytes()) == t["sha"]


@pytest.mark.parametrize("m,n", [(1, 1), (1, 300), (300, 1), (127, 128), (200, 129), (129, 4100), (4100, 129), (2500, 3333),
                                 (7000, 5000)])
def test_traceback_full_vs_oracle(aligner, oracle, m, n):
    import anyseq_b200 as A
    rng = np.random.default_rng(m * 7 + n)
    q = _rand(rng, m)
    s = _related(rng, q, n) if min(m, n) > 50 else _rand(rng, n)
    if min(m, n) > 400:                      # overlap layout: semiglobal and local differ from global
        s = np.concatenate([_rand(rng, n - n // 2), q[: n // 2]])[:n]
        s[rng.integers(0, n, n // 30)] = ACGT[0]
    for mode in MODES:
        for sch in (A.linear_scoring_scheme(2, -1, -1), A.affine_scoring_scheme(2, -1, -2, -1), A.linear_scoring_scheme(3, -2, -4),
                    A.affine_scoring_scheme(5, -4, -10, -1)):
            r = aligner.align_full(mode, q, s, sch)
            sc, aq, as_, st = oracle.traceback_full(mode, q, s, sch.same, sch.diff, sch.gap_init, sch.gap_extend)
            assert r.score == sc and r.start == st, (mode, sch)
            assert (r.aligned_query, r.aligned_subject) == (aq, as_), (mode, sch)


def test_traceback_full_large_and_refusal(aligner):
    """30 k x 25 k (375 MB of predecessors): exact local / semiglobal alignments (column score == score);
    a pair whose matrix cannot fit is refused, not silently truncated"""
    import anyseq_b200 as A
    rng = np.random.default_rng(3)
    core = _rand(rng, 20000)
    q = np.concatenate([_rand(rng, 5000), core, _rand(rng, 5000)])
    s = np.concatenate([_rand(rng, 2000), _related(rng, core, 20000, sub=0.03), _rand(rng, 3000)])
    for mode in ("local", "semiglobal", "global"):
        for sch in (A.linear_scoring_scheme(2, -1, -1), A.affine_scoring_scheme(2, -1, -2, -1)):
            r = aligner.align_full(mode, q, s, sch)
            assert r.score == aligner.score(mode, q, s, sch).score
            aq, as_ = np.frombuffer(r.aligned_query, np.uint8), np.frombuffer(r.aligned_subject, np.uint8)
            keep = ~((aq == 32) & (as_ == 32))
            a, b = aq[keep], as_[keep]
            gq, gs = a == 95, b == 95
            sub = int((np.where(a == b, sch.same, sch.diff) * ~(gq | gs)).sum())
            runs = int((gq[1:] & ~gq[:-1]).sum() + gq[0] + (gs[1:] & ~gs[:-1]).sum() + gs[0])
            col = sub + sch.gap_extend * int(gq.sum() + gs.sum()) + sch.gap_init * runs
            assert col == r.score, (mode, sch, col, r.score)
            dq = bytes(a[~gq]); ds = bytes(b[~gs])
            assert bytes(q)[r.start[0]:r.start[0] + len(dq)] == dq and bytes(s)[r.start[1]:r.start[1] + len(ds)] == ds
            if mode == "local":
                assert len(dq) > 15000          # the planted core is found
    big = np.zeros(3_000_000, np.uint8) + 65
    with pytest.raises(A.AnyseqError) as e:
        aligner.align_full("global", big, big)
    assert e.value.code == -4


def test_batch_packed_16bit_kernels(aligner, oracle):
    """two pairs per warp in 16-bit halves (batch_x2.cu): uniform shapes (every warp packs two DIFFERENT pairs), all
    schemes, linear + Gotoh, odd pair count, large costs near the eligibility bound; must equal the 32-bit kernels
    (option batch_packed = 0) everywhere and the oracle on a sample"""
    import anyseq_b200 as A
    rng = np.random.default_rng(21)
    for (lq, ls, npairs) in [(150, 500, 2001), (37, 90, 501), (1000, 1024, 65), (64, 64, 300), (500, 150, 400)]:
        qs, ss = [], []
        for p in range(npairs):
            q = _rand(rng, lq); s = _rand(rng, ls)
            k = min(lq, ls)
            if p % 3:
                o = int(rng.integers(0, max(ls - k, 0) + 1))
                s[o:o + k] = q[:k]
                s[rng.integers(0, ls, max(1, ls // 15))] = ACGT[p % 4]
            qs.append(q); ss.append(s)
        qd, qo = _pack(qs); sd, so = _pack(ss)
        for sch in (A.affine_scoring_scheme(2, -1, -2, -1), A.linear_scoring_scheme(2, -1, -1), A.affine_scoring_scheme(5, -4, -10, -1),
                    A.linear_scoring_scheme(3, -2, -4)):
            for mode in MODES:
                aligner.set_option("batch_packed", 1)
                got, _ = aligner.score_batch(mode, qd, qo, sd, so, sch)        # four pairs per warp where the columns fit
                aligner.set_option("batch_quad", 0)
                got2, _ = aligner.score_batch(mode, qd, qo, sd, so, sch)       # two pairs per warp
                aligner.set_option("batch_quad", 1)
                assert (got == got2).all(), (lq, ls, mode, sch, np.flatnonzero(got != got2)[:5])
                aligner.set_option("batch_packed", 0)
                ref, _ = aligner.score_batch(mode, qd, qo, sd, so, sch)
                aligner.set_option("batch_packed", 1)
                assert (got == ref).all(), (lq, ls, mode, sch, np.flatnonzero(got != ref)[:5])
                for p in (0, 1, npairs // 2, npairs - 2, npairs - 1):
                    if sch.affine:
                        want = oracle.score_affine(mode, qs[p], ss[p], sch.same, sch.diff, sch.gap_init, sch.gap_extend)[0]
                    else:
                        want = oracle.score_linear(mode, qs[p], ss[p], sch.same, sch.diff, sch.gap_extend)[0]
                    assert got[p] == want, (lq, ls, mode, sch, p)


@pytest.mark.parametrize("npairs", [201, 202, 203])
def test_batch_packed_16bit_kernels_ragged(aligner, oracle, npairs):
    """ragged DNA pairs of at most 512 symbols (four pairs per warp): neighbours of unequal shape, runs of equal
    shape, empty and 1-symbol sequences in both half-warps of the first item, a last item with 1-3 pairs; four and
    two pairs per warp and the 32-bit kernel must agree with each other and with the oracle on every pair"""
    import anyseq_b200 as A
    rng = np.random.default_rng(npairs)
    special = [(0, 37), (1, 0), (0, 0), (1, 1), (150, 0), (1, 512), (0, 1), (512, 1)]     # (lq, ls) of pairs 0..7
    qs, ss = [], []
    for p in range(npairs):
        if p < len(special):
            lq, ls = special[p]
        elif p % 5 == 4:
            lq, ls = len(qs[-1]), len(ss[-1])            # same shape as the previous pair
        else:
            lq = int(rng.integers(2, 201)); ls = int(rng.integers(2, 513))
            if p % 7 == 0:
                lq, ls = ls, lq
        q = _rand(rng, lq); s = _rand(rng, ls)
        k = min(lq, ls)
        if k and p % 3:
            o = int(rng.integers(0, ls - k + 1))
            s[o:o + k] = q[:k]
            s[rng.integers(0, ls, max(1, ls // 15))] = ACGT[p % 4]
        qs.append(q); ss.append(s)
    qd, qo = _pack(qs); sd, so = _pack(ss)
    for sch in (A.linear_scoring_scheme(2, -1, -1), A.affine_scoring_scheme(2, -1, -2, -1), A.affine_scoring_scheme(5, -4, -10, -1)):
        for mode in MODES:
            aligner.set_option("batch_packed", 1)
            quad, _ = aligner.score_batch(mode, qd, qo, sd, so, sch)
            aligner.set_option("batch_quad", 0)
            x2, _ = aligner.score_batch(mode, qd, qo, sd, so, sch)
            aligner.set_option("batch_quad", 1)
            aligner.set_option("batch_packed", 0)
            ref, _ = aligner.score_batch(mode, qd, qo, sd, so, sch)
            aligner.set_option("batch_packed", 1)
            assert (quad == x2).all(), (npairs, mode, sch, np.flatnonzero(quad != x2)[:5])
            assert (quad == ref).all(), (npairs, mode, sch, np.flatnonzero(quad != ref)[:5])
            for p, (q, s) in enumerate(zip(qs, ss)):
                if len(q) == 0 or len(s) == 0:
                    want = aligner.score(mode, q, s, sch).score      # quirk Q12 values, same as the single-pair path
                elif sch.affine:
                    want = oracle.textbook_affine(mode, q, s, sch.same, sch.diff, sch.gap_init, sch.gap_extend)
                else:
                    want = oracle.textbook_linear(mode, q, s, sch.same, sch.diff, sch.gap_extend)
                assert ref[p] == want, (npairs, mode, sch, p, len(q), len(s))


def test_batch_packed2_vs_oracle_and_byte_path(aligner, oracle):
    """anyseq_score_batch_packed2 (2-bit packed DNA, BASELINE configs[3] shape and ragged shapes): host pipeline and
    device-resident entry, uniform strides and explicit offsets/lengths, all schemes -- scores must equal the byte
    path (anyseq_score_batch) and the restated reference (oracle.score_batch)"""
    import torch
    import anyseq_b200 as A
    from anyseq_b200 import capi, workloads as W
    L = capi.load_library()
    # (1) uniform reads x windows, chunked (batch_chunk_pairs small so that several chunks and both slots are used)
    npairs = 5003
    q, qo, s, so = W.read_batch(npairs, 150, 500, seed=11)
    q2 = A.pack2(q.reshape(npairs, 150)); s2 = A.pack2(s.reshape(npairs, 500))
    assert q2.shape == (npairs, 38) and s2.shape == (npairs, 125)
    # the C helper packs like the numpy one
    one = np.zeros(38, dtype=np.uint8)
    assert L.anyseq_pack2(C.c_void_p(q[:150].ctypes.data), 150, C.c_void_p(one.ctypes.data)) == 0
    assert bytes(one) == bytes(q2[0])
    aligner.set_option("batch_chunk_pairs", 1024)
    try:
        for mode in MODES:
            for sch in (A.affine_scoring_scheme(2, -1, -2, -1), A.linear_scoring_scheme(2, -1, -1)):
                want = oracle.score_batch(mode, q, qo, s, so, sch.same, sch.diff, sch.gap_init, sch.gap_extend, threads=8)
                pb = capi.PackedBatch(q2.ctypes.data, s2.ctypes.data, None, None, None, None, 150, 500, 38, 125, npairs)
                got = np.full(npairs, -12345, dtype=np.int32)
                aligner.score_batch_packed2(mode, pb, got.ctypes.data, sch)
                assert np.array_equal(got, want), (mode, sch, np.flatnonzero(got != want)[:5])
                byte_path, _ = aligner.score_batch(mode, q, qo, s, so, sch)
                assert np.array_equal(byte_path, want)
                # device-resident entry
                dq = torch.from_numpy(q2).cuda(); ds = torch.from_numpy(s2).cuda()
                dsc = torch.full((npairs,), -1, dtype=torch.int32, device="cuda")
                pbd = capi.PackedBatch(dq.data_ptr(), ds.data_ptr(), None, None, None, None, 150, 500, 38, 125, npairs)
                aligner.score_batch_packed2(mode, pbd, dsc.data_ptr(), sch, device=True)
                assert np.array_equal(dsc.cpu().numpy(), want)
    finally:
        aligner.set_option("batch_chunk_pairs", 1 << 18)
    # (2) ragged shapes with explicit byte offsets and lengths (incl. empty sequences and lengths not divisible by 4)
    rng = np.random.default_rng(5)
    n2 = 777
    ql = rng.integers(0, 200, n2).astype(np.int32); sl = rng.integers(0, 700, n2).astype(np.int32)
    ql[:3] = (0, 1, 5); sl[:3] = (9, 0, 3)
    qs = [_rand(rng, int(x)) for x in ql]
    ss = []
    for a, x in zip(qs, sl):
        w = _rand(rng, int(x))
        if len(a) and x > len(a) + 5:
            o = int(rng.integers(0, x - len(a)))
            w[o:o + len(a)] = a
            w[o + len(a) // 2] = ord("A")
        ss.append(w)
    qb = np.zeros(n2, dtype=np.int64); sb = np.zeros(n2, dtype=np.int64)
    qparts, sparts = [], []
    qpos = spos = 0
    for i in range(n2):
        qb[i] = qpos; sb[i] = spos
        pq = A.pack2(qs[i]).reshape(-1) if len(qs[i]) else np.zeros(0, dtype=np.uint8)
        ps = A.pack2(ss[i]).reshape(-1) if len(ss[i]) else np.zeros(0, dtype=np.uint8)
        qparts.append(pq); sparts.append(ps)
        qpos += len(pq) + (i % 3)            # gaps between sequences are allowed
        spos += len(ps)
        qparts.append(np.zeros(i % 3, dtype=np.uint8))
    q2r = np.concatenate(qparts + [np.zeros(8, dtype=np.uint8)]); s2r = np.concatenate(sparts + [np.zeros(8, dtype=np.uint8)])
    qcat = np.concatenate(qs); scat = np.concatenate(ss)
    qoff = np.concatenate([[0], np.cumsum(ql)]).astype(np.int64); soff = np.concatenate([[0], np.cumsum(sl)]).astype(np.int64)
    for mode in MODES:
        sch = A.affine_scoring_scheme(2, -1, -3, -1)
        want = oracle.score_batch(mode, qcat, qoff, scat, soff, sch.same, sch.diff, sch.gap_init, sch.gap_extend, threads=8)
        pb = capi.PackedBatch(q2r.ctypes.data, s2r.ctypes.data, qb.ctypes.data, sb.ctypes.data, ql.ctypes.data, sl.ctypes.data,
                              0, 0, 0, 0, n2)
        got = np.full(n2, -12345, dtype=np.int32)
        aligner.score_batch_packed2(mode, pb, got.ctypes.data, sch)
        assert np.array_equal(got, want), (mode, np.flatnonzero(got != want)[:5])


def test_sharded_traceback_equals_single_gpu(oracle):
    """anyseq_align_sharded (multi-GPU linear-space traceback, SURVEY 8e row 3) with 2 and 4 ranks emulated by threads on
    ONE GPU (one engine per rank, the broadcast callback copies between their buffers): the concatenated pieces and the
    merged split rows must be bit-identical to the single-GPU traceback and to the restated reference, for linear and
    Gotoh gaps, all three schemes"""
    import threading
    import torch
    import anyseq_b200 as A
    from anyseq_b200 import capi
    from anyseq_b200.multigpu import ShardedTraceback, _DevView, merge_regions, merge_splits
    rng = np.random.default_rng(21)
    q = _rand(rng, 3111)
    s = _related(rng, q, 5003, sub=0.07)
    for world in (2, 4):
        als = [A.Aligner(0) for _ in range(world)]
        try:
            for sch in (A.linear_scoring_scheme(2, -1, -1), A.affine_scoring_scheme(2, -1, -2, -1)):
                for mode in MODES:
                    bar = threading.Barrier(world)
                    gpu = threading.Lock()      # the emulated ranks share ONE GPU: their persistent (cooperative) kernels
                    slot = {}                   # must never run at the same time, so a rank holds this token while it
                    pieces = [None] * world     # computes and hands it over inside the exchange callback
                    errors = []

                    def make_cb(rank):
                        def cb(user, ptr, nbytes, src):
                            try:
                                gpu.release()               # the engine has synchronised its stream before calling back
                                if rank == src:
                                    slot["ptr"] = ptr
                                bar.wait(timeout=120)
                                if rank != src:
                                    dst = torch.as_tensor(_DevView(ptr, nbytes), device="cuda")
                                    dst.copy_(torch.as_tensor(_DevView(slot["ptr"], nbytes), device="cuda"))
                                    torch.cuda.synchronize()
                                bar.wait(timeout=120)
                                gpu.acquire()
                                return 0
                            except Exception as e:          # pragma: no cover
                                errors.append(e)
                                return 1
                        return capi.BCAST_FN(cb)

                    def worker(rank):
                        try:
                            st = ShardedTraceback(als[rank], rank, world, dist=None)
                            st._cb = make_cb(rank)
                            with gpu:
                                pieces[rank] = st.align(mode, q, s, sch)
                        except Exception as e:
                            errors.append(e)
                            bar.abort()

                    ths = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
                    for t in ths:
                        t.start()
                    for t in ths:
                        t.join()
                    assert not errors, errors
                    aq, as_ = merge_regions(len(q), len(s), [(p[0], p[1], p[2], p[3]) for p in pieces])
                    splits = merge_splits([p[4] for p in pieces])
                    als[0].set_option("align_with_score", 0)
                    one = als[0].align(mode, q, s, sch)
                    assert (aq, as_) == (one.aligned_query, one.aligned_subject), (world, mode, sch)
                    assert splits == als[0].last_splits(), (world, mode, sch)
                    if sch.affine:
                        ref = oracle.traceback_lintime_affine(mode, q, s, sch.same, sch.diff, sch.gap_init, sch.gap_extend)
                    else:
                        ref = oracle.traceback_lintime(mode, q, s, sch.same, sch.diff, sch.gap_extend)
                    assert (aq, as_) == (ref[1], ref[2]), (world, mode, sch)
                    # ranks 0 and 1 always own existing blocks (5003 of 8192 columns: the last of 4 ranks owns none)
                    assert pieces[0][1] > pieces[0][0] and pieces[1][1] > pieces[1][0]
        finally:
            for a in als:
                a.close()


def test_full_size_c3_affine_traceback_against_cpu(aligner):
    """BASELINE.json configs[2] as written: LOCAL, AFFINE, linear-space traceback of the random 1 Mbp pair (seeds 1/2),
    against the frozen result of the restated CPU path (tools/freeze_fullsize.py c3affine, 38 min on 6 cores):
    alignment strings, split rows and vertex types, compared as sha256"""
    import json
    import anyseq_b200 as A
    from anyseq_b200 import workloads as W
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fullsize.json")
    gold = json.load(open(path)).get("c3affine_local")
    if gold is None:
        pytest.skip("tests/golden/fullsize.json has no full-size C3 entry yet")
    q, s = W.random_pair(gold["m"], gold["n"], *gold["seeds"])
    aligner.set_option("align_with_score", 0)
    try:
        r = aligner.align("local", q, s, A.affine_scoring_scheme(*gold["scheme"]))
    finally:
        aligner.set_option("align_with_score", 1)
    assert _sha(r.aligned_query, r.aligned_subject) == gold["sha"]
    assert hashlib.sha256(np.asarray(aligner.last_splits(), dtype=np.int32).tobytes()).hexdigest()[:16] == gold["splits_sha"]
    assert hashlib.sha256(np.asarray(aligner.last_split_types(), dtype=np.int32).tobytes()).hexdigest()[:16] == gold["types_sha"]


@pytest.mark.parametrize("form", [1, 2])
@pytest.mark.parametrize("K", [8, 16, 32])
def test_both_cell_forms_vs_oracle(aligner, oracle, form, K):
    """the decoupled and the mixed cell form of the Gotoh kernels (strip_kernel.cuh: FORM) must both reproduce the
    restated reference on every scheme: the engine picks a form per launch, this forces each one, with several
    bands, 1 - 3 warps per scheduler and ragged widths"""
    import anyseq_b200 as A
    with pytest.raises(A.AnyseqError) as e:           # the coupled cells (0) are not built for these kernels
        aligner.set_option("cell_form", 0)
    assert e.value.code == -2                          # ANYSEQ_ERR_BAD_ARG
    rng = np.random.default_rng(555 + K)
    schemes = [A.affine_scoring_scheme(2, -1, -2, -1), A.affine_scoring_scheme(5, -4, -10, -1), A.affine_scoring_scheme(1, -1, -1, 0)]
    shapes = [(300, 1025), (2100, 32 * K * 3 + 17), (1500, 32 * K * 7), (4099, 2000)]
    aligner.set_option("cell_form", form)
    try:
        for bps, band in ((1, 0), (2, 512), (3, 0)):
            aligner.tune(cols_per_lane=K, band_rows=band, blocks_per_sm=bps, watchdog_ms=10000)
            for (m, n) in shapes:
                q = _rand(rng, m)
                s = _related(rng, q, n, sub=0.12)
                for mode in MODES:
                    for sch in schemes:
                        r = aligner.score(mode, q, s, sch)
                        ref = oracle.score_affine(mode, q, s, sch.same, sch.diff, sch.gap_init, sch.gap_extend)
                        assert r.score == ref[0], (form, K, bps, band, m, n, mode, sch)
                        if mode != "local":
                            assert (r.end_i, r.end_j) == ref[1:], (form, K, bps, band, m, n, mode, sch)
    finally:
        aligner.set_option("cell_form", -1)
        aligner.tune(0, 0, 0, 10000)
