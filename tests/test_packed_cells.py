"""Packed cells (strip_packed.cuh): the global / semiglobal Gotoh strip kernel that keeps two cells in the 16-bit
halves of every register must give the scores and end cells of the 32-bit kernels and of the oracle."""
import numpy as np
import pytest

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
SCHEMES = [(2, -1, -2, -1), (5, -4, -10, -1), (1, -1, -1, 0)]


def _rand(rng, n):
    return ACGT[rng.integers(0, 4, n)]


def _related(rng, q, n, sub):
    s = q[: min(len(q), n)].copy()
    if len(s) < n:
        s = np.concatenate([s, _rand(rng, n - len(s))])
    k = max(1, int(n * sub))
    s[rng.integers(0, n, k)] = _rand(rng, k)
    for _ in range(max(1, n // 400)):
        p = int(rng.integers(0, n))
        s = np.concatenate([s[:p], s[p + 1:], _rand(rng, 1)]) if rng.random() < 0.5 else np.concatenate([s[:p], _rand(rng, 1), s[p:-1]])
    return np.ascontiguousarray(s[:n])


def test_planner_packed_cells_without_a_device():
    """the whole-genome launch runs packed cells; a scheme whose score window no longer fits 16 bits falls back, and
    local mode, linear gaps and multi-GPU slices never use them"""
    import anyseq_b200 as A
    p = A.plan_launch("semiglobal", 4641652, 4600000, affine=True)
    assert p["packed_cells"] == 1 and p["cols_per_lane"] == 32 and p["warps_per_cta"] == 12
    assert A.plan_launch("global", 4641652, 4600000, scheme=(2, -1, -2, -1))["packed_cells"] == 1
    # K = 32: D * (160 + 1024) + constants must stay within 0x3c00; D = same - go = 12 fits, 13 does not
    assert A.plan_launch("semiglobal", 4641652, 4600000, scheme=(9, -1, -2, -1))["packed_cells"] == 1
    assert A.plan_launch("semiglobal", 4641652, 4600000, scheme=(10, -1, -2, -1))["packed_cells"] == 0
    # (5, -4, -10, -1): D = 16 fits the 512-column strips only
    assert A.plan_launch("semiglobal", 1000000, 1000000, scheme=(5, -4, -10, -1))["packed_cells"] == 1
    assert A.plan_launch("semiglobal", 4641652, 4600000, scheme=(5, -4, -10, -1))["packed_cells"] == 0
    assert A.plan_launch("local", 4641652, 4600000, affine=True)["packed_cells"] == 0
    assert A.plan_launch("global", 4641652, 4600000, affine=False)["packed_cells"] == 0
    assert A.plan_launch("semiglobal", 4641652, 575488, affine=True, chained=True)["packed_cells"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("K", [16, 32])
def test_packed_vs_32bit_vs_oracle(aligner, oracle, K):
    """identical, unrelated and mismatch-rich pairs; widths whose ragged last strip ends in the low and in the high
    half; one and several bands; one to three warps per scheduler"""
    import anyseq_b200 as A
    rng = np.random.default_rng(9100 + K)
    SW = 32 * K
    shapes = [(700, 2 * SW + SW // 4 + 3), (1300, 3 * SW + 3 * SW // 4 + 1), (2101, 2 * SW), (97, SW + 5)]
    try:
        for bps, band in ((1, 0), (2, 256), (3, 0)):
            aligner.tune(cols_per_lane=K, band_rows=band, blocks_per_sm=bps, watchdog_ms=10000)
            for (m, n) in shapes:
                q = _rand(rng, m)
                pairs = [(q, np.ascontiguousarray(np.resize(q, n))), (q, _rand(rng, n)), (q, _related(rng, q, n, 0.2))]
                for qq, ss in pairs:
                    for mode in ("global", "semiglobal"):
                        for sch in SCHEMES:
                            sc = A.affine_scoring_scheme(*sch)
                            got = []
                            for packed in (0, 1):
                                aligner.set_option("packed_cells", packed)
                                r = aligner.score(mode, qq, ss, sc)
                                got.append((r.score, r.end_i, r.end_j))
                            ref = oracle.score_affine(mode, qq, ss, *sch)
                            assert got[0] == got[1] == (ref[0], *ref[1:]), (K, bps, band, m, n, mode, sch, got, ref)
    finally:
        aligner.set_option("packed_cells", -1)
        aligner.tune(0, 0, 0, 10000)


@pytest.mark.gpu
def test_packed_large_mismatch_rich(aligner):
    """600 kbp, mismatch- and indel-rich: the packed kernel (K = 16, 32) against the 32-bit kernels, several bands"""
    import anyseq_b200 as A
    rng = np.random.default_rng(4243)
    n = 600_000
    q = _rand(rng, n)
    t = _related(rng, q, n - 7_777, sub=0.25)
    sch = A.affine_scoring_scheme(2, -1, -2, -1)
    try:
        for mode in ("global", "semiglobal"):
            ref = None
            for (K, bps, packed) in ((32, 0, 0), (32, 0, 1), (16, 0, 1), (32, 1, 1), (16, 2, 1)):
                aligner.tune(cols_per_lane=K, blocks_per_sm=bps)
                aligner.set_option("packed_cells", packed)
                r = aligner.score(mode, q, t, sch)
                got = (r.score, r.end_i, r.end_j)
                if ref is None:
                    ref = got
                assert got == ref, (mode, K, bps, packed, got, ref)
    finally:
        aligner.set_option("packed_cells", -1)
        aligner.tune()
