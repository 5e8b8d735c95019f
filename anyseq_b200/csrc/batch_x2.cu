// batch_x2.cu -- the batch kernel with TWO pairs per group of lanes (a warp or a half-warp), packed as 16-bit
// halves of every register.
//
// Short pairs (reads x windows) have scores that fit in 16 bits, and pairs are independent, so the low half
// of each register carries pair A and the high half pair B of the same shape (lenq, lens): the DPX
// instructions VIADDMNMX.S16x2 / VIMNMX3.S16x2 then relax two cells per issue slot.  Everything else is the
// batch kernel of batch.cu: one group per pair of pairs, the longer sequence spread over the group's lanes as
// columns (per-lane column masks per alphabet code in shared memory), the shorter streamed as rows with a lane
// skew, borders from init_scores (src/align.impala:85-86), values only.
//
// Packed arithmetic outside DPX (H + gap_open, diag + sigma) runs as ordinary 32-bit IMADs on the FMA pipe:
// adding c * 65537 adds c to both halves as long as no half goes below zero or above 0x7fff, so all stored H
// values carry a common offset `bias` (host: chosen from the lengths and the scheme; the kernels are only
// used when the whole value range fits).  E and F are touched by DPX only and may be negative.
// Two consecutive pairs of different shape are simply run one after the other (each packed with itself).
#include "batch.cuh"
#include "strip_kernel.cuh"

namespace anyseq {

constexpr int kNeg16 = -30000;     // "minus infinity" of E / F in a signed 16-bit half

struct X2Const {
    int one;
    unsigned ge2;        // (ge, ge) as 16-bit fields (DPX operand)
    int go_c;            // go * 65537 (IMAD operand)
    int dd_c;            // (diff - go) * 65537
    int sd_c;            // low half same - go, high half diff - go
    int dhi;             // (same - diff) << 16
    unsigned floor2;     // local: (bias, bias) = packed zero
};

template <int W>
struct X2State {
    unsigned dd, e, xleft, best, hprev;
    unsigned tm[W];      // match bits of the lane's row: bit 2c = pair A column c, bit 2c+1 = pair B
};

template <bool LOCAL, bool AFFINE, int K, int C>
struct CellX2 {
    template <int KF, int W>
    static __device__ __forceinline__ void run(unsigned (&X)[K], unsigned (&F)[KF], X2State<W>& s, const X2Const& k)
    {
        const unsigned up = X[C];
        const unsigned dd = s.dd;
        if constexpr (C + 1 < K) s.dd = diag_sigma_x2<(2 * (C + 1)) % 32>(s.tm[(2 * (C + 1)) / 32], up, k);
        unsigned h;
        if constexpr (AFFINE) {
            s.e = __viaddmax_s16x2(s.e, k.ge2, s.xleft);
            const unsigned f = __viaddmax_s16x2(F[C], k.ge2, up);
            h = __vimax3_s16x2(dd, s.e, f);
            F[C] = f;
        } else {
            const unsigned tmax = __vmaxs2(s.xleft, up);
            h = __viaddmax_s16x2(tmax, k.ge2, dd);
        }
        if constexpr (LOCAL) {
            h = __vmaxs2(h, k.floor2);
            if constexpr ((C & 1) != 0) s.best = __vimax3_s16x2(s.best, h, s.hprev);
            else s.hprev = h;
        }
        const unsigned x = AFFINE ? (unsigned)imad_add((int)h, k.one, k.go_c) : h;
        X[C] = x;
        s.xleft = x;
        if constexpr (C + 1 < K) CellX2<LOCAL, AFFINE, K, C + 1>::run(X, F, s, k);
    }
};

// colbest = max(colbest, X[idx]) for a warp-uniform run-time idx: a jump into K one-instruction cases instead of
// K compare/select pairs per row
template <int K>
__device__ __forceinline__ void max_column_u(unsigned& best, const unsigned (&X)[K], int idx)
{
    switch (idx) {
#define ANYSEQ_CASE(c) case c: if constexpr (c < K) best = __vmaxs2(best, X[c < K ? c : 0]); break;
        ANYSEQ_CASE(0) ANYSEQ_CASE(1) ANYSEQ_CASE(2) ANYSEQ_CASE(3) ANYSEQ_CASE(4) ANYSEQ_CASE(5) ANYSEQ_CASE(6) ANYSEQ_CASE(7)
        ANYSEQ_CASE(8) ANYSEQ_CASE(9) ANYSEQ_CASE(10) ANYSEQ_CASE(11) ANYSEQ_CASE(12) ANYSEQ_CASE(13) ANYSEQ_CASE(14) ANYSEQ_CASE(15)
        ANYSEQ_CASE(16) ANYSEQ_CASE(17) ANYSEQ_CASE(18) ANYSEQ_CASE(19) ANYSEQ_CASE(20) ANYSEQ_CASE(21) ANYSEQ_CASE(22) ANYSEQ_CASE(23)
        ANYSEQ_CASE(24) ANYSEQ_CASE(25) ANYSEQ_CASE(26) ANYSEQ_CASE(27) ANYSEQ_CASE(28) ANYSEQ_CASE(29) ANYSEQ_CASE(30) ANYSEQ_CASE(31)
#undef ANYSEQ_CASE
        default: break;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// batch_pairs: two pairs per group of LANES lanes, relaxed together in the two halves of every register.
//   LANES = 32: a group is the warp, two pairs per warp, K = 4..32 columns per lane.
//   LANES = 16: a group is a half-warp, four pairs per warp, K = 32 (16 lanes x 32 columns = 512 columns).  The lane
//   skew of a work item is 15 steps instead of 31: a 150-row read costs 165 instead of 181 steps (the 17 % fill/drain
//   of 32 lanes becomes 9 %).  Used when the column sequences have at most 512 symbols (BASELINE configs[3]: 500 bp
//   windows).
// ---------------------------------------------------------------------------------------------------------------
template <int MODE, bool AFFINE, int K, int LANES>
__device__ __forceinline__ void batch_pairs(const BatchArgs& a)
{
    static_assert(LANES == 32 || LANES == 16, "a group is a warp or a half-warp");
    constexpr int G = 32 / LANES;                     // groups per warp; a work item is 2 G consecutive pairs
    constexpr bool LOCAL = MODE == kLocal;
    constexpr bool GLOB = MODE == kGlobal;
    __shared__ uint8_t s_rows[kWarpsPerBlock][G][2][64];
    __shared__ uint8_t s_lut[256];
    extern __shared__ unsigned s_dyn[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = lane / LANES, gl = lane % LANES;  // the lane's group and its lane within the group
    if (!a.packed2) {
        for (int x = threadIdx.x; x < 256; x += kThreads) s_lut[x] = a.lut[x];
    }
    __syncthreads();
    constexpr int W = (2 * K + 31) / 32;              // words of match bits per lane and row
    // [warp][group][pair A/B][code][lane of the group][W]
    unsigned* maskA = s_dyn + ((warp * G + grp) * 2 + 0) * a.ncodes * LANES * W;     // bits 2c
    unsigned* maskB = s_dyn + ((warp * G + grp) * 2 + 1) * a.ncodes * LANES * W;     // bits 2c + 1
    uint8_t* rqA = s_rows[warp][grp][0];
    uint8_t* rqB = s_rows[warp][grp][1];
#pragma unroll
    for (int x = gl; x < 2 * 64; x += LANES) s_rows[warp][grp][0][x] = 0;      // the row rings of both pairs
    __syncwarp();

    const int go = AFFINE ? a.sp.gap_open : 0;
    const int bias = a.bias;
    X2Const k;
    k.one = a.one;
    k.ge2 = pack2(a.sp.gap_extend, a.sp.gap_extend);
    k.go_c = go * 65537;
    k.dd_c = (a.sp.diff - go) * 65537;
    k.sd_c = (a.sp.diff - go) * 65536 + (a.sp.same - go);
    k.dhi = (a.sp.same - a.sp.diff) * 65536;
    k.floor2 = pack2(bias, bias);
    // border(k) = H(k,-1) = H(-1,k) (src/align.impala:85-86, + Gotoh opening), biased
    auto border = [&](int idx) -> int { return (GLOB ? a.sp.gap_open + idx * a.sp.gap_extend : 0) + bias; };

    const long long nitems = (a.npairs + 2 * G - 1) / (2 * G);
    long long wi = (long long)blockIdx.x * kWarpsPerBlock + warp;
    while (wi < nitems) {
        // this group's two pairs (the last item of a batch may have fewer than 2 G)
        const long long p0 = 2 * G * wi + 2 * grp;
        const bool have = p0 < a.npairs;
        // (with one group per item p0 < npairs always holds; saying so keeps pA free of a select)
        const long long pA = (G == 1 || have) ? p0 : a.npairs - 1, pB = min(pA + 1, a.npairs - 1);
        const int lqA = batch_q_len(a, pA), lsA = batch_s_len(a, pA);
        const int lqB = batch_q_len(a, pB), lsB = batch_s_len(a, pB);
        const bool same_shape = lqA == lqB && lsA == lsB;
        // pass 0: (A, B) together when they have one shape, else A with itself; pass 1: B with itself if it was left
        // over.  A warp-wide group runs only the passes it needs (its first pair always exists); the groups of a
        // half-warp item run both passes in step, a group without a pair in the pass keeping the other company.
        const int npass = (G == 1 && same_shape) ? 1 : 2;
        for (int pass = 0; pass < npass; ++pass) {
            const bool active = G == 1 || (have && (pass == 0 || !same_shape));
            if (G > 1 && !__any_sync(kFull, active)) continue;
            const long long pa = (pass == 0) ? pA : pB;
            const long long pb = (pass == 0 && same_shape) ? pB : pa;
            const long long qa0 = batch_q_start(a, pa), sa0 = batch_s_start(a, pa), qb0 = batch_q_start(a, pb), sb0 = batch_s_start(a, pb);
            const int lq = batch_q_len(a, pa), ls = batch_s_len(a, pa);
            const bool empty = lq == 0 || ls == 0;
            int scoreA, scoreB;
            if (G == 1 && empty) {
                scoreA = scoreB = empty_pair_score<MODE>(a, lq, ls);     // a warp-wide group skips the DP
            } else {
                const bool q_is_cols = a.cols_longer ? (lq >= ls) : (lq < ls);
                const uint8_t* colsA = q_is_cols ? a.q + qa0 : a.s + sa0;
                const uint8_t* rowsA = q_is_cols ? a.s + sa0 : a.q + qa0;
                const uint8_t* colsB = q_is_cols ? a.q + qb0 : a.s + sb0;
                const uint8_t* rowsB = q_is_cols ? a.s + sb0 : a.q + qb0;
                const int n = q_is_cols ? lq : ls;                    // columns (<= LANES * K)
                const int m = (active && !empty) ? (q_is_cols ? ls : lq) : 0;     // rows; 0: this group only keeps the warp company
                const bool live = G == 1 || m > 0;    // (a warp-wide group gets here only with a pair to relax)

                unsigned X[K], F[AFFINE ? K : 1];
                const int jl = gl * K;
#pragma unroll
                for (int c = 0; c < K; ++c) { const int b = border(jl + c) + go; X[c] = pack2(b, b); }
                if constexpr (AFFINE) {
#pragma unroll
                    for (int c = 0; c < K; ++c) F[c] = pack2(kNeg16, kNeg16);
                } else {
                    F[0] = 0;
                }
                __syncwarp();
                for (int cd = 0; cd < a.ncodes; ++cd) {
#pragma unroll
                    for (int w = 0; w < W; ++w) { maskA[(cd * LANES + gl) * W + w] = 0u; maskB[(cd * LANES + gl) * W + w] = 0u; }
                }
                if (live) {
#pragma unroll 4
                    for (int c = 0; c < K; ++c) {
                        const int j = jl + c;
                        const int ca = (j < n) ? batch_code(colsA, j, a.packed2, s_lut) : 0;
                        const int cb = (j < n) ? batch_code(colsB, j, a.packed2, s_lut) : 0;
                        if (ca) maskA[(ca * LANES + gl) * W + (2 * c) / 32] |= 1u << ((2 * c) % 32);
                        if (cb) maskB[(cb * LANES + gl) * W + (2 * c) / 32] |= 2u << ((2 * c) % 32);
                    }
                }
                __syncwarp();
                auto row_bits = [&](int i, unsigned (&tm)[W]) {
                    const unsigned* ma = maskA + ((int)rqA[i & 63] * LANES + gl) * W;
                    const unsigned* mb = maskB + ((int)rqB[i & 63] * LANES + gl) * W;
#pragma unroll
                    for (int w = 0; w < W; ++w) tm[w] = ma[w] | mb[w];
                };
                unsigned dcarry;
                { const int b = (gl == 0) ? bias + go : border(jl - 1) + go; dcarry = pack2(b, b); }   // H(-1,-1) = 0
                const int outlane = live ? (n - 1) / K : 0, outc = live ? (n - 1) % K : 0;
                unsigned hr = 0, er = 0;
                unsigned colbest = pack2(kNeg16, kNeg16);    // semiglobal: max over H(i, n-1), kept by lane `outlane`
                X2State<W> st;
                st.dd = 0; st.e = 0; st.xleft = 0;
#pragma unroll
                for (int w = 0; w < W; ++w) st.tm[w] = 0u;
                st.best = k.floor2; st.hprev = k.floor2;
                const int T = live ? m + outlane : 0;
                int Tmax = T;                                // steps of the warp: those of its longest group
                if constexpr (G > 1) Tmax = max(T, __shfl_xor_sync(kFull, T, 16));
                for (int tb = 0; tb < Tmax; tb += 32) {
                    __syncwarp();
                    {
                        // 32 rows of both pairs per batch, G per lane of the group
#pragma unroll
                        for (int u = 0; u < G; ++u) {
                            const int r = tb + gl + u * LANES;
                            uint8_t va = 0, vb = 0;
                            if (r < m) { va = (uint8_t)batch_code(rowsA, r, a.packed2, s_lut); vb = (uint8_t)batch_code(rowsB, r, a.packed2, s_lut); }
                            rqA[r & 63] = va;
                            rqB[r & 63] = vb;
                        }
                        __syncwarp();
                        row_bits(tb - gl, st.tm);
                    }
                    const int tend = min(tb + 32, Tmax);
#pragma unroll 1
                    for (int t = tb; t < tend; ++t) {
                        unsigned xl = __shfl_up_sync(kFull, hr, 1, LANES);
                        unsigned el = 0;
                        if constexpr (AFFINE) el = __shfl_up_sync(kFull, er, 1, LANES);
                        const int i = t - gl;
                        if (gl == 0) { const int b = border(i) + go; xl = pack2(b, b); el = pack2(kNeg16, kNeg16); }
                        unsigned tm_next[W];
                        row_bits(i + 1, tm_next);
                        if ((unsigned)i < (unsigned)m) {
                            st.dd = diag_sigma_x2<0>(st.tm[0], dcarry, k);
                            dcarry = xl;
                            st.xleft = xl;
                            st.e = el;
                            CellX2<LOCAL, AFFINE, K, 0>::run(X, F, st, k);
                            hr = st.xleft;
                            er = st.e;
                            if constexpr (MODE == kSemiglobal) {
                                if (gl == outlane) max_column_u<K>(colbest, X, outc);
                            }
                        }
#pragma unroll
                        for (int w = 0; w < W; ++w) st.tm[w] = tm_next[w];
                    }
                }
                // result extraction: src/scoring.impala:29-137 (values only), per half
                if constexpr (GLOB) {
                    const unsigned v = __shfl_sync(kFull, pick_column(X, outc), outlane, LANES);
                    scoreA = lo16(v) - go - bias;
                    scoreB = hi16(v) - go - bias;
                } else if constexpr (MODE == kSemiglobal) {
                    unsigned best = colbest;
#pragma unroll
                    for (int c = 0; c < K; ++c)
                        if (jl + c < n) best = __vmaxs2(best, X[c]);             // last row H(m-1, j)
#pragma unroll
                    for (int o = LANES / 2; o > 0; o >>= 1) best = __vmaxs2(best, __shfl_xor_sync(kFull, best, o));
                    scoreA = max(lo16(best) - go - bias, 0);                     // candidates H(m-1,-1) = H(-1,n-1) = 0
                    scoreB = max(hi16(best) - go - bias, 0);
                } else {
                    unsigned best = __vmaxs2(st.best, st.hprev);
#pragma unroll
                    for (int o = LANES / 2; o > 0; o >>= 1) best = __vmaxs2(best, __shfl_xor_sync(kFull, best, o));
                    scoreA = lo16(best) - bias;
                    scoreB = hi16(best) - bias;
                }
                if (active && empty) scoreA = scoreB = empty_pair_score<MODE>(a, lq, ls);
            }
            if (active && gl == 0) {
                a.scores[pa] = scoreA;
                if (pb != pa) a.scores[pb] = scoreB;
            }
        }
        unsigned long long nxt = 0;
        if (lane == 0) nxt = atomicAdd(a.counter, 1ull);
        wi = (long long)__shfl_sync(kFull, nxt, 0);
    }
}

// The two lane widths as kernels.  They keep the names, and so the symbols, they had as two separate kernels: profiles
// and the ABI test find them by these.  The minimum block counts set the register caps and with them the occupancy.
template <int MODE, bool AFFINE, int K>
__global__ void __launch_bounds__(kThreads, (K >= 32 ? 4 : (K >= 16 ? 5 : 6))) batch_x2_kernel(const BatchArgs a)
{
    batch_pairs<MODE, AFFINE, K, 32>(a);
}

template <int MODE, bool AFFINE>
__global__ void __launch_bounds__(kThreads, 3) batch_x4_kernel(const BatchArgs a)
{
    batch_pairs<MODE, AFFINE, 32, 16>(a);
}

template <int MODE, bool AFFINE>
static BatchKernelFn pick_x2(int K, int lanes)
{
    if (lanes == 16) return K == 32 ? batch_x4_kernel<MODE, AFFINE> : nullptr;
    switch (K) {
        case 4: return batch_x2_kernel<MODE, AFFINE, 4>;
        case 8: return batch_x2_kernel<MODE, AFFINE, 8>;
        case 16: return batch_x2_kernel<MODE, AFFINE, 16>;
        case 32: return batch_x2_kernel<MODE, AFFINE, 32>;
    }
    return nullptr;
}

BatchKernelFn pick_batch_x2_kernel(int mode, bool affine, int K, int lanes)
{
    switch (mode) {
        case kGlobal: return affine ? pick_x2<kGlobal, true>(K, lanes) : pick_x2<kGlobal, false>(K, lanes);
        case kSemiglobal: return affine ? pick_x2<kSemiglobal, true>(K, lanes) : pick_x2<kSemiglobal, false>(K, lanes);
        default: return affine ? pick_x2<kLocal, true>(K, lanes) : pick_x2<kLocal, false>(K, lanes);
    }
}

}  // namespace anyseq
