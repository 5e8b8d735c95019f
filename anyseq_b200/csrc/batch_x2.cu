// batch_x2.cu -- the batch kernel with TWO pairs per warp, packed as 16-bit halves of every register.
//
// Short pairs (reads x windows) have scores that fit in 16 bits, and pairs are independent, so the low half
// of each register carries pair A and the high half pair B of the same shape (lenq, lens): the DPX
// instructions VIADDMNMX.S16x2 / VIMNMX3.S16x2 then relax two cells per issue slot.  Everything else is the
// batch kernel of batch.cu: one warp per work item, the longer sequence spread over the lanes as columns
// (per-lane column masks per alphabet code in shared memory), the shorter streamed as rows with a 32-step
// lane skew, borders from init_scores (src/align.impala:85-86), values only.
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

template <int K>
__device__ __forceinline__ unsigned pick_column_u(const unsigned (&X)[K], int idx)
{
    unsigned v = X[0];
#pragma unroll
    for (int c = 1; c < K; ++c)
        if (c == idx) v = X[c];
    return v;
}

template <int MODE, bool AFFINE, int K>
__global__ void __launch_bounds__(kThreads, (K >= 32 ? 4 : (K >= 16 ? 5 : 6))) batch_x2_kernel(const BatchArgs a)
{
    constexpr bool LOCAL = MODE == kLocal;
    constexpr bool GLOB = MODE == kGlobal;
    __shared__ uint8_t s_rows[kWarpsPerBlock][2][64];
    __shared__ uint8_t s_lut[256];
    extern __shared__ unsigned s_dyn[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (!a.packed2) {
        for (int x = threadIdx.x; x < 256; x += kThreads) s_lut[x] = a.lut[x];
    }
    __syncthreads();
    constexpr int W = (2 * K + 31) / 32;              // words of match bits per lane and row
    unsigned* maskA = s_dyn + (warp * 2 + 0) * a.ncodes * 32 * W;     // [code][lane][W], bits 2c
    unsigned* maskB = s_dyn + (warp * 2 + 1) * a.ncodes * 32 * W;     // [code][lane][W], bits 2c + 1
    uint8_t* rqA = s_rows[warp][0];
    uint8_t* rqB = s_rows[warp][1];
    rqA[lane] = 0; rqA[32 + lane] = 0; rqB[lane] = 0; rqB[32 + lane] = 0;
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

    const long long npp = (a.npairs + 1) / 2;
    long long pp = (long long)blockIdx.x * kWarpsPerBlock + warp;
    while (pp < npp) {
        const long long pA = 2 * pp, pB = min(2 * pp + 1, a.npairs - 1);
        const int lqA = batch_q_len(a, pA), lsA = batch_s_len(a, pA);
        const int lqB = batch_q_len(a, pB), lsB = batch_s_len(a, pB);
        const bool same_shape = lqA == lqB && lsA == lsB;
        const int npass = same_shape ? 1 : 2;
        for (int pass = 0; pass < npass; ++pass) {
            const long long pa = (same_shape || pass == 0) ? pA : pB;
            const long long pb = same_shape ? pB : pa;
            const long long qa0 = batch_q_start(a, pa), sa0 = batch_s_start(a, pa), qb0 = batch_q_start(a, pb), sb0 = batch_s_start(a, pb);
            const int lq = batch_q_len(a, pa), ls = batch_s_len(a, pa);
            int scoreA, scoreB;
            if (lq == 0 || ls == 0) {
                // quirk Q12 (see engine.cu: empty_result)
                const int L = max(lq, ls);
                scoreA = scoreB = GLOB ? (L > 0 ? a.gap_init + L * a.sp.gap_extend : 0) : (MODE == kSemiglobal ? 0 : kScoreMin);
            } else {
                const bool q_is_cols = a.cols_longer ? (lq >= ls) : (lq < ls);
                const uint8_t* colsA = q_is_cols ? a.q + qa0 : a.s + sa0;
                const uint8_t* rowsA = q_is_cols ? a.s + sa0 : a.q + qa0;
                const uint8_t* colsB = q_is_cols ? a.q + qb0 : a.s + sb0;
                const uint8_t* rowsB = q_is_cols ? a.s + sb0 : a.q + qb0;
                const int n = q_is_cols ? lq : ls;      // columns (<= 32*K)
                const int m = q_is_cols ? ls : lq;      // rows

                unsigned X[K], F[AFFINE ? K : 1];
                const int jl = lane * K;
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
                    for (int w = 0; w < W; ++w) { maskA[(cd * 32 + lane) * W + w] = 0u; maskB[(cd * 32 + lane) * W + w] = 0u; }
                }
#pragma unroll 4
                for (int c = 0; c < K; ++c) {
                    const int j = jl + c;
                    const int ca = (j < n) ? batch_code(colsA, j, a.packed2, s_lut) : 0;
                    const int cb = (j < n) ? batch_code(colsB, j, a.packed2, s_lut) : 0;
                    if (ca) maskA[(ca * 32 + lane) * W + (2 * c) / 32] |= 1u << ((2 * c) % 32);
                    if (cb) maskB[(cb * 32 + lane) * W + (2 * c) / 32] |= 2u << ((2 * c) % 32);
                }
                __syncwarp();
                auto row_bits = [&](int i, unsigned (&tm)[W]) {
                    const unsigned* pa = maskA + ((int)rqA[i & 63] * 32 + lane) * W;
                    const unsigned* pb = maskB + ((int)rqB[i & 63] * 32 + lane) * W;
#pragma unroll
                    for (int w = 0; w < W; ++w) tm[w] = pa[w] | pb[w];
                };
                unsigned dcarry;
                { const int b = (lane == 0) ? bias + go : border(jl - 1) + go; dcarry = pack2(b, b); }   // H(-1,-1) = 0
                const int outlane = (n - 1) / K, outc = (n - 1) % K;
                unsigned hr = 0, er = 0;
                unsigned colbest = pack2(kNeg16, kNeg16);    // semiglobal: max over H(i, n-1), kept by lane `outlane`
                X2State<W> st;
                st.dd = 0; st.e = 0; st.xleft = 0;
#pragma unroll
                for (int w = 0; w < W; ++w) st.tm[w] = 0u;
                st.best = k.floor2; st.hprev = k.floor2;
                const int T = m + outlane;
                for (int tb = 0; tb < T; tb += 32) {
                    __syncwarp();
                    {
                        const int r = tb + lane;
                        uint8_t va = 0, vb = 0;
                        if (r < m) { va = (uint8_t)batch_code(rowsA, r, a.packed2, s_lut); vb = (uint8_t)batch_code(rowsB, r, a.packed2, s_lut); }
                        rqA[r & 63] = va;
                        rqB[r & 63] = vb;
                        __syncwarp();
                        row_bits(tb - lane, st.tm);
                    }
                    const int tend = min(tb + 32, T);
#pragma unroll 1
                    for (int t = tb; t < tend; ++t) {
                        unsigned xl = __shfl_up_sync(kFull, hr, 1);
                        unsigned el = 0;
                        if constexpr (AFFINE) el = __shfl_up_sync(kFull, er, 1);
                        const int i = t - lane;
                        if (lane == 0) { const int b = border(i) + go; xl = pack2(b, b); el = pack2(kNeg16, kNeg16); }
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
                                if (lane == outlane) max_column_u<K>(colbest, X, outc);
                            }
                        }
#pragma unroll
                        for (int w = 0; w < W; ++w) st.tm[w] = tm_next[w];
                    }
                }
                // result extraction: src/scoring.impala:29-137 (values only), per half
                if constexpr (GLOB) {
                    const unsigned v = __shfl_sync(kFull, pick_column_u<K>(X, outc), outlane);
                    scoreA = lo16(v) - go - bias;
                    scoreB = hi16(v) - go - bias;
                } else if constexpr (MODE == kSemiglobal) {
                    unsigned best = colbest;
#pragma unroll
                    for (int c = 0; c < K; ++c)
                        if (jl + c < n) best = __vmaxs2(best, X[c]);             // last row H(m-1, j)
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) best = __vmaxs2(best, __shfl_xor_sync(kFull, best, o));
                    scoreA = max(lo16(best) - go - bias, 0);                     // candidates H(m-1,-1) = H(-1,n-1) = 0
                    scoreB = max(hi16(best) - go - bias, 0);
                } else {
                    unsigned best = __vmaxs2(st.best, st.hprev);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) best = __vmaxs2(best, __shfl_xor_sync(kFull, best, o));
                    scoreA = lo16(best) - bias;
                    scoreB = hi16(best) - bias;
                }
            }
            if (lane == 0) {
                a.scores[pa] = scoreA;
                if (pb != pa) a.scores[pb] = scoreB;
            }
        }
        unsigned long long nxt = 0;
        if (lane == 0) nxt = atomicAdd(a.counter, 1ull);
        pp = (long long)__shfl_sync(kFull, nxt, 0);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// batch_x4_kernel: FOUR pairs per warp.  Each half-warp (16 lanes x 32 columns = 512 columns) relaxes its own pair of
// pairs exactly like batch_x2_kernel does with 32 lanes.  The lane skew of a work item is 15 steps instead of 31: a
// 150-row read costs 165 instead of 181 steps (the 17 % fill/drain of the two-pair kernel becomes 9 %).  Used when the
// column sequences have at most 512 symbols (BASELINE configs[3]: 500 bp windows).
// ---------------------------------------------------------------------------------------------------------------
template <int MODE, bool AFFINE>
__global__ void __launch_bounds__(kThreads, 3) batch_x4_kernel(const BatchArgs a)
{
    constexpr int K = 32;
    constexpr int HL = 16;                           // lanes per pair of pairs
    constexpr bool LOCAL = MODE == kLocal;
    constexpr bool GLOB = MODE == kGlobal;
    __shared__ uint8_t s_rows[kWarpsPerBlock][2][2][64];
    __shared__ uint8_t s_lut[256];
    extern __shared__ unsigned s_dyn[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int half = lane >> 4, hl = lane & (HL - 1);
    if (!a.packed2) {
        for (int x = threadIdx.x; x < 256; x += kThreads) s_lut[x] = a.lut[x];
    }
    __syncthreads();
    constexpr int W = (2 * K + 31) / 32;              // words of match bits per lane and row
    // [warp][half][pair A/B][code][16 lanes][W]
    unsigned* maskA = s_dyn + ((warp * 2 + half) * 2 + 0) * a.ncodes * HL * W;
    unsigned* maskB = s_dyn + ((warp * 2 + half) * 2 + 1) * a.ncodes * HL * W;
    uint8_t* rqA = s_rows[warp][half][0];
    uint8_t* rqB = s_rows[warp][half][1];
    for (int x = hl; x < 64; x += HL) { rqA[x] = 0; rqB[x] = 0; }
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
    auto border = [&](int idx) -> int { return (GLOB ? a.sp.gap_open + idx * a.sp.gap_extend : 0) + bias; };

    const long long nquad = (a.npairs + 3) / 4;       // work items: four consecutive pairs
    long long wi = (long long)blockIdx.x * kWarpsPerBlock + warp;
    while (wi < nquad) {
        // this half's two pairs (the last item of a batch may have fewer than four)
        const long long p0 = 4 * wi + 2 * half;
        const bool have = p0 < a.npairs;
        const long long pA = have ? p0 : a.npairs - 1, pB = min(pA + 1, a.npairs - 1);
        const int lqA = batch_q_len(a, pA), lsA = batch_s_len(a, pA);
        const int lqB = batch_q_len(a, pB), lsB = batch_s_len(a, pB);
        const bool same_shape = lqA == lqB && lsA == lsB;
        for (int pass = 0; pass < 2; ++pass) {
            // pass 0: (A, B) together when they have one shape, else A with itself; pass 1: B with itself if it was left over
            const bool active = have && (pass == 0 || (!same_shape && pB != pA));
            if (!__any_sync(kFull, active)) continue;
            const long long pa = (pass == 0) ? pA : pB;
            const long long pb = (pass == 0 && same_shape) ? pB : pa;
            const long long qa0 = batch_q_start(a, pa), sa0 = batch_s_start(a, pa), qb0 = batch_q_start(a, pb), sb0 = batch_s_start(a, pb);
            const int lq = batch_q_len(a, pa), ls = batch_s_len(a, pa);
            const bool empty = lq == 0 || ls == 0;
            const bool q_is_cols = a.cols_longer ? (lq >= ls) : (lq < ls);
            const uint8_t* colsA = q_is_cols ? a.q + qa0 : a.s + sa0;
            const uint8_t* rowsA = q_is_cols ? a.s + sa0 : a.q + qa0;
            const uint8_t* colsB = q_is_cols ? a.q + qb0 : a.s + sb0;
            const uint8_t* rowsB = q_is_cols ? a.s + sb0 : a.q + qb0;
            const int n = q_is_cols ? lq : ls;      // columns (<= 16*K)
            const int m = (active && !empty) ? (q_is_cols ? ls : lq) : 0;      // rows; 0: this half only keeps the warp company

            unsigned X[K], F[AFFINE ? K : 1];
            const int jl = hl * K;
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
                for (int w = 0; w < W; ++w) { maskA[(cd * HL + hl) * W + w] = 0u; maskB[(cd * HL + hl) * W + w] = 0u; }
            }
            if (m > 0) {
#pragma unroll 4
                for (int c = 0; c < K; ++c) {
                    const int j = jl + c;
                    const int ca = (j < n) ? batch_code(colsA, j, a.packed2, s_lut) : 0;
                    const int cb = (j < n) ? batch_code(colsB, j, a.packed2, s_lut) : 0;
                    if (ca) maskA[(ca * HL + hl) * W + (2 * c) / 32] |= 1u << ((2 * c) % 32);
                    if (cb) maskB[(cb * HL + hl) * W + (2 * c) / 32] |= 2u << ((2 * c) % 32);
                }
            }
            __syncwarp();
            auto row_bits = [&](int i, unsigned (&tm)[W]) {
                const unsigned* pa_ = maskA + ((int)rqA[i & 63] * HL + hl) * W;
                const unsigned* pb_ = maskB + ((int)rqB[i & 63] * HL + hl) * W;
#pragma unroll
                for (int w = 0; w < W; ++w) tm[w] = pa_[w] | pb_[w];
            };
            unsigned dcarry;
            { const int b = (hl == 0) ? bias + go : border(jl - 1) + go; dcarry = pack2(b, b); }   // H(-1,-1) = 0
            const int outlane = m > 0 ? (n - 1) / K : 0, outc = m > 0 ? (n - 1) % K : 0;
            unsigned hr = 0, er = 0;
            unsigned colbest = pack2(kNeg16, kNeg16);
            X2State<W> st;
            st.dd = 0; st.e = 0; st.xleft = 0;
#pragma unroll
            for (int w = 0; w < W; ++w) st.tm[w] = 0u;
            st.best = k.floor2; st.hprev = k.floor2;
            const int T = m > 0 ? m + outlane : 0;
            const int Tmax = max(T, __shfl_xor_sync(kFull, T, 16));
            for (int tb = 0; tb < Tmax; tb += 32) {
                __syncwarp();
                {
                    // 32 rows of both pairs per batch, two per lane of the half
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        const int r = tb + hl + u * HL;
                        uint8_t va = 0, vb = 0;
                        if (r < m) { va = (uint8_t)batch_code(rowsA, r, a.packed2, s_lut); vb = (uint8_t)batch_code(rowsB, r, a.packed2, s_lut); }
                        rqA[r & 63] = va;
                        rqB[r & 63] = vb;
                    }
                    __syncwarp();
                    row_bits(tb - hl, st.tm);
                }
                const int tend = min(tb + 32, Tmax);
#pragma unroll 1
                for (int t = tb; t < tend; ++t) {
                    unsigned xl = __shfl_up_sync(kFull, hr, 1, HL);
                    unsigned el = 0;
                    if constexpr (AFFINE) el = __shfl_up_sync(kFull, er, 1, HL);
                    const int i = t - hl;
                    if (hl == 0) { const int b = border(i) + go; xl = pack2(b, b); el = pack2(kNeg16, kNeg16); }
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
                            if (hl == outlane) max_column_u<K>(colbest, X, outc);
                        }
                    }
#pragma unroll
                    for (int w = 0; w < W; ++w) st.tm[w] = tm_next[w];
                }
            }
            // result extraction per half (src/scoring.impala:29-137, values only)
            int scoreA, scoreB;
            if constexpr (GLOB) {
                const unsigned v = __shfl_sync(kFull, pick_column_u<K>(X, outc), outlane, HL);
                scoreA = lo16(v) - go - bias;
                scoreB = hi16(v) - go - bias;
            } else if constexpr (MODE == kSemiglobal) {
                unsigned best = colbest;
#pragma unroll
                for (int c = 0; c < K; ++c)
                    if (jl + c < n) best = __vmaxs2(best, X[c]);
#pragma unroll
                for (int o = HL / 2; o > 0; o >>= 1) best = __vmaxs2(best, __shfl_xor_sync(kFull, best, o));
                scoreA = max(lo16(best) - go - bias, 0);
                scoreB = max(hi16(best) - go - bias, 0);
            } else {
                unsigned best = __vmaxs2(st.best, st.hprev);
#pragma unroll
                for (int o = HL / 2; o > 0; o >>= 1) best = __vmaxs2(best, __shfl_xor_sync(kFull, best, o));
                scoreA = lo16(best) - bias;
                scoreB = hi16(best) - bias;
            }
            if (active && empty) {
                const int L = max(lq, ls);     // quirk Q12 (see engine.cu: empty_result)
                scoreA = scoreB = GLOB ? (L > 0 ? a.gap_init + L * a.sp.gap_extend : 0) : (MODE == kSemiglobal ? 0 : kScoreMin);
            }
            if (active && hl == 0) {
                a.scores[pa] = scoreA;
                if (pb != pa) a.scores[pb] = scoreB;
            }
        }
        unsigned long long nxt = 0;
        if (lane == 0) nxt = atomicAdd(a.counter, 1ull);
        wi = (long long)__shfl_sync(kFull, nxt, 0);
    }
}

BatchKernelFn pick_batch_x4_kernel(int mode, bool affine)
{
    switch (mode) {
        case kGlobal: return affine ? batch_x4_kernel<kGlobal, true> : batch_x4_kernel<kGlobal, false>;
        case kSemiglobal: return affine ? batch_x4_kernel<kSemiglobal, true> : batch_x4_kernel<kSemiglobal, false>;
        default: return affine ? batch_x4_kernel<kLocal, true> : batch_x4_kernel<kLocal, false>;
    }
}

template <int MODE, bool AFFINE>
static BatchKernelFn pick_x2_k(int K)
{
    switch (K) {
        case 4: return batch_x2_kernel<MODE, AFFINE, 4>;
        case 8: return batch_x2_kernel<MODE, AFFINE, 8>;
        case 16: return batch_x2_kernel<MODE, AFFINE, 16>;
        case 32: return batch_x2_kernel<MODE, AFFINE, 32>;
    }
    return nullptr;
}

BatchKernelFn pick_batch_x2_kernel(int mode, bool affine, int K)
{
    switch (mode) {
        case kGlobal: return affine ? pick_x2_k<kGlobal, true>(K) : pick_x2_k<kGlobal, false>(K);
        case kSemiglobal: return affine ? pick_x2_k<kSemiglobal, true>(K) : pick_x2_k<kSemiglobal, false>(K);
        default: return affine ? pick_x2_k<kLocal, true>(K) : pick_x2_k<kLocal, false>(K);
    }
}

}  // namespace anyseq
