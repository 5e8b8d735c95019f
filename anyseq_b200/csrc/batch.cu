// batch.cu -- batches of independent short pairs (BASELINE.json configs[3]:
// 10^7 reads of 150 bp vs 500 bp windows), score only.
//
// One WARP per pair, the whole DP in registers: the longer sequence of a pair
// (<= 32*K symbols) is spread over the lanes as columns, the shorter one is
// streamed as rows -- the same lane-skewed wavefront and the same DPX/IMAD cell
// as the strip kernel (strip_kernel.cuh: Cell<>), but with no inter-strip
// traffic at all: borders are init_scores (src/align.impala:85-86) generated
// in registers, results are reduced in the warp.  Scores of all three schemes
// are invariant under transposition (linear and Gotoh costs are symmetric in
// the two sequences; the semiglobal scheme of src/scoring.impala:39-77 frees
// the end gaps of both), so picking the orientation per pair is legal for
// score-only work.  Pairs shard over GPUs by contiguous ranges with no
// data-path collective (SURVEY.md 8e).
#include "engine.cuh"
#include "strip_kernel.cuh"
#include "batch.cuh"

#include <algorithm>
#include <cstring>

namespace anyseq {

// stats[0] = max over pairs of max(lenq, lens), stats[1] = max over pairs of min(lenq, lens), stats[2] / stats[3] = max
// over pairs of lenq / lens, clamped to 2^31 - 1; stats[4] = 1 when a pair has a negative length (decreasing offsets)
__global__ void batch_stats_kernel(const BatchArgs a, int* __restrict__ stats)
{
    int mx = 0, mn = 0, mq = 0, ms = 0, neg = 0;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < a.npairs; p += (long long)gridDim.x * blockDim.x) {
        const long long lq = batch_q_len(a, p), ls = batch_s_len(a, p);
        const long long hi = lq > ls ? lq : ls, lo = lq > ls ? ls : lq;
        mx = max(mx, (int)min(hi, (long long)0x7fffffff));
        mn = max(mn, (int)min(lo, (long long)0x7fffffff));
        mq = max(mq, (int)min(lq, (long long)0x7fffffff));
        ms = max(ms, (int)min(ls, (long long)0x7fffffff));
        neg |= lo < 0;
    }
    for (int o = 16; o > 0; o >>= 1) {
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        mn = max(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mq = max(mq, __shfl_xor_sync(0xffffffffu, mq, o));
        ms = max(ms, __shfl_xor_sync(0xffffffffu, ms, o));
        neg |= __shfl_xor_sync(0xffffffffu, neg, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(&stats[0], mx); atomicMax(&stats[1], mn); atomicMax(&stats[2], mq); atomicMax(&stats[3], ms);
        if (neg) stats[4] = 1;
    }
}

template <int MODE, bool AFFINE, int K, bool MASK>
__global__ void __launch_bounds__(kThreads, (K >= 32 ? 4 : (K >= 16 ? 5 : 6))) batch_kernel(const BatchArgs a)
{
    constexpr bool LOCAL = MODE == kLocal;
    constexpr bool GLOB = MODE == kGlobal;
    __shared__ uint8_t s_rows[kWarpsPerBlock][64];
    __shared__ uint8_t s_lut[MASK ? 256 : 4];
    extern __shared__ unsigned s_dyn[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if constexpr (MASK) {
        if (!a.packed2) {
            for (int x = threadIdx.x; x < 256; x += kThreads) s_lut[x] = a.lut[x];
        }
        __syncthreads();
    }
    unsigned* s_mask = s_dyn + warp * a.ncodes * 32;
    uint8_t* rq = s_rows[warp];
    rq[lane] = 0;
    rq[32 + lane] = 0;
    __syncwarp();

    const int go = AFFINE ? a.sp.gap_open : 0;
    StepConst k;
    k.one = a.one;
    k.ge = a.sp.gap_extend;
    k.go = go;
    k.diff_o = a.sp.diff - go;
    k.same_o = a.sp.same - go;
    k.nvalid = K;
    k.outc = K - 1;
    // border(k) = H(k,-1) = H(-1,k): src/align.impala:85-86 (+ Gotoh opening cost)
    auto border = [&](int idx) -> int { return GLOB ? a.sp.gap_open + idx * a.sp.gap_extend : 0; };

    long long pair = (long long)blockIdx.x * kWarpsPerBlock + warp;
    while (pair < a.npairs) {
        const long long q0 = batch_q_start(a, pair), s0 = batch_s_start(a, pair);
        const int lq = batch_q_len(a, pair), ls = batch_s_len(a, pair);
        int score;
        if (lq == 0 || ls == 0) {
            score = empty_pair_score<MODE>(a, lq, ls);
        } else {
            const bool q_is_cols = a.cols_longer ? (lq >= ls) : (lq < ls);
            const uint8_t* cols = q_is_cols ? a.q + q0 : a.s + s0;
            const uint8_t* rows = q_is_cols ? a.s + s0 : a.q + q0;
            const int n = q_is_cols ? lq : ls;      // columns (<= 32*K)
            const int m = q_is_cols ? ls : lq;      // rows

            int X[K], F[AFFINE ? K : 1], sc[MASK ? 1 : K];
            const int jl = lane * K;
#pragma unroll
            for (int c = 0; c < K; ++c) X[c] = border(jl + c) + go;
            if constexpr (AFFINE) {
#pragma unroll
                for (int c = 0; c < K; ++c) F[c] = kNegInf;
            } else {
                F[0] = 0;
            }
            if constexpr (MASK) {
                sc[0] = 0;
                __syncwarp();
                for (int cd = 0; cd < a.ncodes; ++cd) s_mask[cd * 32 + lane] = 0u;
#pragma unroll 4
                for (int c = 0; c < K; ++c) {
                    const int j = jl + c;
                    const int cd = (j < n) ? batch_code(cols, j, a.packed2, s_lut) : 0;
                    if (cd) s_mask[cd * 32 + lane] |= 1u << c;
                }
                __syncwarp();
            } else {
#pragma unroll
                for (int c = 0; c < K; ++c) sc[c] = (jl + c < n) ? (int)cols[jl + c] : 0x7fff;
            }
            int dcarry = (lane == 0) ? go : border(jl - 1) + go;     // H(-1, jl-1) in X form; H(-1,-1) = 0
            const int outlane = (n - 1) / K, outc = (n - 1) % K;
            int hr = 0, er = 0;
            int colbest = kScoreMin;     // semiglobal: max over H(i, n-1), kept by lane `outlane`
            StepState<1> st;
            st.dd = 0; st.e = 0; st.xleft = 0; st.best = kScoreMin; st.hprev = kScoreMin; st.es = 0; st.xs = 0; st.tm[0] = 0u; st.qc = 0;
            auto row_mask = [&](int i) -> unsigned { return s_mask[(int)rq[i & 63] * 32 + lane]; };
            const int T = m + outlane;
            for (int tb = 0; tb < T; tb += 32) {
                __syncwarp();
                {
                    const int r = tb + lane;
                    uint8_t v = 0;
                    if (r < m) v = MASK ? (uint8_t)batch_code(rows, r, a.packed2, s_lut) : rows[r];
                    rq[r & 63] = v;
                    __syncwarp();
                    if constexpr (MASK) st.tm[0] = row_mask(tb - lane);
                }
                const int tend = min(tb + 32, T);
#pragma unroll 1
                for (int t = tb; t < tend; ++t) {
                    int xl = __shfl_up_sync(kFull, hr, 1);
                    int el = 0;
                    if constexpr (AFFINE) el = __shfl_up_sync(kFull, er, 1);
                    const int i = t - lane;
                    if (lane == 0) { xl = border(i) + go; el = kNegInf; }
                    unsigned mask_next = 0u;
                    if constexpr (MASK) mask_next = row_mask(i + 1);
                    if ((unsigned)i < (unsigned)m) {
                        if constexpr (MASK) {
                            st.dd = diag_plus_sigma_mask<0>(st.tm[0], dcarry, k.one, k.diff_o, k.same_o);
                        } else {
                            st.qc = rq[i & 63];
                            st.dd = diag_plus_sigma(st.qc, sc[0], dcarry, k.one, k.diff_o, k.same_o);
                        }
                        dcarry = xl;
                        st.xleft = xl;
                        st.e = el;
                        Cell<LOCAL, AFFINE, K, false, MASK, 1, 0, 0, true>::run(X, F, sc, st, k);    // coupled cells
                        hr = st.xleft;
                        er = st.e;
                        if constexpr (MODE == kSemiglobal) {
                            if (lane == outlane) colbest = max(colbest, pick_column(X, outc));
                        }
                    }
                    if constexpr (MASK) st.tm[0] = mask_next;
                }
            }
            // result extraction: src/scoring.impala:29-137 (values only)
            if constexpr (GLOB) {
                score = __shfl_sync(kFull, pick_column(X, outc), outlane) - go;
            } else if constexpr (MODE == kSemiglobal) {
                int best = colbest;
#pragma unroll
                for (int c = 0; c < K; ++c)
                    if (jl + c < n) best = max(best, X[c]);           // last row H(m-1, j)
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(kFull, best, o));
                score = max(best - go, 0);                             // candidates H(m-1,-1) = H(-1,n-1) = 0
            } else {
                int best = st.best;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(kFull, best, o));
                score = best;
            }
        }
        if (lane == 0) a.scores[pair] = score;
        unsigned long long nxt = 0;
        if (lane == 0) nxt = atomicAdd(a.counter, 1ull);
        pair = (long long)__shfl_sync(kFull, nxt, 0);
    }
}


template <int MODE, bool AFFINE>
static BatchKernelFn pick_batch_kernel_k(int K, bool mask)
{
    if (mask) {
        switch (K) {
            case 4: return batch_kernel<MODE, AFFINE, 4, true>;
            case 8: return batch_kernel<MODE, AFFINE, 8, true>;
            case 16: return batch_kernel<MODE, AFFINE, 16, true>;
            case 32: return batch_kernel<MODE, AFFINE, 32, true>;
        }
    } else {
        switch (K) {
            case 4: return batch_kernel<MODE, AFFINE, 4, false>;
            case 8: return batch_kernel<MODE, AFFINE, 8, false>;
            case 16: return batch_kernel<MODE, AFFINE, 16, false>;
        }
    }
    return nullptr;
}

static BatchKernelFn pick_batch_kernel(int mode, bool affine, int K, bool mask)
{
    switch (mode) {
        case kGlobal: return affine ? pick_batch_kernel_k<kGlobal, true>(K, mask) : pick_batch_kernel_k<kGlobal, false>(K, mask);
        case kSemiglobal: return affine ? pick_batch_kernel_k<kSemiglobal, true>(K, mask) : pick_batch_kernel_k<kSemiglobal, false>(K, mask);
        default: return affine ? pick_batch_kernel_k<kLocal, true>(K, mask) : pick_batch_kernel_k<kLocal, false>(K, mask);
    }
}

// Chooses the batch kernel for pairs of at most (max_long, max_short) symbols (alphabet already analysed: use_mask_,
// ncodes_) and launches it on `st`; ba carries the input description and the score array.
int Engine::launch_batch(const anyseq_scoring& sc, const ScoreParams& sp, bool affine, BatchArgs& ba, int max_long,
                         int max_short, cudaStream_t st)
{
    const long long npairs = ba.npairs;
    // the bound is symmetric in the lengths and grows with both: the longest pair lengths bound every pair
    const int rc = check_score_range(sc, max_long, max_short);
    if (rc) return rc;
    const int limit = use_mask_ ? 1024 : 512;
    int cols_longer, ncols;
    if (max_long <= limit) { cols_longer = 1; ncols = max_long; }
    else if (max_short <= limit) { cols_longer = 0; ncols = max_short; }
    else {
        set_last_error("batch kernel: every pair needs one sequence of at most 1024 symbols (512 for large alphabets); "
                       "use anyseq_score for long pairs");
        return ANYSEQ_ERR_UNSUPPORTED;
    }
    int K = 4;
    while (32 * K < ncols) K *= 2;
    // Packed 16-bit kernels (batch_x2.cu, two pairs per warp): only when every value a pair of these lengths can
    // produce fits a non-negative 16-bit half after adding `bias` (see batch_x2.cu).  Bounds: any cell is at least
    // the all-gap path 2 gi + (rows + cols + 2) ge; at most max(same, diff, 0) * min(rows, cols), since a path has
    // at most min(rows, cols) diagonal steps and its gap steps are <= 0 (diff > same: a run of mismatches is the
    // best path); columns are padded to 32 K.
    int bias = 0;
    bool packed = false;
    if (use_mask_ && tune.batch_packed) {
        const long long rows_max = cols_longer ? max_short : max_long;
        const long long cols_pad = 32LL * K;
        const long long go = affine ? sp.gap_open : 0;
        const long long hmin = 2LL * sc.gap_init + (rows_max + cols_pad + 2) * sc.gap_extend;
        const long long lowest = hmin + go + std::min<long long>(0, std::min(sc.same, sc.diff));
        const long long hmax = std::max<long long>({sc.same, sc.diff, 0}) * std::min(rows_max, cols_pad);
        const long long b = -lowest + 8;
        const long long small = std::max<long long>({std::llabs(sc.same), std::llabs(sc.diff), std::llabs(go), std::llabs(sc.gap_extend)});
        if (b + hmax + 2 * small < 32000 && small < 2000) { packed = true; bias = (int)b; }
    }
    // four pairs per warp (groups of 16 lanes x 32 columns) when the column sequences fit a half-warp
    const bool quad = packed && tune.batch_quad && ncols <= 512;
    const int lanes = quad ? 16 : 32;     // lanes per group; a packed group relaxes two pairs
    if (quad) K = 32;
    BatchKernelFn fn = packed ? pick_batch_x2_kernel(sc.mode, affine, K, lanes) : pick_batch_kernel(sc.mode, affine, K, use_mask_);
    if (!fn) { set_last_error("no batch kernel for this configuration"); return ANYSEQ_ERR_UNSUPPORTED; }
    // one column-mask set per pair of a warp, W words per lane, code and row; packed kernels spread the match bits to
    // every other bit (2 K bits per lane and row)
    const int W = packed ? (2 * K + 31) / 32 : 1;
    const int pairs_per_warp = packed ? 2 * (32 / lanes) : 1;
    const size_t dyn = use_mask_ ? sizeof(unsigned) * lanes * W * (size_t)ncodes_ * pairs_per_warp * kWarpsPerBlock : 0;
    int nb = 0;
    ANYSEQ_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, kThreads, dyn));
    if (nb < 1) { set_last_error("batch kernel does not fit on an SM"); return ANYSEQ_ERR_UNSUPPORTED; }
    const long long units = (npairs + pairs_per_warp - 1) / pairs_per_warp;      // work items claimed by the warps
    const int grid = (int)std::min<long long>((long long)nb * sm_count, (units + kWarpsPerBlock - 1) / kWarpsPerBlock);
    ba.sp = sp;
    ba.gap_init = sc.gap_init;
    ba.mode = sc.mode;
    ba.one = 1;
    ba.ncodes = ncodes_;
    ba.cols_longer = cols_longer;
    ba.bias = bias;
    ba.lut = lut_.as<uint8_t>();
    ba.counter = reinterpret_cast<unsigned long long*>(misc_.as<int>() + kMiscCounter);
    const unsigned long long first = (unsigned long long)grid * kWarpsPerBlock;
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(ba.counter, &first, sizeof(first), cudaMemcpyHostToDevice, st));
    fn<<<grid, kThreads, dyn, st>>>(ba);
    ANYSEQ_CUDA_CHECK(cudaGetLastError());
    return ANYSEQ_OK;
}

int batch_prologue(const anyseq_scoring& sc, int64_t npairs, ScoreParams* sp, bool* affine, anyseq_result* out)
{
    const int rc = make_score_params(sc, sp, affine);
    if (rc) return rc;
    if (out) { std::memset(out, 0, sizeof(*out)); out->end_i = out->end_j = -1; }
    if (npairs > 0 && sc.mode == ANYSEQ_LOCAL && sc.diff > 0) {
        set_last_error("batch local alignment needs diff <= 0 (padded columns must not outscore real ones)");
        return ANYSEQ_ERR_UNSUPPORTED;
    }
    return ANYSEQ_OK;
}

int Engine::batch_len_stats(const BatchArgs& ba, int* max_long, int* max_short, int* max_q, int* max_s, bool* negative)
{
    int* d_stats = misc_.as<int>() + kMiscOut;
    ANYSEQ_CUDA_CHECK(cudaMemsetAsync(d_stats, 0, sizeof(int) * 5, stream_));
    batch_stats_kernel<<<(int)std::min<long long>(sm_count * 8, (ba.npairs + 255) / 256), 256, 0, stream_>>>(ba, d_stats);
    ANYSEQ_CUDA_CHECK(cudaGetLastError());
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(h_misc_ + kMiscOut, d_stats, sizeof(int) * 5, cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(stream_));
    *max_long = h_misc_[kMiscOut];
    *max_short = h_misc_[kMiscOut + 1];
    if (max_q) *max_q = h_misc_[kMiscOut + 2];
    if (max_s) *max_s = h_misc_[kMiscOut + 3];
    if (negative) *negative = h_misc_[kMiscOut + 4] != 0;
    return ANYSEQ_OK;
}

int Engine::batch_epilogue(int launches, anyseq_result* out)
{
    ANYSEQ_CUDA_CHECK(cudaEventRecord(ev1_, stream_));
    ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(stream_));
    float ms = 0.f;
    ANYSEQ_CUDA_CHECK(cudaEventElapsedTime(&ms, ev0_, ev1_));
    if (out) { out->kernel_ms = ms; out->kernel_launches = launches; }
    return ANYSEQ_OK;
}

int Engine::score_batch_device(const anyseq_scoring& sc, const uint8_t* d_q, const int64_t* d_qoff,
                               const uint8_t* d_s, const int64_t* d_soff, int64_t npairs, int32_t* d_scores,
                               anyseq_result* out)
{
    std::lock_guard<std::recursive_mutex> lock(mu_);
    ANYSEQ_CUDA_CHECK(cudaSetDevice(device));
    ScoreParams sp;
    bool affine;
    int rc = batch_prologue(sc, npairs, &sp, &affine, out);
    if (rc || npairs == 0) return rc;
    ANYSEQ_CUDA_CHECK(cudaEventRecord(ev0_, stream_));
    BatchArgs ba;
    std::memset(&ba, 0, sizeof(ba));
    ba.q = d_q;
    ba.qoff = reinterpret_cast<const long long*>(d_qoff);
    ba.s = d_s;
    ba.soff = reinterpret_cast<const long long*>(d_soff);
    ba.npairs = npairs;
    ba.scores = d_scores;
    // totals (for the alphabet scan) and length statistics
    long long tot[2] = {0, 0};
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(&tot[0], d_qoff + npairs, sizeof(long long), cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(&tot[1], d_soff + npairs, sizeof(long long), cudaMemcpyDeviceToHost, stream_));
    int max_long, max_short;
    if ((rc = batch_len_stats(ba, &max_long, &max_short))) return rc;
    if ((rc = analyse_alphabet(d_q, tot[0], d_s, tot[1]))) return rc;
    if ((rc = launch_batch(sc, sp, affine, ba, max_long, max_short, stream_))) return rc;
    return batch_epilogue(5, out);
}

}  // namespace anyseq
