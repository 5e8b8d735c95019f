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

// The body of batch_kernel / batch_ends_kernel, included into both so that each is a kernel of its own code (as a
// shared inline function the body compiles to different SASS for the score-only kernels)
template <int MODE, bool AFFINE, int K, bool MASK>
__global__ void __launch_bounds__(kThreads, (K >= 32 ? 4 : (K >= 16 ? 5 : 6))) batch_kernel(const BatchArgs a)
{
    constexpr bool ENDS = false;
#include "batch_kernel_body.inl"
}

// ENDS: also the end cell of every pair (anyseq_score_batch_ends).  Semiglobal: lane `outlane` keeps the first row
// of the last column's maximum (strict '>'), the warp takes the first column of the last row's maximum, and
// semiglobal_end applies the caller's precedence.  Local: pairs run with the subject as columns and the cells track
// the lane's first maximum in its own row-major order (Cell TRACK); the warp takes the lowest (row, column) among
// the lanes holding the maximum -- the first maximum of the matrix in row-major order (see batch_align.cu).
template <int MODE, bool AFFINE, int K, bool MASK>
__global__ void __launch_bounds__(kThreads, (K >= 32 ? 4 : (K >= 16 ? 5 : 6))) batch_ends_kernel(const BatchArgs a)
{
    constexpr bool ENDS = true;
#include "batch_kernel_body.inl"
}

template <int MODE, bool AFFINE, bool ENDS>
static BatchKernelFn pick_batch_kernel_k(int K, bool mask)
{
#define ANYSEQ_PICK(KK, M) return ENDS ? batch_ends_kernel<MODE, AFFINE, KK, M> : batch_kernel<MODE, AFFINE, KK, M>
    if (mask) {
        switch (K) {
            case 4: ANYSEQ_PICK(4, true);
            case 8: ANYSEQ_PICK(8, true);
            case 16: ANYSEQ_PICK(16, true);
            case 32: ANYSEQ_PICK(32, true);
        }
    } else {
        switch (K) {
            case 4: ANYSEQ_PICK(4, false);
            case 8: ANYSEQ_PICK(8, false);
            case 16: ANYSEQ_PICK(16, false);
        }
    }
#undef ANYSEQ_PICK
    return nullptr;
}

template <int MODE>
static BatchKernelFn pick_batch_kernel_mode(bool affine, int K, bool mask, bool ends)
{
    if (ends) return affine ? pick_batch_kernel_k<MODE, true, true>(K, mask) : pick_batch_kernel_k<MODE, false, true>(K, mask);
    return affine ? pick_batch_kernel_k<MODE, true, false>(K, mask) : pick_batch_kernel_k<MODE, false, false>(K, mask);
}

static BatchKernelFn pick_batch_kernel(int mode, bool affine, int K, bool mask, bool ends)
{
    switch (mode) {
        case kGlobal: return pick_batch_kernel_mode<kGlobal>(affine, K, mask, ends);
        case kSemiglobal: return pick_batch_kernel_mode<kSemiglobal>(affine, K, mask, ends);
        default: return pick_batch_kernel_mode<kLocal>(affine, K, mask, ends);
    }
}

// Chooses the batch kernel for pairs of at most (max_long, max_short) symbols, queries of at most max_q and subjects
// of at most max_s (alphabet already analysed: use_mask_, ncodes_) and launches it on `st`; ba carries the input
// description, the score array and, when ba.ends is set, the end-cell array (the _ends kernels).
int Engine::launch_batch(const anyseq_scoring& sc, const ScoreParams& sp, bool affine, BatchArgs& ba, int max_long,
                         int max_short, int max_q, int max_s, cudaStream_t st)
{
    const long long npairs = ba.npairs;
    // the bound is symmetric in the lengths and grows with both: the longest pair lengths bound every pair
    const int rc = check_score_range(sc, max_long, max_short);
    if (rc) return rc;
    const int limit = use_mask_ ? 1024 : 512;
    const bool ends = ba.ends != nullptr;
    // local end cells follow the row-major order of (query, subject), so those pairs always run with the subject as
    // columns (the kernels ignore cols_longer then)
    const bool subject_cols = ends && sc.mode == ANYSEQ_LOCAL;
    int cols_longer, ncols;
    if (subject_cols) {
        if (max_s > limit) {
            char buf[240];
            std::snprintf(buf, sizeof(buf), "batch end cells of local alignments: a subject of %d symbols is longer than %d; "
                          "score such pairs with anyseq_score and the local_end_cell option", max_s, limit);
            set_last_error(buf);
            return ANYSEQ_ERR_UNSUPPORTED;
        }
        cols_longer = 0;
        ncols = max_s;
    } else if (max_long <= limit) { cols_longer = 1; ncols = max_long; }
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
        const long long rows_max = subject_cols ? max_q : cols_longer ? max_short : max_long;
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
    BatchKernelFn fn = packed ? pick_batch_x2_kernel(sc.mode, affine, K, lanes, ends)
                              : pick_batch_kernel(sc.mode, affine, K, use_mask_, ends);
    if (!fn) { set_last_error("no batch kernel for this configuration"); return ANYSEQ_ERR_UNSUPPORTED; }
    // one column-mask set per pair of a warp, W words per lane, code and row; packed kernels spread the match bits to
    // every other bit (2 K bits per lane and row)
    const int W = packed ? (2 * K + 31) / 32 : 1;
    const int pairs_per_warp = packed ? 2 * (32 / lanes) : 1;
    const size_t dyn = use_mask_ ? sizeof(unsigned) * lanes * W * (size_t)ncodes_ * pairs_per_warp * kWarpsPerBlock : 0;
    if (ends) {
        // the local 16-bit ends kernels keep a row per lane and half in static shared memory (up to 32 KiB a block);
        // with the column masks of a larger alphabet the block then needs more than the default 48 KiB, so these
        // kernels may take up to the opt-in limit (the same value from every caller: no call lowers another's)
        cudaFuncAttributes fa;
        ANYSEQ_CUDA_CHECK(cudaFuncGetAttributes(&fa, fn));
        if (fa.sharedSizeBytes + dyn > (size_t)(48 << 10)) {
            int optin = 0;
            ANYSEQ_CUDA_CHECK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
            if ((size_t)optin > fa.sharedSizeBytes)
                ANYSEQ_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                       optin - (int)fa.sharedSizeBytes));
        }
    }
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
                               anyseq_result* out, int32_t* d_ends)
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
    ba.ends = d_ends;
    // totals (for the alphabet scan) and length statistics
    long long tot[2] = {0, 0};
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(&tot[0], d_qoff + npairs, sizeof(long long), cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(&tot[1], d_soff + npairs, sizeof(long long), cudaMemcpyDeviceToHost, stream_));
    int max_long, max_short, max_q, max_s;
    if ((rc = batch_len_stats(ba, &max_long, &max_short, &max_q, &max_s))) return rc;
    if ((rc = analyse_alphabet(d_q, tot[0], d_s, tot[1]))) return rc;
    if ((rc = launch_batch(sc, sp, affine, ba, max_long, max_short, max_q, max_s, stream_))) return rc;
    return batch_epilogue(5, out);
}

}  // namespace anyseq
