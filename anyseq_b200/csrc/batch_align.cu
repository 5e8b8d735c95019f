// batch_align.cu -- full-matrix tracebacks of batches of short pairs (anyseq_align_batch): for every pair the score,
// end cell, start cell and aligned rows anyseq_align_full gives for that pair alone (traceback_full.cu,
// src/align.impala:190-216), for subjects of at most 1024 symbols.
//
// One warp per pair, one launch for the batch.  The subject is spread over the lanes as columns (K per lane), query
// rows stream through the lane-skewed wavefront of batch_kernel with the borders generated in registers, and every
// cell is fulltb_cell, the cell of fulltb_dp_kernel.  A lane stores the 4 predecessor bits of its K cells of a row as
// one vector store into the warp's slab of global scratch (row-major, 16 K bytes a row).  The warp then finds the end
// cell by the rules of finish_score_kernel / local_end_cell_kernel and walks the slab with fulltb_walk_step, staging
// 32 x 64-cell windows of predecessors through shared memory so that no step waits for a global load.
//
// Pairs are never transposed (unlike score-only batches): the tie order diag > E > F of the walk and the row-major
// rule of the local end cell are not symmetric in the two sequences.  Linear and Gotoh gaps run the same kernel:
// with one block per pair the borders E(i, -1) = F(-1, j) = -inf are the same for both schemes, and linear gaps are
// gi = 0 of the same cell (E and F never extend), so there is no affine flag at all.
#include "engine.cuh"
#include "strip_kernel.cuh"
#include "batch.cuh"
#include "traceback_full.cuh"

#include <algorithm>
#include <cstring>
#include <vector>

namespace anyseq {

constexpr int kWinRows = 32, kWinCols = 64;   // walk window: 32 rows x 64 columns = 32 x 32 bytes of nibbles
constexpr int kMaxAlignBatchSubject = 1024;

// pred: kWarpsPerBlock * gridDim.x slabs of `slab` bytes, one per warp; pair p's aligned rows start at
// alq / als + (q_off[p] - q_off[0]) + (s_off[p] - s_off[0])
template <int MODE, int K>
__global__ void __launch_bounds__(kThreads)
batch_align_kernel(const BatchArgs a, int* __restrict__ ends, int* __restrict__ starts, uint8_t* __restrict__ alq,
                   uint8_t* __restrict__ als, uint8_t* __restrict__ pred_all, size_t slab)
{
    constexpr bool LOCAL = MODE == kLocal;
    constexpr bool GLOB = MODE == kGlobal;
    constexpr int RB = 16 * K;                 // bytes of one predecessor row: 32 lanes x K nibbles
    __shared__ uint8_t s_rows[kWarpsPerBlock][64];
    __shared__ uint4 s_win[kWarpsPerBlock][kWinRows][kWinCols / 32];
    __shared__ uint8_t s_wq[kWarpsPerBlock][kWinRows];
    __shared__ uint8_t s_ws[kWarpsPerBlock][kWinCols];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* rq = s_rows[warp];
    uint8_t* pred = pred_all + (size_t)(blockIdx.x * kWarpsPerBlock + warp) * slab;
    const uint8_t* win = reinterpret_cast<const uint8_t*>(s_win[warp]);
    const int gi = a.gap_init, ge = a.sp.gap_extend, go = a.sp.gap_open, same = a.sp.same, diff = a.sp.diff;
    // H(k, -1) = H(-1, k): src/align.impala:85-86 (+ Gotoh opening cost), as fulltb_dp_kernel
    auto border = [&](int k) -> int { return GLOB ? gi + (k + 1) * ge : 0; };

    long long pair = (long long)blockIdx.x * kWarpsPerBlock + warp;
    while (pair < a.npairs) {
        const long long q0 = a.qoff[pair], s0 = a.soff[pair];
        const int m = (int)(a.qoff[pair + 1] - q0), n = (int)(a.soff[pair + 1] - s0);
        const uint8_t* q = a.q + q0;
        const uint8_t* s = a.s + s0;
        const long long o = (q0 - a.qoff[0]) + (s0 - a.soff[0]);
        int score, ei = m - 1, ej = n - 1, i = -1, j = -1;
        if (m == 0 || n == 0) {
            score = empty_pair_score<MODE>(a, m, n);              // blank rows, start (0, 0): as anyseq_align_full
        } else {
            const int jl = lane * K;
            const int nl = (n - 1) / K + 1;                        // lanes holding real columns
            const int nvalid = n - jl;                             // real columns of this lane (if < K)
            const int outc = (n - 1) - (nl - 1) * K;
            int H[K], F[K];
            unsigned scw[(K + 3) / 4];                             // the lane's subject symbols, four a word
#pragma unroll
            for (int w = 0; w < (K + 3) / 4; ++w) scw[w] = 0u;
#pragma unroll
            for (int c = 0; c < K; ++c) {
                H[c] = border(jl + c);                             // H(-1, j)
                F[c] = kNegInf;
                if (jl + c < n) scw[c >> 2] |= (unsigned)s[jl + c] << (8 * (c & 3));
            }
            int dcarry = lane == 0 ? 0 : border(jl - 1);           // H(-1, jl - 1); H(-1, -1) = 0
            int hr = 0, er = kNegInf;
            int best = kScoreMin, bi = 0x7fffffff, bj = 0;   // local: the lane's first maximum (row, lane column)
            int colbest = kScoreMin, colbest_i = -1;                 // semiglobal: max of H(i, n - 1), lowest i
            const int T = m + nl - 1;
            for (int tb = 0; tb < T; tb += 32) {
                __syncwarp();
                if (tb + lane < m) rq[(tb + lane) & 63] = q[tb + lane];
                __syncwarp();
                const int tend = min(tb + 32, T);
#pragma unroll 1
                for (int t = tb; t < tend; ++t) {
                    int hl = __shfl_up_sync(kFull, hr, 1);
                    int el = __shfl_up_sync(kFull, er, 1);
                    const int r = t - lane;
                    if (lane == 0) { hl = border(r); el = kNegInf; }   // H(r, -1), E(r, -1)
                    if (r >= 0 && r < m && lane < nl) {
                        const int qc = rq[r & 63];
                        int d = dcarry;
                        dcarry = hl;
                        int lft = hl, e = el;
                        unsigned bits[(K + 7) / 8];
#pragma unroll
                        for (int w = 0; w < (K + 7) / 8; ++w) bits[w] = 0u;
#pragma unroll
                        for (int c = 0; c < K; ++c) {
                            const int sc = (int)((scw[c >> 2] >> (8 * (c & 3))) & 0xffu);
                            const int up = H[c];
                            bits[c >> 3] |= fulltb_cell(d + ((qc == sc) ? same : diff), up, lft, e, F[c], go, ge, LOCAL)
                                            << (4 * (c & 7));
                            d = up;
                            H[c] = lft;
                            if constexpr (LOCAL) {
                                if (lft > best && c < nvalid) { best = lft; bi = r; bj = c; }
                            }
                        }
                        hr = lft;
                        er = e;
                        uint8_t* dst = pred + (size_t)r * RB + lane * (K / 2);
                        if constexpr (K == 4) *reinterpret_cast<unsigned short*>(dst) = (unsigned short)bits[0];
                        else if constexpr (K == 8) *reinterpret_cast<unsigned*>(dst) = bits[0];
                        else if constexpr (K == 16) *reinterpret_cast<uint2*>(dst) = make_uint2(bits[0], bits[1]);
                        else *reinterpret_cast<uint4*>(dst) = make_uint4(bits[0], bits[1], bits[2], bits[3]);
                        if constexpr (MODE == kSemiglobal) {
                            if (lane == nl - 1) {
                                const int v = pick_column(H, outc);
                                if (v > colbest) { colbest = v; colbest_i = r; }
                            }
                        }
                    }
                }
            }
            // end cell: get_score_pos() (src/scoring.impala:29-137) as the single-pair path reports it
            if constexpr (GLOB) {
                score = __shfl_sync(kFull, pick_column(H, outc), nl - 1);
            } else if constexpr (MODE == kSemiglobal) {
                // finish_score_kernel: the last row first (lowest j, the j = -1 candidate of value 0 winning ties),
                // then the last column only if strictly greater (lowest i)
                int rv = kScoreMin, rj = 0x7fffffff;
#pragma unroll
                for (int c = 0; c < K; ++c)
                    if (c < nvalid && H[c] > rv) { rv = H[c]; rj = jl + c; }
                for (int x = 16; x > 0; x >>= 1) {
                    const int ov = __shfl_xor_sync(kFull, rv, x), oj = __shfl_xor_sync(kFull, rj, x);
                    if (ov > rv || (ov == rv && oj < rj)) { rv = ov; rj = oj; }
                }
                int cs = __shfl_sync(kFull, colbest, nl - 1), ci = __shfl_sync(kFull, colbest_i, nl - 1);
                if (0 >= rv) { rv = 0; rj = -1; }
                if (0 >= cs) { cs = 0; ci = -1; }
                score = rv; ei = m - 1; ej = rj;
                if (cs > score) { score = cs; ei = ci; ej = n - 1; }
            } else {
                // local_end_cell_kernel keeps one maximum per 1024 x 1024 block and picks, among the blocks holding
                // the overall maximum, the smallest (slot, diagonal) with slot = min(bi + bj, nbi - 1) - bi, then the
                // block's first maximum in row-major order.  With n <= 1024 every block lies in block column bj = 0,
                // so slot = 0 and the diagonal is bi: the first block row holding the maximum wins, and inside it the
                // first cell in row-major order -- together the first maximum of the whole matrix in row-major order.
                // Each lane keeps its first maximum with strict '>' (rows arrive in order, columns ascend within a
                // row); the warp takes the maximum value, then the smallest (i, j).
                bj += jl;
                for (int x = 16; x > 0; x >>= 1) {
                    const int ov = __shfl_xor_sync(kFull, best, x), oi = __shfl_xor_sync(kFull, bi, x);
                    const int oj = __shfl_xor_sync(kFull, bj, x);
                    if (ov > best || (ov == best && (oi < bi || (oi == bi && oj < bj)))) { best = ov; bi = oi; bj = oj; }
                }
                score = best; ei = bi; ej = bj;
            }

            // the walk (fulltb_walk_kernel) from the end cell, through shared-memory windows of the slab
            __syncwarp();                                          // the pair's predecessor rows are visible
            uint8_t* oq = alq + o;
            uint8_t* os = als + o;
            i = ei; j = ej;
            int state = 0, going = 1;
            while (going && i >= 0 && j >= 0) {
                const int r0 = max(0, i - (kWinRows - 1));
                const int c0 = max(0, ((j >> 5) - 1) << 5);        // 16-byte aligned; j - c0 < 64
                const int rr = r0 + lane;
                if (rr <= i) {
                    const uint4* src = reinterpret_cast<const uint4*>(pred + (size_t)rr * RB + (c0 >> 1));
                    s_win[warp][lane][0] = __ldcg(src);
                    s_win[warp][lane][1] = __ldcg(src + 1);
                    s_wq[warp][lane] = q[rr];
                }
                if (c0 + lane <= j) s_ws[warp][lane] = s[c0 + lane];
                if (c0 + 32 + lane <= j) s_ws[warp][32 + lane] = s[c0 + 32 + lane];
                __syncwarp();
                if (lane == 0) {
                    while (i >= r0 && j >= c0) {
                        const int cc = j - c0;
                        const unsigned p = (win[(i - r0) * (kWinCols / 2) + (cc >> 1)] >> (4 * (cc & 1))) & 15u;
                        if (!fulltb_walk_step(p, i, j, state, s_wq[warp][i - r0], s_ws[warp][cc], oq, os)) { going = 0; break; }
                    }
                }
                i = __shfl_sync(kFull, i, 0);
                j = __shfl_sync(kFull, j, 0);
                state = __shfl_sync(kFull, state, 0);
                going = __shfl_sync(kFull, going, 0);
                __syncwarp();                                      // the window is read before it is reloaded
            }
            if (GLOB && going) {                                   // border row / column: gaps to (-1, -1)
                for (int k = lane; k <= j; k += 32) { oq[k] = '_'; os[k] = s[k]; }
                for (int k = lane; k <= i; k += 32) { oq[k] = q[k]; os[k] = '_'; }
                i = j = -1;
            }
        }
        if (lane == 0) {
            a.scores[pair] = score;
            if (ends) { ends[2 * pair] = ei; ends[2 * pair + 1] = ej; }
            if (starts) { starts[2 * pair] = i + 1; starts[2 * pair + 1] = j + 1; }
        }
        unsigned long long nxt = 0;
        if (lane == 0) nxt = atomicAdd(a.counter, 1ull);
        pair = (long long)__shfl_sync(kFull, nxt, 0);
    }
}

using AlignBatchKernelFn = void (*)(const BatchArgs, int*, int*, uint8_t*, uint8_t*, uint8_t*, size_t);

template <int MODE>
static AlignBatchKernelFn pick_align_batch_kernel_k(int K)
{
    switch (K) {
        case 4: return batch_align_kernel<MODE, 4>;
        case 8: return batch_align_kernel<MODE, 8>;
        case 16: return batch_align_kernel<MODE, 16>;
        default: return batch_align_kernel<MODE, 32>;
    }
}

int Engine::align_batch_device(const anyseq_scoring& sc, const uint8_t* d_q, const int64_t* d_qoff, const uint8_t* d_s,
                               const int64_t* d_soff, int64_t npairs, int32_t* d_scores, int32_t* d_ends,
                               int32_t* d_starts, char* d_alq, char* d_als, anyseq_result* out)
{
    std::lock_guard<std::recursive_mutex> lock(mu_);
    ANYSEQ_CUDA_CHECK(cudaSetDevice(device));
    ScoreParams sp;
    bool affine;
    int rc = make_score_params(sc, &sp, &affine);
    if (rc) return rc;
    if (out) { std::memset(out, 0, sizeof(*out)); out->end_i = out->end_j = -1; }
    if (npairs == 0) return ANYSEQ_OK;
    BatchArgs ba;
    std::memset(&ba, 0, sizeof(ba));
    ba.q = d_q;
    ba.qoff = reinterpret_cast<const long long*>(d_qoff);
    ba.s = d_s;
    ba.soff = reinterpret_cast<const long long*>(d_soff);
    ba.npairs = npairs;
    ba.scores = d_scores;
    ba.sp = sp;
    ba.gap_init = sc.gap_init;
    ba.mode = sc.mode;
    long long bounds[4] = {0, 0, 0, 0};   // q_off[0], q_off[npairs], s_off[0], s_off[npairs]
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(&bounds[0], d_qoff, sizeof(long long), cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(&bounds[1], d_qoff + npairs, sizeof(long long), cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(&bounds[2], d_soff, sizeof(long long), cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(&bounds[3], d_soff + npairs, sizeof(long long), cudaMemcpyDeviceToHost, stream_));
    int max_long, max_short, max_q, max_s;
    bool negative;
    if ((rc = batch_len_stats(ba, &max_long, &max_short, &max_q, &max_s, &negative))) return rc;
    if (negative) { set_last_error("batch offsets must be non-decreasing"); return ANYSEQ_ERR_BAD_ARG; }
    if (max_s > kMaxAlignBatchSubject) {
        char buf[200];
        std::snprintf(buf, sizeof(buf), "batch traceback: a subject of %d symbols is longer than %d; "
                      "align such pairs with anyseq_align_full", max_s, kMaxAlignBatchSubject);
        set_last_error(buf);
        return ANYSEQ_ERR_UNSUPPORTED;
    }
    int K = 4;
    while (32 * K < max_s) K *= 2;
    AlignBatchKernelFn fn = sc.mode == ANYSEQ_GLOBAL ? pick_align_batch_kernel_k<kGlobal>(K)
                          : sc.mode == ANYSEQ_SEMIGLOBAL ? pick_align_batch_kernel_k<kSemiglobal>(K)
                          : pick_align_batch_kernel_k<kLocal>(K);
    int nb = 0;
    ANYSEQ_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, kThreads, 0));
    if (nb < 1) { set_last_error("batch traceback kernel does not fit on an SM"); return ANYSEQ_ERR_UNSUPPORTED; }
    // one predecessor slab per warp: max_q rows of 16 K bytes; the grid shrinks until the slabs fit
    const size_t slab = (size_t)std::max(max_q, 1) * 16 * K;
    const size_t per_block = slab * kWarpsPerBlock;
    size_t free_b = 0, total_b = 0;
    ANYSEQ_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    const size_t have = free_b + batch_pred_.bytes, reserve = 64u << 20;
    const long long fit = have > reserve ? (long long)((have - reserve) / per_block) : 0;
    const long long want = std::min<long long>((long long)nb * sm_count, (npairs + kWarpsPerBlock - 1) / kWarpsPerBlock);
    const int grid = (int)std::min(want, fit);
    if (grid < 1) {
        char buf[240];
        std::snprintf(buf, sizeof(buf), "batch traceback: queries of %d symbols need %.2f GB of predecessor scratch per "
                      "block (%.2f GB free); split the batch", max_q, per_block / 1e9, have / 1e9);
        set_last_error(buf);
        return ANYSEQ_ERR_UNSUPPORTED;
    }
    if (batch_pred_.ensure(per_block * grid)) return ANYSEQ_ERR_NO_DEVICE;
    const size_t total = (size_t)(bounds[1] - bounds[0]) + (size_t)(bounds[3] - bounds[2]);
    ba.counter = reinterpret_cast<unsigned long long*>(misc_.as<int>() + kMiscCounter);
    const unsigned long long first = (unsigned long long)grid * kWarpsPerBlock;
    ANYSEQ_CUDA_CHECK(cudaEventRecord(ev0_, stream_));
    if (total) {                                           // src/traceback.impala:20-23
        ANYSEQ_CUDA_CHECK(cudaMemsetAsync(d_alq, ' ', total, stream_));
        ANYSEQ_CUDA_CHECK(cudaMemsetAsync(d_als, ' ', total, stream_));
    }
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(ba.counter, &first, sizeof(first), cudaMemcpyHostToDevice, stream_));
    fn<<<grid, kThreads, 0, stream_>>>(ba, d_ends, d_starts, reinterpret_cast<uint8_t*>(d_alq),
                                       reinterpret_cast<uint8_t*>(d_als), batch_pred_.as<uint8_t>(), slab);
    ANYSEQ_CUDA_CHECK(cudaGetLastError());
    return batch_epilogue(2, out);
}

int Engine::align_batch_host(const anyseq_scoring& sc, const char* q, const int64_t* qoff, const char* s,
                             const int64_t* soff, int64_t npairs, int32_t* scores, int32_t* ends, int32_t* starts,
                             char* alq, char* als, anyseq_result* out)
{
    if (npairs < 0 || !qoff || !soff) { set_last_error("bad arguments"); return ANYSEQ_ERR_BAD_ARG; }
    for (int64_t p = 0; p < npairs; ++p) {
        if (qoff[p + 1] < qoff[p] || soff[p + 1] < soff[p]) {
            set_last_error("batch offsets must be non-decreasing");
            return ANYSEQ_ERR_BAD_ARG;
        }
    }
    const long long qt = qoff[npairs] - qoff[0], st = soff[npairs] - soff[0];
    const size_t total = (size_t)qt + (size_t)st;
    if ((npairs > 0 && !scores) || (qt > 0 && !q) || (st > 0 && !s) || (total > 0 && (!alq || !als))) {
        set_last_error("bad arguments");
        return ANYSEQ_ERR_BAD_ARG;
    }
    ScoreParams sp;
    bool affine;
    int rc = make_score_params(sc, &sp, &affine);
    if (rc) return rc;
    if (out) { std::memset(out, 0, sizeof(*out)); out->end_i = out->end_j = -1; }
    if (npairs == 0) return ANYSEQ_OK;
    std::lock_guard<std::recursive_mutex> lock(mu_);
    ANYSEQ_CUDA_CHECK(cudaSetDevice(device));

    // one device block: sequences, offsets (rebased to 0), scores, ends, starts, aligned rows
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t n1 = (size_t)npairs + 1;
    const size_t b_q = up((size_t)qt), b_s = up((size_t)st), b_off = up(sizeof(int64_t) * n1);
    const size_t b_sc = up(sizeof(int32_t) * npairs), b_pair = up(sizeof(int32_t) * 2 * npairs), b_al = up(total);
    const size_t bytes = b_q + b_s + 2 * b_off + b_sc + 2 * b_pair + 2 * b_al;
    size_t free_b = 0, total_b = 0;
    ANYSEQ_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    const size_t have = free_b + batch_io_.bytes;
    if (bytes + (64u << 20) > have) {
        char buf[200];
        std::snprintf(buf, sizeof(buf), "batch traceback of %lld pairs needs %.2f GB of device memory for its inputs and "
                      "outputs (%.2f GB free); split the batch", (long long)npairs, bytes / 1e9, have / 1e9);
        set_last_error(buf);
        return ANYSEQ_ERR_UNSUPPORTED;
    }
    if (batch_io_.ensure(bytes)) return ANYSEQ_ERR_NO_DEVICE;
    uint8_t* base = batch_io_.as<uint8_t>();
    uint8_t* d_q = base;
    uint8_t* d_s = d_q + b_q;
    int64_t* d_qoff = reinterpret_cast<int64_t*>(d_s + b_s);
    int64_t* d_soff = reinterpret_cast<int64_t*>(reinterpret_cast<uint8_t*>(d_qoff) + b_off);
    int32_t* d_scores = reinterpret_cast<int32_t*>(reinterpret_cast<uint8_t*>(d_soff) + b_off);
    int32_t* d_ends = reinterpret_cast<int32_t*>(reinterpret_cast<uint8_t*>(d_scores) + b_sc);
    int32_t* d_starts = reinterpret_cast<int32_t*>(reinterpret_cast<uint8_t*>(d_ends) + b_pair);
    char* d_alq = reinterpret_cast<char*>(d_starts) + b_pair;
    char* d_als = d_alq + b_al;
    std::vector<int64_t> ro(2 * n1);
    for (size_t p = 0; p < n1; ++p) { ro[p] = qoff[p] - qoff[0]; ro[n1 + p] = soff[p] - soff[0]; }
    if (qt) ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(d_q, q + qoff[0], (size_t)qt, cudaMemcpyHostToDevice, stream_));
    if (st) ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(d_s, s + soff[0], (size_t)st, cudaMemcpyHostToDevice, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(d_qoff, ro.data(), sizeof(int64_t) * n1, cudaMemcpyHostToDevice, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(d_soff, ro.data() + n1, sizeof(int64_t) * n1, cudaMemcpyHostToDevice, stream_));
    rc = align_batch_device(sc, d_q, d_qoff, d_s, d_soff, npairs, d_scores, ends ? d_ends : nullptr,
                            starts ? d_starts : nullptr, d_alq, d_als, out);
    if (rc) return rc;
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(scores, d_scores, sizeof(int32_t) * npairs, cudaMemcpyDeviceToHost, stream_));
    if (ends) ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(ends, d_ends, sizeof(int32_t) * 2 * npairs, cudaMemcpyDeviceToHost, stream_));
    if (starts) ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(starts, d_starts, sizeof(int32_t) * 2 * npairs, cudaMemcpyDeviceToHost, stream_));
    if (total) {
        ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(alq, d_alq, total, cudaMemcpyDeviceToHost, stream_));
        ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(als, d_als, total, cudaMemcpyDeviceToHost, stream_));
    }
    ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(stream_));
    return ANYSEQ_OK;
}

}  // namespace anyseq
