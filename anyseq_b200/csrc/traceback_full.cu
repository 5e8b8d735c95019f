// traceback_full.cu -- full-matrix traceback for pairs whose m*n/2 predecessor bytes fit in HBM
// (SURVEY 8f.4; reference: traceback_full, src/align.impala:190-216, exported as
// construct_*_alignment_fulltb, src/export.impala:38,94,151).
//
// Unlike the linear-space path this one gives the exact semiglobal and local alignments: one walk from
// scoring.get_score_pos() through the whole predecessor matrix until PRED_NONE (src/traceback.impala:47-80).
//
// Three device passes:
//   1. the ordinary strip-kernel score pass with 128-column strips (K = 4), which additionally keeps every
//      strip's right edge column (H and E per row): the score, the end cell (local: the reference's block
//      slot rule, see local_end_cell_kernel) and the left borders of all 128-column blocks;
//   2. fulltb_dp_kernel: one warp per 128-column block re-relaxes its block over all rows from those borders
//      and stores 4 predecessor bits per cell (H source in the reference's numbering, E-extends, F-extends)
//      -- blocks are independent now, rows stream through the warp with a 32-step lane skew;
//   3. fulltb_walk_kernel: the walk.  Linear gaps are gap_init == 0 of the same machine: E never extends
//      (H(i,j-1) >= E(i,j-1)), so the walk and the tie order NO_GAP > GAP_Q > GAP_S are the reference's.
// The Gotoh variant is build-defined like every affine entry point (parity unpinned vs the reference).
#include "engine.cuh"
#include "traceback_full.cuh"

#include <algorithm>
#include <cstring>

namespace anyseq {

constexpr int kFullBlockW = 128;

// pred16[i * pitch + b * 32 + lane] = 4 cells x 4 bits of row i, columns 128 b + 4 lane ...
__global__ void __launch_bounds__(128)
fulltb_dp_kernel(const uint8_t* __restrict__ q, const uint8_t* __restrict__ s, int m, int n, int nblocks,
                 const int2* __restrict__ edges, int local, int glob, int affine, int same, int diff, int gi, int ge,
                 unsigned short* __restrict__ pred16)
{
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= nblocks) return;
    const int go = gi + ge;
    const int oj = b * kFullBlockW;
    const size_t pitch = (size_t)nblocks * 32;
    const int2* left = b > 0 ? edges + (size_t)(b - 1) * m : nullptr;
    int H[4], F[4], sc[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int j = oj + lane * 4 + c;
        H[c] = glob ? gi + (j + 1) * ge : 0;                          // H(-1, j)
        F[c] = kNegInf;
        sc[c] = j < n ? (int)s[j] : 0x7fff;
    }
    // H(-1, first column of the lane - 1); H(-1,-1) = 0
    int dcarry = (oj + lane * 4 == 0) ? 0 : (glob ? gi + (oj + lane * 4) * ge : 0);
    int hr = 0, er = kNegInf;
    int2 rec = make_int2(0, kNegInf);
    for (int t = 0; t < m + 31; ++t) {
        if (left && (t & 31) == 0) {                                  // lane 0's next 32 border rows, coalesced
            const int r = t + lane;
            rec = r < m ? __ldcg(left + r) : make_int2(0, kNegInf);
        }
        int hl = __shfl_up_sync(0xffffffffu, hr, 1);
        int el = __shfl_up_sync(0xffffffffu, er, 1);
        const int bh = __shfl_sync(0xffffffffu, rec.x, t & 31);
        const int be = __shfl_sync(0xffffffffu, rec.y, t & 31);
        const int i = t - lane;
        if (lane == 0) {
            if (left) { hl = bh; el = affine ? be : kNegInf; }
            else { hl = glob ? gi + (i + 1) * ge : 0; el = kNegInf; }  // H(i,-1), E(i,-1)
        }
        if (i >= 0 && i < m) {
            const int qc = q[i];
            int d = dcarry;
            dcarry = hl;
            int lft = hl, e = el;
            unsigned bits = 0;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int up = H[c];
                bits |= fulltb_cell(d + ((qc == sc[c]) ? same : diff), up, lft, e, F[c], go, ge, local) << (4 * c);
                d = up;
                H[c] = lft;
            }
            hr = lft;
            er = e;
            pred16[(size_t)i * pitch + (size_t)b * 32 + lane] = (unsigned short)bits;
        }
    }
}

// the walk of traceback_offset (src/traceback.impala:47-80) as a 3-state machine; one thread.
// out[2] = get_alignment_start() = (i + 1, j + 1) where it stopped.
__global__ void fulltb_walk_kernel(const uint8_t* __restrict__ q, const uint8_t* __restrict__ s, int end_i, int end_j,
                                   int glob, int nblocks, const unsigned short* __restrict__ pred16,
                                   uint8_t* __restrict__ out_q, uint8_t* __restrict__ out_s, int* __restrict__ start)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const size_t pitch = (size_t)nblocks * 32;
    int i = end_i, j = end_j, state = 0;                              // 0 = H, 1 = E, 2 = F
    for (;;) {
        if (i < 0 && j < 0) break;
        const size_t pos = (size_t)(i + j + 1);
        if (i < 0) {                                                   // border row: GAP_Q for global, else NONE
            if (!glob) break;
            out_q[pos] = '_'; out_s[pos] = s[j]; --j; continue;
        }
        if (j < 0) {                                                   // border column: GAP_S for global, else NONE
            if (!glob) break;
            out_q[pos] = q[i]; out_s[pos] = '_'; --i; continue;
        }
        const unsigned p = (pred16[(size_t)i * pitch + (size_t)(j >> 2)] >> (4 * (j & 3))) & 15u;
        if (!fulltb_walk_step(p, i, j, state, q[i], s[j], out_q, out_s)) break;
    }
    start[0] = i + 1;
    start[1] = j + 1;
}

int Engine::align_full_host(const anyseq_scoring& sc, const char* q, int m, const char* s, int n, char* alq, char* als,
                            anyseq_result* out, int* start2)
{
    if (m < 0 || n < 0 || !out || !alq || !als || (m > 0 && !q) || (n > 0 && !s)) { set_last_error("bad arguments"); return ANYSEQ_ERR_BAD_ARG; }
    ScoreParams sp;
    bool affine;
    int rc = make_score_params(sc, &sp, &affine);
    if (rc) return rc;
    const size_t total = (size_t)m + (size_t)n;
    std::memset(alq, ' ', total);                                     // src/traceback.impala:20-23
    std::memset(als, ' ', total);
    if (start2) start2[0] = start2[1] = 0;
    if (m == 0 || n == 0) return score_host(sc, q, m, s, n, out);     // nothing to relax: degenerate result, blank rows
    std::lock_guard<std::recursive_mutex> lock(mu_);
    ANYSEQ_CUDA_CHECK(cudaSetDevice(device));

    const int nb = (n + kFullBlockW - 1) / kFullBlockW;
    const size_t pred_bytes = sizeof(unsigned short) * 32 * (size_t)nb * (size_t)m;
    const size_t edge_bytes = sizeof(int2) * (size_t)nb * (size_t)m;
    size_t free_b = 0, total_b = 0;
    ANYSEQ_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    const size_t have = free_b + pred_.bytes + edges_.bytes;
    if (pred_bytes + edge_bytes + (64u << 20) > have) {
        char buf[200];
        std::snprintf(buf, sizeof(buf), "full-matrix traceback of %d x %d needs %.1f GB of device memory (%.1f GB free); "
                      "use anyseq_align (linear space)", m, n, (pred_bytes + edge_bytes) / 1e9, have / 1e9);
        set_last_error(buf);
        return ANYSEQ_ERR_UNSUPPORTED;
    }
    if (seq_q_.ensure((size_t)m + 64) || seq_s_.ensure((size_t)n + 64)) return ANYSEQ_ERR_NO_DEVICE;
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(seq_q_.ptr, q, (size_t)m, cudaMemcpyHostToDevice, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(seq_s_.ptr, s, (size_t)n, cudaMemcpyHostToDevice, stream_));

    // pass 1: score + end cell + block borders
    anyseq_result res;
    {
        struct Scope { Engine* e; ~Scope() { e->want_edges_ = false; e->force_track_ = false; } } scope{this};
        want_edges_ = true;
        force_track_ = sc.mode == ANYSEQ_LOCAL;
        rc = score_device(sc, seq_q_.as<uint8_t>(), m, seq_s_.as<uint8_t>(), n, &res);
    }
    if (rc) return rc;

    // passes 2 + 3
    if (pred_.ensure(pred_bytes) || aux_.ensure(2 * total + 64)) return ANYSEQ_ERR_NO_DEVICE;
    uint8_t* d_oq = aux_.as<uint8_t>();
    uint8_t* d_os = d_oq + total;
    int* d_start = misc_.as<int>() + kMiscOut + 4;
    cudaEvent_t e0 = ev0_, e1 = ev1_;
    ANYSEQ_CUDA_CHECK(cudaEventRecord(e0, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemsetAsync(d_oq, ' ', 2 * total, stream_));
    fulltb_dp_kernel<<<(nb + 3) / 4, 128, 0, stream_>>>(seq_q_.as<uint8_t>(), seq_s_.as<uint8_t>(), m, n, nb,
                                                        edges_.as<int2>(), sc.mode == ANYSEQ_LOCAL, sc.mode == ANYSEQ_GLOBAL,
                                                        affine ? 1 : 0, sc.same, sc.diff, sc.gap_init, sc.gap_extend,
                                                        pred_.as<unsigned short>());
    ANYSEQ_CUDA_CHECK(cudaGetLastError());
    fulltb_walk_kernel<<<1, 32, 0, stream_>>>(seq_q_.as<uint8_t>(), seq_s_.as<uint8_t>(), res.end_i, res.end_j,
                                              sc.mode == ANYSEQ_GLOBAL, nb, pred_.as<unsigned short>(), d_oq, d_os, d_start);
    ANYSEQ_CUDA_CHECK(cudaGetLastError());
    ANYSEQ_CUDA_CHECK(cudaEventRecord(e1, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(alq, d_oq, total, cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(als, d_os, total, cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(h_misc_ + kMiscOut + 4, d_start, sizeof(int) * 2, cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(stream_));
    float ms = 0.f;
    ANYSEQ_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    if (start2) { start2[0] = h_misc_[kMiscOut + 4]; start2[1] = h_misc_[kMiscOut + 5]; }
    last_start_[0] = h_misc_[kMiscOut + 4];
    last_start_[1] = h_misc_[kMiscOut + 5];
    *out = res;
    out->kernel_ms = res.kernel_ms + ms;
    out->kernel_launches = res.kernel_launches + 3;
    return ANYSEQ_OK;
}

}  // namespace anyseq
