// traceback.cu -- linear-space traceback on the GPU, linear and Gotoh gaps.
//
// Same algorithm and the same results as the reference's CPU build of
// traceback_lintime (src/align.impala:237-311):
//   * iterative Hirschberg over SUBJECT halves: every level relaxes, for every
//     part, the left half forward and the right half on reversed sequences
//     (iteration_partitioned, src/iteration_cpu.impala:59-119;
//     get_sequence_acc_half, src/traceback_lintime.impala:137-148) -- here all
//     halves of a level are jobs of ONE persistent strip-kernel launch,
//   * hb_sum (src/traceback_lintime.impala:44-135) picks the split row of every
//     part; ties are resolved in the reference CPU build's candidate order
//     (sub-blocks of BLOCK_WIDTH = 1024, src/iteration_cpu.impala:1), which
//     decides which co-optimal alignment comes out (SURVEY.md A.5, Q10),
//   * final pass: every 128-column block is relaxed from fresh borders with
//     predecessors (iteration_blockwise :121-157, get_iteration_acc_tb_device
//     src/scoring_cpu.impala:125-157) and walked from its bottom-right cell
//     until PRED_NONE (traceback_offset, src/traceback.impala:47-80).
// Quirks Q2/Q3/Q4 of SURVEY.md Appendix B follow from doing exactly that.
//
// Gotoh gaps are BUILD-DEFINED: the reference has no affine path
// (src/align.impala:153-166 is an uncalled stub), so parity with the reference is
// unpinned; the behaviour is pinned bit for bit against the CPU restatement kept
// with the tests (its affine traceback).  Linear gaps are Gotoh with gi = 0, and
// one driver runs both.  What Gotoh adds to the reference's shape (Myers & Miller
// 1988, adapted to splitting the SUBJECT):
//   * the right edge records of a half already carry E next to H ({H,tag,E,tag}),
//   * a split vertex has a type, H or E (a horizontal gap runs through it);
//     candidates per row i, scanned H first then E, strict '>':
//         H: LH(i) + RH(len-i-2)        E: LE(i) + RE(len-i-2) - gi
//     (linear runs scan the H candidates only, so every type stays H),
//   * a block whose start (end) vertex has type E gets a free gap opening on its
//     top border (on the top border of its reversed problem): Job::top_open,
//   * final blocks keep 4 predecessor bits per cell (H source, E ext, F ext) and
//     are walked with a 3-state machine.  With gi = 0, E(i,j-1) <= H(i,j-1) and
//     F(i-1,j) <= H(i-1,j), so no gap extends, and the H sources in the order
//     diag > E > F are the reference's NO_GAP > GAP_Q > GAP_S: the walk steps
//     exactly as the reference's 2-bit one.
#include "engine.cuh"
#include "strip_kernel.cuh"

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>

namespace anyseq {

constexpr int kMinPartW = 128;      // MIN_PART_WIDTH_HB, src/align.impala:18
constexpr int kRefBlockW = 1024;    // BLOCK_WIDTH of the reference CPU build

enum : int { kSrcNone = 0, kSrcE = 1, kSrcF = 2, kSrcDiag = 3 };   // numbering of src/align.impala:37-40

__global__ void reverse_bytes_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int n)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        dst[n - 1 - i] = src[i];
}

struct HbPart {          // one part of a Hirschberg level
    int off, len;        // row range [off, off+len)
    int split_slot;      // splits / types slot that receives the result
    int rhw;             // width of the right half (clipped by the subject end)
    int open_l, open_r;  // opening cost on the top border of the left half / of the reversed right half
};

// hb_sum: argmax over split rows of L(i) + R(len-i-2) with the two border
// candidates, in the reference's candidate order; AFFINE also weighs the E
// joins, each right after the H candidate of its row.  One CTA per part.  A
// template flag rather than an argument: the top levels run one CTA over all
// rows, where loading H and E of a row together saves a memory round trip.
template <bool AFFINE>
__global__ void hb_sum_kernel(const HbPart* __restrict__ parts, int nparts, const int4* __restrict__ colL,
                              const int4* __restrict__ colR, int* __restrict__ splits /* [0] = slot -1 */,
                              int* __restrict__ types, int half, int bpp2, int glob, int gi, int ge)
{
    __shared__ unsigned long long s_key[32];
    __shared__ int s_idx[32];
    for (int p = blockIdx.x; p < nparts; p += gridDim.x) {
        const HbPart P = parts[p];
        const int len = P.len;
        // last-column records of the two halves: .x = H, .z = E
        auto rec = [&](const int4* base, int i) -> int4 { return __ldcg(base + P.off + i); };
        // key = (value, -priority): larger wins; priority = position in the reference's scan
        unsigned long long best = 0ull;   // below every real candidate
        int best_idx = -2;                // packed: 2 * (idx + 1) + type
        auto consider = [&](int val, unsigned prio, int idx, int type) {
            const unsigned long long key =
                ((unsigned long long)((unsigned)val ^ 0x80000000u) << 32) | (unsigned long long)(0xffffffffu - prio);
            if (key > best) { best = key; best_idx = 2 * (idx + 1) + type; }
        };
        const unsigned per_block = (unsigned)(len / bpp2 + 4);
        if (len > 0 && threadIdx.x == 0) {
            const int4 rl = rec(colR, len - 1);
            const int4 ll = rec(colL, len - 1);
            const int bl = glob ? P.open_l + half * ge : 0;          // init_scores(lhw - 1)
            const int br = glob ? P.open_r + P.rhw * ge : 0;         // init_scores(rhw - 1)
            consider(bl + rl.x, 0u, -1, 0);
            if (AFFINE && glob) consider(bl + rl.z - gi, 1u, -1, 1);
            consider(ll.x + br, 2u, len - 1, 0);
            if (AFFINE && glob) consider(ll.z + br - gi, 3u, len - 1, 1);
        }
        for (int i = threadIdx.x; i < len - 1; i += blockDim.x) {
            const int4 l = rec(colL, i);
            const int4 r = rec(colR, len - i - 2);
            const unsigned prio = 2u * ((unsigned)(i % bpp2) * per_block + (unsigned)(i / bpp2) + 2u);
            consider(l.x + r.x, prio, i, 0);
            if (AFFINE) consider(l.z + r.z - gi, prio + 1u, i, 1);
        }
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long ok = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, best_idx, o);
            if (ok > best) { best = ok; best_idx = oi; }
        }
        if ((threadIdx.x & 31) == 0) { s_key[threadIdx.x >> 5] = best; s_idx[threadIdx.x >> 5] = best_idx; }
        __syncthreads();
        if (threadIdx.x < 32) {
            const int nw = blockDim.x >> 5;
            best = threadIdx.x < nw ? s_key[threadIdx.x] : 0ull;
            best_idx = threadIdx.x < nw ? s_idx[threadIdx.x] : -2;
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long ok = __shfl_xor_sync(0xffffffffu, best, o);
                const int oi = __shfl_xor_sync(0xffffffffu, best_idx, o);
                if (ok > best) { best = ok; best_idx = oi; }
            }
            if (threadIdx.x == 0) {
                int idx = -1, type = 0;
                if (best_idx >= 0) { idx = (best_idx >> 1) - 1; type = best_idx & 1; }
                splits[P.split_slot + 1] = P.off + idx + 1;
                types[P.split_slot + 1] = type;
            }
        }
        __syncthreads();
    }
}

// Final pass, one WARP per 128-column block: lane l owns columns 4l..4l+3, lane
// skew as in the strip kernel (relax_global / relax_local, src/align.impala:46-79).
// pred16[(off + i) * 32 + lane] = 4 cells x {H source (2 bits), E ext, F ext}.
// blk_end[2b], [2b+1] = H and E of the block's bottom-right cell.
__global__ void trace_dp_kernel(const uint8_t* __restrict__ q, const uint8_t* __restrict__ s,
                                const int* __restrict__ blk_off, const int* __restrict__ blk_h,
                                const int* __restrict__ blk_open_top, int nblocks, int n, int local, int glob,
                                int same, int diff, int gi, int ge, unsigned short* __restrict__ pred16,
                                int* __restrict__ blk_end)
{
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    const int go = gi + ge;
    for (int b = blockIdx.x * wpb + (threadIdx.x >> 5); b < nblocks; b += gridDim.x * wpb) {
        const int off = blk_off[b], h = blk_h[b];
        if (h < 0) continue;                                          // block of another rank (sharded traceback)
        const int open_top = blk_open_top[b];
        const int oj = b * kMinPartW;
        const int w = min(kMinPartW, n - oj);
        int H[4], F[4], sc[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int j = lane * 4 + c;
            H[c] = glob ? open_top + (j + 1) * ge : 0;                // H(-1, j)
            F[c] = kNegInf;
            sc[c] = (oj + j < n) ? (int)s[oj + j] : 0x7fff;
        }
        int dcarry = (lane == 0) ? 0 : (glob ? open_top + (lane * 4) * ge : 0);   // H(-1, 4l-1); H(-1,-1) = 0
        int hr = 0, er = kNegInf;
        const int endlane = (w - 1) >> 2, endc = (w - 1) & 3;
        for (int t = 0; t < h + 31; ++t) {
            int hl = __shfl_up_sync(0xffffffffu, hr, 1);
            int el = __shfl_up_sync(0xffffffffu, er, 1);
            const int i = t - lane;
            if (lane == 0) { hl = glob ? gi + (i + 1) * ge : 0; el = kNegInf; }   // H(i,-1), E(i,-1)
            if (i >= 0 && i < h) {
                const int qc = q[off + i];
                int d = dcarry;
                dcarry = hl;
                int left = hl, e = el;
                unsigned bits = 0;
                int hend = 0, eend = 0;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int up = H[c];
                    int eext = 0, fext = 0;
                    int eo = left + go;
                    if (e + ge > eo) { eo = e + ge; eext = 1; }
                    e = eo;
                    int fo = up + go;
                    if (F[c] + ge > fo) { fo = F[c] + ge; fext = 1; }
                    int score = d + ((qc == sc[c]) ? same : diff);
                    int src = kSrcDiag;
                    if (e > score) { score = e; src = kSrcE; }
                    if (fo > score) { score = fo; src = kSrcF; }
                    if (local && 0 > score) { score = 0; src = kSrcNone; }
                    bits |= (unsigned)(src | (eext << 2) | (fext << 3)) << (4 * c);
                    d = up;
                    H[c] = score;
                    F[c] = fo;
                    left = score;
                    if (c == endc) { hend = score; eend = e; }
                }
                hr = left;
                er = e;
                pred16[(size_t)(off + i) * 32 + lane] = (unsigned short)bits;
                if (i == h - 1 && lane == endlane) { blk_end[2 * b] = hend; blk_end[2 * b + 1] = eend; }
            }
        }
    }
}

// traceback_offset (src/traceback.impala:47-80) as a 3-state walk, one thread per
// block.  The borders step as init_predc_* (src/align.impala:88-90,
// src/mapping_cpu.impala:70-78): gaps in global mode, the end otherwise.
__global__ void trace_walk_kernel(const uint8_t* __restrict__ q, const uint8_t* __restrict__ s,
                                  const int* __restrict__ blk_off, const int* __restrict__ blk_h,
                                  const int* __restrict__ blk_end_type, const int* __restrict__ blk_end, int nblocks,
                                  int n, int glob, int gi, const unsigned short* __restrict__ pred16,
                                  uint8_t* __restrict__ out_q, uint8_t* __restrict__ out_s)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const int off = blk_off[b], h = blk_h[b];
    if (h < 0) return;                                                // block of another rank (sharded traceback)
    const int oj = b * kMinPartW;
    const int w = min(kMinPartW, n - oj);
    int i = h - 1, j = w - 1;
    int state = 0;                                    // 0 = H, 1 = E, 2 = F
    if (blk_end_type[b] && h > 0 && w > 0 && blk_end[2 * b + 1] - gi > blk_end[2 * b]) state = 1;
    const size_t ob = (size_t)off + (size_t)oj;
    for (;;) {
        if (i < 0 && j < 0) break;
        const size_t pos = ob + (size_t)(i + j + 1);
        if (i < 0) {                                  // top border: horizontal gap (global only)
            if (!glob) break;
            out_q[pos] = '_'; out_s[pos] = s[oj + j]; --j; continue;
        }
        if (j < 0) {                                  // left border: vertical gap (global only)
            if (!glob) break;
            out_q[pos] = q[off + i]; out_s[pos] = '_'; --i; continue;
        }
        const unsigned p = (pred16[(size_t)(off + i) * 32 + (j >> 2)] >> (4 * (j & 3))) & 15u;
        if (state == 0) {
            const int src = p & 3;
            if (src == kSrcNone) break;
            if (src == kSrcDiag) { out_q[pos] = q[off + i]; out_s[pos] = s[oj + j]; --i; --j; }
            else state = (src == kSrcE) ? 1 : 2;
        } else if (state == 1) {
            out_q[pos] = '_'; out_s[pos] = s[oj + j];
            state = ((p >> 2) & 1) ? 1 : 0; --j;
        } else {
            out_q[pos] = q[off + i]; out_s[pos] = '_';
            state = ((p >> 3) & 1) ? 2 : 0; --i;
        }
    }
}

// which rank relaxes half `h` (= 2 * part + side) of a level with `np_full` parts (see TracebackShard)
int traceback_half_owner(int h, int np_full, int world)
{
    const int halves = 2 * np_full;
    return halves >= world ? h / (halves / world) : h * (world / halves);
}

static int next_pow_2(int i)   // src/utils.impala:19-28
{
    if (i == 0) return 0;
    int n = i - 1, r = 1;
    while (n > 0) { n >>= 1; r <<= 1; }
    return r;
}

int Engine::align_host(const anyseq_scoring& sc, const char* q, int m, const char* s, int n, char* alq,
                       char* als, anyseq_result* out)
{
    if (m < 0 || n < 0 || !out || (m > 0 && !q) || (n > 0 && !s)) { set_last_error("bad arguments"); return ANYSEQ_ERR_BAD_ARG; }
    std::lock_guard<std::recursive_mutex> lock(mu_);
    ANYSEQ_CUDA_CHECK(cudaSetDevice(device));
    ScoreParams sp;
    bool affine;
    int rc = make_score_params(sc, &sp, &affine);
    if (rc) return rc;
    const size_t outlen = (size_t)m + (size_t)n;
    std::memset(out, 0, sizeof(*out));
    out->end_i = -1;
    out->end_j = -1;
    if (outlen == 0) return ANYSEQ_OK;
    if (m == 0 || n == 0) {
        // no block ever runs in the reference; global borders still produce the
        // all-gap alignment of the non-empty subject (Q4-style), nothing else does
        std::memset(alq, ' ', outlen);
        std::memset(als, ' ', outlen);
        if (sc.mode == ANYSEQ_GLOBAL && m == 0)
            for (int j = 0; j < n; ++j) { alq[j] = '_'; als[j] = s[j]; }
        anyseq_result tmp;
        rc = score_host(sc, q, m, s, n, &tmp);
        if (rc) return rc;
        out->score = tmp.score;
        return ANYSEQ_OK;
    }
    if ((rc = check_score_range(sc, m, n))) return rc;

    const bool local = sc.mode == ANYSEQ_LOCAL;
    const int glob = sc.mode == ANYSEQ_GLOBAL;
    const int gi = sc.gap_init, ge = sc.gap_extend;     // linear: gi = 0
    int launches = 0;
    float total_ms = 0.f;

    // true optimal score of the scheme (the reference returns the value of a
    // never-relaxed object here, quirk Q1; the legacy symbols reproduce that)
    const int srank = shard_ ? shard_->rank : 0, sworld = shard_ ? shard_->world : 1;
    if (tune.align_with_score && !shard_) {
        anyseq_result tmp;
        rc = score_host(sc, q, m, s, n, &tmp);
        if (rc) return rc;
        out->score = tmp.score;
        out->end_i = tmp.end_i;
        out->end_j = tmp.end_j;
        launches += tmp.kernel_launches;
        total_ms += tmp.kernel_ms;
    }

    // sequences + reversed copies
    if (seq_q_.ensure((size_t)m + 64) || seq_s_.ensure((size_t)n + 64) || seq_qr_.ensure((size_t)m + 64) ||
        seq_sr_.ensure((size_t)n + 64))
        return ANYSEQ_ERR_NO_DEVICE;
    ANYSEQ_CUDA_CHECK(cudaEventRecord(ev0_, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(seq_q_.ptr, q, (size_t)m, cudaMemcpyHostToDevice, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(seq_s_.ptr, s, (size_t)n, cudaMemcpyHostToDevice, stream_));
    reverse_bytes_kernel<<<std::min(1024, (m + 255) / 256), 256, 0, stream_>>>(seq_q_.as<uint8_t>(), seq_qr_.as<uint8_t>(), m);
    reverse_bytes_kernel<<<std::min(1024, (n + 255) / 256), 256, 0, stream_>>>(seq_s_.as<uint8_t>(), seq_sr_.as<uint8_t>(), n);
    launches += 2;
    const uint8_t* d_q = seq_q_.as<uint8_t>();
    const uint8_t* d_s = seq_s_.as<uint8_t>();
    const uint8_t* d_qr = seq_qr_.as<uint8_t>();
    const uint8_t* d_sr = seq_sr_.as<uint8_t>();

    // Splits: src/traceback_lintime.impala:9-42 (index -1 stored at [0]), and the type of every split vertex
    int part_width = next_pow_2(n);
    const int nb = (n + kMinPartW - 1) / kMinPartW;
    int bpp = part_width / kMinPartW;
    const int full_width = part_width;
    std::vector<int> splits((size_t)nb + 1, shard_ ? -1 : 0), types((size_t)nb + 1, 0);   // sharded: -1 = another rank's split
    splits[0] = 0;
    splits[nb] = m;
    auto part_dims = [&](int part, int* off, int* h, int* start_slot, int* end_slot) {
        const int start = part * bpp - 1;
        const int end = std::min((part + 1) * bpp - 1, nb - 1);
        *off = splits[start + 1];
        *h = splits[end + 1] - *off;
        *start_slot = start;
        *end_slot = end;
    };

    const size_t rowlen = (size_t)std::max(part_width, kMinPartW) + 1024;
    if (col_.ensure(sizeof(int4) * (size_t)m) || col2_.ensure(sizeof(int4) * (size_t)m) ||
        rowH_.ensure(sizeof(int) * rowlen) || (affine && rowF_.ensure(sizeof(int) * rowlen)) ||
        aux_.ensure(sizeof(int) * 2 * ((size_t)nb + 1)))
        return ANYSEQ_ERR_NO_DEVICE;
    int* d_splits = aux_.as<int>();
    int* d_types = d_splits + (nb + 1);
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(d_splits, splits.data(), sizeof(int) * splits.size(), cudaMemcpyHostToDevice, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(d_types, types.data(), sizeof(int) * types.size(), cudaMemcpyHostToDevice, stream_));

    rc = analyse_alphabet(d_q, m, d_s, n);
    if (rc) return rc;
    launches += 3;
    // a rank of a sharded traceback relaxes 1 / world of the columns of every level: strips for ITS schedulers
    const int Ktop = pick_K_levels(n / sworld);
    std::vector<Job> jobs;
    std::vector<HbPart> parts;

    const bool trace_levels = std::getenv("ANYSEQ_TRACE_LEVELS") != nullptr;   // development: per-level host time on stderr
    while (part_width > kMinPartW) {
        const auto lvl_t0 = std::chrono::steady_clock::now();
        const int half = part_width / 2;
        const int num_halfs = (n + half - 1) / part_width * 2;
        const int nparts = num_halfs / 2;
        const int K = std::max(4, std::min(Ktop, half / kWarp));
        const int SW = kWarp * K;

        // sharded traceback: who relaxes which half of this level (TracebackShard)
        const int np_full = full_width / part_width;
        const bool shared_level = sworld > 1 && np_full < sworld;       // the halves of a part sit on different ranks
        jobs.clear();
        parts.clear();
        long long strip_total = 0;
        for (int p = 0; p < nparts; ++p) {
            const int own_l = sworld > 1 ? traceback_half_owner(2 * p, np_full, sworld) : 0;
            const int own_r = sworld > 1 ? traceback_half_owner(2 * p + 1, np_full, sworld) : 0;
            if (!shared_level && own_l != srank) continue;              // a whole part of another rank
            int off, len, s0, s1;
            part_dims(p, &off, &len, &s0, &s1);
            const int c_left = 2 * p * half;
            const int c_right = c_left + half;
            const int rhw = std::min(half, n - c_right);
            HbPart hp;
            hp.off = off; hp.len = len; hp.rhw = rhw;
            hp.split_slot = p * bpp + bpp / 2 - 1;
            hp.open_l = types[s0 + 1] ? 0 : gi;
            hp.open_r = types[s1 + 1] ? 0 : gi;
            parts.push_back(hp);
            if (len <= 0) continue;
            for (int side = 0; side < 2; ++side) {
                if ((side == 0 ? own_l : own_r) != srank) continue;
                Job J;
                std::memset(&J, 0, sizeof(J));
                const int w = side == 0 ? half : rhw;
                const int c0 = side == 0 ? c_left : c_right;
                J.q = side == 0 ? d_q + off : d_qr + (m - off - len);
                J.s = side == 0 ? d_s + c0 : d_sr + (n - c0 - w);
                J.h = len;
                J.w = w;
                J.nstrips = (w + SW - 1) / SW;
                J.col = (side == 0 ? col_.as<int4>() : col2_.as<int4>()) + off;
                J.rowH = rowH_.as<int>() + c0;
                if (affine) J.rowF = rowF_.as<int>() + c0;
                J.item_begin = strip_total;
                strip_total += J.nstrips;
                J.best = misc_.as<int>() + kMiscBest;
                J.init_global = glob;
                J.top_open = (side == 0 ? hp.open_l : hp.open_r) + ge;
                jobs.push_back(J);
            }
        }
        if (!jobs.empty()) {
            if (corner_.ensure(sizeof(int) * (size_t)strip_total) || progress_.ensure(sizeof(int) * (size_t)strip_total))
                return ANYSEQ_ERR_NO_DEVICE;
            for (Job& J : jobs) {
                J.corner = corner_.as<int>() + J.item_begin;
                J.progress = progress_.as<int>() + J.item_begin;
            }
            init_col0_ = 0;
            rc = run_jobs(jobs, sp, local, affine, K, &launches);
            if (rc) return rc;
        }
        if (shared_level) {
            // every rank needs the last-column records of BOTH halves of every part of this level (H, and E for the
            // Gotoh joins): broadcast them from the ranks that relaxed them (16 bytes per query row and half; NVLink)
            ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(stream_));
            for (int p = 0; p < (int)parts.size(); ++p) {
                const HbPart& hp = parts[(size_t)p];
                if (hp.len <= 0) continue;
                rc = shard_->bcast(shard_->user, col_.as<int4>() + hp.off, (int64_t)sizeof(int4) * hp.len,
                                   traceback_half_owner(2 * p, np_full, sworld));
                if (!rc) rc = shard_->bcast(shard_->user, col2_.as<int4>() + hp.off, (int64_t)sizeof(int4) * hp.len,
                                            traceback_half_owner(2 * p + 1, np_full, sworld));
                if (rc) { set_last_error("sharded traceback: the broadcast callback failed"); return ANYSEQ_ERR_BAD_ARG; }
            }
        }
        const int nparts_here = (int)parts.size();      // all parts of a shared level, else the parts of this rank
        if (aux2_.ensure(sizeof(HbPart) * (size_t)std::max(nparts_here, 1))) return ANYSEQ_ERR_NO_DEVICE;
        ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(aux2_.ptr, parts.data(), sizeof(HbPart) * (size_t)nparts_here, cudaMemcpyHostToDevice, stream_));
        const int bpp2 = part_width / std::min(kRefBlockW, part_width);
        const auto hb_sum = affine ? hb_sum_kernel<true> : hb_sum_kernel<false>;
        if (nparts_here > 0)
        hb_sum<<<std::min(nparts_here, 4096), 256, 0, stream_>>>(aux2_.as<HbPart>(), nparts_here, col_.as<int4>(),
                                                            col2_.as<int4>(), d_splits, d_types, half, bpp2, glob, gi, ge);
        ANYSEQ_CUDA_CHECK(cudaGetLastError());
        launches += 1;
        ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(splits.data(), d_splits, sizeof(int) * splits.size(), cudaMemcpyDeviceToHost, stream_));
        ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(types.data(), d_types, sizeof(int) * types.size(), cudaMemcpyDeviceToHost, stream_));
        ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(stream_));
        ANYSEQ_CUDA_CHECK(cudaMemcpy(h_misc_, misc_.ptr, sizeof(int) * 4, cudaMemcpyDeviceToHost));
        if (h_misc_[kMiscStatus] != kStatusOk) {
            set_last_error("strip kernel watchdog fired during a Hirschberg level");
            return ANYSEQ_ERR_KERNEL_TIMEOUT;
        }
        if (trace_levels) {
            const double lvl_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - lvl_t0).count();
            std::fprintf(stderr, "[anyseq level] part_width=%d parts=%d jobs=%zu K=%d: %.2f ms\n", part_width, nparts, jobs.size(), K, lvl_ms);
        }
        part_width /= 2;
        bpp /= 2;
    }

    // final pass: blockwise relaxation with predecessors + walks.  Per block: offset, height, opening cost on the
    // top border, end vertex type
    std::vector<int> blk(4 * (size_t)nb);
    const int blocks_full = std::max(1, full_width / kMinPartW);
    long long out_lo = (long long)outlen, out_hi = 0;
    for (int b = 0; b < nb; ++b) {
        const int owner = (sworld > 1 && blocks_full >= sworld) ? b / (blocks_full / sworld) : 0;
        if (owner != srank) { blk[b] = 0; blk[nb + b] = -1; blk[2 * nb + b] = 0; blk[3 * nb + b] = 0; continue; }   // skipped by the kernels
        int off, h, s0, s1;
        part_dims(b, &off, &h, &s0, &s1);   // bpp == 1 here, or 0 for n <= 64 (quirk Q4: height 0)
        blk[b] = off;
        blk[nb + b] = h;
        blk[2 * nb + b] = types[s0 + 1] ? 0 : gi;
        blk[3 * nb + b] = types[s1 + 1];
        // the block writes output columns [off + 128 b, off + h + 128 b + w) only
        out_lo = std::min(out_lo, (long long)off + (long long)b * kMinPartW);
        out_hi = std::max(out_hi, (long long)off + h + (long long)b * kMinPartW + std::min(kMinPartW, n - b * kMinPartW));
    }
    if (shard_) {
        // the ranges of the ranks tile [0, m + n): the first rank starts at 0, the last one ends at m + n
        if (out_lo > out_hi) out_lo = out_hi = 0;
        shard_->out_lo = out_lo;
        shard_->out_hi = out_hi;
    }
    if (aux2_.ensure(sizeof(int) * 6 * (size_t)nb) || pred_.ensure((size_t)m * 64 + 128) || tb_out_.ensure(2 * outlen + 64))
        return ANYSEQ_ERR_NO_DEVICE;
    int* d_blk = aux2_.as<int>();
    int* d_blk_end = d_blk + 4 * nb;
    uint8_t* d_out = tb_out_.as<uint8_t>();
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(d_blk, blk.data(), sizeof(int) * blk.size(), cudaMemcpyHostToDevice, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemsetAsync(d_blk_end, 0, sizeof(int) * 2 * (size_t)nb, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemsetAsync(d_out, ' ', 2 * outlen, stream_));
    {
        const int wpb = 4;
        const int grid = std::min((nb + wpb - 1) / wpb, sm_count * 16);
        trace_dp_kernel<<<grid, wpb * 32, 0, stream_>>>(d_q, d_s, d_blk, d_blk + nb, d_blk + 2 * nb, nb, n, local ? 1 : 0,
                                                        glob, sp.same, sp.diff, gi, ge, pred_.as<unsigned short>(), d_blk_end);
        ANYSEQ_CUDA_CHECK(cudaGetLastError());
        trace_walk_kernel<<<(nb + 127) / 128, 128, 0, stream_>>>(d_q, d_s, d_blk, d_blk + nb, d_blk + 3 * nb, d_blk_end, nb,
                                                                 n, glob, gi, pred_.as<unsigned short>(), d_out, d_out + outlen);
        ANYSEQ_CUDA_CHECK(cudaGetLastError());
        launches += 2;
    }
    ANYSEQ_CUDA_CHECK(cudaEventRecord(ev1_, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(alq, d_out, outlen, cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(als, d_out + outlen, outlen, cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(stream_));
    float ms = 0.f;
    ANYSEQ_CUDA_CHECK(cudaEventElapsedTime(&ms, ev0_, ev1_));
    out->kernel_ms = total_ms + ms;
    out->kernel_launches = launches;
    last_splits_ = splits;
    last_types_ = affine ? types : std::vector<int>();
    return ANYSEQ_OK;
}

int Engine::align_host_sharded(const anyseq_scoring& sc, const char* q, int m, const char* s, int n, char* alq, char* als,
                               anyseq_result* out, TracebackShard* shard)
{
    if (!shard || shard->world < 1 || (shard->world & (shard->world - 1)) != 0 || shard->rank < 0 || shard->rank >= shard->world ||
        (shard->world > 1 && !shard->bcast)) {
        set_last_error("sharded traceback: world must be a power of two, 0 <= rank < world, and a broadcast callback is needed");
        return ANYSEQ_ERR_BAD_ARG;
    }
    if (m < 1 || n < 1) { set_last_error("sharded traceback: empty sequence"); return ANYSEQ_ERR_BAD_ARG; }
    std::lock_guard<std::recursive_mutex> lock(mu_);
    struct Scope { TracebackShard*& p; ~Scope() { p = nullptr; } } scope{shard_};
    shard_ = shard;
    shard->out_lo = shard->out_hi = 0;
    return align_host(sc, q, m, s, n, alq, als, out);
}

}  // namespace anyseq
