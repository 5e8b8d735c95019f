// engine.cu -- score-only path: job construction, launches, result extraction.
#include "engine.cuh"
#include "strip_kernel.cuh"

#include <algorithm>
#include <cstdlib>
#include <cstring>

namespace anyseq {

static thread_local std::string g_last_error;
void set_last_error(const std::string& s) { g_last_error = s; }
const char* last_error_cstr() { return g_last_error.c_str(); }

// ---------------------------------------------------------------------------
// border initialisation: create_scoring_matrix_linmem (src/scoring.impala:218-242)
// and create_scoring_hb_matrix_linmem (:261-299) -- column/row/corner vectors
// from init_scores (src/align.impala:85-86).  border(k) = H(k, -1) = H(-1, k).
// ---------------------------------------------------------------------------
__global__ void init_jobs_kernel(const Job* __restrict__ jobs, int njobs, ScoreParams sp, int SW,
                                 int col0)
{
    for (int jb = blockIdx.y; jb < njobs; jb += gridDim.y) {
        const Job J = jobs[jb];
        const int wpad = J.nstrips * SW;
        const int n = max(max(J.h, wpad), J.nstrips);
        for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += gridDim.x * blockDim.x) {
            if (idx < J.h) {
                // left matrix border as records tagged 0: {H(idx,-1), 0, E(idx,-1) = -inf, 0}
                J.col[idx] = make_int4(J.init_global ? sp.gap_open + idx * sp.gap_extend : 0, 0, kNegInf, 0);
            }
            if (idx < wpad) {
                J.rowH[idx] = J.init_global ? J.top_open + (col0 + idx) * sp.gap_extend : 0;
                if (J.rowF) J.rowF[idx] = kNegInf;
            }
            if (idx < J.nstrips) {
                const int c = col0 + idx * SW - 1;   // column left of the strip
                J.corner[idx] = (J.init_global && c >= 0) ? J.top_open + c * sp.gap_extend : 0;
                J.progress[idx] = 0;
            }
            if (idx == 0 && J.best) *J.best = kScoreMin;
        }
    }
}

// ---------------------------------------------------------------------------
// result extraction: get_{global,semiglobal,local}_scoring_linmem
// (src/scoring.impala:29-137).  reduce_max of the reference returns the LOWEST
// index attaining the maximum (src/utils.impala:30-49,
// src/iteration_cpu.impala:205-250); arg_max_lowest reproduces that.
// ---------------------------------------------------------------------------
__device__ void arg_max_lowest(const int* __restrict__ v, int n, int stride, int& best, int& best_i)
{
    __shared__ int s_v[32];
    __shared__ int s_i[32];
    int bv = kScoreMin, bi = 0x7fffffff;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int x = __ldcg(v + (size_t)i * stride);
        if (x > bv) { bv = x; bi = i; }   // ascending i per thread: first max kept
    }
    for (int o = 16; o > 0; o >>= 1) {
        const int ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = bv; s_i[threadIdx.x >> 5] = bi; }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int nw = (blockDim.x + 31) / 32;
        bv = threadIdx.x < nw ? s_v[threadIdx.x] : kScoreMin;
        bi = threadIdx.x < nw ? s_i[threadIdx.x] : 0x7fffffff;
        for (int o = 16; o > 0; o >>= 1) {
            const int ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
    }
    __syncthreads();
    best = bv;
    best_i = bi;   // valid in thread 0
}

// out[0]=score out[1]=pos_i out[2]=pos_j ; partial (multi-GPU) results in out[3..7]:
// row_best,row_best_j,col_best,col_best_i ; local_best in out[0]
__global__ void finish_score_kernel(const Job* __restrict__ jobs, int mode, int col0, int n_total,
                                    int* __restrict__ out)
{
    const Job J = jobs[blockIdx.x];          // one block per job, 8 result words each
    out += 8 * blockIdx.x;
    int rv, ri, cv, ci;
    const int* colH = reinterpret_cast<const int*>(J.col);      // .x of every 16-byte record
    arg_max_lowest(J.rowH, J.w, 1, rv, ri);
    arg_max_lowest(colH, J.h, 4, cv, ci);
    if (threadIdx.x == 0) {
        out[3] = rv; out[4] = ri + col0; out[5] = cv; out[6] = ci;
        out[7] = __ldcg(colH + 4 * (size_t)(J.h - 1));
        if (mode == kGlobal) {
            out[0] = __ldcg(colH + 4 * (size_t)(J.h - 1));
            out[1] = J.h - 1; out[2] = n_total - 1;
        } else if (mode == kSemiglobal) {
            // candidates -1 (value init = 0) come first and win ties
            // (src/scoring.impala:51-63: row first, column only if strictly greater)
            int score = kScoreMin, pi = -1, pj = -1;
            int rs = rv, rj = ri + col0;
            if (0 >= rs) { rs = 0; rj = -1; }
            if (rs > score) { score = rs; pi = J.h - 1; pj = rj; }
            int cs = cv, cidx = ci;
            if (0 >= cs) { cs = 0; cidx = -1; }
            if (cs > score) { score = cs; pi = cidx; pj = n_total - 1; }
            out[0] = score; out[1] = pi; out[2] = pj;
        } else {
            out[0] = *J.best; out[1] = -1; out[2] = -1;
        }
    }
}

// Local end cell by the reference's rule.  The reference keeps one (maximum, position) slot per index
// INSIDE a block anti-diagonal (slot = block_dia_j, src/scoring_cpu.impala:56-73), updates a slot with
// strict '>' as the diagonals go by, and get_score_pos() takes the lowest slot holding the overall
// maximum (src/scoring.impala:103-110 -> reduce_max, src/utils.impala:30-49).  So among the 1024 x 1024
// blocks that contain the maximum M the winner has the smallest slot, then the smallest diagonal; inside
// a block the first cell in row-major order (src/scoring_cpu.impala:48-54).  blockmax holds, per block,
// (value ^ sign, 0xfffff - row-major position) written by the tracking strip kernels.
__global__ void local_end_cell_kernel(const unsigned long long* __restrict__ blockmax, int nbi, int nbj,
                                      int* __restrict__ out)
{
    __shared__ unsigned long long s_red[32];
    const long long nblk = (long long)nbi * nbj;
    auto block_reduce = [&](unsigned long long v, bool want_max) {
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long u = __shfl_xor_sync(0xffffffffu, v, o);
            v = want_max ? (u > v ? u : v) : (u < v ? u : v);
        }
        __syncthreads();
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
        __syncthreads();
        v = s_red[0];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) {
            const unsigned long long u = s_red[w];
            v = want_max ? (u > v ? u : v) : (u < v ? u : v);
        }
        return v;
    };
    unsigned long long top = 0ull;
    for (long long b = threadIdx.x; b < nblk; b += blockDim.x) {
        const unsigned long long v = blockmax[b] >> 32;
        top = v > top ? v : top;
    }
    top = block_reduce(top, true);
    unsigned long long pick = ~0ull;            // (slot, diagonal) of the winning block
    for (long long b = threadIdx.x; b < nblk; b += blockDim.x) {
        if ((blockmax[b] >> 32) != top) continue;
        const int bi = (int)(b / nbj), bj = (int)(b % nbj);
        const int d = bi + bj;
        const int slot = min(d, nbi - 1) - bi;
        const unsigned long long key = ((unsigned long long)(unsigned)slot << 32) | (unsigned)d;
        pick = key < pick ? key : pick;
    }
    pick = block_reduce(pick, false);
    if (threadIdx.x == 0 && top != 0ull) {
        const int slot = (int)(pick >> 32), d = (int)(pick & 0xffffffffu);
        const int bi = min(d, nbi - 1) - slot, bj = d - bi;
        const unsigned pos = 0xfffffu - (unsigned)(blockmax[(size_t)bi * nbj + bj] & 0xfffffu);
        out[1] = bi * 1024 + (int)(pos >> 10);
        out[2] = bj * 1024 + (int)(pos & 1023u);
    }
}

// ---------------------------------------------------------------------------
// kernel dispatch (instantiations live in strip_inst_*.cu)
// ---------------------------------------------------------------------------
using KernelFn = StripKernelFn;

static KernelFn pick_kernel(bool local, bool affine, int K, bool mask, bool track, int form)
{
    if (form == 3) return get_strip_kernel_01p(K);
    if (local && track) return affine ? get_strip_kernel_11t(K, mask) : get_strip_kernel_10t(K, mask);
    if (local) return affine ? get_strip_kernel_11(K, mask, form) : get_strip_kernel_10(K, mask, form);
    return affine ? get_strip_kernel_01(K, mask, form) : get_strip_kernel_00(K, mask, form);
}

// Cell form of a launch (strip_kernel.cuh: 1 = decoupled, 2 = mixed).  Measured on B200s with the warps of a
// scheduler on adjacent strips, semiglobal Gotoh, GCUPS, coupled / decoupled / mixed: 4.6 Mbp pair, three warps per
// scheduler: 3853 / 3864-3885 on four different boxes / 3974 on one box, 3753-3758 on three others (local Gotoh:
// 3315 / 3038 / 3302-3505); 575 k-column slice, two per scheduler: 2846 / 3195 / 3159; lone warps (K = 32 slice):
// 2214 / 2885 / 2753; 1 Mbp x 1 Mbp: 2500 / 3157 / 2654.  So: the decoupled cells everywhere -- they are the fastest or
// within 2 % of it and the most repeatable -- except for wide LOCAL Gotoh launches, whose decoupled cell needs one more
// instruction; those run the mixed cells.  The coupled cells, never ahead by more than noise, are not built for these
// kernels.  cell_form 1 / 2 forces a form, any other value picks per launch.
static int pick_form(const Tuning& tune, bool affine, bool mask, int K, long long strips_total, int sm_count, bool local)
{
    const bool has_mixed = affine && mask && K >= 16;
    if (tune.cell_form == 1) return 1;
    if (tune.cell_form == 2) return has_mixed ? 2 : 1;
    return (has_mixed && local && strips_total >= 24LL * sm_count) ? 2 : 1;
}

// Packed cells (strip_packed.cuh) hold a warp's scores as 16-bit halves around a re-centred offset.  With go = gi + ge,
// a step right or down changes H by a value in [go, same - go], so every value alive in a warp is within
// D = max(same - go, -go) per row or column of the others: the warp's live window is 128 rows (64 lanes of two-row
// tiles) plus 32 rows of drift between two re-centrings, by the strip's 32 * K columns.  It must fit, with the
// sigma / go constants, into [0x400, 0x7c00] around the centre 0x4000 -- far from 0 and 0xffff, where the IMAD of a
// packed add would carry into the other half.
static bool packed_fits(const ScoreParams& sp, int K)
{
    if (K != 16 && K != 32) return false;
    if (sp.gap_open > 0 || sp.gap_extend > 0 || sp.gap_open > sp.gap_extend || sp.same < sp.diff) return false;
    const long long D = std::max<long long>((long long)sp.same - sp.gap_open, -(long long)sp.gap_open);
    const long long constants = 4LL * (std::llabs(sp.same) + std::llabs(sp.diff) + std::llabs(sp.gap_open));
    return D * (128 + 32 + 32LL * K) + constants <= 0x3c00;
}

// Packed cells for a global / semiglobal Gotoh score launch (MASK kernels, K = 16 or 32) whose window fits; the
// option packed_cells = 0 keeps the 32-bit decoupled cells.
static bool use_packed(const Tuning& tune, const ScoreParams& sp, bool local, bool affine, bool mask, bool track, int K)
{
    return tune.packed_cells != 0 && !local && affine && mask && !track && packed_fits(sp, K);
}

// rows per lane and step of the kernel variant (strip_kernel.cuh: StripRows)
static int rows_per_step(int K, bool mask, bool track)
{
    if (!mask || track) return 1;      // end-cell tracking runs on the single-row kernels
    return K >= 32 ? ANYSEQ_ROWS_K32 : (K >= 16 ? ANYSEQ_ROWS_K16 : (K >= 8 ? ANYSEQ_ROWS_K8 : ANYSEQ_ROWS_K4));
}

// CTAs per SM actually launched.  Multi-row tiles carry R dependent chains per
// warp, so 2-3 warps per scheduler saturate the issue slots; and never more warps
// than strips: at most one warp works on a strip at a time, the others would only
// poll and add spread to the progress of the busy ones -- which is what the
// strip-to-strip pipeline is sensitive to (measured: profiles/).
static int default_blocks_per_sm(int K, bool mask, bool track, int occupancy_max, long long nstrips, int sm_count)
{
    int nb = occupancy_max;
    if (rows_per_step(K, mask, track) >= 2) {
        const long long per_round = 4LL * sm_count;              // warps of one CTA per SM
        // Enough warps for every strip to have its own (single-band launches), at most three per scheduler (measured
        // on the 4.6 Mbp pair, decoupled cells: 3736 GCUPS with two, 3883 with three; linear gaps 5376 / 5687) -- but
        // only if that loads the schedulers evenly: in a single-band chain the most loaded scheduler sets the pace of
        // every strip to its right (1218 strips as 3+2+2+2 per SM: 2470 GCUPS; 1124 strips as 2+2+2+2: 3214).  A launch
        // that would fill less than 80 % of the warps runs with one warp less and several bands.
        int want = (int)std::max<long long>(1, (nstrips + per_round - 1) / per_round);
        if (want > 1 && nstrips * 10 < (long long)want * per_round * 8) --want;
        nb = std::min(nb, std::min(3, want));
    }
    return nb;
}

// dynamic shared memory of the MASK kernels: [warps][ncodes][32 lanes][W words] spread column masks (packed cells:
// one set per half of the strip)
static size_t mask_smem_bytes(bool mask, bool track, int ncodes, int K, int warps, int form)
{
    if (!mask) return 0;
    const int words = std::max(1, rows_per_step(K, mask, track) * K / 32) * (form == 3 ? 2 : 1);
    return sizeof(unsigned) * 32 * (size_t)ncodes * warps * words;
}

// Launch shape of a strip kernel: the end-cell tracking kernels run `nb` CTAs of 4 warps per SM, all others ONE CTA of
// 4 * nb warps per SM (strip_kernel.cuh: the warps of a scheduler take adjacent strips).  Returns the largest nb <= want
// that fits, 0 if none does.
static int fit_blocks_per_sm(KernelFn fn, bool track, bool mask, int ncodes, int K, int want, int form)
{
    for (int nb = want; nb >= 1; --nb) {
        int got = 0;
        const int warps = track ? kWarpsPerBlock : kWarpsPerBlock * nb;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&got, fn, warps * kWarp, mask_smem_bytes(mask, track, ncodes, K, warps, form)) != cudaSuccess)
            return 0;
        if (track ? got >= nb : got >= 1) return nb;
    }
    return 0;
}

// Grid of a strip-kernel launch with `total` items and nb warps per scheduler: ONE CTA per SM for the ordinary kernels
// (nb CTAs of 4 warps for the tracking kernels); with few items, just enough warps per CTA that every item of the first
// round has one, spread evenly over all SMs.
static void launch_shape(bool track, int nb, int sm_count, long long total, int* grid, int* warps_per_cta, long long* first_items)
{
    const int wpb = track ? kWarpsPerBlock : kWarpsPerBlock * nb;
    int wpb_used = wpb;
    int g;
    if (track) {
        g = (int)std::min<long long>((long long)nb * sm_count, std::max<long long>((total + wpb - 1) / wpb, 1));
    } else {
        g = (int)std::min<long long>(sm_count, std::max<long long>((total + kWarpsPerBlock - 1) / kWarpsPerBlock, 1));
        const long long per_cta = (total + g - 1) / g;                   // items of the fullest CTA
        wpb_used = (int)std::min<long long>(wpb, (per_cta + kWarpsPerBlock - 1) / kWarpsPerBlock * kWarpsPerBlock);
    }
    *grid = g;
    *warps_per_cta = wpb_used;
    *first_items = std::min<long long>(total, (long long)g * wpb_used);
}

// ---------------------------------------------------------------------------
// alphabet analysis for the MASK kernels.  Symbols are compared as raw bytes
// (src/align.impala:132), so any equality-preserving recoding is legal: bytes
// that occur in BOTH sequences get codes 1..A, every other byte gets code 0,
// which matches nothing (its column mask is empty).
// ---------------------------------------------------------------------------
__global__ void alphabet_presence_kernel(const uint8_t* __restrict__ p, long long n, unsigned* __restrict__ bits /* [8] */)
{
    __shared__ unsigned s_bits[8];
    if (threadIdx.x < 8) s_bits[threadIdx.x] = 0u;
    __syncthreads();
    unsigned loc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const unsigned b = p[i];
#pragma unroll
        for (int w = 0; w < 8; ++w) loc[w] |= ((b >> 5) == (unsigned)w) ? (1u << (b & 31)) : 0u;
    }
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        unsigned v = loc[w];
        for (int o = 16; o > 0; o >>= 1) v |= __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0 && v) atomicOr(&s_bits[w], v);
    }
    __syncthreads();
    if (threadIdx.x < 8 && s_bits[threadIdx.x]) atomicOr(&bits[threadIdx.x], s_bits[threadIdx.x]);
}

// bits_q/bits_s [8] -> lut_q/lut_s [256], *ncodes = 1 + number of shared symbols
__global__ void build_lut_kernel(const unsigned* __restrict__ bits_q, const unsigned* __restrict__ bits_s,
                                 uint8_t* __restrict__ lut_q, uint8_t* __restrict__ lut_s, int* __restrict__ ncodes)
{
    if (threadIdx.x == 0) {
        int next = 1;
        for (int b = 0; b < 256; ++b) {
            const bool both = ((bits_q[b >> 5] >> (b & 31)) & 1u) && ((bits_s[b >> 5] >> (b & 31)) & 1u);
            int code = 0;
            if (both) { code = next < 255 ? next : 255; ++next; }
            lut_q[b] = (uint8_t)code;
            lut_s[b] = (uint8_t)code;
        }
        *ncodes = next;
    }
}

int Engine::init(int dev)
{
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        set_last_error("no CUDA device available (libanyseq_b200 has no CPU fallback)");
        return ANYSEQ_ERR_NO_DEVICE;
    }
    if (dev < 0) ANYSEQ_CUDA_CHECK(cudaGetDevice(&dev));
    ANYSEQ_CUDA_CHECK(cudaSetDevice(dev));
    device = dev;
    cudaDeviceProp prop;
    ANYSEQ_CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
    sm_count = prop.multiProcessorCount;
    std::strncpy(name, prop.name, sizeof(name) - 1);
    if (prop.major < 10) {
        set_last_error(std::string("device ") + prop.name + " is not sm_100-class; this library is built for sm_100a only");
        return ANYSEQ_ERR_NO_DEVICE;
    }
    ANYSEQ_CUDA_CHECK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
    ANYSEQ_CUDA_CHECK(cudaEventCreate(&ev0_));
    ANYSEQ_CUDA_CHECK(cudaEventCreate(&ev1_));
    if (misc_.ensure(sizeof(int) * kMiscWords)) return ANYSEQ_ERR_NO_DEVICE;
    ANYSEQ_CUDA_CHECK(cudaMallocHost(&h_misc_, sizeof(int) * kMiscWords + 512));    // + the host-built byte -> code tables
    const char* env;
    if ((env = std::getenv("ANYSEQ_K"))) tune.cols_per_lane = std::atoi(env);
    if ((env = std::getenv("ANYSEQ_BAND"))) tune.band_rows = std::atoi(env);
    if ((env = std::getenv("ANYSEQ_BLOCKS_PER_SM"))) tune.blocks_per_sm = std::atoi(env);
    if ((env = std::getenv("ANYSEQ_WATCHDOG_MS"))) tune.watchdog_ms = std::atoi(env);
    if ((env = std::getenv("ANYSEQ_ALIGN_SCORE"))) tune.align_with_score = std::atoi(env) != 0;
    if ((env = std::getenv("ANYSEQ_FORCE_GENERIC"))) tune.force_generic = std::atoi(env) != 0;
    if ((env = std::getenv("ANYSEQ_CELL_FORM"))) tune.cell_form = std::atoi(env);
    if ((env = std::getenv("ANYSEQ_PACKED_CELLS"))) tune.packed_cells = std::atoi(env);
    if ((env = std::getenv("ANYSEQ_SMALL_MODEL"))) tune.small_model = std::atoi(env) != 0;
    if ((env = std::getenv("ANYSEQ_BATCH_PACKED"))) tune.batch_packed = std::atoi(env) != 0;
    if ((env = std::getenv("ANYSEQ_BATCH_QUAD"))) tune.batch_quad = std::atoi(env) != 0;
    if ((env = std::getenv("ANYSEQ_LOCAL_END_CELL"))) tune.local_end_cell = std::atoi(env) != 0;
    return ANYSEQ_OK;
}

void Engine::destroy()
{
    if (device >= 0) cudaSetDevice(device);
    DeviceBuffer* bufs[] = {&seq_q_, &seq_s_, &seq_qr_, &seq_sr_, &col_, &rowH_, &rowF_, &corner_,
                            &progress_, &jobs_, &misc_, &lut_, &col2_, &aux_, &aux2_, &pred_,
                            &tb_out_, &blockmax_, &edges_, &multi_, &p2_[0], &p2_[1], &batch_pred_, &batch_io_};
    drop_host_batch_stream();
    for (DeviceBuffer* b : bufs) b->release();
    if (h_misc_) cudaFreeHost(h_misc_);
    if (ev0_) cudaEventDestroy(ev0_);
    if (ev1_) cudaEventDestroy(ev1_);
    if (stream_) cudaStreamDestroy(stream_);
    if (copy_stream_) cudaStreamDestroy(copy_stream_);
    for (int i = 0; i < 2; ++i) {
        if (p2_ready_[i]) cudaEventDestroy(p2_ready_[i]);
        if (p2_done_[i]) cudaEventDestroy(p2_done_[i]);
        p2_ready_[i] = p2_done_[i] = nullptr;
    }
    copy_stream_ = nullptr;
    h_misc_ = nullptr; ev0_ = ev1_ = nullptr; stream_ = nullptr;
}

#ifdef ANYSEQ_PROFILE
// measurement builds only (tools/build_variants.sh): per-strip timeline + the time of the strip kernel alone
static unsigned long long* g_trace = nullptr;
static cudaEvent_t g_ev_k0 = nullptr, g_ev_k1 = nullptr;
static int g_trace_strips = 0;
#endif

int Engine::resident_warps(int K, bool local, bool affine, long long nstrips)
{
    const int form = pick_form(tune, affine, use_mask_, K, nstrips, sm_count, local);
    KernelFn fn = pick_kernel(local, affine, K, use_mask_, track_ && local, form);
    if (!fn) return 0;
    const bool track = track_ && local;
    int want = tune.blocks_per_sm > 0 ? tune.blocks_per_sm : default_blocks_per_sm(K, use_mask_, track, track ? 6 : 3, nstrips, sm_count);
    if (!track) want = std::min(want, kMaxStripWarps / kWarpsPerBlock);
    return fit_blocks_per_sm(fn, track, use_mask_, ncodes_, K, want, form) * kWarpsPerBlock * sm_count;
}

// Decide between the MASK and the generic kernels for a (query, subject) pair
// that is resident in device memory; builds the byte -> code tables.
int Engine::analyse_alphabet(const uint8_t* d_q, long long m, const uint8_t* d_s, long long n)
{
    if (alphabet_ready_) { alphabet_ready_ = false; return ANYSEQ_OK; }     // done on the host for this very pair
    if (lut_.ensure(512 + 64 + 16)) return ANYSEQ_ERR_NO_DEVICE;
    unsigned* bits = reinterpret_cast<unsigned*>(lut_.as<uint8_t>() + 512);   // [16] presence, then ncodes
    int* d_ncodes = reinterpret_cast<int*>(bits + 16);
    ANYSEQ_CUDA_CHECK(cudaMemsetAsync(bits, 0, sizeof(unsigned) * 17, stream_));
    const int gq = (int)std::min<long long>(sm_count * 8, (m + 255) / 256);
    const int gs = (int)std::min<long long>(sm_count * 8, (n + 255) / 256);
    alphabet_presence_kernel<<<std::max(gq, 1), 256, 0, stream_>>>(d_q, m, bits);
    alphabet_presence_kernel<<<std::max(gs, 1), 256, 0, stream_>>>(d_s, n, bits + 8);
    build_lut_kernel<<<1, 32, 0, stream_>>>(bits, bits + 8, lut_.as<uint8_t>(), lut_.as<uint8_t>() + 256, d_ncodes);
    ANYSEQ_CUDA_CHECK(cudaGetLastError());
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(h_misc_ + kMiscWords - 1, d_ncodes, sizeof(int), cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(stream_));
    ncodes_ = h_misc_[kMiscWords - 1];
    use_mask_ = ncodes_ <= kMaxCodes && !tune.force_generic;
    if (!use_mask_) ncodes_ = 1;
    return ANYSEQ_OK;
}

// The same analysis for sequences that are still in HOST memory (score_host / align_host): a pass over the bytes on the
// CPU and one small upload instead of three kernels and a device -> host round trip -- which is most of the fixed cost
// of a small alignment (align -r 10000: ~50 us of 1.5 ms).  The next analyse_alphabet() call is then skipped.
int Engine::analyse_alphabet_host(const uint8_t* q, long long m, const uint8_t* s, long long n)
{
    if (lut_.ensure(512 + 64 + 16)) return ANYSEQ_ERR_NO_DEVICE;
    bool in_q[256] = {false}, in_s[256] = {false};
    for (long long i = 0; i < m; ++i) in_q[q[i]] = true;
    for (long long j = 0; j < n; ++j) in_s[s[j]] = true;
    uint8_t* lut = reinterpret_cast<uint8_t*>(h_misc_ + kMiscWords);     // pinned scratch behind the misc mirror
    int next = 1;
    for (int b = 0; b < 256; ++b) {
        int code = 0;
        if (in_q[b] && in_s[b]) { code = next < 255 ? next : 255; ++next; }
        lut[b] = (uint8_t)code;
        lut[256 + b] = (uint8_t)code;
    }
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(lut_.ptr, lut, 512, cudaMemcpyHostToDevice, stream_));
    ncodes_ = next;
    use_mask_ = ncodes_ <= kMaxCodes && !tune.force_generic;
    if (!use_mask_) ncodes_ = 1;
    alphabet_ready_ = true;
    return ANYSEQ_OK;
}

// Strip width for launches whose jobs advance together (Hirschberg levels: all halves of a level, `n` columns in
// total): the widest strips that still give every scheduler a warp -- measured on the 1 Mbp traceback, K = 32 against
// K = 16 per level: 140 vs 170 ms, 68 vs 78, 34.5 vs 38, 17.5 vs 20.
int Engine::pick_K_levels(int n_total) const
{
    if (tune.cols_per_lane == 4 || tune.cols_per_lane == 8 || tune.cols_per_lane == 16 || tune.cols_per_lane == 32)
        return tune.cols_per_lane;
    const long long want = 4LL * sm_count;             // one warp per scheduler
    for (int K = use_mask_ ? 32 : 16; K > 4; K /= 2)
        if ((long long)n_total / (kWarp * K) >= want) return K;
    return 4;
}

int Engine::pick_K(int n, bool chained, int m, bool affine) const
{
    (void)chained;
    if (tune.cols_per_lane == 4 || tune.cols_per_lane == 8 || tune.cols_per_lane == 16 ||
        tune.cols_per_lane == 32)
        return tune.cols_per_lane;
    // The widest strips that still give every scheduler about two warps (which then sit on adjacent strips): wider
    // strips have less per-step overhead and a shorter chain, but at most one warp works on a strip at a time.
    // B200, semiglobal Gotoh, GCUPS: 575 k columns: 3188 at K = 16 (1124 strips) vs 2890 at K = 32, 3008 at K = 8;
    // 1.15 M: 3513 at K = 32 (1124 strips) vs 3375 at K = 16; 1 M x 1 M: 3157 at K = 16 vs 2624 at K = 8.
    const long long want = 7LL * sm_count;             // ~1040 strips on a B200
    for (int K = use_mask_ ? 32 : 16; K > 4; K /= 2)   // generic kernels keep subject bytes in registers: K <= 16
        if ((long long)n / (kWarp * K) >= want) return K;
    // Small problems -- every strip has a scheduler to itself even at K = 4 -- are bound by the critical path of the strip
    // chain, not by throughput:  time = a_K * rows + lag_K * strips_K  (the last strip's own rows plus the start-up lag of
    // every strip before it: lane skew + one 32-row border batch + the L2 hand-over).  Measured on the B200 over nine
    // shapes from 64 x 9011 to 32348 x 9011 (profiles/r02_c1_table_fit.log; the fit reproduces every entry within 5 %
    // and ranks the three widths correctly for every shape, linear and Gotoh):
    //                          linear gaps                        Gotoh
    //      K   rows/step   a_K (ns/row)  lag_K (us/strip)   a_K (ns/row)  lag_K (us/strip)
    //      4       2           55.5            9.4              67.4            9.2
    //      8       4           64             15.5              84             16.2
    //     16       2           96             11.4             131.8           13.6
    // e.g. 8087 x 9011 linear (the reference CLI's default): 1185 / 1168 / 1056 us; 8087 x 18022: 1815 / 1742 / 1272 us;
    // 32348 x 9011: 2646 / 2766 / 3389 us; 1024 x 9011 Gotoh: 769 / 750 / 451 us.
    if (tune.small_model && m > 0 && use_mask_ && !track_ && (n + kWarp * 4 - 1) / (kWarp * 4) <= 4LL * sm_count) {
        static const struct { int K; double a_ns[2], lag_ns[2]; } kFit[] = {
            {4, {55.5, 67.4}, {9400.0, 9200.0}}, {8, {64.0, 84.0}, {15500.0, 16200.0}}, {16, {96.0, 131.8}, {11400.0, 13600.0}}};
        int best = 4;
        double tbest = 0.0;
        for (const auto& f : kFit) {
            const double t = f.a_ns[affine ? 1 : 0] * m + f.lag_ns[affine ? 1 : 0] * ((n + kWarp * f.K - 1) / (kWarp * f.K));
            if (f.K == 4 || t < tbest) { best = f.K; tbest = t; }
        }
        return best;
    }
    return 4;
}

// Number of row bands of a launch.  Items are taken in index order (band, job, strip) by `resident` warps, i.e. by a
// window of `resident` consecutive strips of one band, each `lag` rows behind its left neighbour (lane skew + the
// 32-row publish and fetch batches).  When every strip of the launch has its own warp there is ONE band: a strip is
// then relaxed top to bottom by one warp, and the distance to its left neighbour -- which drifts upwards as random
// delays accumulate (measured: ~290 rows in the middle of a band for lone warps, against 105-136 at the start) --
// costs nothing.  Otherwise a band must be high enough for the whole window to overlap with slack for that drift:
// band_h = band_slack * lag * window; the price of higher bands is only the last, partially filled round of items.
int Engine::plan_bands(int max_h, long long strips_total, int resident, int K, bool chained) const
{
    if (tune.band_rows > 0) {
        const int bh = std::max(32, (tune.band_rows + 31) / 32 * 32);
        return std::max(1, (max_h + bh - 1) / bh);
    }
    if (strips_total <= resident) return 1;
    const long long lag = 32LL * rows_per_step(K, use_mask_, track_) + 96;
    // a rank of a multi-GPU wavefront: the next rank can only start when this rank's LAST strip has begun its first
    // band, i.e. about one band time after the launch -- lower bands there (slack 1 costs 1 % on one GPU: 3671 vs 3710)
    const long long slack = chained ? 1 : tune.band_slack;
    const long long target = std::max<long long>(lag * resident * slack, 4096);
    return (int)std::max<long long>(1, (max_h + target - 1) / target);
}

// More strips than warps even with three warps per scheduler: the launch runs in bands, and the warps go through the
// (band, strip) items in rounds -- the last round may be nearly empty.  1 Mbp x 1 Mbp (1953 strips of 512 columns): three
// warps per scheduler = 2 bands = 3906 items = 2.2 rounds of 1776 warps, 2585 GCUPS; two per scheduler = 3 bands = 5859
// items = 4.95 rounds of 1184, 3166 GCUPS (profiles/r02_perf_1m_warps_per_scheduler.log).  So: the fill of the rounds times
// the full-width rate of the two shapes (3883 vs 3736 GCUPS on the 4.6 Mbp pair, which keeps three: 22.8 rounds).
int Engine::balance_warps(int nb, int max_h, long long strips_total, int K, bool chained) const
{
    if (nb < 3 || tune.blocks_per_sm > 0 || strips_total <= (long long)nb * kWarpsPerBlock * sm_count) return nb;
    auto rate = [&](int w) {
        const long long resident = (long long)w * kWarpsPerBlock * sm_count;
        const long long items = (long long)plan_bands(max_h, strips_total, (int)resident, K, chained) * strips_total;
        const long long rounds = (items + resident - 1) / resident;
        return (double)items / (double)(rounds * resident) * (w == 3 ? 1.04 : 1.0);
    };
    return rate(2) > rate(3) ? 2 : 3;
}

// The launch run_jobs() would make for ONE lenq x lens score-only problem (column-mask kernels, default tuning unless
// this engine's `tune` says otherwise) on a GPU with `sms` SMs -- host logic only, no CUDA call: what the CPU tests and
// tools/plan.py look at.  The occupancy query of the real path (fit_blocks_per_sm) is taken as granted; the shipped
// kernels fit 12 warps per SM.
int Engine::plan_launch(int sms, int mode, bool affine, int m, int n, bool chained, const ScoreParams& sp,
                        anyseq_launch_plan* out)
{
    if (sms < 1 || m < 1 || n < 1 || mode < 0 || mode > 2 || !out) { set_last_error("bad plan request"); return ANYSEQ_ERR_BAD_ARG; }
    sm_count = sms;
    use_mask_ = true;
    track_ = false;
    const bool local = mode == ANYSEQ_LOCAL;
    const int K = pick_K(n, chained, chained ? 0 : m, affine);
    const long long strips = ((long long)n + kWarp * K - 1) / (kWarp * K);
    const int form = pick_form(tune, affine, true, K, strips, sms, local);
    int nb = tune.blocks_per_sm > 0 ? tune.blocks_per_sm : default_blocks_per_sm(K, true, false, 3, strips, sms);
    nb = std::max(1, std::min(nb, kMaxStripWarps / kWarpsPerBlock));
    nb = balance_warps(nb, m, strips, K, chained);
    const int resident = nb * kWarpsPerBlock * sms;
    const int nbands = plan_bands(m, strips, resident, K, chained);
    const int bh = (m + nbands - 1) / nbands;
    int grid, wpb;
    long long first;
    launch_shape(false, nb, sms, (long long)nbands * strips, &grid, &wpb, &first);
    out->cols_per_lane = K;
    out->rows_per_step = rows_per_step(K, true, false);
    out->cell_form = form;
    out->strips = (int)std::min<long long>(strips, 0x7fffffff);
    out->warps_per_scheduler = nb;
    out->bands = nbands;
    out->band_rows = std::max(32, (bh + 31) / 32 * 32);
    out->grid = grid;
    out->warps_per_cta = wpb;
    out->first_items = first;
    out->packed_cells = (!chained && use_packed(tune, sp, local, affine, true, false, K)) ? 1 : 0;
    return ANYSEQ_OK;
}

// Launch init + strip kernels for a job list that is already in host memory.
int Engine::run_jobs(std::vector<Job>& jobs, const ScoreParams& sp, bool local, bool affine, int K,
                     int* launches, bool packed_ok)
{
    const int njobs = (int)jobs.size();
    long long strips_total = 0;
    int max_h = 1;
    for (Job& j : jobs) {
        j.item_begin = strips_total;           // launch-wide index of the job's first strip
        strips_total += j.nstrips;
        max_h = std::max(max_h, j.h);
    }
    if (strips_total > 0x7fffffff) { set_last_error("too many strips in one launch"); return ANYSEQ_ERR_UNSUPPORTED; }

    const bool track = track_ && local;
    bool chained = false;
    for (const Job& j : jobs) chained = chained || j.in != nullptr || j.out != nullptr;
    const bool packed = packed_ok && !chained && use_packed(tune, sp, local, affine, use_mask_, track, K);
    const int form = packed ? 3 : pick_form(tune, affine, use_mask_, K, strips_total, sm_count, local);
    KernelFn fn = pick_kernel(local, affine, K, use_mask_, track_ && local, form);
    if (!fn) { set_last_error("unsupported columns-per-lane"); return ANYSEQ_ERR_BAD_ARG; }
    int want = tune.blocks_per_sm > 0 ? tune.blocks_per_sm : default_blocks_per_sm(K, use_mask_, track, track ? 6 : 3, strips_total, sm_count);
    if (!track) want = balance_warps(std::min(want, kMaxStripWarps / kWarpsPerBlock), max_h, strips_total, K, chained);
    const int nb = fit_blocks_per_sm(fn, track, use_mask_, ncodes_, K, want, form);
    if (nb < 1) { set_last_error("strip kernel does not fit on an SM"); return ANYSEQ_ERR_UNSUPPORTED; }
    const int resident = nb * kWarpsPerBlock * sm_count;

    // bands: the same number for every job of the launch (items are ordered band, job, strip)
    const int nbands = plan_bands(max_h, strips_total, resident, K, chained);
    for (Job& j : jobs) {
        const int bh = (j.h + nbands - 1) / nbands;
        j.band_h = std::max(32, (bh + 31) / 32 * 32);
        j.nbands = nbands;
    }
    const long long total = (long long)nbands * strips_total;

    // jobs + the strip -> job table in one upload
    const size_t jobs_bytes = (sizeof(Job) * (size_t)njobs + 255) / 256 * 256;
    if (jobs_.ensure(jobs_bytes + sizeof(int) * (size_t)strips_total)) return ANYSEQ_ERR_NO_DEVICE;
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(jobs_.ptr, jobs.data(), sizeof(Job) * (size_t)njobs,
                                      cudaMemcpyHostToDevice, stream_));
    int* d_strip2job = reinterpret_cast<int*>(jobs_.as<uint8_t>() + jobs_bytes);
    if (njobs > 1) {
        strip2job_.resize((size_t)strips_total);
        for (int j = 0; j < njobs; ++j)
            std::fill(strip2job_.begin() + jobs[(size_t)j].item_begin, strip2job_.begin() + jobs[(size_t)j].item_begin + jobs[(size_t)j].nstrips, j);
        ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(d_strip2job, strip2job_.data(), sizeof(int) * (size_t)strips_total,
                                          cudaMemcpyHostToDevice, stream_));
    }
    ANYSEQ_CUDA_CHECK(cudaMemsetAsync(misc_.ptr, 0, sizeof(int) * 4, stream_));
#ifdef ANYSEQ_PROFILE
    ANYSEQ_CUDA_CHECK(cudaMemsetAsync(misc_.as<int>() + 20, 0, sizeof(int) * 16, stream_));
    if (!g_trace) {
        ANYSEQ_CUDA_CHECK(cudaMalloc(&g_trace, sizeof(unsigned long long) * 4 * kTraceStrips));
        ANYSEQ_CUDA_CHECK(cudaEventCreate(&g_ev_k0));
        ANYSEQ_CUDA_CHECK(cudaEventCreate(&g_ev_k1));
    }
    ANYSEQ_CUDA_CHECK(cudaMemsetAsync(g_trace, 0, sizeof(unsigned long long) * 4 * kTraceStrips, stream_));
    g_trace_strips = (int)std::min<long long>(strips_total, kTraceStrips);
#endif

    // launch shape: ONE CTA per SM for the ordinary kernels (nb CTAs of 4 warps for the tracking kernels); with few
    // items, just enough warps per CTA that every item of the first round has one, spread evenly over all SMs
    int wpb_used, grid;
    long long first_items;
    launch_shape(track, nb, sm_count, total, &grid, &wpb_used, &first_items);

    {
        int maxlen = 1;
        for (const Job& j : jobs) maxlen = std::max(maxlen, std::max(j.h, j.nstrips * kWarp * K));
        dim3 g((unsigned)std::min(1024, (maxlen + 255) / 256), (unsigned)std::min(njobs, 32768));
        init_jobs_kernel<<<g, 256, 0, stream_>>>(jobs_.as<Job>(), njobs, sp, kWarp * K, init_col0_);
        ANYSEQ_CUDA_CHECK(cudaGetLastError());
    }
    KernelArgs ka;
    ka.jobs = jobs_.as<Job>();
    ka.njobs = njobs;
    ka.total_items = total;
    ka.sp = sp;
    ka.one = 1;
    ka.ncodes = ncodes_;
    ka.lut_q = lut_.as<uint8_t>();
    ka.lut_s = lut_.as<uint8_t>() + 256;
    ka.status = misc_.as<int>() + kMiscStatus;
    ka.next_item = reinterpret_cast<unsigned long long*>(misc_.as<int>() + kMiscCounter);
    {
        const unsigned long long first = (unsigned long long)first_items;
        ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(ka.next_item, &first, sizeof(first), cudaMemcpyHostToDevice, stream_));
    }
    ka.timeout_ns = (unsigned long long)tune.watchdog_ms * 1000000ull;
    ka.strips_total = (int)strips_total;
    ka.strip2job = d_strip2job;
    ka.first_items = first_items;
    void* args[] = {&ka};
#ifdef ANYSEQ_PROFILE
    ka.trace = g_trace;
    ANYSEQ_CUDA_CHECK(cudaEventRecord(g_ev_k0, stream_));
#endif
    ANYSEQ_CUDA_CHECK(cudaLaunchCooperativeKernel((const void*)fn, dim3(grid), dim3(wpb_used * kWarp), args,
                                                  mask_smem_bytes(use_mask_, track, ncodes_, K, wpb_used, form), stream_));
#ifdef ANYSEQ_PROFILE
    ANYSEQ_CUDA_CHECK(cudaEventRecord(g_ev_k1, stream_));
    std::fprintf(stderr, "[anyseq profile] launch: grid=%d warps/CTA=%d items=%lld bands=%d form=%d\n", grid, wpb_used, total, nbands, form);
#endif
    if (launches) *launches += 2;
    return ANYSEQ_OK;
}

// Cells are 32-bit with minus infinity kNegInf = -2^30.  lo and hi bound every H of an m x n problem: hi is the score
// of a path with min(m, n) diagonal steps of the best symbol score, lo the larger of an all-gap path and a diagonal-then-
// gap path (global), of the diagonal from the border and a single gap from the border (semiglobal), or 0 (local).  E
// and F stay within [lo + go, hi].  The 4 P margin covers the few additions a cell makes (+ sigma, + go, + ge, the
// decoupled X = H + go), so kNegInf + ge stays below every real candidate and no sum wraps.  Padded cells only feed
// padded cells, so the real lengths decide.  The Hirschberg joins add two halves of one alignment through the split
// (plus -gi for an E join), which the whole problem's bound covers.
int check_score_range(const anyseq_scoring& sc, long long m, long long n)
{
    const long long same = sc.same, diff = sc.diff, gi = sc.gap_init, ge = sc.gap_extend;
    const long long P = std::max({std::llabs(same), std::llabs(diff), std::llabs(gi), std::llabs(ge)});
    bool ok = P <= (1LL << 24);
    if (ok) {                         // P <= 2^24 and lengths < 2^31: every product below fits 64 bits
        const long long k = std::min(m, n), sigma = std::min({0LL, same, diff});
        const long long hi = std::max({same, diff, 0LL}) * k;
        long long lo = 0;
        if (sc.mode == ANYSEQ_GLOBAL) lo = std::max(2 * gi + (m + n) * ge, sigma * k + gi + (std::max(m, n) - 1) * ge);
        else if (sc.mode == ANYSEQ_SEMIGLOBAL) lo = std::max(sigma * k, gi + k * ge);
        ok = hi <= 0x7fffffffLL - 4 * P && lo >= (long long)kNegInf + 4 * P;
    }
    if (ok) return ANYSEQ_OK;
    char buf[256];
    std::snprintf(buf, sizeof(buf), "scores of a %lld x %lld problem under (%d, %d, %d, %d) leave the 32-bit cell range: "
                  "|same|, |diff|, |gap_init|, |gap_extend| <= 2^24 and every score within [-2^30 + 4 P, 2^31 - 1 - 4 P] "
                  "(P = the largest of them)", m, n, sc.same, sc.diff, sc.gap_init, sc.gap_extend);
    set_last_error(buf);
    return ANYSEQ_ERR_UNSUPPORTED;
}

int make_score_params(const anyseq_scoring& sc, ScoreParams* sp, bool* affine)
{
    if (sc.mode < 0 || sc.mode > 2 || sc.gap_init > 0 || sc.gap_extend > 0) {
        set_last_error("bad scoring scheme (mode in 0..2, gap costs must be <= 0)");
        return ANYSEQ_ERR_BAD_ARG;
    }
    // an empty problem: only the magnitude limit of the cell range applies (gap_init + gap_extend must not wrap)
    const int rc = check_score_range(sc, 0, 0);
    if (rc) return rc;
    *affine = sc.gap_init != 0;
    sp->same = sc.same;
    sp->diff = sc.diff;
    sp->gap_extend = sc.gap_extend;
    sp->gap_open = sc.gap_init + sc.gap_extend;   // linear: == gap
    return ANYSEQ_OK;
}

// Degenerate inputs, following the reference's storage (SURVEY quirk Q12):
// global -> the init value left in the column vector; semiglobal -> 0;
// local -> SCORE_MIN (no block ever ran).
static void empty_result(const anyseq_scoring& sc, int m, int n, anyseq_result* out)
{
    const int L = std::max(m, n);
    int64_t v;
    if (sc.mode == ANYSEQ_GLOBAL) v = L > 0 ? (int64_t)sc.gap_init + (int64_t)L * sc.gap_extend : 0;
    else if (sc.mode == ANYSEQ_SEMIGLOBAL) v = 0;
    else v = kScoreMin;
    out->score = v;
    out->end_i = m - 1;
    out->end_j = n - 1;
    out->kernel_ms = 0.f;
    out->kernel_launches = 0;
}

int Engine::score_device(const anyseq_scoring& sc, const uint8_t* d_q, int m, const uint8_t* d_s, int n,
                         anyseq_result* out)
{
    anyseq_strip_partial part;
    if (m < 0 || n < 0 || !out) { set_last_error("bad lengths"); return ANYSEQ_ERR_BAD_ARG; }
    if (m == 0 || n == 0) { empty_result(sc, m, n, out); return ANYSEQ_OK; }
    // held across the result read: h_misc_ is shared by every call on this context
    std::lock_guard<std::recursive_mutex> lock(mu_);
    int rc = score_strip_device(sc, d_q, m, d_s, 0, n, n, nullptr, nullptr, &part);
    if (rc) return rc;
    out->score = h_misc_[kMiscOut + 0];
    out->end_i = h_misc_[kMiscOut + 1];
    out->end_j = h_misc_[kMiscOut + 2];
    out->kernel_ms = part.kernel_ms;
    out->kernel_launches = part.kernel_launches;
    return ANYSEQ_OK;
}

int Engine::score_strip_device(const anyseq_scoring& sc, const uint8_t* d_q, int m,
                               const uint8_t* d_s_slice, int col_begin, int col_end, int n_total,
                               Inbox* inbox, Inbox* next_inbox, anyseq_strip_partial* out)
{
    std::lock_guard<std::recursive_mutex> lock(mu_);
    ANYSEQ_CUDA_CHECK(cudaSetDevice(device));
    ScoreParams sp;
    bool affine;
    int rc = make_score_params(sc, &sp, &affine);
    if (rc) return rc;
    affine = affine || tune.force_affine;
    const int w = col_end - col_begin;
    if (m < 1 || w < 1 || col_begin < 0 || col_end > n_total) { set_last_error("bad strip range"); return ANYSEQ_ERR_BAD_ARG; }
    // the whole problem, not the slice: a rank's narrow slice of an out-of-range problem is out of range too
    if ((rc = check_score_range(sc, m, n_total))) return rc;
    // the strips read / write one border record per query row of the inboxes (the next rank's lives in PEER memory)
    if ((inbox && m > inbox->rows) || (next_inbox && m > next_inbox->rows)) {
        set_last_error("query longer than the rows the inbox was created with");
        return ANYSEQ_ERR_BAD_ARG;
    }
    const bool local = sc.mode == ANYSEQ_LOCAL;
    // the end cell of a local alignment needs the whole matrix in one job (reference block grid)
    const bool track = local && (tune.local_end_cell || force_track_) && !inbox && !next_inbox && col_begin == 0 && col_end == n_total;
    struct TrackScope { bool& t; ~TrackScope() { t = false; } } track_scope{track_};
    track_ = track;
    ANYSEQ_CUDA_CHECK(cudaEventRecord(ev0_, stream_));
    rc = analyse_alphabet(d_q, m, d_s_slice, w);
    if (rc) return rc;
    // edge columns are wanted per 128-column block; whole single-GPU problems may use the small-problem fit (pick_K)
    const bool whole = !inbox && !next_inbox && col_begin == 0 && col_end == n_total;
    const int K = want_edges_ ? 4 : pick_K(w, !whole, whole ? m : 0, affine);
    const int SW = kWarp * K;
    const int nstrips = (w + SW - 1) / SW;

    const size_t wpad = (size_t)nstrips * SW;
    if (col_.ensure(sizeof(int4) * (size_t)m) || rowH_.ensure(sizeof(int) * wpad) ||
        corner_.ensure(sizeof(int) * (size_t)nstrips) || progress_.ensure(sizeof(int) * (size_t)nstrips))
        return ANYSEQ_ERR_NO_DEVICE;
    if (affine && rowF_.ensure(sizeof(int) * wpad)) return ANYSEQ_ERR_NO_DEVICE;

    Job J;
    std::memset(&J, 0, sizeof(J));
    J.q = d_q;
    J.s = d_s_slice;
    J.h = m;
    J.w = w;
    J.nstrips = nstrips;              // bands are planned by run_jobs
    J.col = col_.as<int4>();
    J.rowH = rowH_.as<int>();
    J.rowF = affine ? rowF_.as<int>() : nullptr;
    J.corner = corner_.as<int>();
    J.progress = progress_.as<int>();
    J.best = misc_.as<int>() + kMiscBest;
    J.init_global = sc.mode == ANYSEQ_GLOBAL;
    J.top_open = sp.gap_open;
    const int nbi = (m + 1023) / 1024, nbj = (w + 1023) / 1024;
    if (track) {
        const size_t bytes = sizeof(unsigned long long) * (size_t)nbi * nbj;
        if (blockmax_.ensure(bytes)) return ANYSEQ_ERR_NO_DEVICE;
        ANYSEQ_CUDA_CHECK(cudaMemsetAsync(blockmax_.ptr, 0, bytes, stream_));
        J.blockmax = blockmax_.as<unsigned long long>();
        J.nbj = nbj;
    }
    if (want_edges_) {
        if (edges_.ensure(sizeof(int2) * (size_t)nstrips * (size_t)m)) return ANYSEQ_ERR_NO_DEVICE;
        J.edges = edges_.as<int2>();
    }
    // the tag of a run is agreed without communication: both ends count their uses of the inbox
    if (inbox) { J.in = inbox->records; J.in_tag = 0x40000000 + (++inbox->uses_in & 0xffffff); }
    if (next_inbox) { J.out = next_inbox->records; J.out_tag = 0x40000000 + (++next_inbox->uses_out & 0xffffff); }

    std::vector<Job> jobs(1, J);
    int launches = 0;
    init_col0_ = col_begin;
    launches += 3;   // alphabet analysis
    // packed cells for whole single-GPU score problems (not for the edge columns of a full-matrix traceback)
    rc = run_jobs(jobs, sp, local, affine, K, &launches, whole && !want_edges_);
    init_col0_ = 0;
    if (rc) return rc;
    finish_score_kernel<<<1, 1024, 0, stream_>>>(jobs_.as<Job>(), sc.mode, col_begin, n_total,
                                                  misc_.as<int>() + kMiscOut);
    ANYSEQ_CUDA_CHECK(cudaGetLastError());
    launches += 1;
    if (track) {
        local_end_cell_kernel<<<1, 1024, 0, stream_>>>(blockmax_.as<unsigned long long>(), nbi, nbj,
                                                        misc_.as<int>() + kMiscOut);
        ANYSEQ_CUDA_CHECK(cudaGetLastError());
        launches += 1;
    }
    ANYSEQ_CUDA_CHECK(cudaEventRecord(ev1_, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(h_misc_, misc_.ptr, sizeof(int) * kMiscWords, cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(stream_));
    if (h_misc_[kMiscStatus] != kStatusOk) {
        char buf[160];
        std::snprintf(buf, sizeof(buf), "strip kernel watchdog fired (status %d, need %d, saw %d)",
                      h_misc_[kMiscStatus], h_misc_[kMiscStatus + 1], h_misc_[kMiscStatus + 2]);
        set_last_error(buf);
        return ANYSEQ_ERR_KERNEL_TIMEOUT;
    }
    float ms = 0.f;
    ANYSEQ_CUDA_CHECK(cudaEventElapsedTime(&ms, ev0_, ev1_));
#ifdef ANYSEQ_PROFILE
    {
        const unsigned long long* pc = reinterpret_cast<const unsigned long long*>(h_misc_ + 20);
        const double nb = (double)pc[3] > 0 ? (double)pc[3] : 1.0;
        std::fprintf(stderr, "[anyseq profile] K=%d batches=%llu cycles/batch: wait=%.0f io=%.0f steps=%.0f | items=%llu "
                             "cycles/item: bandwait=%.0f total=%.0f\n", K, pc[3], pc[0] / nb, pc[1] / nb, pc[2] / nb, pc[6],
                     pc[6] ? (double)pc[4] / pc[6] : 0.0, pc[6] ? (double)pc[5] / pc[6] : 0.0);
        float pre = 0.f, ker = 0.f, post = 0.f;
        cudaEventElapsedTime(&pre, ev0_, g_ev_k0);
        cudaEventElapsedTime(&ker, g_ev_k0, g_ev_k1);
        cudaEventElapsedTime(&post, g_ev_k1, ev1_);
        std::fprintf(stderr, "[anyseq profile] phases (us): before the strip kernel %.1f, strip kernel %.1f, after %.1f\n",
                     pre * 1e3, ker * 1e3, post * 1e3);
        if (const char* tf = std::getenv("ANYSEQ_TRACE_FILE")) {
            std::vector<unsigned long long> tr((size_t)4 * g_trace_strips);
            cudaMemcpy(tr.data(), g_trace, sizeof(unsigned long long) * tr.size(), cudaMemcpyDeviceToHost);
            unsigned long long t0 = ~0ull;
            for (int i = 0; i < g_trace_strips; ++i) if (tr[4 * i]) t0 = std::min(t0, tr[4 * i]);
            if (FILE* f = std::fopen(tf, "a")) {
                std::fprintf(f, "{\"m\": %d, \"w\": %d, \"K\": %d, \"kernel_us\": %.1f, \"strips\": [", m, w, K, ker * 1e3);
                for (int i = 0; i < g_trace_strips; ++i)
                    std::fprintf(f, "%s[%lld, %lld, %lld, %llu]", i ? ", " : "", (long long)(tr[4 * i] - t0), (long long)(tr[4 * i + 1] - t0),
                                 (long long)(tr[4 * i + 2] - t0), tr[4 * i + 3]);
                std::fprintf(f, "]}\n");
                std::fclose(f);
            }
        }
    }
#endif
    if (out) {
        out->row_best = h_misc_[kMiscOut + 3];
        out->row_best_j = h_misc_[kMiscOut + 4];
        out->col_best = h_misc_[kMiscOut + 5];
        out->col_best_i = h_misc_[kMiscOut + 6];
        out->corner = h_misc_[kMiscOut + 7];
        out->local_best = h_misc_[kMiscBest];
        out->kernel_ms = ms;
        out->kernel_launches = launches;
        out->lenq = m;
        out->lens_total = n_total;
    }
    return ANYSEQ_OK;
}

// Several pairs of one shape in ONE persistent launch (items ordered band, pair, strip).  Used by the streamed
// multi-GPU wavefront: a rank's slice of two consecutive alignments gives the kernel twice the strips, so all
// warps have work (one slice alone feeds 1.9 warps per scheduler, profiles/r01_summary.md).  Every pair has its
// own border records, bottom rows, corners, progress counters, inboxes and partial result.
int Engine::score_strip_device_multi(const anyseq_scoring& sc, int npairs, const uint8_t* const* d_q, int m,
                                     const uint8_t* const* d_s_slice, int col_begin, int col_end, int n_total,
                                     Inbox* const* inbox, Inbox* const* next_inbox, anyseq_strip_partial* out)
{
    if (npairs < 1 || npairs > 8 || !d_q || !d_s_slice || !out) { set_last_error("bad pair list"); return ANYSEQ_ERR_BAD_ARG; }
    if (npairs == 1)
        return score_strip_device(sc, d_q[0], m, d_s_slice[0], col_begin, col_end, n_total, inbox ? inbox[0] : nullptr,
                                  next_inbox ? next_inbox[0] : nullptr, out);
    std::lock_guard<std::recursive_mutex> lock(mu_);
    ANYSEQ_CUDA_CHECK(cudaSetDevice(device));
    ScoreParams sp;
    bool affine;
    int rc = make_score_params(sc, &sp, &affine);
    if (rc) return rc;
    affine = affine || tune.force_affine;
    const int w = col_end - col_begin;
    if (m < 1 || w < 1 || col_begin < 0 || col_end > n_total) { set_last_error("bad strip range"); return ANYSEQ_ERR_BAD_ARG; }
    if ((rc = check_score_range(sc, m, n_total))) return rc;
    for (int p = 0; p < npairs; ++p) {
        if ((inbox && inbox[p] && m > inbox[p]->rows) || (next_inbox && next_inbox[p] && m > next_inbox[p]->rows)) {
            set_last_error("query longer than the rows the inbox was created with");
            return ANYSEQ_ERR_BAD_ARG;
        }
    }
    const bool local = sc.mode == ANYSEQ_LOCAL;
    ANYSEQ_CUDA_CHECK(cudaEventRecord(ev0_, stream_));
    // one alphabet for all pairs: presence bits accumulate over every sequence
    {
        if (lut_.ensure(512 + 64 + 16)) return ANYSEQ_ERR_NO_DEVICE;
        unsigned* bits = reinterpret_cast<unsigned*>(lut_.as<uint8_t>() + 512);
        int* d_ncodes = reinterpret_cast<int*>(bits + 16);
        ANYSEQ_CUDA_CHECK(cudaMemsetAsync(bits, 0, sizeof(unsigned) * 17, stream_));
        const int gq = (int)std::min<long long>(sm_count * 8, (m + 255) / 256);
        const int gs = (int)std::min<long long>(sm_count * 8, (w + 255) / 256);
        for (int p = 0; p < npairs; ++p) {
            alphabet_presence_kernel<<<std::max(gq, 1), 256, 0, stream_>>>(d_q[p], m, bits);
            alphabet_presence_kernel<<<std::max(gs, 1), 256, 0, stream_>>>(d_s_slice[p], w, bits + 8);
        }
        build_lut_kernel<<<1, 32, 0, stream_>>>(bits, bits + 8, lut_.as<uint8_t>(), lut_.as<uint8_t>() + 256, d_ncodes);
        ANYSEQ_CUDA_CHECK(cudaGetLastError());
        ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(h_misc_ + kMiscWords - 1, d_ncodes, sizeof(int), cudaMemcpyDeviceToHost, stream_));
        ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(stream_));
        ncodes_ = h_misc_[kMiscWords - 1];
        use_mask_ = ncodes_ <= kMaxCodes && !tune.force_generic;
        if (!use_mask_) ncodes_ = 1;
    }
    const bool chained = inbox != nullptr || next_inbox != nullptr;
    // the strips of all pairs feed the warps together: choose the strip width for the combined width
    const int K = pick_K((int)std::min<long long>((long long)w * npairs, 0x7fffffff), chained);
    const int SW = kWarp * K;
    const int nstrips = (w + SW - 1) / SW;

    // per-pair storage carved out of one buffer: col records, rowH, rowF, corner, progress, result words
    const size_t wpad = (size_t)nstrips * SW;
    auto align256 = [](size_t x) { return (x + 255) / 256 * 256; };
    const size_t b_col = align256(sizeof(int4) * (size_t)m), b_row = align256(sizeof(int) * wpad),
                 b_small = align256(sizeof(int) * (size_t)nstrips);
    const size_t per_pair = b_col + 2 * b_row + 2 * b_small;
    const size_t b_res = align256(sizeof(int) * 16 * (size_t)npairs);
    if (multi_.ensure(per_pair * (size_t)npairs + b_res)) return ANYSEQ_ERR_NO_DEVICE;
    uint8_t* base = multi_.as<uint8_t>();
    int* d_res = reinterpret_cast<int*>(base + per_pair * (size_t)npairs);       // [npairs][8] finish words, then [npairs] best
    int* d_best = d_res + 8 * npairs;
    ANYSEQ_CUDA_CHECK(cudaMemsetAsync(d_res, 0, b_res, stream_));

    std::vector<Job> jobs((size_t)npairs);
    for (int p = 0; p < npairs; ++p) {
        Job& J = jobs[(size_t)p];
        std::memset(&J, 0, sizeof(J));
        uint8_t* pb = base + per_pair * (size_t)p;
        J.q = d_q[p];
        J.s = d_s_slice[p];
        J.h = m;
        J.w = w;
        J.nstrips = nstrips;
        J.col = reinterpret_cast<int4*>(pb);
        J.rowH = reinterpret_cast<int*>(pb + b_col);
        J.rowF = affine ? reinterpret_cast<int*>(pb + b_col + b_row) : nullptr;
        J.corner = reinterpret_cast<int*>(pb + b_col + 2 * b_row);
        J.progress = reinterpret_cast<int*>(pb + b_col + 2 * b_row + b_small);
        J.best = d_best + p;
        J.init_global = sc.mode == ANYSEQ_GLOBAL;
        J.top_open = sp.gap_open;
        Inbox* in = inbox ? inbox[p] : nullptr;
        Inbox* nx = next_inbox ? next_inbox[p] : nullptr;
        if (in) { J.in = in->records; J.in_tag = 0x40000000 + (++in->uses_in & 0xffffff); }
        if (nx) { J.out = nx->records; J.out_tag = 0x40000000 + (++nx->uses_out & 0xffffff); }
    }
    int launches = 2 * npairs + 1;   // alphabet analysis
    init_col0_ = col_begin;
    rc = run_jobs(jobs, sp, local, affine, K, &launches);
    init_col0_ = 0;
    if (rc) return rc;
    finish_score_kernel<<<npairs, 1024, 0, stream_>>>(jobs_.as<Job>(), sc.mode, col_begin, n_total, d_res);
    ANYSEQ_CUDA_CHECK(cudaGetLastError());
    launches += 1;
    ANYSEQ_CUDA_CHECK(cudaEventRecord(ev1_, stream_));
    std::vector<int> h_res((size_t)9 * npairs);
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(h_res.data(), d_res, sizeof(int) * 9 * (size_t)npairs, cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(h_misc_, misc_.ptr, sizeof(int) * 4, cudaMemcpyDeviceToHost, stream_));
    ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(stream_));
    if (h_misc_[kMiscStatus] != kStatusOk) {
        char buf[160];
        std::snprintf(buf, sizeof(buf), "strip kernel watchdog fired (status %d, need %d, saw %d)",
                      h_misc_[kMiscStatus], h_misc_[kMiscStatus + 1], h_misc_[kMiscStatus + 2]);
        set_last_error(buf);
        return ANYSEQ_ERR_KERNEL_TIMEOUT;
    }
    float ms = 0.f;
    ANYSEQ_CUDA_CHECK(cudaEventElapsedTime(&ms, ev0_, ev1_));
    for (int p = 0; p < npairs; ++p) {
        const int* r = h_res.data() + 8 * p;
        out[p].row_best = r[3];
        out[p].row_best_j = r[4];
        out[p].col_best = r[5];
        out[p].col_best_i = r[6];
        out[p].corner = r[7];
        out[p].local_best = h_res[(size_t)8 * npairs + p];
        out[p].kernel_ms = ms;
        out[p].kernel_launches = p == 0 ? launches : 0;
        out[p].lenq = m;
        out[p].lens_total = n_total;
    }
    return ANYSEQ_OK;
}

int Engine::score_strip_host(const anyseq_scoring& sc, const char* q, int m, const char* s_slice, int col_begin, int col_end,
                             int n_total, Inbox* inbox, Inbox* next_inbox, anyseq_strip_partial* out)
{
    const int w = col_end - col_begin;
    if (m < 1 || w < 1 || !q || !s_slice || !out) { set_last_error("bad arguments"); return ANYSEQ_ERR_BAD_ARG; }
    std::lock_guard<std::recursive_mutex> lock(mu_);
    ANYSEQ_CUDA_CHECK(cudaSetDevice(device));
    if (seq_q_.ensure((size_t)m + 64) || seq_s_.ensure((size_t)w + 64)) return ANYSEQ_ERR_NO_DEVICE;
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(seq_q_.ptr, q, (size_t)m, cudaMemcpyHostToDevice, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(seq_s_.ptr, s_slice, (size_t)w, cudaMemcpyHostToDevice, stream_));
    return score_strip_device(sc, seq_q_.as<uint8_t>(), m, seq_s_.as<uint8_t>(), col_begin, col_end, n_total, inbox,
                              next_inbox, out);
}

int Engine::score_host(const anyseq_scoring& sc, const char* q, int m, const char* s, int n,
                       anyseq_result* out)
{
    if (m < 0 || n < 0 || !out || (m > 0 && !q) || (n > 0 && !s)) { set_last_error("bad arguments"); return ANYSEQ_ERR_BAD_ARG; }
    if (m == 0 || n == 0) { empty_result(sc, m, n, out); return ANYSEQ_OK; }
    std::lock_guard<std::recursive_mutex> lock(mu_);
    ANYSEQ_CUDA_CHECK(cudaSetDevice(device));
    if (seq_q_.ensure((size_t)m + 64) || seq_s_.ensure((size_t)n + 64)) return ANYSEQ_ERR_NO_DEVICE;
    // sequence_to_device: src/mapping_acc.impala:125-131
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(seq_q_.ptr, q, (size_t)m, cudaMemcpyHostToDevice, stream_));
    ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(seq_s_.ptr, s, (size_t)n, cudaMemcpyHostToDevice, stream_));
    if ((long long)m + n <= kHostAlphabetLimit) {
        const int rc = analyse_alphabet_host(reinterpret_cast<const uint8_t*>(q), m, reinterpret_cast<const uint8_t*>(s), n);
        if (rc) return rc;
    }
    const int rc = score_device(sc, seq_q_.as<uint8_t>(), m, seq_s_.as<uint8_t>(), n, out);
    alphabet_ready_ = false;
    return rc;
}

}  // namespace anyseq
