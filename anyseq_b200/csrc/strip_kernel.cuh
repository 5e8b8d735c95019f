// strip_kernel.cuh -- the DP relaxation hot path, hand-written for sm_100a.
//
// Replaces the reference's iteration_{cpu,acc} / scoring_{cpu,acc} /
// mapping_{cpu,acc} layer (src/iteration_acc.impala:16-172,
// src/scoring_acc.impala:1-181, src/mapping_acc.impala) -- same recurrences
// (relax_global / relax_local, src/align.impala:46-79), different machine
// mapping:
//
//   * one WARP owns a column strip of 32*K subject columns; each lane keeps K
//     columns of H (and F for Gotoh) in registers for the whole band,
//   * lane l works on row t-l at step t (anti-diagonal across lanes); the
//     right edge (H, E) moves to lane l+1 with warp shuffles,
//   * the cell update is DPX on the ALU pipe (VIADDMNMX, VIMNMX3[.RELU]) with
//     every plain add moved to the FMA pipe as IMAD -- the B200 issues both
//     pipes side by side at 64 lanes/clk/SM each (microbench.cu),
//   * symbol comparison: MASK kernels keep, per lane, one 32-bit column mask
//     per alphabet code in shared memory; the row's query code selects a mask
//     (one LDS, prefetched a row ahead) and the per-cell predicate is a bit
//     test that ptxas folds into R2P (7 predicates per instruction); generic
//     kernels (alphabets with > 32 shared symbols) compare byte registers,
//   * strips are chained through HBM/L2: lane 31's edge is staged in shared
//     memory and published 32 rows at a time (coalesced, .cg) with a
//     release/acquire row counter per strip -- no kernel relaunch, no grid
//     barrier (the reference relaunches per block anti-diagonal),
//   * a persistent grid claims (band, strip) items in dependency order, so all
//     waits are on lower-numbered items: deadlock-free when co-resident.
//
// Score domain: signed 32-bit, identical to the reference (Score = i32,
// src/dynprog.impala:10).  For Gotoh the registers hold X = H + gap_open so
// that E and F need one VIADDMNMX each:  E' = max(E + ge, X_left).
#pragma once

#include <type_traits>

#include "common.cuh"

namespace anyseq {

// Cell formulations:
//   "coupled":   E' = max(E+ge, X_left); H = max3(diag, E', F); X = H+go  -- 3 ALU + 3 FMA ops per Gotoh cell, but the
//                loop-carried chain along a row is VIADDMNMX -> VIMNMX3 -> IMAD (about 14 cycles per cell), so a warp
//                needs several independent rows or several co-resident warps to fill the issue slots.
//   "decoupled": M = max(F+go, diag) (no horizontal input), E' = max(E+ge, M_left), X = max(E'+go, M)  -- 4 ALU + 2 FMA,
//                the loop-carried chain is ONE VIADDMNMX (4 cycles): valid because the E term inside H(i,j-1) can never
//                win the maximum that forms E(i,j) (E+go <= E+ge).  A lone warp saturates its scheduler's ALU pipe, so
//                half as many (twice as fast) warps are needed -- which is what the strip-to-strip chain, narrow
//                problems and multi-GPU slices are sensitive to.
// The strip kernels build them as template parameter FORM (engine.cu: pick_form, use_packed):
//   1  decoupled cells: the default (linear and Gotoh gaps, every strip width).
//   2  "mixed": even rows coupled, odd rows decoupled -- wide local Gotoh launches (two-row MASK tiles).
//   3  "packed": the decoupled cell on 16-bit halves, two cells per DPX instruction (strip_packed.cuh) -- global and
//      semiglobal Gotoh with column masks, when the scheme's score window fits 16 bits.
// The end-cell tracking kernels (TRACK) run coupled cells: they need H itself to find where the maximum is reached.

constexpr int kWarpsPerBlock = 4;                       // batch kernels, end-cell tracking strip kernels
constexpr int kThreads = kWarpsPerBlock * kWarp;
// The strip kernels run ONE CTA per SM with 4, 8 or 12 warps (1 - 3 per scheduler; warp w issues on scheduler w % 4):
// the warps that share a scheduler take ADJACENT strips.  When the right one of them has to wait for its left
// neighbour, the neighbour is the warp that inherits its issue slots, so a pair (or triple) of strips behaves like one
// wide strip with two (three) instruction streams instead of two unrelated streams that disturb each other's pace.
constexpr int kMaxStripWarps = 12;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kMaxCodes = 32;      // MASK kernels: alphabet codes incl. code 0 = "matches nothing"

struct KernelArgs {
    const Job* jobs;
    int njobs;
    long long total_items;
    ScoreParams sp;
    int one;                        // == 1, opaque to the compiler (see imad_add)
    int ncodes;                     // MASK kernels: number of alphabet codes (<= kMaxCodes)
    const uint8_t* lut_q;           // MASK kernels: byte -> code for query / subject symbols
    const uint8_t* lut_s;
    int* status;                    // [0] StatusCode, [1..3] diagnostics
    unsigned long long* next_item;  // work counter, initialised to the number of resident warps
    unsigned long long timeout_ns;  // watchdog for dependency waits
    // Work items are ordered (band, job, strip): all jobs of a launch have the same NUMBER of bands (a short job's last
    // bands may be empty) and advance together; strip2job maps a launch-wide strip index to its job, whose
    // Job::item_begin is the launch-wide index of its first strip.
    int strips_total;
    const int* strip2job;
    long long first_items;          // items of the static first round (<= gridDim.x * warps per CTA), spread evenly over the CTAs
#ifdef ANYSEQ_PROFILE
    unsigned long long* trace;      // measurement builds: [kTraceStrips][4] = item start, first border batch seen, end of the steps (ns), SM
#endif
};
#ifdef ANYSEQ_PROFILE
constexpr int kTraceStrips = 4096;
#endif

__device__ __forceinline__ int ld_acquire_gpu(const int* p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int ld_acquire_sys(const int* p)
{
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_gpu(int* p, int v)
{
    asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(int* p, int v)
{
    asm volatile("st.relaxed.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// a + b on the FMA pipe: IMAD with a multiplier the compiler cannot fold (one == 1
// at run time).  Every add moved here is an ALU slot freed for VIADDMNMX / VIMNMX3.
__device__ __forceinline__ int imad_add(int a, int one, int b)
{
    int r;
    asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(one), "r"(b));
    return r;
}
// d + (q == s ? same : diff): one compare (ALU) and two IMADs, the second one
// predicated -- no SEL.
__device__ __forceinline__ int diag_plus_sigma(int qc, int sc, int d, int one, int diff, int same)
{
    int dd;
    asm("{\n\t.reg .pred p;\n\tsetp.eq.s32 p, %1, %2;\n\tmad.lo.s32 %0, %3, %4, %5;\n\t@p mad.lo.s32 %0, %3, %4, %6;\n\t}"
        : "=&r"(dd)
        : "r"(qc), "r"(sc), "r"(d), "r"(one), "r"(diff), "r"(same));
    return dd;
}
// same with the match predicate taken from bit C of the row's column mask
template <int C>
__device__ __forceinline__ int diag_plus_sigma_mask(unsigned mask, int d, int one, int diff, int same)
{
    int dd;
    asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %1, %2;\n\tsetp.ne.u32 p, t, 0;\n\tmad.lo.s32 %0, %3, %4, %5;\n\t@p mad.lo.s32 %0, %3, %4, %6;\n\t}"
        : "=&r"(dd)
        : "r"(mask), "n"(1u << C), "r"(d), "r"(one), "r"(diff), "r"(same));
    return dd;
}

// dst = src if bit C of `mask` is set -- as a predicated IMAD (FMA pipe) whose predicate ptxas takes from R2P, like the
// match bits above.  Ragged strips use it to keep the edge column's values: 1/7 ALU instruction per cell instead of
// ISETP + SEL per cell.
template <int C>
__device__ __forceinline__ void capture_if_bit(unsigned mask, int& dst, int src, int one)
{
    asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %1, %2;\n\tsetp.ne.u32 p, t, 0;\n\t@p mad.lo.s32 %0, %3, %4, 0;\n\t}"
        : "+r"(dst)
        : "r"(mask), "n"(1u << C), "r"(src), "r"(one));
}

__device__ __forceinline__ int ld_relaxed_gpu(const int* p)
{
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int ld_relaxed_sys(const int* p)
{
    int v;
    asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

struct StepConst;
// bit (BASE + r) of a tile mask, r in 0..3 known after unrolling
template <int BASE, int W>
__device__ __forceinline__ int diag_mask_bit(const unsigned (&tm)[W], int r, int d, const StepConst& k);

// Wait until *flag >= need.  Executed by all lanes of a warp (same address:
// one transaction).  Fast path: one acquire load.  Slow path: relaxed polls (an
// acquire load costs a CCTL.IVALL -- a whole-L1 invalidate -- per poll), then one
// acquire load to order the following border loads.  Returns false if the
// watchdog fired or another warp already reported a failure -- the caller then
// leaves the kernel, so a logic error shows up as a status code instead of a
// hung GPU.
__device__ __forceinline__ bool wait_rows(const int* flag, int need, bool sys, int* status,
                                          unsigned long long timeout_ns)
{
    // common case: already published -- a single acquire load
    int v = sys ? ld_acquire_sys(flag) : ld_acquire_gpu(flag);
    if (v >= need) return true;
    bool ok = true;
    const unsigned long long t0 = global_timer_ns();
    unsigned spins = 0;
    while (true) {
        v = sys ? ld_relaxed_sys(flag) : ld_relaxed_gpu(flag);
        if (v >= need) break;
        ++spins;
#ifndef ANYSEQ_SPIN_NOSLEEP
        if (spins > 8u) __nanosleep(spins > 64u ? 400 : 40);
#endif
        if ((spins & 127u) == 0u) {
            if (*(volatile int*)status != kStatusOk) { ok = false; break; }
            if (global_timer_ns() - t0 > timeout_ns) {
                if (atomicCAS(status, kStatusOk, kStatusTimeout) == kStatusOk) {
                    status[1] = need; status[2] = v;
                }
                ok = false;
                break;
            }
        }
    }
    // the poll was relaxed: order the border loads after it
    v = sys ? ld_acquire_sys(flag) : ld_acquire_gpu(flag);
    return __all_sync(kFull, ok && v >= need);
}

template <int K>
__device__ __forceinline__ void load_row_ints(const int* __restrict__ p, int (&dst)[K])
{
#pragma unroll
    for (int c = 0; c < K; c += 4) {
        const int4 v = __ldcg(reinterpret_cast<const int4*>(p + c));
        dst[c] = v.x; dst[c + 1] = v.y; dst[c + 2] = v.z; dst[c + 3] = v.w;
    }
}

// Tile mask (MASK kernels): bit (c*R + r) of the W-word mask says "subject column c
// equals the query symbol of row r of the lane's current R-row group"; it is the
// sum over r of (spread column mask of row r's code) << r.  Consecutive cells of
// the 2-D wavefront read consecutive bits, which ptxas turns into R2P (seven
// predicates per instruction) instead of one LOP3 per cell.
template <int R, int K>
struct TileWords {
    static constexpr int value = (R * K + 31) / 32;
};

// state of one lane during one single-row chain
template <int W>
struct StepState {
    int dd;          // H(i-1, j-1) + sigma of the cell about to be relaxed
    int e;           // E of the cell to the left
    int xleft;       // X (= H [+ open]) of the cell to the left
    int best;        // LOCAL: running maximum
    int hprev;       // LOCAL: H of the previous (even) column, folded pairwise with VIMNMX3
    int es;          // PARTIAL: E of the edge column
    int xs;          // PARTIAL: X of the edge column
    int bpos;        // TRACK: row * K + column (within the item, within the lane) of the first cell attaining best
    int rowpos;      // TRACK: row * K of the row being relaxed
    unsigned tm[W];  // MASK: tile mask of the lane's current row group
    int qc;          // !MASK: the row's query byte
};

struct StepConst {
    int one, ge, go, diff_o, same_o;
    int nvalid, outc;   // PARTIAL only
    unsigned capmask;   // PARTIAL only: bit outc
    int diff_c, same_c; // FORM 2: sigma - go for the coupled rows of a mixed tile
};

template <int BASE, int W>
__device__ __forceinline__ int diag_mask_bit_c(const unsigned (&tm)[W], int r, int d, int one, int diff_o, int same_o)
{
    switch (r) {
        case 0: return diag_plus_sigma_mask<(BASE + 0) % 32>(tm[(BASE + 0) / 32 < W ? (BASE + 0) / 32 : 0], d, one, diff_o, same_o);
        case 1: return diag_plus_sigma_mask<(BASE + 1) % 32>(tm[(BASE + 1) / 32 < W ? (BASE + 1) / 32 : 0], d, one, diff_o, same_o);
        case 2: return diag_plus_sigma_mask<(BASE + 2) % 32>(tm[(BASE + 2) / 32 < W ? (BASE + 2) / 32 : 0], d, one, diff_o, same_o);
        default: return diag_plus_sigma_mask<(BASE + 3) % 32>(tm[(BASE + 3) / 32 < W ? (BASE + 3) / 32 : 0], d, one, diff_o, same_o);
    }
}

template <int BASE, int W>
__device__ __forceinline__ int diag_mask_bit(const unsigned (&tm)[W], int r, int d, const StepConst& k)
{
    // r is a compile-time constant after unrolling; the switch folds away
    switch (r) {
        case 0: return diag_plus_sigma_mask<(BASE + 0) % 32>(tm[(BASE + 0) / 32 < W ? (BASE + 0) / 32 : 0], d, k.one, k.diff_o, k.same_o);
        case 1: return diag_plus_sigma_mask<(BASE + 1) % 32>(tm[(BASE + 1) / 32 < W ? (BASE + 1) / 32 : 0], d, k.one, k.diff_o, k.same_o);
        case 2: return diag_plus_sigma_mask<(BASE + 2) % 32>(tm[(BASE + 2) / 32 < W ? (BASE + 2) / 32 : 0], d, k.one, k.diff_o, k.same_o);
        default: return diag_plus_sigma_mask<(BASE + 3) % 32>(tm[(BASE + 3) / 32 < W ? (BASE + 3) / 32 : 0], d, k.one, k.diff_o, k.same_o);
    }
}

// Cell C of the lane's K columns, then cell C+1, ... (compile-time recursion so
// that the mask bit is an immediate).  Per cell (SASS, cuobjdump):
//   Gotoh : VIADDMNMX (E), VIADDMNMX (F), VIMNMX3[.RELU] + 1/7 R2P | IMAD, @p IMAD, IMAD
//   linear: VIMNMX, VIADDMNMX[.RELU]               + 1/7 R2P | IMAD, @p IMAD
// The diagonal term of cell C+1 is formed before X[C] is overwritten, so the
// old value dies in place and no register moves are needed.
// RS / RO: the row is row RO of an RS-row group (selects its bits in the tile mask).
// COUPLED: the coupled cell (the end-cell tracking strip kernels and the one-pair-per-warp batch kernels), otherwise
// the decoupled one.
// TRACK (local scheme, coupled cells): also remember WHERE the lane's maximum was first reached, in the
// lane's own row-major order (strict '>'), for the reference's end-cell rule (src/scoring_cpu.impala:48-72).
template <bool LOCAL, bool AFFINE, int K, int PARTIAL, bool MASK, int RS, int RO, int C, bool COUPLED, bool TRACK = false>
struct Cell {
    static_assert(!TRACK || (LOCAL && COUPLED), "end-cell tracking: local scheme, coupled cells");
    template <int KF, int KS, int W>
    static __device__ __forceinline__ void run(int (&X)[K], int (&F)[KF], const int (&sc)[KS], StepState<W>& s,
                                               const StepConst& k)
    {
        const int up = X[C];
        const int dd = s.dd;
        if constexpr (C + 1 < K) {
            constexpr int BIT = (C + 1) * RS + RO;
            if constexpr (MASK) s.dd = diag_plus_sigma_mask<BIT % 32>(s.tm[BIT / 32], up, k.one, k.diff_o, k.same_o);
            else s.dd = diag_plus_sigma(s.qc, sc[C + 1], up, k.one, k.diff_o, k.same_o);
        }
        if constexpr (!COUPLED) {
            // decoupled form: s.xleft carries M of the cell to the left (X of the left neighbour for the lane's first
            // column -- both are valid second operands of E' = max(E + ge, .)), dd = X_diag + sigma (X form throughout)
            int x;
            if constexpr (AFFINE) {
                const int f = __viaddmax_s32(F[C], k.ge, up);
                int mp;
                if constexpr (LOCAL) mp = __vimax3_s32(imad_add(f, k.one, k.go), dd, k.go);   // H >= 0  <=>  X >= go
                else mp = __viaddmax_s32(f, k.go, dd);
                s.e = __viaddmax_s32(s.e, k.ge, s.xleft);
                if constexpr (PARTIAL != 0) capture_if_bit<C>(k.capmask, s.es, s.e, k.one);
                x = __viaddmax_s32(s.e, k.go, mp);
                F[C] = f;
                s.xleft = (C + 1 < K) ? mp : x;        // the lane hands X (not M) to its right neighbour
            } else {
                const int nn = LOCAL ? __viaddmax_s32_relu(up, k.ge, dd) : __viaddmax_s32(up, k.ge, dd);
                x = __viaddmax_s32(s.xleft, k.ge, nn);
                s.xleft = x;
            }
            if constexpr (LOCAL) {
                if constexpr (PARTIAL) {
                    if (C < k.nvalid) s.best = max(s.best, x);
                } else if constexpr ((C & 1) != 0) {
                    s.best = __vimax3_s32(s.best, s.hprev, x);
                } else {
                    s.hprev = x;
                }
            }
            X[C] = x;
            if constexpr (PARTIAL != 0) capture_if_bit<C>(k.capmask, s.xs, x, k.one);
            if constexpr (C + 1 < K) Cell<LOCAL, AFFINE, K, PARTIAL, MASK, RS, RO, C + 1, COUPLED, TRACK>::run(X, F, sc, s, k);
            return;
        }
        int h;
        if constexpr (AFFINE) {
            s.e = __viaddmax_s32(s.e, k.ge, s.xleft);
            if constexpr (PARTIAL != 0) capture_if_bit<C>(k.capmask, s.es, s.e, k.one);
            const int f = __viaddmax_s32(F[C], k.ge, up);
            h = LOCAL ? __vimax3_s32_relu(dd, s.e, f) : __vimax3_s32(dd, s.e, f);
            F[C] = f;
        } else {
            const int tmax = max(s.xleft, up);
            h = LOCAL ? __viaddmax_s32_relu(tmax, k.ge, dd) : __viaddmax_s32(tmax, k.ge, dd);
        }
        if constexpr (LOCAL && TRACK) {
            if ((!PARTIAL || C < k.nvalid) && h > s.best) { s.best = h; s.bpos = s.rowpos + C; }
        } else if constexpr (LOCAL) {
            if constexpr (PARTIAL) {
                if (C < k.nvalid) s.best = max(s.best, h);
            } else if constexpr ((C & 1) != 0) {
                s.best = __vimax3_s32(s.best, s.hprev, h);
            } else {
                s.hprev = h;
            }
        }
        const int x = AFFINE ? imad_add(h, k.one, k.go) : h;
        X[C] = x;
        s.xleft = x;
        if constexpr (PARTIAL != 0) capture_if_bit<C>(k.capmask, s.xs, x, k.one);
        if constexpr (C + 1 < K) Cell<LOCAL, AFFINE, K, PARTIAL, MASK, RS, RO, C + 1, COUPLED, TRACK>::run(X, F, sc, s, k);
    }
};

// R rows of one lane per step (R = 2 or 4): cells (r, C) for r = 0..R-1, then
// column C+1.  Row r is one column behind row r-1 (its F and its diagonal come
// from the row r-1 cell just relaxed), so a lane carries R dependent chains in a
// small 2-D wavefront instead of one chain: R times the instruction-level
// parallelism, 1/R of the per-cell step overhead, and one such warp per
// scheduler is enough to keep the issue slots busy.
template <int R, int W>
struct StepStateR {
    int dd[R];           // diag + sigma of the R cells about to be relaxed
    int e[R];            // E to the left, per row
    int x[R];            // X to the left, per row
    unsigned tm[W];      // MASK: tile mask of the group
    int qc[R];           // !MASK: query bytes of the R rows
    int best;            // LOCAL
    int xs[R], es[R];    // PARTIAL: X and E of the edge column, per row
};

template <bool LOCAL, bool AFFINE, int K, int PARTIAL, bool MASK, int R, int C, int FORM>
struct CellR {
    template <int KF, int KS, int W>
    static __device__ __forceinline__ void run(int (&X)[K], int (&F)[KF], const int (&sc)[KS], StepStateR<R, W>& s,
                                               const StepConst& k)
    {
        int above_x = X[C];                      // X of the cell above (row -1 of this group: the stored row)
        int above_f = 0;
        if constexpr (AFFINE) above_f = F[C];
        int hrow[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int dd = s.dd[r];
            // FORM 2 ("mixed", Gotoh two-row tiles): even rows coupled (3 ALU-pipe ops per cell), odd rows decoupled (4) --
            // the decoupled kernel is ALU-pipe bound (94 % busy, ncu), the coupled one latency bound; half and half has
            // 12 % less ALU work than the one and a short chain in every other row unlike the other
            const bool coupled_row = FORM == 2 && (r & 1) == 0;
            if constexpr (C + 1 < K) {
                // diagonal term of cell (r, C+1): H(r-1, C) = the cell above this one
                if constexpr (MASK) {
                    if (coupled_row) s.dd[r] = diag_mask_bit_c<(C + 1) * R>(s.tm, r, above_x, k.one, k.diff_c, k.same_c);
                    else s.dd[r] = diag_mask_bit<(C + 1) * R>(s.tm, r, above_x, k);
                } else {
                    s.dd[r] = diag_plus_sigma(s.qc[r], sc[C + 1], above_x, k.one, k.diff_o, k.same_o);
                }
            }
            int h, x;
            if (coupled_row) {
                s.e[r] = __viaddmax_s32(s.e[r], k.ge, s.x[r]);
                const int f = __viaddmax_s32(above_f, k.ge, above_x);
                h = LOCAL ? __vimax3_s32_relu(dd, s.e[r], f) : __vimax3_s32(dd, s.e[r], f);
                x = imad_add(h, k.one, k.go);
                above_f = f;
                hrow[r] = x;                    // the local maximum is tracked on X in this form
                s.x[r] = x;
                above_x = x;
                if constexpr (PARTIAL != 0) {
                    capture_if_bit<C>(k.capmask, s.xs[r], x, k.one);
                    capture_if_bit<C>(k.capmask, s.es[r], s.e[r], k.one);
                }
                continue;
            }
            if constexpr (AFFINE) {
                // decoupled form (see Cell): s.x[r] carries M of the cell to the left, hrow holds X (= H + go)
                const int f = __viaddmax_s32(above_f, k.ge, above_x);
                int mp;
                if constexpr (LOCAL) mp = __vimax3_s32(imad_add(f, k.one, k.go), dd, k.go);
                else mp = __viaddmax_s32(f, k.go, dd);
                s.e[r] = __viaddmax_s32(s.e[r], k.ge, s.x[r]);
                x = __viaddmax_s32(s.e[r], k.go, mp);
                h = x;
                above_f = f;
                hrow[r] = h;
                s.x[r] = (C + 1 < K) ? mp : x;
                above_x = x;
                if constexpr (PARTIAL != 0) {
                    capture_if_bit<C>(k.capmask, s.xs[r], x, k.one);
                    capture_if_bit<C>(k.capmask, s.es[r], s.e[r], k.one);
                }
                continue;
            } else {
                const int nn = LOCAL ? __viaddmax_s32_relu(above_x, k.ge, dd) : __viaddmax_s32(above_x, k.ge, dd);
                h = __viaddmax_s32(s.x[r], k.ge, nn);
                x = h;
            }
            hrow[r] = h;
            s.x[r] = x;
            above_x = x;
            if constexpr (PARTIAL != 0) capture_if_bit<C>(k.capmask, s.xs[r], x, k.one);
        }
        if constexpr (LOCAL) {
            if constexpr (PARTIAL) {
                if (C < k.nvalid) {
#pragma unroll
                    for (int r = 0; r + 1 < R; r += 2) s.best = __vimax3_s32(s.best, hrow[r], hrow[r + 1]);
                }
            } else {
#pragma unroll
                for (int r = 0; r + 1 < R; r += 2) s.best = __vimax3_s32(s.best, hrow[r], hrow[r + 1]);
            }
        }
        X[C] = above_x;
        if constexpr (AFFINE) F[C] = above_f;
        if constexpr (C + 1 < K) CellR<LOCAL, AFFINE, K, PARTIAL, MASK, R, C + 1, FORM>::run(X, F, sc, s, k);
    }
};

// shared memory of one warp: a batch is always 32 rows (32/R steps)
struct alignas(16) WarpSmem {
    int2 in[32];        // left border rows of the current batch (X form, E)
    int2 out[64];       // right edge rows waiting to be published (ring of two batches)
    uint8_t q[256];     // query symbols (MASK: codes) of the last 64*R rows (ring; packed cells: the last 256 rows)
    int boff[8];        // packed cells: the warp's score offset of each of the last 8 batches (strip_packed.cuh)
};

__device__ __forceinline__ int4 ld_record(const int4* p)
{
    int4 v;
    asm volatile("ld.volatile.global.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p)
                 : "memory");
    return v;
}
__device__ __forceinline__ void st_record(int4* p, int4 v)
{
    asm volatile("st.volatile.global.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}

// One (band, strip) item.  PARTIAL != 0: the strip is cut by the right matrix edge
// (only the last strip of a job can be): the columns past the edge compute
// don't-care values (dependencies only run left->right, so they never reach a
// valid cell), the edge column is picked out for the output, and the local
// maximum is masked.  R = rows per lane and step (PARTIAL items use R = 1).
template <bool LOCAL, bool AFFINE, int K, int PARTIAL, bool MASK, int R, bool TRACK, int FORM>
__device__ __forceinline__ bool process_item(const Job& J, const int band, const int strip,
                                             const KernelArgs& a, WarpSmem& sm,
                                             unsigned* __restrict__ s_mask /* [ncodes][32][W] spread column masks */,
                                             const uint8_t* __restrict__ s_lut /* [2][256] */,
                                             const int lane)
{
    static_assert(R == 1 || R == 2 || R == 4, "rows per step");
    static_assert(!TRACK || (LOCAL && R == 1), "end-cell tracking: local scheme, single-row kernels");
    constexpr int SW = kWarp * K;
    constexpr int B = 32 / R;              // steps per batch (a batch = 32 rows)
    constexpr int QM = 64 * R - 1;         // query ring mask
    constexpr int W = TileWords<R, K>::value;
    const int i0 = band * J.band_h;
    const int hb = min(J.band_h, J.h - i0);
    const int j0 = strip * SW;
    const int wv = min(SW, J.w - j0);
    const bool last_strip = (strip == J.nstrips - 1);
    const int go = AFFINE ? a.sp.gap_open : 0;
    StepConst k;
    k.one = a.one;
    k.ge = a.sp.gap_extend;
    k.go = go;
    // coupled form: dd = H_diag + sigma = X_diag + (sigma - go); decoupled form: dd = X_diag + sigma
    k.diff_o = TRACK ? a.sp.diff - go : a.sp.diff;
    k.same_o = TRACK ? a.sp.same - go : a.sp.same;
    k.diff_c = a.sp.diff - go;
    k.same_c = a.sp.same - go;
    static_assert(FORM == 1 || (FORM == 2 && MASK && AFFINE && R == 2), "decoupled cells, or mixed cells: Gotoh two-row MASK tiles");
    int* const status = a.status;
    const unsigned long long timeout_ns = a.timeout_ns;

    // border records this strip consumes / produces
    const bool from_inbox = (strip == 0) && (J.in != nullptr);
    const int4* lin = (from_inbox ? J.in : J.col) + i0;
    const int expect = from_inbox ? J.in_tag : strip;
    const int my_tag = strip + 1;
    int4* const colout = J.col + i0;
    const bool mirror = last_strip && (J.out != nullptr);
    const uint8_t* qrow = J.q + i0;

#ifdef ANYSEQ_PROFILE
    const long long pf_item0 = clock64();
#endif
    // the band above must be complete (its bottom border is our top border)
    if (band > 0) {
        if (!wait_rows(J.progress + strip, i0, false, status, timeout_ns)) return false;
    }
#ifdef ANYSEQ_PROFILE
    const long long pf_band = clock64() - pf_item0;
    const long long pf_slot = J.item_begin + strip;
    const bool pf_trace = a.trace && band == 0 && pf_slot < kTraceStrips && lane == 0;
    if (pf_trace) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        a.trace[4 * pf_slot + 0] = global_timer_ns();
        a.trace[4 * pf_slot + 3] = smid;
    }
#endif

    int X[K], F[AFFINE ? K : 1], sc[MASK ? 1 : K];
    const int jl = j0 + lane * K;
    load_row_ints<K>(J.rowH + jl, X);
    if constexpr (AFFINE) {
        load_row_ints<K>(J.rowF + jl, F);
#pragma unroll
        for (int c = 0; c < K; ++c) X[c] += go;
    } else {
        F[0] = 0;
    }
    if constexpr (MASK) {
        // per-lane column masks, one per alphabet code, spread by R (column c -> bit c*R);
        // code 0 matches nothing
        sc[0] = 0;
        __syncwarp();
        for (int cd = 0; cd < a.ncodes; ++cd)
#pragma unroll
            for (int w = 0; w < W; ++w) s_mask[(cd * 32 + lane) * W + w] = 0u;
#pragma unroll 4
        for (int c = 0; c < K; ++c) {
            const int j = jl + c;
            const int cd = (j < J.w) ? (int)s_lut[256 + J.s[j]] : 0;
            if (cd) s_mask[(cd * 32 + lane) * W + (c * R) / 32] |= 1u << ((c * R) % 32);
        }
        __syncwarp();
    } else {
#pragma unroll
        for (int c = 0; c < K; ++c) {
            const int j = jl + c;
            sc[c] = (j < J.w) ? (int)J.s[j] : 0x7fff;   // never equals a byte
        }
    }

    // H(i0-1, first column - 1) in X form
    int dcarry = __shfl_up_sync(kFull, X[K - 1], 1);
    if (lane == 0) dcarry = __ldcg(J.corner + strip) + go;

    const int outlane = PARTIAL ? (wv - 1) / K : 31;
    k.outc = PARTIAL ? (wv - 1) % K : K - 1;
    k.nvalid = PARTIAL ? max(0, min(K, wv - lane * K)) : K;
    k.capmask = PARTIAL ? (1u << k.outc) : 0u;
    const int ngroups = (hb + R - 1) / R;  // row groups of R rows
    const int T = ngroups + outlane;       // number of steps
    int hr[R], er[R];
    unsigned tm_cur[W];
#pragma unroll
    for (int r = 0; r < R; ++r) { hr[r] = 0; er[r] = 0; }
#pragma unroll
    for (int w = 0; w < W; ++w) tm_cur[w] = 0u;
    int flushed = 0;                       // rows published so far
    StepState<W> st;
    st.dd = 0; st.e = 0; st.xleft = 0; st.best = kScoreMin; st.hprev = kScoreMin; st.es = 0; st.xs = 0; st.qc = 0;
    st.bpos = 0; st.rowpos = 0;
#pragma unroll
    for (int w = 0; w < W; ++w) st.tm[w] = 0u;
    int vbest = kScoreMin;                 // TRACK: value maximum over the flushed block rows
    // TRACK: fold the lane's (maximum, first position) of the current 1024-row block row into the per-block table;
    // key order = larger value first, then smaller row-major position inside the 1024 x 1024 block
    auto flush_track = [&]() {
        if (st.best > kScoreMin) {
            const int row = st.bpos / K, c = st.bpos % K;
            const int absrow = i0 + row, abscol = jl + c;
            const unsigned pos = ((unsigned)(absrow & 1023) << 10) | (unsigned)(abscol & 1023);
            const unsigned long long key =
                ((unsigned long long)((unsigned)st.best ^ 0x80000000u) << 32) | (unsigned long long)(0xfffffu - pos);
            atomicMax(J.blockmax + (size_t)(absrow >> 10) * J.nbj + (abscol >> 10), key);
            vbest = max(vbest, st.best);
        }
        st.best = kScoreMin;
    };

    // rows [base, base+32) of the out lane's edge -> tagged records (coalesced 16-byte stores, no fence)
    auto flush32 = [&](int base) {
        const int r = base + lane;
        if (r < hb) {
            const int2 v = sm.out[r & 63];
            st_record(colout + r, make_int4(v.x - go, my_tag, v.y, my_tag));
            if (mirror) st_record(J.out + i0 + r, make_int4(v.x - go, J.out_tag, v.y, J.out_tag));
            if (J.edges) __stcg(J.edges + (size_t)strip * J.h + i0 + r, make_int2(v.x - go, v.y));
        }
    };
    // MASK: tile mask of row group g = sum over its rows of (spread mask of the row's code) << r
    auto tile_mask = [&](int g, unsigned (&tm)[W]) {
#pragma unroll
        for (int w = 0; w < W; ++w) tm[w] = 0u;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const unsigned* mp = s_mask + ((int)sm.q[(R * g + r) & QM] * 32 + lane) * W;
#pragma unroll
            for (int w = 0; w < W; ++w) tm[w] += mp[w] << r;
        }
    };

    // one row of one lane (single chain): used for R = 1 and for the guarded steps of R > 1
    auto relax_row = [&](auto ro_tag, const int row, const int xl, const int el, int& hro, int& ero) {
        constexpr int RO = decltype(ro_tag)::value;
        if constexpr (TRACK) {
            if (((i0 + row) & 1023) == 0) flush_track();      // a new 1024-row block row of the reference starts
            st.rowpos = row * K;
        }
        if constexpr (MASK) {
#pragma unroll
            for (int w = 0; w < W; ++w) st.tm[w] = tm_cur[w];
            st.dd = diag_plus_sigma_mask<RO>(st.tm[0], dcarry, k.one, k.diff_o, k.same_o);
        } else {
            st.qc = sm.q[row & QM];
            st.dd = diag_plus_sigma(st.qc, sc[0], dcarry, k.one, k.diff_o, k.same_o);
        }
        dcarry = xl;
        st.xleft = xl;
        st.e = el;
        Cell<LOCAL, AFFINE, K, PARTIAL, MASK, R, RO, 0, TRACK, TRACK>::run(X, F, sc, st, k);     // coupled iff tracking
        hro = st.xleft;
        ero = st.e;
        if constexpr (PARTIAL != 0) {
            if (lane == outlane) sm.out[row & 63] = make_int2(st.xs, st.es);
        } else {
            if (lane == 31) sm.out[row & 63] = make_int2(hro, ero);
        }
    };

    // one anti-diagonal step; GUARD = some rows of some lanes may be outside [0, hb)
    auto step = [&](auto guard_tag, const int t) {
        constexpr bool GUARD = decltype(guard_tag)::value;
        int xl[R], el[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            xl[r] = __shfl_up_sync(kFull, hr[r], 1);
            el[r] = 0;
            if constexpr (AFFINE) el[r] = __shfl_up_sync(kFull, er[r], 1);
        }
        {
            const int2* bp = &sm.in[R * (t & (B - 1))];
            if constexpr (R == 1) {
                const int2 bnd = bp[0];
                if (lane == 0) { xl[0] = bnd.x; el[0] = bnd.y; }
            } else {
#pragma unroll
                for (int r = 0; r < R; r += 2) {
                    const int4 bnd = *reinterpret_cast<const int4*>(bp + r);
                    if (lane == 0) { xl[r] = bnd.x; el[r] = bnd.y; xl[r + 1] = bnd.z; el[r + 1] = bnd.w; }
                }
            }
        }
        const int g = t - lane;                 // row group of this lane
        unsigned tm_next[W];
#pragma unroll
        for (int w = 0; w < W; ++w) tm_next[w] = 0u;
        if constexpr (MASK) tile_mask(g + 1, tm_next);            // prefetch, off the critical path
        if constexpr (!GUARD && R > 1) {
            StepStateR<R, W> s2;
            s2.best = st.best;
#pragma unroll
            for (int w = 0; w < W; ++w) s2.tm[w] = tm_cur[w];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                s2.qc[r] = 0;
                const int dg = (r == 0) ? dcarry : xl[r - 1];      // H(row-1, first column - 1)
                if constexpr (MASK) {
                    if (FORM == 2 && (r & 1) == 0) s2.dd[r] = diag_mask_bit_c<0>(s2.tm, r, dg, k.one, k.diff_c, k.same_c);
                    else s2.dd[r] = diag_mask_bit<0>(s2.tm, r, dg, k);
                } else {
                    s2.qc[r] = sm.q[(R * g + r) & QM];
                    s2.dd[r] = diag_plus_sigma(s2.qc[r], sc[0], dg, k.one, k.diff_o, k.same_o);
                }
                s2.x[r] = xl[r];
                s2.e[r] = el[r];
            }
            dcarry = xl[R - 1];
#pragma unroll
            for (int r = 0; r < R; ++r) { s2.xs[r] = 0; s2.es[r] = 0; }
            CellR<LOCAL, AFFINE, K, PARTIAL, MASK, R, 0, FORM>::run(X, F, sc, s2, k);
#pragma unroll
            for (int r = 0; r < R; ++r) { hr[r] = s2.x[r]; er[r] = s2.e[r]; }
            st.best = s2.best;
            if (lane == outlane) {
#pragma unroll
                for (int r = 0; r < R; r += 2) {
                    const int4 v = PARTIAL != 0 ? make_int4(s2.xs[r], s2.es[r], s2.xs[r + 1], s2.es[r + 1])
                                                : make_int4(hr[r], er[r], hr[r + 1], er[r + 1]);
                    *reinterpret_cast<int4*>(&sm.out[(R * g + r) & 63]) = v;
                }
            }
        } else {
            const int row0 = R * g;
            if (!GUARD || (unsigned)row0 < (unsigned)hb)
                relax_row(std::integral_constant<int, 0>{}, row0, xl[0], el[0], hr[0], er[0]);
            if constexpr (R > 1) {
                if ((unsigned)(row0 + 1) < (unsigned)hb)
                    relax_row(std::integral_constant<int, 1>{}, row0 + 1, xl[R > 1 ? 1 : 0], el[R > 1 ? 1 : 0], hr[R > 1 ? 1 : 0], er[R > 1 ? 1 : 0]);
            }
            if constexpr (R > 2) {
                if ((unsigned)(row0 + 2) < (unsigned)hb)
                    relax_row(std::integral_constant<int, 2>{}, row0 + 2, xl[R > 2 ? 2 : 0], el[R > 2 ? 2 : 0], hr[R > 2 ? 2 : 0], er[R > 2 ? 2 : 0]);
                if ((unsigned)(row0 + 3) < (unsigned)hb)
                    relax_row(std::integral_constant<int, 3>{}, row0 + 3, xl[R > 2 ? 3 : 0], el[R > 2 ? 3 : 0], hr[R > 2 ? 3 : 0], er[R > 2 ? 3 : 0]);
            }
        }
        // also on steps where this lane is still above the band: its first row
        // group must find its tile mask in place
#pragma unroll
        for (int w = 0; w < W; ++w) tm_cur[w] = tm_next[w];
    };

#ifdef ANYSEQ_PROFILE
    long long pf_wait = 0, pf_io = 0, pf_steps = 0, pf_t;
#define PF_BEGIN() pf_t = clock64()
#define PF_END(acc) acc += clock64() - pf_t
#else
#define PF_BEGIN()
#define PF_END(acc)
#endif
    // speculative prefetch of the first batch of border records and query symbols
    int4 rec = make_int4(0, expect, kNegInf, expect);
    uint8_t qsym = 0;
    if (lane < hb) {
        rec = ld_record(lin + lane);
        qsym = qrow[lane];
    }
    for (int tb = 0; tb < T; tb += B) {
        __syncwarp();
        PF_BEGIN();
        const int rb = R * tb;                  // first row of the batch
        // (1) publish the edge rows the out lane finished so far
        {
            const int completed = min(max(R * (tb - outlane), 0), hb);
            while (completed - flushed >= 32) {
                flush32(flushed);
                flushed += 32;
            }
        }
        PF_END(pf_io);
        // (2) the batch's border records were prefetched a batch ago; a record is
        //     valid when both of its tags are the expected one
        if (rb < hb) {
            PF_BEGIN();
            const int r = rb + lane;
            bool ok = (r >= hb) || (rec.y == expect && (!AFFINE || rec.w == expect));
            if (!__all_sync(kFull, ok)) {
                const unsigned long long t0 = global_timer_ns();
                unsigned spins = 0;
                while (true) {
                    if (r < hb) rec = ld_record(lin + r);
                    ok = (r >= hb) || (rec.y == expect && (!AFFINE || rec.w == expect));
                    if (__all_sync(kFull, ok)) break;
                    if ((++spins & 63u) == 0u) {
                        bool fail = *(volatile int*)status != kStatusOk;
                        if (!fail && global_timer_ns() - t0 > timeout_ns) {
                            if (atomicCAS(status, kStatusOk, kStatusTimeout) == kStatusOk) {
                                status[1] = expect; status[2] = rec.y; status[3] = strip;
                            }
                            fail = true;
                        }
                        if (__any_sync(kFull, fail)) return false;
                    }
                }
            }
            PF_END(pf_wait);
#ifdef ANYSEQ_PROFILE
            if (pf_trace && tb == 0) a.trace[4 * pf_slot + 1] = global_timer_ns();
#endif
            PF_BEGIN();
            sm.in[lane] = make_int2(rec.x + go, rec.z);
            sm.q[r & QM] = MASK ? s_lut[qsym] : qsym;
            // prefetch the next batch (its records may not be there yet: checked next time)
            const int rn = r + 32;
            if (rn < hb) {
                rec = ld_record(lin + rn);
                qsym = qrow[rn];
            }
            __syncwarp();
            if constexpr (MASK) tile_mask(tb - lane, tm_cur);     // row group of this lane at step tb
            PF_END(pf_io);
        }
        PF_BEGIN();
        // (3) B anti-diagonal steps; batches in which every row of every lane is
        //     inside the band run the unguarded body
        if (tb >= 31 && R * (tb + B) <= hb) {
#pragma unroll 1
            for (int t = tb; t < tb + B; ++t) step(std::false_type{}, t);
        } else {
            const int tend = min(tb + B, T);
#pragma unroll 1
            for (int t = tb; t < tend; ++t) step(std::true_type{}, t);
        }
        PF_END(pf_steps);
    }
#ifdef ANYSEQ_PROFILE
    if (lane == 0) {
        unsigned long long* pc = reinterpret_cast<unsigned long long*>(a.status + 20);
        atomicAdd(pc + 0, (unsigned long long)pf_wait);
        atomicAdd(pc + 1, (unsigned long long)pf_io);
        atomicAdd(pc + 2, (unsigned long long)pf_steps);
        atomicAdd(pc + 3, (unsigned long long)((T + B - 1) / B));
        atomicAdd(pc + 4, (unsigned long long)pf_band);
        atomicAdd(pc + 5, (unsigned long long)(clock64() - pf_item0));
        atomicAdd(pc + 6, 1ull);
    }
    if (pf_trace) a.trace[4 * pf_slot + 2] = global_timer_ns();
#endif

    // drain: remaining edge rows, bottom border, corner, local maximum
    __syncwarp();
    while (flushed < hb) {
        flush32(flushed);
        flushed += 32;
    }
#pragma unroll
    for (int c = 0; c < K; c += 4) {
        __stcg(reinterpret_cast<int4*>(J.rowH + jl + c),
               make_int4(X[c] - go, X[c + 1] - go, X[c + 2] - go, X[c + 3] - go));
        if constexpr (AFFINE)
            __stcg(reinterpret_cast<int4*>(J.rowF + jl + c), make_int4(F[c], F[c + 1], F[c + 2], F[c + 3]));
    }
    if (lane == 0) __stcg(J.corner + strip, dcarry - go);
    if constexpr (LOCAL) {
        if constexpr (TRACK) { flush_track(); st.best = vbest; }
        int best = st.best;
        if constexpr (!PARTIAL) best = max(best, st.hprev);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(kFull, best, o));
        if constexpr (!TRACK && AFFINE) {
            if (best > kScoreMin) best -= go;             // the decoupled (and mixed) Gotoh cells track X = H + go
        }
        if (lane == 0) atomicMax(J.best, best);
    }
    // band hand-over: bottom border + corner are visible before the row counter
    __syncwarp();
    if (lane == 0) {
        __threadfence();
        st_relaxed_gpu(J.progress + strip, i0 + hb);
    }
    return true;
}

}  // namespace anyseq

#include "strip_packed.cuh"

namespace anyseq {

// rows per lane and step of each kernel variant
#ifndef ANYSEQ_ROWS_K32
#define ANYSEQ_ROWS_K32 2
#endif
#ifndef ANYSEQ_ROWS_K16
#define ANYSEQ_ROWS_K16 2
#endif
#ifndef ANYSEQ_ROWS_K8
#define ANYSEQ_ROWS_K8 4     // narrow problems have few strips: four chains per warp make the lone warps fast
#endif
#ifndef ANYSEQ_ROWS_K4
#define ANYSEQ_ROWS_K4 2     // small problems are latency-bound: two rows per step cost 123 instead of 2 x 107 cycles (SASS issue model)
#endif
template <int K, bool MASK>
struct StripRows {
    static constexpr int value = !MASK ? 1 : (K >= 32 ? ANYSEQ_ROWS_K32 : (K >= 16 ? ANYSEQ_ROWS_K16 : (K >= 8 ? ANYSEQ_ROWS_K8 : ANYSEQ_ROWS_K4)));
};

// CTAs per SM the register allocation is capped for.  Single-row kernels need
// >= 4 warps per scheduler to hide the 3-deep dependent chain per cell; multi-row
// tiles carry R chains per warp and run with 1-3 CTAs per SM (engine.cu), so
// they may use more registers.
template <int K, bool MASK>
constexpr int strip_min_blocks()
{
    constexpr int R = StripRows<K, MASK>::value;
    if (R >= 4) return 1;
    if (R == 2) return K >= 32 ? 2 : (K >= 16 ? 3 : 4);
    return K >= 32 ? 4 : (K >= 16 ? 5 : 6);
}

template <bool LOCAL, bool AFFINE, int K, bool MASK, bool TRACK = false, int FORM = 1>
__global__ void __launch_bounds__(TRACK ? kThreads : kMaxStripWarps * kWarp, TRACK ? (K >= 32 ? 4 : (K >= 16 ? 5 : 6)) : 1)
strip_kernel(const KernelArgs a)
{
    constexpr int R = TRACK ? 1 : StripRows<K, MASK>::value;
    __shared__ WarpSmem s_warp[TRACK ? kWarpsPerBlock : kMaxStripWarps];
    __shared__ uint8_t s_lut[MASK ? 512 : 4];
    extern __shared__ unsigned s_dyn[];          // MASK: [warps][ncodes][32][W] spread column masks

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    constexpr int SW = kWarp * K;
    if constexpr (MASK) {
        for (int x = threadIdx.x; x < 256; x += blockDim.x) {
            s_lut[x] = a.lut_q[x];
            s_lut[256 + x] = a.lut_s[x];
        }
        __syncthreads();
    }
    static_assert(FORM != 3 || (!LOCAL && AFFINE && MASK && !TRACK && R == 2), "packed cells: global / semiglobal Gotoh two-row MASK tiles");
    // packed cells keep one mask per half of the strip
    unsigned* s_mask = s_dyn + warp * a.ncodes * 32 * TileWords<R, K>::value * (FORM == 3 ? 2 : 1);
    // the query ring is read one row ahead (mask prefetch): never let an
    // uninitialised byte be used as a code
    for (int x = lane; x < 256; x += 32) s_warp[warp].q[x] = 0;
    __syncwarp();

    // Items are claimed in index order from a global counter (the first round is
    // the static assignment): every item only waits on lower-numbered items, which
    // were claimed earlier by warps that are resident, so no wait can be circular.
    int jcur = 0;
    // First round: static.  CTA b gets items [ceil(b F / G), ceil((b + 1) F / G)) (F = a.first_items, G = gridDim.x: every SM gets its
    // share even when there are fewer items than warps); inside the CTA the items go to the schedulers in runs, so the warps
    // of one scheduler (w, w + 4, w + 8) work on neighbouring strips.  A warp without an item claims one dynamically.
    long long item;
    {
        // (rounded up: when the items do not divide evenly, the LAST CTAs get one item less -- the last item of a launch is
        // its ragged strip, the slowest one, and this way it tends to have a scheduler to itself)
        const long long lo = ((long long)blockIdx.x * a.first_items + gridDim.x - 1) / gridDim.x;
        const int cnt = (int)(((long long)(blockIdx.x + 1) * a.first_items + gridDim.x - 1) / gridDim.x - lo);
        const int sch = warp & 3, slot = warp >> 2;
        const int base = cnt >> 2, rem = cnt & 3;
        const int mine = base + (sch < rem ? 1 : 0);           // items of this scheduler
        const int off = sch * base + min(sch, rem);
        if (slot < mine) {
            item = lo + off + slot;
        } else {
            unsigned long long nxt = 0;
            if (lane == 0) nxt = atomicAdd(a.next_item, 1ull);
            item = (long long)__shfl_sync(kFull, nxt, 0);
        }
    }
    for (; item < a.total_items;) {
        const int band = (int)(item / a.strips_total);
        const int rem = (int)(item % a.strips_total);
        jcur = a.njobs > 1 ? a.strip2job[rem] : 0;
        const int strip = rem - (int)a.jobs[jcur].item_begin;
        const Job& J = a.jobs[jcur];
        const bool partial = (strip + 1) * SW > J.w;
        bool ok = true;
        if ((long long)band * J.band_h >= J.h) {
            // a band past the end of a short job: nothing to relax
        } else if constexpr (FORM == 3) {
            if (partial) ok = process_item_packed<K, 1>(J, band, strip, a, s_warp[warp], s_mask, s_lut, lane);
            else ok = process_item_packed<K, 0>(J, band, strip, a, s_warp[warp], s_mask, s_lut, lane);
        } else if (partial) {
            ok = process_item<LOCAL, AFFINE, K, 1, MASK, R, TRACK, FORM>(J, band, strip, a, s_warp[warp], s_mask, s_lut, lane);
        } else {
            ok = process_item<LOCAL, AFFINE, K, 0, MASK, R, TRACK, FORM>(J, band, strip, a, s_warp[warp], s_mask, s_lut, lane);
        }
        if (!ok) return;
        unsigned long long nxt = 0;
        if (lane == 0) nxt = atomicAdd(a.next_item, 1ull);
        item = (long long)__shfl_sync(kFull, nxt, 0);
    }
}

using StripKernelFn = void (*)(const KernelArgs);
// defined in strip_inst_*.cu (one translation unit per (LOCAL, AFFINE) pair)
// form: 1 = decoupled cells, 2 = mixed cells (Gotoh MASK kernels with K = 16 / 32 only)
StripKernelFn get_strip_kernel_00(int K, bool mask, int form);
StripKernelFn get_strip_kernel_01(int K, bool mask, int form);
StripKernelFn get_strip_kernel_10(int K, bool mask, int form);
StripKernelFn get_strip_kernel_11(int K, bool mask, int form);
StripKernelFn get_strip_kernel_10t(int K, bool mask);   // local + end-cell tracking
StripKernelFn get_strip_kernel_11t(int K, bool mask);
StripKernelFn get_strip_kernel_01p(int K);              // global / semiglobal Gotoh, packed cells (strip_packed.cuh)

}  // namespace anyseq
