// strip_packed.cuh -- packed cells: the global / semiglobal Gotoh strip item with TWO cells per DPX instruction.
//
// The decoupled Gotoh cell costs four 32-bit DPX operations, and the strip kernel is ALU-pipe bound (DESIGN.md 3.1).
// Here every register holds two 16-bit halves, so VIADDMNMX.S16x2 relaxes two cells per issue slot.  Genome scores do
// not fit in 16 bits, but a warp never needs them absolutely: with go = gi + ge <= 0, ge <= 0 and same >= diff, a step
// right or down changes H by a value in [go, same - go], so every value alive in a warp lies within D * (rows + columns)
// of any other (D = max(same - go, -go)).  The registers therefore hold values relative to a warp-uniform 32-bit offset
// `off`, re-centred once per 32-row batch; the border records, rowH / rowF, the corners and everything the other
// kernels read stay absolute 32-bit.  engine.cu (packed_fits) only launches this form when that window fits.
//
// Layout (strip of 32 * K columns, K2 = K / 2 packed registers per lane):
//   low halves:  columns j0 + l * K2 + c            (left half of the strip)
//   high halves: columns j0 + 32 * K2 + l * K2 + c  (right half)
// The high halves run 32 steps behind the low halves, so the warp acts as one chain of 64 lanes: lane l hands its right
// edge to lane l + 1 with a rotating shuffle, and lane 0 merges the border record (low half) with lane 31's low-half
// edge (high half) in one PRMT.  Lane 31's high half is the strip's right edge.  Match bits of column c, row r of the
// two-row tile sit at bit 4c + 2r (low half) and 4c + 2r + 1 (high half), so that the predicates still come from R2P
// and sigma is three IMADs per pair (diag_sigma_x2).
//
// Values that pass through an IMAD (X, the diagonal term) must stay inside [0, 0x7fff], or the add of c * 65537 would
// carry across the halves: the centre is 0x4000, and "minus infinity" (E / F borders) is clamped to kFloor16, far
// below the window and far above the wrap-around at -0x8000.
#pragma once

namespace anyseq {

constexpr int kCentre16 = 0x4000;
constexpr int kFloor16 = -0x7000;

__device__ __forceinline__ unsigned pack2(int lo, int hi) { return ((unsigned)lo & 0xffffu) | ((unsigned)hi << 16); }
__device__ __forceinline__ int lo16(unsigned v) { return (int)(short)(v & 0xffffu); }
__device__ __forceinline__ int hi16(unsigned v) { return (int)(short)(v >> 16); }

// diag + sigma for both halves: base, override when the low half matches, add when the high half matches (3 IMADs,
// no SEL).  The match bits of a cell pair sit next to each other (bit BIT: low half, BIT + 1: high half).
// KC: any constant block with one, dd_c = base * 65537, sd_c = base * 65536 + low-match value, dhi = (match - base) << 16.
template <int BIT, class KC>
__device__ __forceinline__ unsigned diag_sigma_x2(unsigned m, unsigned d, const KC& k)
{
    unsigned dd = (unsigned)diag_plus_sigma_mask<BIT>(m, (int)d, k.one, k.dd_c, k.sd_c);
    asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %1, %2;\n\tsetp.ne.u32 p, t, 0;\n\t@p mad.lo.s32 %0, %3, %4, %0;\n\t}"
        : "+r"(dd)
        : "r"(m), "n"(2u << BIT), "r"(k.one), "r"(k.dhi));
    return dd;
}

// absolute 32-bit value -> 16-bit half relative to `off`, clamped to [kFloor16, 0x7fff] (only the borders' minus
// infinity is ever clamped: every finite value is inside the window)
__device__ __forceinline__ unsigned rel16(int v, int off)
{
    return (unsigned)max(kFloor16, min(v - off, 0x7fff)) & 0xffffu;
}

struct PackedConst {
    int one;
    unsigned ge2, go2;           // (ge, ge), (go, go): DPX operands
    int dd_c, sd_c, dhi;         // sigma, see diag_sigma_x2
    unsigned capmask;            // PARTIAL: bit of the edge column
};

template <int W>
struct PackedState {
    unsigned dd[2];              // diag + sigma of the cells about to be relaxed, per row of the tile
    unsigned e[2];               // E to the left
    unsigned x[2];               // M (X for the lane's first column) to the left
    unsigned tm[W];              // match bits of the tile
    int xs[2], es[2];            // PARTIAL: X and E of the edge column
};

// One decoupled Gotoh cell pair (see Cell, FORM 1): row RO of the tile, column C of the lane's K2 packed columns.
// ax / af: X and F of the cell above on entry, of this cell on exit.  Four DPX (ALU) + three IMADs (FMA) per pair.
template <int K2, int PARTIAL, int C, int RO, int W>
__device__ __forceinline__ void packed_cell(unsigned& ax, unsigned& af, PackedState<W>& s, const int r, const PackedConst& k)
{
    const unsigned dd = s.dd[r];
    if constexpr (C + 1 < K2) {
        constexpr int BIT = 4 * (C + 1) + 2 * RO;
        s.dd[r] = diag_sigma_x2<BIT % 32>(s.tm[BIT / 32], ax, k);
    }
    const unsigned f = __viaddmax_s16x2(af, k.ge2, ax);
    const unsigned mp = __viaddmax_s16x2(f, k.go2, dd);
    s.e[r] = __viaddmax_s16x2(s.e[r], k.ge2, s.x[r]);
    const unsigned x = __viaddmax_s16x2(s.e[r], k.go2, mp);
    s.x[r] = (C + 1 < K2) ? mp : x;      // the lane hands X (not M) to its right neighbour
    af = f;
    ax = x;
    if constexpr (PARTIAL != 0) {
        capture_if_bit<C>(k.capmask, s.xs[r], (int)x, k.one);
        capture_if_bit<C>(k.capmask, s.es[r], (int)s.e[r], k.one);
    }
}

// the two-row tile: cells (0, C), (1, C), then column C + 1
template <int K2, int PARTIAL, int C>
struct PackedTile {
    template <int W>
    static __device__ __forceinline__ void run(unsigned (&X)[K2], unsigned (&F)[K2], PackedState<W>& s, const PackedConst& k)
    {
        unsigned ax = X[C], af = F[C];
        packed_cell<K2, PARTIAL, C, 0>(ax, af, s, 0, k);
        packed_cell<K2, PARTIAL, C, 1>(ax, af, s, 1, k);
        X[C] = ax;
        F[C] = af;
        if constexpr (C + 1 < K2) PackedTile<K2, PARTIAL, C + 1>::run(X, F, s, k);
    }
};

// one row of the tile alone (guarded steps), state in slot 0
template <int K2, int PARTIAL, int RO, int C>
struct PackedRow {
    template <int W>
    static __device__ __forceinline__ void run(unsigned (&X)[K2], unsigned (&F)[K2], PackedState<W>& s, const PackedConst& k)
    {
        unsigned ax = X[C], af = F[C];
        packed_cell<K2, PARTIAL, C, RO>(ax, af, s, 0, k);
        X[C] = ax;
        F[C] = af;
        if constexpr (C + 1 < K2) PackedRow<K2, PARTIAL, RO, C + 1>::run(X, F, s, k);
    }
};

// One (band, strip) item of a global / semiglobal Gotoh launch with column masks and two-row tiles (process_item's
// contract: same border records, rowH / rowF, corner and progress counter, all absolute).
template <int K, int PARTIAL>
__device__ __forceinline__ bool process_item_packed(const Job& J, const int band, const int strip, const KernelArgs& a,
                                                    WarpSmem& sm,
                                                    unsigned* __restrict__ s_mask /* [ncodes][32][2 halves][W] */,
                                                    const uint8_t* __restrict__ s_lut, const int lane)
{
    constexpr int K2 = K / 2;
    constexpr int SW = kWarp * K;
    constexpr int HW = kWarp * K2;             // columns of one half of the strip
    constexpr int B = 16;                      // steps per batch (a batch = 32 rows)
    constexpr int QM = 255;                    // query ring: the high halves read 64 rows behind the low halves
    constexpr int W = TileWords<2, K>::value;  // 4 * K2 bits of match bits per lane
    static_assert(K == 16 || K == 32, "packed cells: K = 16 or 32");
    const int i0 = band * J.band_h;
    const int hb = min(J.band_h, J.h - i0);
    const int j0 = strip * SW;
    const int wv = min(SW, J.w - j0);
    const bool last_strip = (strip == J.nstrips - 1);
    const int go = a.sp.gap_open;
    PackedConst k;
    k.one = a.one;
    k.ge2 = pack2(a.sp.gap_extend, a.sp.gap_extend);
    k.go2 = pack2(go, go);
    k.dd_c = a.sp.diff * 65537;
    k.sd_c = a.sp.diff * 65536 + a.sp.same;
    k.dhi = (a.sp.same - a.sp.diff) * 65536;
    const unsigned floor2 = pack2(kFloor16, kFloor16);
    int* const status = a.status;
    const unsigned long long timeout_ns = a.timeout_ns;

    const bool from_inbox = (strip == 0) && (J.in != nullptr);
    const int4* lin = (from_inbox ? J.in : J.col) + i0;
    const int expect = from_inbox ? J.in_tag : strip;
    const int my_tag = strip + 1;
    int4* const colout = J.col + i0;
    const bool mirror = last_strip && (J.out != nullptr);
    const uint8_t* qrow = J.q + i0;

    if (band > 0) {
        if (!wait_rows(J.progress + strip, i0, false, status, timeout_ns)) return false;
    }

    // the offset puts X of the strip's first column on the top border at the centre
    int off = __ldcg(J.rowH + j0) + go - kCentre16;
    unsigned X[K2], F[K2];
    const int jlo = j0 + lane * K2, jhi = jlo + HW;
    {
        int lo[K2], hi[K2];
        load_row_ints<K2>(J.rowH + jlo, lo);
        load_row_ints<K2>(J.rowH + jhi, hi);
#pragma unroll
        for (int c = 0; c < K2; ++c) X[c] = rel16(lo[c] + go, off) | (rel16(hi[c] + go, off) << 16);
        load_row_ints<K2>(J.rowF + jlo, lo);
        load_row_ints<K2>(J.rowF + jhi, hi);
#pragma unroll
        for (int c = 0; c < K2; ++c) F[c] = rel16(lo[c], off) | (rel16(hi[c], off) << 16);
    }
    // per-lane column masks, one pair (low, high half) per alphabet code: column c -> bit 4c (low) / 4c + 1 (high)
    __syncwarp();
    for (int cd = 0; cd < a.ncodes; ++cd)
#pragma unroll
        for (int w = 0; w < 2 * W; ++w) s_mask[(cd * 32 + lane) * 2 * W + w] = 0u;
#pragma unroll 4
    for (int c = 0; c < K2; ++c) {
        const int cl = (jlo + c < J.w) ? (int)s_lut[256 + J.s[jlo + c]] : 0;
        const int ch = (jhi + c < J.w) ? (int)s_lut[256 + J.s[jhi + c]] : 0;
        if (cl) s_mask[(cl * 32 + lane) * 2 * W + (4 * c) / 32] |= 1u << ((4 * c) % 32);
        if (ch) s_mask[(ch * 32 + lane) * 2 * W + W + (4 * c) / 32] |= 2u << ((4 * c) % 32);
    }
    __syncwarp();

    // hand-over from lane l - 1 (rotating): lane 0 takes the border value as its low half and lane 31's low half
    // (the left half's right edge, one step old) as its high half
    const int src = (lane + 31) & 31;
    const unsigned sel = lane == 0 ? 0x1054u : 0x3210u;
    // H(i0 - 1, first column - 1) in X form, per half
    unsigned dcarry = __byte_perm(__shfl_sync(kFull, X[K2 - 1], src), rel16(__ldcg(J.corner + strip) + go, off), sel);

    // the edge column: half, lane and column of the strip's last valid column
    const int lastc = wv - 1;
    const int outhalf = PARTIAL ? (lastc >= HW ? 1 : 0) : 1;
    const int outlane = PARTIAL ? (lastc % HW) / K2 : 31;
    k.capmask = PARTIAL ? (1u << (lastc % K2)) : 0u;
    const int outpos = 32 * outhalf + outlane;    // steps the edge cells lag lane 0's low half
    const int ngroups = (hb + 1) / 2;
    const int T = ngroups + outpos;
    unsigned hr[2] = {floor2, floor2}, er[2] = {floor2, floor2};
    unsigned tm_cur[W];
#pragma unroll
    for (int w = 0; w < W; ++w) tm_cur[w] = 0u;
    int flushed = 0;

    // rows [base, base + 32) of the edge -> absolute tagged records; a row written at step t carries the offset of
    // t's batch
    auto flush32 = [&](int base) {
        const int r = base + lane;
        if (r < hb) {
            const int2 v = sm.out[r & 63];
            const int o = sm.boff[((r / 2 + outpos) >> 4) & 7];
            const int x = (outhalf ? hi16((unsigned)v.x) : lo16((unsigned)v.x)) + o - go;
            const int e = (outhalf ? hi16((unsigned)v.y) : lo16((unsigned)v.y)) + o;
            st_record(colout + r, make_int4(x, my_tag, e, my_tag));
            if (mirror) st_record(J.out + i0 + r, make_int4(x, J.out_tag, e, J.out_tag));
            if (J.edges) __stcg(J.edges + (size_t)strip * J.h + i0 + r, make_int2(x, e));
        }
    };
    // match bits of the lane's tile at low-half row group g (high half: group g - 32)
    auto tile_mask = [&](int g, unsigned (&tm)[W]) {
        const int r0 = 2 * g;
        const unsigned* l0 = s_mask + ((int)sm.q[r0 & QM] * 32 + lane) * 2 * W;
        const unsigned* l1 = s_mask + ((int)sm.q[(r0 + 1) & QM] * 32 + lane) * 2 * W;
        const unsigned* h0 = s_mask + ((int)sm.q[(r0 - 64) & QM] * 32 + lane) * 2 * W + W;
        const unsigned* h1 = s_mask + ((int)sm.q[(r0 - 63) & QM] * 32 + lane) * 2 * W + W;
#pragma unroll
        for (int w = 0; w < W; ++w) tm[w] = l0[w] + (l1[w] << 2) + h0[w] + (h1[w] << 2);
    };

    // row RO of the tile of step t alone; a half whose row is outside [0, hb) is left untouched
    auto relax_row = [&](auto ro_tag, const int t, const unsigned xl, const unsigned el) {
        constexpr int RO = decltype(ro_tag)::value;
        const int rlo = 2 * (t - lane) + RO, rhi = rlo - 64;
        const unsigned keep = ((unsigned)rlo < (unsigned)hb ? 0x0000ffffu : 0u) | ((unsigned)rhi < (unsigned)hb ? 0xffff0000u : 0u);
        if (keep == 0u) return;
        unsigned X0[K2], F0[K2];
#pragma unroll
        for (int c = 0; c < K2; ++c) { X0[c] = X[c]; F0[c] = F[c]; }
        PackedState<W> s;
#pragma unroll
        for (int w = 0; w < W; ++w) s.tm[w] = tm_cur[w];
        s.dd[0] = diag_sigma_x2<2 * RO>(s.tm[0], dcarry, k);
        s.x[0] = xl;
        s.e[0] = el;
        s.xs[0] = 0; s.es[0] = 0;
        PackedRow<K2, PARTIAL, RO, 0>::run(X, F, s, k);
#pragma unroll
        for (int c = 0; c < K2; ++c) { X[c] = (X[c] & keep) | (X0[c] & ~keep); F[c] = (F[c] & keep) | (F0[c] & ~keep); }
        dcarry = (xl & keep) | (dcarry & ~keep);
        hr[RO] = s.x[0];
        er[RO] = s.e[0];
        const int ro = outhalf ? rhi : rlo;
        if (lane == outlane && (unsigned)ro < (unsigned)hb)
            sm.out[ro & 63] = PARTIAL ? make_int2(s.xs[0], s.es[0]) : make_int2((int)s.x[0], (int)s.e[0]);
    };

    // one anti-diagonal step; GUARD = some row of some half of some lane may be outside [0, hb)
    auto step = [&](auto guard_tag, const int t) {
        constexpr bool GUARD = decltype(guard_tag)::value;
        unsigned xl[2], el[2];
        {
            const int4 bnd = *reinterpret_cast<const int4*>(&sm.in[2 * (t & (B - 1))]);
            xl[0] = __byte_perm(__shfl_sync(kFull, hr[0], src), (unsigned)bnd.x, sel);
            el[0] = __byte_perm(__shfl_sync(kFull, er[0], src), (unsigned)bnd.y, sel);
            xl[1] = __byte_perm(__shfl_sync(kFull, hr[1], src), (unsigned)bnd.z, sel);
            el[1] = __byte_perm(__shfl_sync(kFull, er[1], src), (unsigned)bnd.w, sel);
        }
        const int g = t - lane;
        unsigned tm_next[W];
        tile_mask(g + 1, tm_next);                 // prefetch, off the critical path
        if constexpr (!GUARD) {
            PackedState<W> s;
#pragma unroll
            for (int w = 0; w < W; ++w) s.tm[w] = tm_cur[w];
            s.dd[0] = diag_sigma_x2<0>(s.tm[0], dcarry, k);
            s.dd[1] = diag_sigma_x2<2>(s.tm[0], xl[0], k);
#pragma unroll
            for (int r = 0; r < 2; ++r) { s.x[r] = xl[r]; s.e[r] = el[r]; s.xs[r] = 0; s.es[r] = 0; }
            dcarry = xl[1];
            PackedTile<K2, PARTIAL, 0>::run(X, F, s, k);
#pragma unroll
            for (int r = 0; r < 2; ++r) { hr[r] = s.x[r]; er[r] = s.e[r]; }
            if (lane == outlane) {
                const int ro = 2 * (g - 32 * outhalf);
                *reinterpret_cast<int4*>(&sm.out[ro & 63]) = PARTIAL ? make_int4(s.xs[0], s.es[0], s.xs[1], s.es[1])
                                                                     : make_int4((int)hr[0], (int)er[0], (int)hr[1], (int)er[1]);
            }
        } else {
            relax_row(std::integral_constant<int, 0>{}, t, xl[0], el[0]);
            relax_row(std::integral_constant<int, 1>{}, t, xl[1], el[1]);
        }
#pragma unroll
        for (int w = 0; w < W; ++w) tm_cur[w] = tm_next[w];
    };

    int4 rec = make_int4(0, expect, kNegInf, expect);
    uint8_t qsym = 0;
    if (lane < hb) {
        rec = ld_record(lin + lane);
        qsym = qrow[lane];
    }
    for (int tb = 0; tb < T; tb += B) {
        __syncwarp();
        const int rb = 2 * tb;
        {
            const int completed = min(max(2 * (tb - outpos), 0), hb);
            while (completed - flushed >= 32) {
                flush32(flushed);
                flushed += 32;
            }
        }
        // re-centre: lane 0's first low-half column goes back to the centre (warp-uniform shift; the floor keeps the
        // clamped minus infinity from wrapping)
        {
            const int d = lo16(__shfl_sync(kFull, X[0], 0)) - kCentre16;
            if (d != 0) {
                const unsigned nd = pack2(-d, -d);
                off += d;
#pragma unroll
                for (int c = 0; c < K2; ++c) { X[c] = __viaddmax_s16x2(X[c], nd, floor2); F[c] = __viaddmax_s16x2(F[c], nd, floor2); }
#pragma unroll
                for (int r = 0; r < 2; ++r) { hr[r] = __viaddmax_s16x2(hr[r], nd, floor2); er[r] = __viaddmax_s16x2(er[r], nd, floor2); }
                dcarry = __viaddmax_s16x2(dcarry, nd, floor2);
            }
            if (lane == 0) sm.boff[(tb >> 4) & 7] = off;
        }
        if (rb < hb) {
            const int r = rb + lane;
            bool ok = (r >= hb) || (rec.y == expect && rec.w == expect);
            if (!__all_sync(kFull, ok)) {
                const unsigned long long t0 = global_timer_ns();
                unsigned spins = 0;
                while (true) {
                    if (r < hb) rec = ld_record(lin + r);
                    ok = (r >= hb) || (rec.y == expect && rec.w == expect);
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
            sm.in[lane] = r < hb ? make_int2((int)rel16(rec.x + go, off), (int)rel16(rec.z, off))
                                 : make_int2((int)floor2, (int)floor2);
            sm.q[r & QM] = s_lut[qsym];
            const int rn = r + 32;
            if (rn < hb) {
                rec = ld_record(lin + rn);
                qsym = qrow[rn];
            }
            __syncwarp();
            tile_mask(tb - lane, tm_cur);
        }
        // batches in which both halves of every lane are inside the band run the unguarded body
        if (tb >= 63 && 2 * (tb + B) <= hb) {
#pragma unroll 1
            for (int t = tb; t < tb + B; ++t) step(std::false_type{}, t);
        } else {
            const int tend = min(tb + B, T);
#pragma unroll 1
            for (int t = tb; t < tend; ++t) step(std::true_type{}, t);
        }
    }

    // drain: remaining edge rows, bottom border, corner -- back to absolute values
    __syncwarp();
    while (flushed < hb) {
        flush32(flushed);
        flushed += 32;
    }
#pragma unroll
    for (int c = 0; c < K2; c += 4) {
        const int o = off - go;
        __stcg(reinterpret_cast<int4*>(J.rowH + jlo + c),
               make_int4(lo16(X[c]) + o, lo16(X[c + 1]) + o, lo16(X[c + 2]) + o, lo16(X[c + 3]) + o));
        __stcg(reinterpret_cast<int4*>(J.rowH + jhi + c),
               make_int4(hi16(X[c]) + o, hi16(X[c + 1]) + o, hi16(X[c + 2]) + o, hi16(X[c + 3]) + o));
        __stcg(reinterpret_cast<int4*>(J.rowF + jlo + c),
               make_int4(lo16(F[c]) + off, lo16(F[c + 1]) + off, lo16(F[c + 2]) + off, lo16(F[c + 3]) + off));
        __stcg(reinterpret_cast<int4*>(J.rowF + jhi + c),
               make_int4(hi16(F[c]) + off, hi16(F[c + 1]) + off, hi16(F[c + 2]) + off, hi16(F[c + 3]) + off));
    }
    if (lane == 0) __stcg(J.corner + strip, lo16(dcarry) + off - go);
    __syncwarp();
    if (lane == 0) {
        __threadfence();
        st_relaxed_gpu(J.progress + strip, i0 + hb);
    }
    return true;
}

}  // namespace anyseq
