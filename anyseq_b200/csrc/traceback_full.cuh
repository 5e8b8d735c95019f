// traceback_full.cuh -- the predecessor encoding and the walk of the full-matrix traceback, shared by the single-pair
// kernels (traceback_full.cu) and the batch kernel (batch_align.cu)
#pragma once
#include "common.cuh"

namespace anyseq {

// 4 predecessor bits per cell: bits 0-1 the H source in the reference's numbering, bit 2 E extends, bit 3 F extends
enum : int { kFSrcNone = 0, kFSrcE = 1, kFSrcF = 2, kFSrcDiag = 3 };   // src/align.impala:37-40

// One cell: H(i, j) from dsig = H(i-1, j-1) + sigma(q[i], s[j]), up = H(i-1, j), lft = H(i, j-1), e = E(i, j-1) and
// f = F(i-1, j); leaves H(i, j) in lft, E(i, j) in e, F(i, j) in f and returns the cell's predecessor nibble.  Sources
// are taken in the order diag > E > F with strict '>' (the reference's NO_GAP > GAP_Q > GAP_S); linear gaps are
// gi = 0 (go = ge), where E and F never extend.
__device__ __forceinline__ unsigned fulltb_cell(int dsig, int up, int& lft, int& e, int& f, int go, int ge, bool local)
{
    int eext = 0, fext = 0;
    int eo = lft + go;
    if (e + ge > eo) { eo = e + ge; eext = 1; }
    e = eo;
    int fo = up + go;
    if (f + ge > fo) { fo = f + ge; fext = 1; }
    f = fo;
    int score = dsig;
    int src = kFSrcDiag;
    if (e > score) { score = e; src = kFSrcE; }
    if (fo > score) { score = fo; src = kFSrcF; }
    if (local && 0 > score) { score = 0; src = kFSrcNone; }
    lft = score;
    return (unsigned)(src | (eext << 2) | (fext << 3));
}

// One step of the walk of traceback_offset (src/traceback.impala:47-80) as a 3-state machine (0 = H, 1 = E, 2 = F) at
// a cell inside the matrix (i, j >= 0) with predecessor nibble p; qc = q[i], sc = s[j].  Writes column i + j + 1 of
// the aligned rows when the step emits one and moves (i, j).  Returns false where the walk stops (state H, source
// NONE).  The border row and column are the caller's: there only global alignments go on, with gaps.
__device__ __forceinline__ bool fulltb_walk_step(unsigned p, int& i, int& j, int& state, uint8_t qc, uint8_t sc,
                                                 uint8_t* __restrict__ out_q, uint8_t* __restrict__ out_s)
{
    const size_t pos = (size_t)(i + j + 1);
    if (state == 0) {
        const int src = (int)(p & 3u);
        if (src == kFSrcNone) return false;
        if (src == kFSrcDiag) { out_q[pos] = qc; out_s[pos] = sc; --i; --j; }
        else state = (src == kFSrcE) ? 1 : 2;
    } else if (state == 1) {
        out_q[pos] = '_'; out_s[pos] = sc;
        state = ((p >> 2) & 1u) ? 1 : 0; --j;
    } else {
        out_q[pos] = qc; out_s[pos] = '_';
        state = ((p >> 3) & 1u) ? 2 : 0; --i;
    }
    return true;
}

}  // namespace anyseq
