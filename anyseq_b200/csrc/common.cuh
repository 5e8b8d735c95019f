// common.cuh -- shared definitions of the B200 alignment engine (sm_100a only).
#pragma once

#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>

namespace anyseq {

constexpr int kWarp = 32;
// "minus infinity" for the affine E/F borders (SURVEY.md A.7: MIN/2 so that
// adding gap costs cannot wrap).  check_score_range (engine.cu) refuses problems whose scores come near it or INT_MAX.
constexpr int kNegInf = -(1 << 30);
// reference SCORE_MIN_VALUE: src/align.impala:16
constexpr int kScoreMin = -2147483647;

enum Mode : int { kGlobal = 0, kSemiglobal = 1, kLocal = 2 };

// status words written by kernels (device -> host)
enum StatusCode : int {
    kStatusOk = 0,
    kStatusTimeout = 1,     // a dependency wait exceeded the watchdog
};

// One DP rectangle ("job"): rows = query symbols q[0..h), columns = subject
// symbols s[0..w).  A single score() call is one job; one Hirschberg level is
// one job per half (forward halves on the forward copies, reversed halves on
// the reversed copies of the sequences).  A job is cut into column strips of
// 32*K columns (one warp each) and row bands of band_h rows; (band, strip)
// pairs are the work items.
//
// Boundary storage mirrors the reference's O(m+n) scheme (column vector, row
// vector, corners: src/scoring.impala:218-259), re-laid for streaming:
//   col[h]        one 16-byte BORDER RECORD per row: {H, tag, E, tag}.  Strip x
//                 consumes the records tagged x (tag 0 = the matrix border,
//                 written by the init kernel) and overwrites them with its own
//                 right edge tagged x+1.  Data and tag share an 8-byte word
//                 (stored atomically), so a consumer that sees the tag has the
//                 value: no flag, no fence, and the next batch of records can be
//                 prefetched speculatively (the NCCL "LL" protocol idea).
//   rowH/rowF[w'] item (b,x) loads its top border from it and stores its
//                 bottom border back (w' = w rounded up to the strip width).
//   corner[x]     H(i0-1, j0-1) for the next band of strip x.
//   progress[x]   rows of strip x completed band-wise (release/acquire): only
//                 the band hand-over (once per item) uses it.
struct Job {
    const uint8_t* q;
    const uint8_t* s;
    int h, w;
    int band_h;
    int nstrips, nbands;
    long long item_begin;    // launch-wide index of the job's first strip (prefix sum of nstrips over the jobs of a launch)
    int4* col;
    int* rowH;
    int* rowF;
    int* corner;
    int* progress;
    int* best;               // local mode: running maximum (atomicMax)
    unsigned long long* blockmax;   // local end-cell tracking: per 1024 x 1024 reference block (value, -position) keys
    int nbj;                 // number of 1024-column blocks (row pitch of blockmax)
    int2* edges;             // optional [nstrips][h]: (H, E) of every strip's last column, kept for the full-matrix traceback
    // multi-GPU chaining (null on a single GPU): strip 0 consumes the records
    // tagged in_tag from `in` (this rank's inbox, written by the previous rank
    // over NVLink); the last strip mirrors its right edge into `out` (the next
    // rank's inbox, peer memory) tagged out_tag.
    const int4* in;
    int4* out;
    int in_tag;
    int out_tag;
    // initialisation of the borders (init kernel)
    int init_global;         // 1: gap multiples (global), 0: zeros
    int top_open;            // global: H(-1, j) = top_open + j * gap_extend (cost of the first gap symbol on
                             // the top border; smaller for Gotoh traceback blocks entered inside a gap)
};

struct ScoreParams {
    int same, diff;
    int gap_extend;          // linear: the gap cost; affine: ge
    int gap_open;            // affine: gi + ge (cost of the first gap symbol); linear: unused
};

#define ANYSEQ_CUDA_CHECK(expr)                                                        \
    do {                                                                               \
        cudaError_t err__ = (expr);                                                    \
        if (err__ != cudaSuccess) {                                                    \
            std::fprintf(stderr, "anyseq_b200: CUDA error %s at %s:%d: %s\n",          \
                         cudaGetErrorName(err__), __FILE__, __LINE__,                  \
                         cudaGetErrorString(err__));                                   \
            return -(int)err__ - 1000;                                                 \
        }                                                                              \
    } while (0)

}  // namespace anyseq
