// batch.cuh -- argument block and device helpers shared by the batch kernels (batch.cu, batch_x2.cu)
#pragma once
#include "common.cuh"

namespace anyseq {

struct BatchArgs {
    const uint8_t* q;
    const long long* qoff;
    const uint8_t* s;
    const long long* soff;
    long long npairs;
    int* scores;
    ScoreParams sp;
    int gap_init;
    int mode;
    int one;
    int ncodes;
    int cols_longer;               // 1: columns = longer sequence of a pair, 0: shorter
    const uint8_t* lut;            // byte -> code (shared by both sequences)
    unsigned long long* counter;   // next pair (packed kernels: pair of pairs) to claim
    int bias;                      // packed 16-bit kernels: offset that keeps every stored value non-negative
    // 2-bit packed DNA input (anyseq_score_batch_packed2): four symbols per byte, least significant bits first, every
    // sequence starting on a byte boundary.  q / s then hold packed bytes, qoff / soff BYTE offsets of the sequences
    // (nullptr: sequence p starts at p * stride) and the lengths come from qlen / slen (nullptr: uniform length).
    int packed2;
    const int* qlen;
    const int* slen;
    int qlen_u, slen_u;
    long long qstride, sstride;
};

// where pair p's sequences start (symbol offset, or byte offset for 2-bit input) and how many symbols they have
__device__ __forceinline__ long long batch_q_start(const BatchArgs& a, long long p) { return a.qoff ? a.qoff[p] : p * a.qstride; }
__device__ __forceinline__ long long batch_s_start(const BatchArgs& a, long long p) { return a.soff ? a.soff[p] : p * a.sstride; }
// 64-bit so that the length statistics see a pair of 2^31 or more symbols as too long; the kernels take it as int
__device__ __forceinline__ long long batch_q_len(const BatchArgs& a, long long p)
{
    return a.packed2 ? (a.qlen ? a.qlen[p] : a.qlen_u) : a.qoff[p + 1] - a.qoff[p];
}
__device__ __forceinline__ long long batch_s_len(const BatchArgs& a, long long p)
{
    return a.packed2 ? (a.slen ? a.slen[p] : a.slen_u) : a.soff[p + 1] - a.soff[p];
}
// alphabet code of symbol idx of a sequence: byte -> code table, or the 2-bit value + 1 (code 0 matches nothing)
__device__ __forceinline__ int batch_code(const uint8_t* __restrict__ base, int idx, int packed2, const uint8_t* lut)
{
    if (packed2) return (int)((base[idx >> 2] >> (2 * (idx & 3))) & 3u) + 1;
    return (int)lut[base[idx]];
}

// score of a pair with an empty sequence, following the reference's storage (quirk Q12, see engine.cu: empty_result)
template <int MODE>
__device__ __forceinline__ int empty_pair_score(const BatchArgs& a, int lq, int ls)
{
    const int L = max(lq, ls);
    return MODE == kGlobal ? (L > 0 ? a.gap_init + L * a.sp.gap_extend : 0) : (MODE == kSemiglobal ? 0 : kScoreMin);
}

// value of X[idx] for a run-time idx (one lane needs it; jump table, not K selects)
template <typename T, int K>
__device__ __forceinline__ T pick_column(const T (&X)[K], int idx)
{
    T v = X[0];
#pragma unroll
    for (int c = 1; c < K; ++c)
        if (c == idx) v = X[c];
    return v;
}

using BatchKernelFn = void (*)(const BatchArgs);
// packed 16-bit kernels (batch_x2.cu): two pairs per group of `lanes` lanes (32: K = 4, 8, 16, 32; 16: K = 32, four
// pairs per warp); nullptr for other combinations
BatchKernelFn pick_batch_x2_kernel(int mode, bool affine, int K, int lanes);

}  // namespace anyseq
