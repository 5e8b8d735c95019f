// batch_packed2.cu -- batches of short pairs whose sequences arrive 2-bit packed (four DNA symbols per byte).
//
// BASELINE.json configs[3] (10^7 reads of 150 bp vs 500 bp windows) is bound by the host->device copy when every
// symbol travels as a byte (round 1: 2.38 TCUPS end to end vs 3.74 in the kernel).  Packed input is a quarter of
// the bytes, needs no alphabet analysis (codes are value + 1, code 0 = "matches nothing" for padded columns) and the
// batch kernels unpack it while they build their per-lane column masks (batch.cuh: batch_code).  The reference
// stages sequences one byte per symbol (sequence_to_device, src/mapping_acc.impala:125-131); comparison is by value
// (src/align.impala:132), so the scores are those of the unpacked sequences.
//
// Host variant: the caller's (ideally pinned) arrays are copied chunk by chunk on a copy stream into one of two
// device slots while the previous chunk is relaxed on the compute stream -- no staging memcpy, no helper threads.
#include "engine.cuh"
#include "batch.cuh"

#include <algorithm>
#include <cstring>

namespace anyseq {

// the caller's description of a 2-bit batch and its score array
static int check_packed_batch(const anyseq_packed_batch& b, const int32_t* scores)
{
    if (b.npairs < 0 || (b.npairs > 0 && (!b.q2 || !b.s2))) { set_last_error("packed batch: null sequence arrays"); return ANYSEQ_ERR_BAD_ARG; }
    if ((!b.q_len && b.q_len_uniform < 0) || (!b.s_len && b.s_len_uniform < 0)) { set_last_error("packed batch: negative length"); return ANYSEQ_ERR_BAD_ARG; }
    if ((!b.q_boff && b.q_stride < (b.q_len ? 0 : (b.q_len_uniform + 3) / 4)) ||
        (!b.s_boff && b.s_stride < (b.s_len ? 0 : (b.s_len_uniform + 3) / 4))) {
        set_last_error("packed batch: stride shorter than a packed sequence");
        return ANYSEQ_ERR_BAD_ARG;
    }
    if (b.npairs > 0 && !scores) { set_last_error("packed batch: null score array"); return ANYSEQ_ERR_BAD_ARG; }
    return ANYSEQ_OK;
}

int Engine::use_2bit_alphabet()
{
    use_mask_ = true;
    ncodes_ = 5;
    return lut_.ensure(512 + 64 + 16) ? ANYSEQ_ERR_NO_DEVICE : ANYSEQ_OK;
}

static void fill_args(BatchArgs& ba, const anyseq_packed_batch& b, int32_t* d_scores)
{
    std::memset(&ba, 0, sizeof(ba));
    ba.q = b.q2;
    ba.s = b.s2;
    ba.qoff = reinterpret_cast<const long long*>(b.q_boff);
    ba.soff = reinterpret_cast<const long long*>(b.s_boff);
    ba.qlen = b.q_len;
    ba.slen = b.s_len;
    ba.qlen_u = b.q_len_uniform;
    ba.slen_u = b.s_len_uniform;
    ba.qstride = b.q_stride;
    ba.sstride = b.s_stride;
    ba.packed2 = 1;
    ba.npairs = b.npairs;
    ba.scores = d_scores;
}

int Engine::score_batch_packed2_device(const anyseq_scoring& sc, const anyseq_packed_batch& b, int32_t* d_scores,
                                       anyseq_result* out)
{
    std::lock_guard<std::recursive_mutex> lock(mu_);
    ANYSEQ_CUDA_CHECK(cudaSetDevice(device));
    ScoreParams sp;
    bool affine;
    int rc = check_packed_batch(b, d_scores);
    if (rc) return rc;
    rc = batch_prologue(sc, b.npairs, &sp, &affine, out);
    if (rc || b.npairs == 0) return rc;
    ANYSEQ_CUDA_CHECK(cudaEventRecord(ev0_, stream_));
    BatchArgs ba;
    fill_args(ba, b, d_scores);
    int max_long = std::max(b.q_len_uniform, b.s_len_uniform), max_short = std::min(b.q_len_uniform, b.s_len_uniform);
    int launches = 1;
    if (b.q_len || b.s_len) {
        if ((rc = batch_len_stats(ba, &max_long, &max_short))) return rc;
        launches += 1;
    }
    if ((rc = use_2bit_alphabet())) return rc;
    if ((rc = launch_batch(sc, sp, affine, ba, max_long, max_short, stream_))) return rc;
    return batch_epilogue(launches, out);
}

int Engine::score_batch_packed2_host(const anyseq_scoring& sc, const anyseq_packed_batch& b, int32_t* scores,
                                     anyseq_result* out)
{
    std::lock_guard<std::recursive_mutex> lock(mu_);
    ANYSEQ_CUDA_CHECK(cudaSetDevice(device));
    ScoreParams sp;
    bool affine;
    int rc = check_packed_batch(b, scores);
    if (rc) return rc;
    const int64_t np = b.npairs;
    rc = batch_prologue(sc, np, &sp, &affine, out);
    if (rc || np == 0) return rc;
    // length statistics + byte extent of every sequence array (host pass over the metadata only)
    auto qlen = [&](int64_t p) { return b.q_len ? b.q_len[p] : b.q_len_uniform; };
    auto slen = [&](int64_t p) { return b.s_len ? b.s_len[p] : b.s_len_uniform; };
    auto qbeg = [&](int64_t p) { return b.q_boff ? b.q_boff[p] : p * b.q_stride; };
    auto sbeg = [&](int64_t p) { return b.s_boff ? b.s_boff[p] : p * b.s_stride; };
    int max_long = 0, max_short = 0;
    if (!b.q_len && !b.s_len) {
        max_long = std::max(b.q_len_uniform, b.s_len_uniform);
        max_short = std::min(b.q_len_uniform, b.s_len_uniform);
    } else {
        for (int64_t p = 0; p < np; ++p) {
            const int a = qlen(p), c = slen(p);
            if (a < 0 || c < 0) { set_last_error("packed batch: negative length"); return ANYSEQ_ERR_BAD_ARG; }
            max_long = std::max(max_long, std::max(a, c));
            max_short = std::max(max_short, std::min(a, c));
        }
    }
    if (b.q_boff || b.s_boff) {
        for (int64_t p = 0; p + 1 < np; ++p) {
            if ((b.q_boff && b.q_boff[p + 1] < b.q_boff[p]) || (b.s_boff && b.s_boff[p + 1] < b.s_boff[p])) {
                set_last_error("packed batch: byte offsets must be non-decreasing");
                return ANYSEQ_ERR_BAD_ARG;
            }
        }
    }
    if ((rc = use_2bit_alphabet())) return rc;
    if (!copy_stream_) {
        ANYSEQ_CUDA_CHECK(cudaStreamCreateWithFlags(&copy_stream_, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            ANYSEQ_CUDA_CHECK(cudaEventCreateWithFlags(&p2_ready_[i], cudaEventDisableTiming));
            ANYSEQ_CUDA_CHECK(cudaEventCreateWithFlags(&p2_done_[i], cudaEventDisableTiming));
        }
    }
    // chunks of pairs: a chunk's sequences are contiguous byte ranges of the caller's arrays (offsets are monotone)
    const int64_t chunk_pairs = std::max<int64_t>(1024, std::min<int64_t>(tune.batch_chunk_pairs, (np + 3) / 4));
    auto align16 = [](size_t x) { return (x + 255) / 256 * 256; };
    auto q_end = [&](int64_t p) { return qbeg(p) + (qlen(p) + 3) / 4; };     // exclusive byte end of sequence p
    auto s_end = [&](int64_t p) { return sbeg(p) + (slen(p) + 3) / 4; };
    size_t slot_bytes = 0;
    for (int64_t p0 = 0; p0 < np; p0 += chunk_pairs) {
        const int64_t p1 = std::min(np, p0 + chunk_pairs), n = p1 - p0;
        const size_t need = align16((size_t)(q_end(p1 - 1) - qbeg(p0))) + align16((size_t)(s_end(p1 - 1) - sbeg(p0))) +
                            align16(sizeof(int32_t) * (size_t)n) +
                            (b.q_boff ? align16(sizeof(int64_t) * (size_t)n) : 0) + (b.s_boff ? align16(sizeof(int64_t) * (size_t)n) : 0) +
                            (b.q_len ? align16(sizeof(int32_t) * (size_t)n) : 0) + (b.s_len ? align16(sizeof(int32_t) * (size_t)n) : 0);
        slot_bytes = std::max(slot_bytes, need);
    }
    if (p2_[0].ensure(slot_bytes + 1024) || p2_[1].ensure(slot_bytes + 1024)) return ANYSEQ_ERR_NO_DEVICE;

    ANYSEQ_CUDA_CHECK(cudaEventRecord(ev0_, stream_));
    int launches = 0;
    int64_t h2d = 0;
    int c = 0;
    for (int64_t p0 = 0; p0 < np; p0 += chunk_pairs, ++c) {
        const int64_t p1 = std::min(np, p0 + chunk_pairs), n = p1 - p0;
        const int slot = c & 1;
        uint8_t* base = p2_[slot].as<uint8_t>();
        // the slot is free once the kernel AND the score copy of the chunk two steps back have finished
        if (c >= 2) ANYSEQ_CUDA_CHECK(cudaStreamWaitEvent(copy_stream_, p2_done_[slot], 0));
        const int64_t qb0 = qbeg(p0), sb0 = sbeg(p0);
        const size_t qbytes = (size_t)(q_end(p1 - 1) - qb0), sbytes = (size_t)(s_end(p1 - 1) - sb0);
        size_t off = 0;
        uint8_t* d_q = base + off; off += align16(qbytes);
        uint8_t* d_s = base + off; off += align16(sbytes);
        int32_t* d_sc = reinterpret_cast<int32_t*>(base + off); off += align16(sizeof(int32_t) * (size_t)n);
        ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(d_q, b.q2 + qb0, qbytes, cudaMemcpyHostToDevice, copy_stream_));
        ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(d_s, b.s2 + sb0, sbytes, cudaMemcpyHostToDevice, copy_stream_));
        h2d += (int64_t)(qbytes + sbytes);
        anyseq_packed_batch d = b;
        d.npairs = n;
        // the kernels index with the caller's ABSOLUTE byte offsets: shift the base pointers instead of the offsets
        d.q2 = d_q - (b.q_boff ? qb0 : 0);
        d.s2 = d_s - (b.s_boff ? sb0 : 0);
        auto up = [&](const void* src, size_t bytes) -> void* {
            void* dst = base + off;
            off += align16(bytes);
            cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, copy_stream_);
            h2d += (int64_t)bytes;
            return dst;
        };
        if (b.q_boff) d.q_boff = static_cast<const int64_t*>(up(b.q_boff + p0, sizeof(int64_t) * (size_t)n));
        if (b.s_boff) d.s_boff = static_cast<const int64_t*>(up(b.s_boff + p0, sizeof(int64_t) * (size_t)n));
        if (b.q_len) d.q_len = static_cast<const int32_t*>(up(b.q_len + p0, sizeof(int32_t) * (size_t)n));
        if (b.s_len) d.s_len = static_cast<const int32_t*>(up(b.s_len + p0, sizeof(int32_t) * (size_t)n));
        ANYSEQ_CUDA_CHECK(cudaGetLastError());
        ANYSEQ_CUDA_CHECK(cudaEventRecord(p2_ready_[slot], copy_stream_));
        ANYSEQ_CUDA_CHECK(cudaStreamWaitEvent(stream_, p2_ready_[slot], 0));
        BatchArgs ba;
        fill_args(ba, d, d_sc);
        rc = launch_batch(sc, sp, affine, ba, max_long, max_short, stream_);
        if (rc) { cudaStreamSynchronize(copy_stream_); cudaStreamSynchronize(stream_); return rc; }
        ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(scores + p0, d_sc, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, stream_));
        ANYSEQ_CUDA_CHECK(cudaEventRecord(p2_done_[slot], stream_));
        launches += 1;
    }
    rc = batch_epilogue(launches, out);
    ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(copy_stream_));
    return rc;
}

}  // namespace anyseq

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
extern "C" {


int anyseq_score_batch_packed2(anyseq_ctx* ctx, const anyseq_scoring* sc, const anyseq_packed_batch* host_batch,
                               int32_t* scores, anyseq_result* out)
{
    if (!ctx || !sc || !host_batch) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.score_batch_packed2_host(*sc, *host_batch, scores, out);
}


int anyseq_score_batch_packed2_device(anyseq_ctx* ctx, const anyseq_scoring* sc, const anyseq_packed_batch* device_batch,
                                      int32_t* d_scores, anyseq_result* out)
{
    if (!ctx || !sc || !device_batch) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.score_batch_packed2_device(*sc, *device_batch, d_scores, out);
}


int64_t anyseq_pack2(const char* seq, int64_t n, uint8_t* out)
{
    int64_t bad = 0;
    for (int64_t i = 0; i < n; i += 4) {
        unsigned v = 0;
        for (int k = 0; k < 4 && i + k < n; ++k) {
            unsigned code = 0;
            switch (seq[i + k]) {
                case 'A': case 'a': code = 0; break;
                case 'C': case 'c': code = 1; break;
                case 'G': case 'g': code = 2; break;
                case 'T': case 't': code = 3; break;
                default: ++bad; break;
            }
            v |= code << (2 * k);
        }
        out[i >> 2] = (uint8_t)v;
    }
    return bad;
}

}  // extern "C"
