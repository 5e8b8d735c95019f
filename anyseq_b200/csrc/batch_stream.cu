// batch_stream.cu -- streaming front end of the batch path (SURVEY 8f.2).
//
// A stream owns a small ring of chunk slots.  Each slot has PINNED host buffers
// (packed queries / subjects, their offset arrays, the scores) and matching
// device buffers.  A producer thread fills a slot (parsing FASTA/FASTQ records
// straight into it, or copying from caller memory), submit() starts the H2D
// copies on the stream's own copy stream, and the consumer's collect() runs
// the batch kernel of that chunk on the engine's stream and brings the scores
// back.  Filling and copying chunk c+1 therefore overlap the kernel of chunk c;
// no slot is touched by two stages at once (free -> filling -> submitted ->
// done -> free).  The reference's reader offers the same producer/consumer
// split on the host (next()/skip() under a mutex, src/sequence_io.cpp:13-41);
// it has no batch path of its own.
#include "engine.cuh"

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <thread>
#include <vector>

namespace anyseq {

struct PinnedBuffer {
    void* ptr = nullptr;
    size_t bytes = 0;
    int ensure(size_t n)
    {
        if (n <= bytes) return 0;
        if (ptr) cudaFreeHost(ptr);
        ptr = nullptr;
        bytes = 0;
        if (cudaMallocHost(&ptr, n) != cudaSuccess) { cudaGetLastError(); return 1; }
        bytes = n;
        return 0;
    }
    void release()
    {
        if (ptr) cudaFreeHost(ptr);
        ptr = nullptr;
        bytes = 0;
    }
};

struct BatchSlot {
    enum State { kFree, kFilling, kSubmitted, kDone } state = kFree;
    PinnedBuffer hq, hs, hqo, hso, hscores;
    DeviceBuffer dq, ds, dqo, dso, dscores;
    cudaEvent_t ready = nullptr;     // H2D of this slot's chunk has finished
    int64_t npairs = 0;
    float kernel_ms = 0.f;
    int launches = 0;
};

class BatchStream {
public:
    BatchStream(Engine* eng, const anyseq_scoring& sc) : eng_(eng), sc_(sc) {}
    ~BatchStream() { destroy(); }

    // reuse of an idle stream (every slot free) for another batch: pinned allocations are expensive
    bool reusable(int64_t cap_pairs, int64_t cap_q, int64_t cap_s) const
    {
        return !slots_.empty() && !failed_ && cap_pairs <= cap_pairs_ && cap_q <= cap_q_ && cap_s <= cap_s_;
    }
    void restart(const anyseq_scoring& sc)
    {
        std::lock_guard<std::mutex> lk(mu_);
        sc_ = sc;
        order_.clear();
        for (BatchSlot& s : slots_) s.state = BatchSlot::kFree;
        finished_ = false;
        next_fill_ = 0;
        kernel_ms_ = 0.f;
        launches_ = 0;
        h2d_bytes_ = 0;
        d2h_bytes_ = 0;
    }

    int init(int64_t cap_pairs, int64_t cap_q, int64_t cap_s, int nslots)
    {
        cap_pairs_ = std::max<int64_t>(1, cap_pairs);
        cap_q_ = std::max<int64_t>(1, cap_q);
        cap_s_ = std::max<int64_t>(1, cap_s);
        ANYSEQ_CUDA_CHECK(cudaSetDevice(eng_->device));
        ANYSEQ_CUDA_CHECK(cudaStreamCreateWithFlags(&copy_stream_, cudaStreamNonBlocking));
        slots_.resize((size_t)std::max(2, std::min(nslots, 8)));
        const size_t no = sizeof(int64_t) * (size_t)(cap_pairs_ + 1), ns = sizeof(int32_t) * (size_t)cap_pairs_;
        for (BatchSlot& s : slots_) {
            if (s.hq.ensure((size_t)cap_q_) || s.hs.ensure((size_t)cap_s_) || s.hqo.ensure(no) || s.hso.ensure(no) ||
                s.hscores.ensure(ns)) {
                set_last_error("batch stream: out of pinned host memory");
                return ANYSEQ_ERR_NO_DEVICE;
            }
            if (s.dq.ensure((size_t)cap_q_ + 64) || s.ds.ensure((size_t)cap_s_ + 64) || s.dqo.ensure(no) || s.dso.ensure(no) ||
                s.dscores.ensure(ns))
                return ANYSEQ_ERR_NO_DEVICE;
            ANYSEQ_CUDA_CHECK(cudaEventCreateWithFlags(&s.ready, cudaEventDisableTiming));
        }
        return ANYSEQ_OK;
    }

    void destroy()
    {
        if (eng_ && eng_->device >= 0) cudaSetDevice(eng_->device);
        if (copy_stream_) cudaStreamSynchronize(copy_stream_);
        for (BatchSlot& s : slots_) {
            s.hq.release(); s.hs.release(); s.hqo.release(); s.hso.release(); s.hscores.release();
            s.dq.release(); s.ds.release(); s.dqo.release(); s.dso.release(); s.dscores.release();
            if (s.ready) cudaEventDestroy(s.ready);
            s.ready = nullptr;
        }
        slots_.clear();
        if (copy_stream_) cudaStreamDestroy(copy_stream_);
        copy_stream_ = nullptr;
    }

    // producer: a free slot to fill (blocks while every slot is in flight)
    int acquire(anyseq_batch_chunk* c)
    {
        std::unique_lock<std::mutex> lk(mu_);
        int idx = -1;
        cv_.wait(lk, [&] {
            for (size_t i = 0; i < slots_.size(); ++i) {
                const size_t k = (next_fill_ + i) % slots_.size();
                if (slots_[k].state == BatchSlot::kFree) { idx = (int)k; return true; }
            }
            return failed_;
        });
        if (failed_) return ANYSEQ_ERR_BAD_ARG;
        BatchSlot& s = slots_[(size_t)idx];
        s.state = BatchSlot::kFilling;
        next_fill_ = ((size_t)idx + 1) % slots_.size();
        std::memset(c, 0, sizeof(*c));
        c->queries = static_cast<char*>(s.hq.ptr);
        c->subjects = static_cast<char*>(s.hs.ptr);
        c->q_off = static_cast<int64_t*>(s.hqo.ptr);
        c->s_off = static_cast<int64_t*>(s.hso.ptr);
        c->cap_pairs = cap_pairs_;
        c->cap_query_bytes = cap_q_;
        c->cap_subject_bytes = cap_s_;
        c->slot = idx;
        return ANYSEQ_OK;
    }

    // producer: chunk is filled (npairs, offsets[0..npairs]); start its H2D copies
    int submit(const anyseq_batch_chunk* c)
    {
        if (!c || c->slot < 0 || c->slot >= (int)slots_.size()) { set_last_error("batch stream: bad chunk"); return ANYSEQ_ERR_BAD_ARG; }
        BatchSlot& s = slots_[(size_t)c->slot];
        const int64_t np = c->npairs;
        if (s.state != BatchSlot::kFilling || np < 0 || np > cap_pairs_ || (np > 0 && (c->q_off[0] != 0 || c->s_off[0] != 0)) ||
            (np > 0 && (c->q_off[np] > cap_q_ || c->s_off[np] > cap_s_))) {
            set_last_error("batch stream: chunk exceeds the slot capacity or was not acquired");
            fail();
            return ANYSEQ_ERR_BAD_ARG;
        }
        ANYSEQ_CUDA_CHECK(cudaSetDevice(eng_->device));
        s.npairs = np;
        if (np > 0) {
            const size_t no = sizeof(int64_t) * (size_t)(np + 1);
            ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(s.dq.ptr, s.hq.ptr, (size_t)c->q_off[np], cudaMemcpyHostToDevice, copy_stream_));
            ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(s.ds.ptr, s.hs.ptr, (size_t)c->s_off[np], cudaMemcpyHostToDevice, copy_stream_));
            ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(s.dqo.ptr, s.hqo.ptr, no, cudaMemcpyHostToDevice, copy_stream_));
            ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(s.dso.ptr, s.hso.ptr, no, cudaMemcpyHostToDevice, copy_stream_));
            h2d_bytes_ += (long long)c->q_off[np] + (long long)c->s_off[np] + 2 * (long long)no;
        }
        ANYSEQ_CUDA_CHECK(cudaEventRecord(s.ready, copy_stream_));
        {
            std::lock_guard<std::mutex> lk(mu_);
            s.state = BatchSlot::kSubmitted;
            order_.push_back(c->slot);
        }
        cv_.notify_all();
        return ANYSEQ_OK;
    }

    // producer: no more chunks will be submitted
    void finish()
    {
        { std::lock_guard<std::mutex> lk(mu_); finished_ = true; }
        cv_.notify_all();
    }

    // consumer: next chunk in submission order -> kernel + scores; ANYSEQ_EOF after finish()
    int collect(anyseq_batch_chunk* c)
    {
        int idx;
        {
            std::unique_lock<std::mutex> lk(mu_);
            cv_.wait(lk, [&] { return !order_.empty() || finished_ || failed_; });
            if (failed_) return ANYSEQ_ERR_BAD_ARG;
            if (order_.empty()) return ANYSEQ_EOF;
            idx = order_.front();
            order_.pop_front();
        }
        BatchSlot& s = slots_[(size_t)idx];
        ANYSEQ_CUDA_CHECK(cudaSetDevice(eng_->device));
        anyseq_result r;
        std::memset(&r, 0, sizeof(r));
        if (s.npairs > 0) {
            ANYSEQ_CUDA_CHECK(cudaStreamWaitEvent(eng_->stream(), s.ready, 0));
            int rc = eng_->score_batch_device(sc_, s.dq.as<uint8_t>(), s.dqo.as<int64_t>(), s.ds.as<uint8_t>(),
                                              s.dso.as<int64_t>(), s.npairs, s.dscores.as<int32_t>(), &r);
            if (rc) { fail(); return rc; }
            ANYSEQ_CUDA_CHECK(cudaMemcpyAsync(s.hscores.ptr, s.dscores.ptr, sizeof(int32_t) * (size_t)s.npairs,
                                              cudaMemcpyDeviceToHost, eng_->stream()));
            ANYSEQ_CUDA_CHECK(cudaStreamSynchronize(eng_->stream()));
            d2h_bytes_ += (long long)sizeof(int32_t) * s.npairs;
        }
        s.kernel_ms = r.kernel_ms;
        s.launches = r.kernel_launches;
        kernel_ms_ += r.kernel_ms;
        launches_ += r.kernel_launches;
        {
            std::lock_guard<std::mutex> lk(mu_);
            s.state = BatchSlot::kDone;
        }
        std::memset(c, 0, sizeof(*c));
        c->npairs = s.npairs;
        c->scores = static_cast<const int32_t*>(s.hscores.ptr);
        c->kernel_ms = s.kernel_ms;
        c->slot = idx;
        return ANYSEQ_OK;
    }

    // consumer: scores of the chunk have been used, its slot may be refilled
    int release(const anyseq_batch_chunk* c)
    {
        if (!c || c->slot < 0 || c->slot >= (int)slots_.size()) return ANYSEQ_ERR_BAD_ARG;
        {
            std::lock_guard<std::mutex> lk(mu_);
            if (slots_[(size_t)c->slot].state != BatchSlot::kDone) return ANYSEQ_ERR_BAD_ARG;
            slots_[(size_t)c->slot].state = BatchSlot::kFree;
        }
        cv_.notify_all();
        return ANYSEQ_OK;
    }

    void fail()
    {
        { std::lock_guard<std::mutex> lk(mu_); failed_ = true; }
        cv_.notify_all();
    }

    void stats(anyseq_result* out, long long* h2d, long long* d2h) const
    {
        if (out) { std::memset(out, 0, sizeof(*out)); out->end_i = out->end_j = -1; out->kernel_ms = kernel_ms_; out->kernel_launches = launches_; }
        if (h2d) *h2d = h2d_bytes_.load();
        if (d2h) *d2h = d2h_bytes_.load();
    }
    int64_t cap_pairs() const { return cap_pairs_; }
    int64_t cap_q() const { return cap_q_; }
    int64_t cap_s() const { return cap_s_; }

private:
    Engine* eng_;
    anyseq_scoring sc_;
    cudaStream_t copy_stream_ = nullptr;
    std::vector<BatchSlot> slots_;
    std::deque<int> order_;
    std::mutex mu_;
    std::condition_variable cv_;
    size_t next_fill_ = 0;
    bool finished_ = false, failed_ = false;
    int64_t cap_pairs_ = 0, cap_q_ = 0, cap_s_ = 0;
    float kernel_ms_ = 0.f;
    int launches_ = 0;
    std::atomic<long long> h2d_bytes_{0}, d2h_bytes_{0};      // producer / consumer threads
};

// ---------------------------------------------------------------------------
// anyseq_score_batch with host buffers = a stream whose producer copies ranges
// of the caller's (pageable) arrays into the pinned slots with a few threads.
// ---------------------------------------------------------------------------
static void parallel_copy(char* dst, const char* src, size_t n, int threads)
{
    if (n < (size_t)(4 << 20) || threads <= 1) { std::memcpy(dst, src, n); return; }
    std::vector<std::thread> th;
    const size_t per = (n + (size_t)threads - 1) / (size_t)threads;
    for (int t = 1; t < threads; ++t) {
        const size_t b = std::min(n, per * (size_t)t), e = std::min(n, b + per);
        if (e > b) th.emplace_back([=] { std::memcpy(dst + b, src + b, e - b); });
    }
    std::memcpy(dst, src, std::min(n, per));
    for (std::thread& x : th) x.join();
}

int Engine::score_batch_host(const anyseq_scoring& sc, const char* q, const int64_t* qoff, const char* s,
                             const int64_t* soff, int64_t npairs, int32_t* scores, anyseq_result* out)
{
    ScoreParams sp;
    bool affine;
    int rc = batch_prologue(sc, npairs, &sp, &affine, out);
    if (rc || npairs == 0) return rc;
    // chunk = up to 64 MiB of packed symbols; a single pair is at most ~2 GiB, far above any slot, so the
    // slot capacity follows the largest pair when one exceeds the default
    const int64_t total = (qoff[npairs] - qoff[0]) + (soff[npairs] - soff[0]);
    int64_t max_pair_q = 0, max_pair_s = 0;
    for (int64_t p = 0; p < npairs; ++p) {
        if (qoff[p + 1] < qoff[p] || soff[p + 1] < soff[p]) { set_last_error("batch offsets must be non-decreasing"); return ANYSEQ_ERR_BAD_ARG; }
        max_pair_q = std::max(max_pair_q, qoff[p + 1] - qoff[p]);
        max_pair_s = std::max(max_pair_s, soff[p + 1] - soff[p]);
    }
    const int64_t target = std::min<int64_t>(std::max<int64_t>(total / 2 + 1, 1 << 20), (int64_t)tune.batch_chunk_bytes);
    const double fq = total > 0 ? (double)(qoff[npairs] - qoff[0]) / (double)total : 0.5;
    const int64_t cap_q = std::max<int64_t>(max_pair_q, (int64_t)(target * fq) + 1) + 64;
    const int64_t cap_s = std::max<int64_t>(max_pair_s, (int64_t)(target * (1.0 - fq)) + 1) + 64;
    const int64_t cap_pairs = std::min<int64_t>(npairs, std::max<int64_t>(1, (int64_t)tune.batch_chunk_pairs));

    // one cached stream per engine: its pinned + device slots survive between calls
    std::lock_guard<std::recursive_mutex> lock(mu_);
    BatchStream* cached = static_cast<BatchStream*>(host_batch_stream_);
    if (cached && !cached->reusable(cap_pairs, cap_q, cap_s)) {
        delete cached;
        cached = nullptr;
        host_batch_stream_ = nullptr;
    }
    if (!cached) {
        cached = new BatchStream(this, sc);
        rc = cached->init(std::max<int64_t>(cap_pairs, std::min<int64_t>(tune.batch_chunk_pairs, 1 << 18)), cap_q, cap_s, 3);
        if (rc) { delete cached; return rc; }
        host_batch_stream_ = cached;
    }
    cached->restart(sc);
    BatchStream& st = *cached;
    // chunk limits of THIS call (the cached stream's slots may be larger)
    const int64_t chunk_pairs = cap_pairs, chunk_q = cap_q, chunk_s = cap_s;
    const int copy_threads = std::max(1, std::min(tune.batch_copy_threads, (int)std::thread::hardware_concurrency()));
    int producer_rc = ANYSEQ_OK;
    std::thread producer([&] {
        int64_t p = 0;
        while (p < npairs) {
            anyseq_batch_chunk c;
            if ((producer_rc = st.acquire(&c)) != ANYSEQ_OK) break;
            int64_t e = p;
            while (e < npairs && e - p < chunk_pairs && qoff[e + 1] - qoff[p] <= chunk_q && soff[e + 1] - soff[p] <= chunk_s) ++e;
            const int64_t np = e - p;
            for (int64_t i = 0; i <= np; ++i) { c.q_off[i] = qoff[p + i] - qoff[p]; c.s_off[i] = soff[p + i] - soff[p]; }
            parallel_copy(c.queries, q + qoff[p], (size_t)(qoff[e] - qoff[p]), copy_threads);
            parallel_copy(c.subjects, s + soff[p], (size_t)(soff[e] - soff[p]), copy_threads);
            c.npairs = np;
            if ((producer_rc = st.submit(&c)) != ANYSEQ_OK) break;
            p = e;
        }
        st.finish();
        if (producer_rc != ANYSEQ_OK) st.fail();
    });
    int64_t done = 0;
    int crc = ANYSEQ_OK;
    for (;;) {
        anyseq_batch_chunk c;
        crc = st.collect(&c);
        if (crc != ANYSEQ_OK) break;
        std::memcpy(scores + done, c.scores, sizeof(int32_t) * (size_t)c.npairs);
        done += c.npairs;
        st.release(&c);
    }
    if (crc != ANYSEQ_EOF) st.fail();
    producer.join();
    if (crc != ANYSEQ_EOF || producer_rc != ANYSEQ_OK) {     // do not reuse a stream that failed
        delete cached;
        host_batch_stream_ = nullptr;
    }
    if (crc != ANYSEQ_EOF) return crc;
    if (producer_rc != ANYSEQ_OK) return producer_rc;
    if (done != npairs) { set_last_error("batch stream lost pairs"); return ANYSEQ_ERR_BAD_ARG; }
    st.stats(out, nullptr, nullptr);
    return ANYSEQ_OK;
}

void Engine::drop_host_batch_stream()
{
    delete static_cast<BatchStream*>(host_batch_stream_);
    host_batch_stream_ = nullptr;
}

}  // namespace anyseq

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
struct anyseq_batch_stream {
    anyseq::BatchStream* impl;
};

extern "C" {

int anyseq_batch_stream_open(anyseq_ctx* ctx, const anyseq_scoring* sc, int64_t cap_pairs, int64_t cap_query_bytes,
                             int64_t cap_subject_bytes, int slots, anyseq_batch_stream** out)
{
    if (!ctx || !sc || !out || cap_pairs < 1 || cap_query_bytes < 1 || cap_subject_bytes < 1) {
        anyseq::set_last_error("batch stream: bad arguments");
        return ANYSEQ_ERR_BAD_ARG;
    }
    *out = nullptr;
    anyseq::ScoreParams sp;
    bool affine;
    int rc = anyseq::make_score_params(*sc, &sp, &affine);
    if (rc) return rc;
    anyseq::BatchStream* impl = new anyseq::BatchStream(&ctx->eng, *sc);
    rc = impl->init(cap_pairs, cap_query_bytes, cap_subject_bytes, slots <= 0 ? 3 : slots);
    if (rc) { delete impl; return rc; }
    *out = new anyseq_batch_stream{impl};
    return ANYSEQ_OK;
}

int anyseq_batch_stream_acquire(anyseq_batch_stream* st, anyseq_batch_chunk* chunk)
{
    if (!st || !chunk) return ANYSEQ_ERR_BAD_ARG;
    return st->impl->acquire(chunk);
}

int anyseq_batch_stream_submit(anyseq_batch_stream* st, const anyseq_batch_chunk* chunk)
{
    if (!st || !chunk) return ANYSEQ_ERR_BAD_ARG;
    return st->impl->submit(chunk);
}

int anyseq_batch_stream_finish(anyseq_batch_stream* st)
{
    if (!st) return ANYSEQ_ERR_BAD_ARG;
    st->impl->finish();
    return ANYSEQ_OK;
}

int anyseq_batch_stream_collect(anyseq_batch_stream* st, anyseq_batch_chunk* chunk)
{
    if (!st || !chunk) return ANYSEQ_ERR_BAD_ARG;
    return st->impl->collect(chunk);
}

int anyseq_batch_stream_release(anyseq_batch_stream* st, const anyseq_batch_chunk* chunk)
{
    if (!st || !chunk) return ANYSEQ_ERR_BAD_ARG;
    return st->impl->release(chunk);
}

int anyseq_batch_stream_stats(anyseq_batch_stream* st, anyseq_result* out, int64_t* h2d_bytes, int64_t* d2h_bytes)
{
    if (!st) return ANYSEQ_ERR_BAD_ARG;
    long long a = 0, b = 0;
    st->impl->stats(out, &a, &b);
    if (h2d_bytes) *h2d_bytes = a;
    if (d2h_bytes) *d2h_bytes = b;
    return ANYSEQ_OK;
}

void anyseq_batch_stream_close(anyseq_batch_stream* st)
{
    if (!st) return;
    delete st->impl;
    delete st;
}

}  // extern "C"
