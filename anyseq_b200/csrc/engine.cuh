// engine.cuh -- host-side engine: workspace, job construction, launches.
#pragma once

#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"
#include "../../include/anyseq.h"

namespace anyseq {

struct BatchArgs;   // batch.cuh

// grow-only device allocation
struct DeviceBuffer {
    void* ptr = nullptr;
    size_t bytes = 0;
    int ensure(size_t need)
    {
        if (need <= bytes) return 0;
        if (ptr) ANYSEQ_CUDA_CHECK(cudaFree(ptr));
        ptr = nullptr;
        bytes = 0;
        size_t cap = need + need / 8 + 256;
        ANYSEQ_CUDA_CHECK(cudaMalloc(&ptr, cap));
        bytes = cap;
        return 0;
    }
    void release()
    {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(ptr); }
};

struct Tuning {
    int cols_per_lane = 0;   // K, 0 = auto
    int band_rows = 0;       // 0 = auto
    int blocks_per_sm = 0;   // 0 = occupancy maximum
    int watchdog_ms = 20000;
    int cell_form = -1;      // -1 = per launch (engine.cu: pick_form), 1 = decoupled, 2 = mixed cells
    int packed_cells = -1;   // -1 / 1 = packed cells where the score window fits (engine.cu: packed_fits), 0 = never
    int band_slack = 2;      // band height = band_slack * lag * (resident warps) when the strips outnumber the warps
    bool force_generic = false;     // never use the MASK kernels (testing)
    bool force_affine = false;      // score path: run the Gotoh kernels even for gap_init == 0 (testing: must equal the linear kernels)
    bool local_end_cell = false;    // local scores also report the reference's end cell (single-row kernels)
    bool align_with_score = true;   // anyseq_align also computes the optimal score (one more m*n pass)
    bool small_model = true;        // small problems: strip width from the measured critical-path fit (engine.cu: pick_K)
    int batch_chunk_bytes = 64 << 20;    // host batches: packed symbols per pipeline chunk
    int batch_chunk_pairs = 1 << 18;     // host batches: pairs per pipeline chunk
    bool batch_quad = true;              // packed batches with columns <= 512: four pairs per warp (half-warps)
    bool batch_packed = true;            // batches: two pairs per warp in 16-bit halves when the scores fit
    int batch_copy_threads = 4;          // host batches: threads staging caller memory into pinned slots
};

// word layout of the small device "misc" block
enum MiscWord : int {
    kMiscStatus = 0,     // 4 words
    kMiscBest = 4,       // local running maximum
    kMiscOut = 8,        // 8 words: finish kernel output
    kMiscCounter = 16,   // 2 words (8-byte aligned): work-item counter of the strip kernel
    kMiscWords = 40
};

struct Inbox {            // left-border mailbox of a rank (multi-GPU wavefront): one 16-byte record per row
    int4* records = nullptr;
    int rows = 0;
    bool owned = false;   // false: opened from a peer's IPC handle
    int uses_in = 0;      // runs that consumed from it (this process)
    int uses_out = 0;     // runs that produced into it (this process)
    static size_t bytes_for(int rows) { return sizeof(int4) * (size_t)rows + 256; }
};

// Multi-GPU linear-space traceback (one process per GPU, SURVEY 8e row 3): the halves of a Hirschberg level are
// independent DP problems (iteration_partitioned, src/iteration_cpu.impala:59-119), so they are dealt out to the ranks:
// half h of a level with P parts belongs to rank h / (2P / world) once 2P >= world (a rank then owns whole parts and
// needs nothing from anybody), and to rank h * (world / 2P) on the first log2(world) levels, where the two halves of a
// part sit on different ranks and their last-column records are broadcast before hb_sum
// (src/traceback_lintime.impala:44-135) runs on every rank.  Every rank finally emits the 128-column blocks of its parts.
struct TracebackShard {
    int rank = 0, world = 1;
    anyseq_bcast_fn bcast = nullptr;   // broadcast of a device buffer from src_rank to all ranks (caller: NCCL)
    void* user = nullptr;
    long long out_lo = 0, out_hi = 0;  // [out] index range of the output strings this rank produced
};

class Engine {
public:
    int init(int device);
    void destroy();

    int score_device(const anyseq_scoring& sc, const uint8_t* d_q, int m, const uint8_t* d_s, int n,
                     anyseq_result* out);
    int score_host(const anyseq_scoring& sc, const char* q, int m, const char* s, int n,
                   anyseq_result* out);
    int score_strip_device(const anyseq_scoring& sc, const uint8_t* d_q, int m,
                           const uint8_t* d_s_slice, int col_begin, int col_end, int n_total,
                           Inbox* inbox, Inbox* next_inbox, anyseq_strip_partial* out);
    int score_strip_host(const anyseq_scoring& sc, const char* q, int m, const char* s_slice, int col_begin, int col_end,
                         int n_total, Inbox* inbox, Inbox* next_inbox, anyseq_strip_partial* out);
    // several pairs of the SAME shape (lenq, slice) in one launch, their items interleaved band by band: a narrow
    // multi-GPU slice has too few strips to fill the SMs, two of them side by side do (engine.cu)
    int score_strip_device_multi(const anyseq_scoring& sc, int npairs, const uint8_t* const* d_q, int m,
                                 const uint8_t* const* d_s_slice, int col_begin, int col_end, int n_total,
                                 Inbox* const* inbox, Inbox* const* next_inbox, anyseq_strip_partial* out);
    int align_host(const anyseq_scoring& sc, const char* q, int m, const char* s, int n,
                   char* alq, char* als, anyseq_result* out);
    // this rank's share of a traceback spread over `shard.world` GPUs (traceback.cu); alq/als are full-size buffers of
    // which only [shard.out_lo, shard.out_hi) is meaningful afterwards
    int align_host_sharded(const anyseq_scoring& sc, const char* q, int m, const char* s, int n,
                           char* alq, char* als, anyseq_result* out, TracebackShard* shard);
    // full-matrix traceback (traceback_full.cu); start2 = get_alignment_start()
    int align_full_host(const anyseq_scoring& sc, const char* q, int m, const char* s, int n,
                        char* alq, char* als, anyseq_result* out, int* start2);
    int score_batch_device(const anyseq_scoring& sc, const uint8_t* d_q, const int64_t* d_qoff,
                           const uint8_t* d_s, const int64_t* d_soff, int64_t npairs,
                           int32_t* d_scores, anyseq_result* out);
    int score_batch_host(const anyseq_scoring& sc, const char* q, const int64_t* qoff,
                         const char* s, const int64_t* soff, int64_t npairs, int32_t* scores,
                         anyseq_result* out);
    // full-matrix tracebacks of a batch of pairs with subjects of at most 1024 symbols (batch_align.cu): per pair what
    // align_full_host gives; ends / starts may be null
    int align_batch_device(const anyseq_scoring& sc, const uint8_t* d_q, const int64_t* d_qoff, const uint8_t* d_s,
                           const int64_t* d_soff, int64_t npairs, int32_t* d_scores, int32_t* d_ends, int32_t* d_starts,
                           char* d_alq, char* d_als, anyseq_result* out);
    int align_batch_host(const anyseq_scoring& sc, const char* q, const int64_t* qoff, const char* s, const int64_t* soff,
                         int64_t npairs, int32_t* scores, int32_t* ends, int32_t* starts, char* alq, char* als,
                         anyseq_result* out);
    // 2-bit packed DNA batches (batch_packed2.cu)
    int score_batch_packed2_device(const anyseq_scoring& sc, const anyseq_packed_batch& b, int32_t* d_scores,
                                   anyseq_result* out);
    int score_batch_packed2_host(const anyseq_scoring& sc, const anyseq_packed_batch& b, int32_t* scores,
                                 anyseq_result* out);
    int measure_int_peak(int kind, double* ops_per_s, float* sm_mhz);
    // launch planning without a device (engine.cu); usable on an Engine that was never init()ed
    int plan_launch(int sms, int mode, bool affine, int m, int n, bool chained, const ScoreParams& sp,
                    anyseq_launch_plan* out);

    int inbox_create(int rows, Inbox** out, void* handle64);
    int inbox_open(const void* handle64, int rows, Inbox** out);
    int inbox_reset(Inbox* box);
    void inbox_destroy(Inbox* box);

    Tuning tune;
    const std::vector<int>& last_splits() const { return last_splits_; }
    const std::vector<int>& last_types() const { return last_types_; }
    const int* last_start() const { return last_start_; }
    int device = -1;
    int sm_count = 0;
    char name[64] = {0};
    int resident_warps(int K, bool local, bool affine, long long nstrips = 1LL << 40);
    cudaStream_t stream() const { return stream_; }
    void drop_host_batch_stream();       // batch_stream.cu: the cached pipeline of score_batch_host

private:
    int run_jobs(std::vector<Job>& jobs, const ScoreParams& sp, bool local, bool affine, int K, int* launches,
                 bool packed_ok = false);
    int pick_K(int n, bool chained = false, int m = 0, bool affine = false) const;
    int pick_K_levels(int n_total) const;
    int analyse_alphabet(const uint8_t* d_q, long long m, const uint8_t* d_s, long long n);
    int analyse_alphabet_host(const uint8_t* q, long long m, const uint8_t* s, long long n);
    int plan_bands(int max_h, long long strips_total, int resident, int K, bool chained) const;
    int balance_warps(int nb, int max_h, long long strips_total, int K, bool chained) const;
    int launch_batch(const anyseq_scoring& sc, const ScoreParams& sp, bool affine, BatchArgs& ba, int max_long,
                     int max_short, cudaStream_t st);
    // batch.cu: max over pairs of the longer and of the shorter length, optionally of the query and of the subject
    // length and whether some pair has a negative length (synchronises stream_)
    int batch_len_stats(const BatchArgs& ba, int* max_long, int* max_short, int* max_q = nullptr, int* max_s = nullptr,
                        bool* negative = nullptr);
    // batch.cu: ends a timed batch call on stream_ (ev0_ .. ev1_) and reports the time and launch count in *out
    int batch_epilogue(int launches, anyseq_result* out);
    // batch_packed2.cu: 2-bit input has codes 1..4 (0 matches nothing) and always runs the column-mask kernels
    int use_2bit_alphabet();

    cudaStream_t stream_ = nullptr;
    cudaEvent_t ev0_ = nullptr, ev1_ = nullptr;
    DeviceBuffer seq_q_, seq_s_, seq_qr_, seq_sr_;
    DeviceBuffer col_, rowH_, rowF_, corner_, progress_, jobs_, misc_;
    DeviceBuffer lut_;                // byte -> code tables of the MASK kernels + presence bits
    DeviceBuffer col2_;               // second column-record set (Hirschberg right halves)
    DeviceBuffer aux_, aux2_, pred_;  // traceback scratch
    DeviceBuffer tb_out_;             // linear-space traceback: the two output rows on the device
    DeviceBuffer multi_;         // score_strip_device_multi: per-pair border/row/corner/progress/result storage
    DeviceBuffer edges_;         // full-matrix traceback: right edge column (H, E) of every 128-column strip
    DeviceBuffer blockmax_;      // local end-cell tracking: one key per 1024 x 1024 reference block
    DeviceBuffer p2_[2];         // packed2 host pipeline: two device chunk slots
    DeviceBuffer batch_pred_;    // batch tracebacks: one predecessor slab per resident warp
    DeviceBuffer batch_io_;      // batch tracebacks from host memory: inputs and outputs on the device
    cudaStream_t copy_stream_ = nullptr;                     // packed2 host pipeline: H2D of chunk c+1 under the kernel of chunk c
    cudaEvent_t p2_ready_[2] = {nullptr, nullptr}, p2_done_[2] = {nullptr, nullptr};
    int* h_misc_ = nullptr;           // pinned mirror of misc_
    std::vector<int> strip2job_;      // run_jobs: launch-wide strip index -> job
    std::vector<int> last_splits_;    // split rows of the last traceback (slot -1 first)
    std::vector<int> last_types_;     // Gotoh traceback: vertex types of the split rows (0 = H, 1 = E)
    int ncodes_ = 1;                  // alphabet codes of the current pair (MASK kernels)
    bool use_mask_ = false;
    bool alphabet_ready_ = false;     // the tables of the pair about to be relaxed were built on the host
    static constexpr long long kHostAlphabetLimit = 8 << 20;     // host-side alphabet pass up to this many symbols
    void* host_batch_stream_ = nullptr;  // BatchStream* reused by score_batch_host
    bool want_edges_ = false;    // the running score call keeps the strips' edge columns (K = 4)
    bool force_track_ = false;   // ... and tracks the local end cell whatever the option says
    int last_start_[2] = {0, 0}; // get_alignment_start() of the last full-matrix traceback
    bool track_ = false;         // the running score call tracks the local end cell
    int init_col0_ = 0;               // absolute column of the job's first column (multi-GPU)
    TracebackShard* shard_ = nullptr; // set while align_host_sharded runs
    std::recursive_mutex mu_;
};

void set_last_error(const std::string& s);
int make_score_params(const anyseq_scoring& sc, ScoreParams* sp, bool* affine);
// batch.cu: the checks every batch entry point starts with -- the scheme, a cleared *out, and local alignment with
// diff > 0 refused for a non-empty batch (padded columns must not outscore real ones)
int batch_prologue(const anyseq_scoring& sc, int64_t npairs, ScoreParams* sp, bool* affine, anyseq_result* out);

}  // namespace anyseq

// the opaque context of the C ABI (include/anyseq.h)
struct anyseq_ctx {
    anyseq::Engine eng;
};
