/*
 * anyseq.h -- C ABI of libanyseq_b200.so, the B200-native (sm_100a CUDA)
 * replacement for the DP-relaxation hot path of DasNaCl/anyseq.
 *
 * Drop-in boundary.  The reference's host program (src/main.cpp) reaches its
 * kernels through six C symbols declared in src/import.h:14-41 and defined by
 * the Impala `extern fn`s of src/export.impala:5-147.  Section 1 re-declares
 * exactly those symbols (same names, same argument meaning, same ownership
 * rules: src/main.cpp:31-36,73-76).  Section 2 is the parametrised surface the
 * reference keeps internal (linear_scoring_scheme / affine_scoring_scheme and
 * global/semiglobal/local_scheme, src/align.impala:96-166) plus what a B200
 * deployment needs: device-resident inputs, batches, multi-GPU strips.
 *
 * Plain pointers and sizes only; no C++/torch types.  All functions are
 * blocking.  There is NO CPU fallback: if no CUDA device is usable every
 * entry point fails loudly (status < 0; the legacy symbols abort()).
 */
#ifndef ANYSEQ_B200_H_
#define ANYSEQ_B200_H_

#include <stdint.h>

#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif
#ifdef __cplusplus
extern "C" {
#endif

/* score storage type of the reference's C interface: src/datatypes.h:14 */
typedef int64_t score_t;

/* ---------------------------------------------------------------------------
 * 1. Legacy symbols -- replace src/import.h:14-41 one for one.
 *    Scoring is the reference's hard-wired linear_scoring_scheme(2,-1,-1)
 *    (src/export.impala:14,33,70,89,126,145).
 *    construct_*: alQuery/alSubject are caller buffers of lenq+lens bytes,
 *    overwritten with ' ' and then with the alignment columns at index i+j+1,
 *    gaps as '_' (src/traceback.impala:1-2,47-80), linear-space traceback
 *    (traceback_lintime, src/align.impala:237-311).  Their return value follows
 *    the reference (score of the never-relaxed scoring object, SURVEY quirk
 *    Q1: -lenq / 0 / -2147483647) unless ANYSEQ_TRUE_SCORE=1 is set in the
 *    environment, in which case the optimal score is returned.
 * ------------------------------------------------------------------------- */
score_t global_alignment_score(const char* query, int lenq, const char* subject, int lens);
score_t semiglobal_alignment_score(const char* query, int lenq, const char* subject, int lens);
score_t local_alignment_score(const char* query, int lenq, const char* subject, int lens);

score_t construct_global_alignment(const char* query, int lenq, const char* subject, int lens,
                                   char* alQuery, char* alSubject);
score_t construct_semiglobal_alignment(const char* query, int lenq, const char* subject, int lens,
                                       char* alQuery, char* alSubject);
score_t construct_local_alignment(const char* query, int lenq, const char* subject, int lens,
                                  char* alQuery, char* alSubject);

/* The full-matrix variants the Impala side also exports (src/export.impala:38,94,151; not declared in
 * src/import.h): traceback_full, src/align.impala:190-216 -- the whole predecessor matrix and ONE walk from
 * get_score_pos(), i.e. the exact semiglobal / local alignments the linear-space path does not give.
 * Same buffers and output layout; they return the real score (the scoring object is relaxed there).
 * Memory is m*n/2 bytes of HBM: pairs up to roughly 400 k x 400 k on a 180 GB B200; abort()s beyond. */
score_t construct_global_alignment_fulltb(const char* query, int lenq, const char* subject, int lens,
                                          char* alQuery, char* alSubject);
score_t construct_semiglobal_alignment_fulltb(const char* query, int lenq, const char* subject, int lens,
                                              char* alQuery, char* alSubject);
score_t construct_local_alignment_fulltb(const char* query, int lenq, const char* subject, int lens,
                                         char* alQuery, char* alSubject);

/* ---------------------------------------------------------------------------
 * 2. Parametrised surface.
 * ------------------------------------------------------------------------- */
enum {                       /* alignment schemes: src/align.impala:96-124 */
    ANYSEQ_GLOBAL = 0,
    ANYSEQ_SEMIGLOBAL = 1,
    ANYSEQ_LOCAL = 2
};

enum {                       /* status codes (0 = ok, < 0 = failure) */
    ANYSEQ_EOF = 1,          /* anyseq_batch_stream_collect: every submitted chunk has been collected */
    ANYSEQ_OK = 0,
    ANYSEQ_ERR_NO_DEVICE = -1,
    ANYSEQ_ERR_BAD_ARG = -2,
    ANYSEQ_ERR_KERNEL_TIMEOUT = -3,
    ANYSEQ_ERR_UNSUPPORTED = -4
    /* <= -1000: -(cudaError_t) - 1000 */
};

/* Scoring scheme.  gap_init == 0 selects linear gaps with cost gap_extend per
 * gap symbol (linear_scoring_scheme(same,diff,gap), src/align.impala:144);
 * gap_init < 0 selects Gotoh affine gaps: a gap of length L costs
 * gap_init + L*gap_extend (parameter names of affine_scoring_scheme,
 * src/align.impala:153-154; the recurrence itself is defined by this build,
 * see DESIGN.md -- the reference only ships an uncalled stub). */
typedef struct anyseq_scoring {
    int32_t mode;            /* ANYSEQ_GLOBAL / SEMIGLOBAL / LOCAL */
    int32_t same;            /* score of equal symbols (bytes compared raw) */
    int32_t diff;            /* score of different symbols */
    int32_t gap_init;        /* <= 0 */
    int32_t gap_extend;      /* <= 0 */
} anyseq_scoring;

typedef struct anyseq_result {
    int64_t score;
    int32_t end_i;           /* end cell of the alignment (row = query index), -1 if unknown */
    int32_t end_j;           /* end cell (column = subject index) */
    float   kernel_ms;       /* device time of the DP kernels of this call (CUDA events) */
    int32_t kernel_launches; /* number of kernels this call launched */
} anyseq_result;

typedef struct anyseq_ctx anyseq_ctx;   /* one per (process, GPU) */

/* Create / destroy an engine bound to CUDA device `device` (-1: current). */
int anyseq_ctx_create(int device, anyseq_ctx** out);
void anyseq_ctx_destroy(anyseq_ctx* ctx);
const char* anyseq_last_error(void);

/* Tuning knobs (0 = automatic): columns per lane K in {4,8,16,32}, band height
 * in rows, persistent blocks per SM, dependency-wait watchdog in ms. */
int anyseq_ctx_tune(anyseq_ctx* ctx, int cols_per_lane, int band_rows, int blocks_per_sm, int watchdog_ms);

/* Named options: "cols_per_lane", "band_rows", "blocks_per_sm" (warps per scheduler of the strip kernels, 1-3),
 * "watchdog_ms" (> 0), "band_slack" (band height = slack * lag * resident warps when a launch has more strips than
 * warps; default 2), "cell_form" (-1 = per launch, 1 = decoupled, 2 = mixed Gotoh cells: identical results,
 * different instruction mixes -- see DESIGN.md 3.1; other values are refused),
 * "force_generic" (1: byte-register kernels even for small alphabets), "force_affine" (1: the score path runs the
 * Gotoh kernels even for gap_init == 0 -- must equal the linear kernels; testing),
 * "align_with_score" (0: anyseq_align skips the extra score pass),
 * "small_model" (0: small problems keep 128-column strips instead of the width the measured critical-path
 * fit prefers -- engine.cu: pick_K),
 * "batch_chunk_bytes" / "batch_chunk_pairs" / "batch_copy_threads" (pipeline of
 * anyseq_score_batch with host buffers), "batch_packed" (0: never use the 16-bit two-pairs-per-warp
 * batch kernels), "batch_quad" (0: never use the four-pairs-per-warp variant of them),
 * "local_end_cell" (1: local scores also fill end_i/end_j with the cell the
 * reference's get_score_pos() reports -- src/scoring.impala:103-110 with the
 * slot order of src/scoring_cpu.impala:48-73; runs the single-row kernels,
 * measured 2.29 vs 3.44 TCUPS on the whole-genome pair; default 0: end_i = end_j = -1
 * for the local scheme). */
int anyseq_ctx_set_option(anyseq_ctx* ctx, const char* name, int value);

/* Score only: score() of src/align.impala:218-235 with host buffers (the call
 * copies them to the device) ... */
int anyseq_score(anyseq_ctx* ctx, const anyseq_scoring* sc,
                 const char* query, int lenq, const char* subject, int lens,
                 anyseq_result* out);
/* ... or with sequences already resident in HBM (device pointers, lenq/lens
 * bytes; must stay valid until the call returns). */
int anyseq_score_device(anyseq_ctx* ctx, const anyseq_scoring* sc,
                        const void* d_query, int lenq, const void* d_subject, int lens,
                        anyseq_result* out);

/* Linear-space traceback.  Linear gaps: traceback_lintime of
 * src/align.impala:237-311, bit-exact with the reference CPU build (hb_sum
 * candidate order for BLOCK_WIDTH = 1024).  Gotoh gaps (gap_init < 0): the same
 * driver with Myers-Miller joins -- defined by this build (the reference has no
 * affine path), optimal for the global scheme; see DESIGN.md.  Output buffers as
 * for construct_*.  out->score is the true optimal score of the scheme. */
int anyseq_align(anyseq_ctx* ctx, const anyseq_scoring* sc,
                 const char* query, int lenq, const char* subject, int lens,
                 char* alQuery, char* alSubject, anyseq_result* out);

/* Split rows chosen by the last anyseq_align / construct_* call of this ctx
 * (the reference's Splits vector, src/traceback_lintime.impala:9-42): element 0
 * is slot -1 (= 0), then one entry per 128-column block.  Returns the number of
 * entries (writes at most cap). */
int anyseq_last_splits(anyseq_ctx* ctx, int32_t* out, int cap);

/* Gotoh traceback only: type of every split vertex (0 = ordinary, 1 = a horizontal
 * gap runs through it), same indexing as anyseq_last_splits; empty after a
 * linear-gap traceback. */
int anyseq_last_split_types(anyseq_ctx* ctx, int32_t* out, int cap);

/* traceback_full() with a parametrised scheme (Gotoh: build-defined, parity unpinned).  start[2] (optional)
 * receives get_alignment_start() = the cell after which the walk stopped; out->end_i/end_j the cell it
 * began at (get_score_pos()).  ANYSEQ_ERR_UNSUPPORTED when the predecessor matrix does not fit. */
int anyseq_align_full(anyseq_ctx* ctx, const anyseq_scoring* sc,
                      const char* query, int lenq, const char* subject, int lens,
                      char* alQuery, char* alSubject, anyseq_result* out, int32_t* start);

/* Full-matrix traceback of a batch of independent pairs (traceback_full per pair, as anyseq_align_full).
 * Pair p is queries[q_off[p] .. q_off[p+1]) vs subjects[s_off[p] .. s_off[p+1]); every subject <= 1024 symbols.
 * Pair p's aligned rows occupy alQuery/alSubject[o_p .. o_p + lq + ls) with
 * o_p = (q_off[p] - q_off[0]) + (s_off[p] - s_off[0]), i.e. both buffers hold
 * (q_off[npairs] - q_off[0]) + (s_off[npairs] - s_off[0]) bytes.
 * scores[npairs]; ends[2*npairs] = get_score_pos(), starts[2*npairs] = get_alignment_start() (either may be NULL).
 * Pairs are not transposed.  ANYSEQ_ERR_UNSUPPORTED for a subject longer than 1024 (use anyseq_align_full) and
 * when the batch's scratch or outputs do not fit in device memory (split the batch); ANYSEQ_ERR_BAD_ARG for
 * decreasing offsets.  The _device variant takes device pointers for every array. */
int anyseq_align_batch(anyseq_ctx* ctx, const anyseq_scoring* sc, const char* queries, const int64_t* q_off,
                       const char* subjects, const int64_t* s_off, int64_t npairs, int32_t* scores,
                       int32_t* ends, int32_t* starts, char* alQuery, char* alSubject, anyseq_result* out);
int anyseq_align_batch_device(anyseq_ctx* ctx, const anyseq_scoring* sc, const void* d_queries,
                              const int64_t* d_q_off, const void* d_subjects, const int64_t* d_s_off,
                              int64_t npairs, int32_t* d_scores, int32_t* d_ends, int32_t* d_starts,
                              char* d_alQuery, char* d_alSubject, anyseq_result* out);

/* Derived view of an alignment pair: CIGAR string (=/X/I/D run-length, I = gap
 * in the query ('_' in alQuery), D = gap in the subject), skipping blank
 * columns.  Returns the length written (excluding the NUL) or -needed if cap is
 * too small. */
int64_t anyseq_cigar(const char* alQuery, const char* alSubject, int64_t len, char* out, int64_t cap);

/* Batch of independent pairs (score only).  Sequences are packed back to back;
 * pair p is queries[q_off[p] .. q_off[p+1]) vs subjects[s_off[p] .. s_off[p+1]).
 * Host buffers; scores[npairs] is written.  Every scheme the single-pair calls take is scored exactly, except
 * local alignment with diff > 0: ANYSEQ_ERR_UNSUPPORTED (the kernels pad columns, and padding must not outscore
 * real symbols).  The same holds for the packed and streaming batch entries below. */
int anyseq_score_batch(anyseq_ctx* ctx, const anyseq_scoring* sc,
                       const char* queries, const int64_t* q_off,
                       const char* subjects, const int64_t* s_off,
                       int64_t npairs, int32_t* scores, anyseq_result* out);
int anyseq_score_batch_device(anyseq_ctx* ctx, const anyseq_scoring* sc,
                              const void* d_queries, const int64_t* d_q_off,
                              const void* d_subjects, const int64_t* d_s_off,
                              int64_t npairs, int32_t* d_scores, anyseq_result* out);

/* 2-bit packed batches (DNA reads x windows, BASELINE configs[3]; the packed staging of the reference is
 * sequence_to_device, src/mapping_acc.impala:125-131, one byte per symbol).  Four symbols per byte, least significant
 * bits first, A/C/G/T (either case) = 0/1/2/3; every sequence starts on a byte boundary.  Symbols are compared by
 * value, exactly like the byte path compares bytes (src/align.impala:132), so scores equal those of the unpacked
 * sequences.  Sequence p of the queries starts at byte q_boff[p] (q_boff == NULL: at p * q_stride) and has q_len[p]
 * symbols (q_len == NULL: q_len_uniform); same for the subjects.  A quarter of the bytes of the byte path cross
 * PCIe, and no alphabet analysis pass is needed.  Host variant: chunks are copied straight from the caller's memory
 * (pin it for full H2D speed) on a copy stream while the previous chunk is relaxed; scores land in `scores`. */
typedef struct anyseq_packed_batch {
    const uint8_t* q2;
    const uint8_t* s2;
    const int64_t* q_boff;
    const int64_t* s_boff;
    const int32_t* q_len;
    const int32_t* s_len;
    int32_t q_len_uniform, s_len_uniform;
    int64_t q_stride, s_stride;
    int64_t npairs;
} anyseq_packed_batch;
int anyseq_score_batch_packed2(anyseq_ctx* ctx, const anyseq_scoring* sc, const anyseq_packed_batch* host_batch,
                               int32_t* scores, anyseq_result* out);
int anyseq_score_batch_packed2_device(anyseq_ctx* ctx, const anyseq_scoring* sc, const anyseq_packed_batch* device_batch,
                                      int32_t* d_scores, anyseq_result* out);
/* Producer-side helper: packs n symbols (A/C/G/T, either case) into ceil(n/4) bytes of out; returns the number of
 * symbols that are not A/C/G/T (they cannot be represented: use the byte path for such sequences). */
int64_t anyseq_pack2(const char* seq, int64_t n, uint8_t* out);

/* Streaming batches (SURVEY 8f.2: many-record FASTA/FASTQ x windows ingestion that is not H2D-bound).
 * A stream owns `slots` chunk slots of PINNED host memory + device memory.  One producer thread
 *   acquire (blocks for a free slot) -> fill queries/q_off/subjects/s_off/npairs -> submit (starts H2D)
 * and one consumer thread
 *   collect (next chunk in submission order: kernel + D2H of the scores; ANYSEQ_EOF after finish)
 *   -> use chunk.scores -> release (slot becomes free)
 * run concurrently, so parsing/copying chunk c+1 overlaps the kernel of chunk c.  The reference's host
 * reader has the same producer/consumer shape (next()/skip() under a mutex, src/sequence_io.cpp:13-41).
 * anyseq_score_batch() with host buffers is a stream fed from the caller's arrays.  Offsets of a chunk
 * are chunk-relative (q_off[0] == s_off[0] == 0). */
typedef struct anyseq_batch_stream anyseq_batch_stream;
typedef struct anyseq_batch_chunk {
    char* queries;             /* acquire: pinned buffer of cap_query_bytes */
    int64_t* q_off;            /* acquire: cap_pairs + 1 offsets */
    char* subjects;
    int64_t* s_off;
    int64_t cap_pairs, cap_query_bytes, cap_subject_bytes;
    int64_t npairs;            /* producer sets it before submit; collect returns it */
    const int32_t* scores;     /* collect: npairs scores (pinned, valid until release) */
    float kernel_ms;           /* collect: device time of this chunk */
    int32_t slot;              /* internal */
} anyseq_batch_chunk;
int anyseq_batch_stream_open(anyseq_ctx* ctx, const anyseq_scoring* sc, int64_t cap_pairs,
                             int64_t cap_query_bytes, int64_t cap_subject_bytes, int slots,
                             anyseq_batch_stream** out);
int anyseq_batch_stream_acquire(anyseq_batch_stream* st, anyseq_batch_chunk* chunk);
int anyseq_batch_stream_submit(anyseq_batch_stream* st, const anyseq_batch_chunk* chunk);
int anyseq_batch_stream_finish(anyseq_batch_stream* st);
int anyseq_batch_stream_collect(anyseq_batch_stream* st, anyseq_batch_chunk* chunk);
int anyseq_batch_stream_release(anyseq_batch_stream* st, const anyseq_batch_chunk* chunk);
int anyseq_batch_stream_stats(anyseq_batch_stream* st, anyseq_result* totals, int64_t* h2d_bytes, int64_t* d2h_bytes);
void anyseq_batch_stream_close(anyseq_batch_stream* st);

/* Multi-GPU column-strip wavefront for one long pair (one process per GPU).
 * Rank r of `nranks` owns subject columns [col_begin, col_end).  Its left
 * border arrives in this rank's `inbox` (device memory this rank allocates with
 * anyseq_strip_inbox_create and exports as a CUDA IPC handle); its right edge
 * is written straight into the next rank's inbox over NVLink (peer pointer
 * obtained with anyseq_strip_inbox_open).  No host in the loop. */
typedef struct anyseq_inbox anyseq_inbox;
int anyseq_strip_inbox_create(anyseq_ctx* ctx, int rows, anyseq_inbox** out, void* ipc_handle_64B);
int anyseq_strip_inbox_open(anyseq_ctx* ctx, const void* ipc_handle_64B, int rows, anyseq_inbox** out);
int anyseq_strip_inbox_reset(anyseq_ctx* ctx, anyseq_inbox* box);
void anyseq_strip_inbox_destroy(anyseq_ctx* ctx, anyseq_inbox* box);
/* Partial result of a rank: best of the last-row slice it owns (semiglobal),
 * last column (last rank), running maximum (local); combine with
 * anyseq_strip_combine on any rank. */
typedef struct anyseq_strip_partial {
    int32_t row_best, row_best_j;      /* semiglobal: max over H(m-1, j) of owned columns (lowest j) */
    int32_t col_best, col_best_i;      /* semiglobal, last rank: max over H(i, n-1) (lowest i) */
    int32_t local_best;                /* local: max over owned cells */
    int32_t corner;                    /* last rank: H(m-1, n-1) */
    float   kernel_ms;
    int32_t kernel_launches;
    int32_t lenq, lens_total;          /* the whole matrix (filled by the engine): combine reports end cells like a single-GPU run */
} anyseq_strip_partial;
int anyseq_score_strip_device(anyseq_ctx* ctx, const anyseq_scoring* sc,
                              const void* d_query, int lenq,
                              const void* d_subject_slice, int col_begin, int col_end, int lens_total,
                              anyseq_inbox* inbox /* NULL on rank 0 */,
                              anyseq_inbox* next_inbox /* NULL on the last rank */,
                              anyseq_strip_partial* out);
/* The same with HOST buffers (the rank's query and its slice of the subject): the call copies them to the device,
 * like anyseq_score does on one GPU (sequence_to_device, src/mapping_acc.impala:125-131). */
int anyseq_score_strip(anyseq_ctx* ctx, const anyseq_scoring* sc,
                       const char* query, int lenq,
                       const char* subject_slice, int col_begin, int col_end, int lens_total,
                       anyseq_inbox* inbox, anyseq_inbox* next_inbox, anyseq_strip_partial* out);
/* The same for `npairs` (<= 8) pairs of ONE shape (lenq, column range) in a single persistent launch, their work
 * items interleaved band by band.  A narrow slice alone has too few strips to occupy a B200; the slices of two
 * consecutive alignments of a stream side by side do.  Arrays of npairs device pointers / inboxes (inbox arrays may be
 * NULL on the first / last rank); out[npairs]. */
int anyseq_score_strip_device_multi(anyseq_ctx* ctx, const anyseq_scoring* sc, int npairs,
                                    const void* const* d_query, int lenq,
                                    const void* const* d_subject_slice, int col_begin, int col_end, int lens_total,
                                    anyseq_inbox* const* inbox, anyseq_inbox* const* next_inbox,
                                    anyseq_strip_partial* out);
int anyseq_strip_combine(const anyseq_scoring* sc, const anyseq_strip_partial* parts, int nranks,
                         anyseq_result* out);

/* Multi-GPU linear-space traceback (SURVEY 8e: the halves of a Hirschberg level are independent, src/align.impala:254-259,
 * src/iteration_cpu.impala:59-119).  Every rank (one process per GPU, world a power of two) calls it with the SAME
 * sequences; the halves of every level are dealt out to the ranks, on the first log2(world) levels the last-column
 * records of the halves are exchanged through `bcast` (the caller's collective, e.g. ncclBroadcast on the given device
 * buffer; it must be complete when it returns), afterwards the ranks work independently.  alQuery / alSubject are
 * lenq+lens-byte buffers of which this rank fills [*out_lo, *out_hi) -- the columns of its 128-column blocks; the
 * ranges of all ranks tile [0, lenq+lens) in rank order, so concatenating them gives exactly the single-GPU strings.
 * anyseq_last_splits afterwards holds -1 in the slots other ranks decided.  The optimal score is not computed here
 * (use the strip wavefront, anyseq_score_strip*): out->score = 0. */
typedef int (*anyseq_bcast_fn)(void* user, void* d_buffer, int64_t nbytes, int src_rank);
int anyseq_align_sharded(anyseq_ctx* ctx, const anyseq_scoring* sc,
                         const char* query, int lenq, const char* subject, int lens,
                         int rank, int world, anyseq_bcast_fn bcast, void* user,
                         char* alQuery, char* alSubject, int64_t* out_lo, int64_t* out_hi, anyseq_result* out);

/* Measured integer-pipe peak of this GPU for the DP instruction mix (the
 * roofline denominator, SURVEY.md 8d): runs dependency-free loops of the named
 * mix and returns 32-bit lane-operations per second. kind: 0 = VIMNMX/VIADDMNMX
 * only (ALU pipe), 1 = the 5-op linear cell mix, 2 = the 7-op affine cell mix,
 * 3 = IMAD only (FMA pipe), 4 = ALU+IMAD interleaved; 5 / 6 = the strip kernel's own
 * Gotoh / linear cell instruction sequence (both pipes), returned as CELLS per second. */
int anyseq_measure_int_peak(anyseq_ctx* ctx, int kind, double* ops_per_s, float* sm_mhz_est);

/* Device properties the bench reports. */
int anyseq_device_info(anyseq_ctx* ctx, int* sm_count, int* resident_warps, char* name64);

/* The launch the engine makes for ONE lenq x lens score-only problem on a GPU with sm_count SMs (148 on a B200):
 * strip width, tile height, cell form, bands and grid.  Pure host logic -- needs no device and no context -- so the
 * planner can be tested on a CPU-only machine and inspected from tools (tools/plan.py).  It answers for the column-mask
 * kernels (alphabets of at most 31 shared symbols) with default tuning; chained != 0: the problem is one rank's column
 * slice of a multi-GPU wavefront.  This replaces what the reference fixes at compile time (BLOCK_WIDTH / BLOCK_HEIGHT,
 * src/mapping_acc.impala:1-12) and its per-anti-diagonal launch loop (src/iteration_acc.impala:120-172). */
typedef struct anyseq_launch_plan {
    int32_t cols_per_lane;        /* K: a strip is 32 * K subject columns wide */
    int32_t rows_per_step;        /* R: query rows a lane relaxes per anti-diagonal step */
    int32_t cell_form;            /* 1 decoupled, 2 mixed (DESIGN.md 3.1) */
    int32_t strips;
    int32_t warps_per_scheduler;  /* 1..3: resident warps = 4 * this * sm_count */
    int32_t bands;                /* row bands; 1 when every strip has a warp of its own */
    int32_t band_rows;
    int32_t grid;                 /* CTAs (one per SM at most) */
    int32_t warps_per_cta;
    int64_t first_items;          /* (band, strip) items assigned statically; the rest is claimed from a counter */
    int32_t packed_cells;         /* 1: the decoupled Gotoh cells run as 16-bit pairs, two per DPX instruction (DESIGN.md 3.1) */
} anyseq_launch_plan;
/* anyseq_plan_launch answers for the scheme (same, diff, gap_init, gap_extend) = (2, -1, -2, -1) (gap_init = 0 when
 * affine == 0); anyseq_plan_launch_scheme for any scheme (packed_cells depends on it). */
int anyseq_plan_launch(int sm_count, int mode, int affine, int lenq, int lens, int chained, anyseq_launch_plan* out);
int anyseq_plan_launch_scheme(int sm_count, const anyseq_scoring* sc, int lenq, int lens, int chained, anyseq_launch_plan* out);

#ifdef __cplusplus
}
#endif
#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#endif /* ANYSEQ_B200_H_ */
