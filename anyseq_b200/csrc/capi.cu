// capi.cu -- the C ABI of libanyseq_b200.so (include/anyseq.h).
#include "engine.cuh"

#include <cstdlib>
#include <cstring>
#include <string>

namespace anyseq {
const char* last_error_cstr();
}

struct anyseq_inbox {
    anyseq::Inbox box;
};

using anyseq::Engine;
using anyseq::set_last_error;

extern "C" {

const char* anyseq_last_error(void) { return anyseq::last_error_cstr(); }

int anyseq_ctx_create(int device, anyseq_ctx** out)
{
    if (!out) return ANYSEQ_ERR_BAD_ARG;
    *out = nullptr;
    anyseq_ctx* c = new anyseq_ctx();
    int rc = c->eng.init(device);
    if (rc) {
        c->eng.destroy();
        delete c;
        return rc;
    }
    *out = c;
    return ANYSEQ_OK;
}

void anyseq_ctx_destroy(anyseq_ctx* ctx)
{
    if (!ctx) return;
    ctx->eng.destroy();
    delete ctx;
}

int anyseq_ctx_tune(anyseq_ctx* ctx, int cols_per_lane, int band_rows, int blocks_per_sm, int watchdog_ms)
{
    if (!ctx) return ANYSEQ_ERR_BAD_ARG;
    if (cols_per_lane != 0 && cols_per_lane != 4 && cols_per_lane != 8 && cols_per_lane != 16 &&
        cols_per_lane != 32) {
        set_last_error("cols_per_lane must be 0, 4, 8, 16 or 32");
        return ANYSEQ_ERR_BAD_ARG;
    }
    ctx->eng.tune.cols_per_lane = cols_per_lane;
    ctx->eng.tune.band_rows = band_rows;
    ctx->eng.tune.blocks_per_sm = blocks_per_sm;
    if (watchdog_ms > 0) ctx->eng.tune.watchdog_ms = watchdog_ms;
    return ANYSEQ_OK;
}

int anyseq_ctx_set_option(anyseq_ctx* ctx, const char* name, int value)
{
    if (!ctx || !name) return ANYSEQ_ERR_BAD_ARG;
    const std::string n(name);
    anyseq::Tuning& t = ctx->eng.tune;
    if (n == "cols_per_lane") t.cols_per_lane = value;
    else if (n == "band_rows") t.band_rows = value;
    else if (n == "blocks_per_sm") t.blocks_per_sm = value;
    else if (n == "watchdog_ms") {
        // 0 would time every slow-path wait out, a negative value would disable the watchdog (anyseq_ctx_tune rejects both too)
        if (value <= 0) { anyseq::set_last_error("watchdog_ms must be > 0"); return ANYSEQ_ERR_BAD_ARG; }
        t.watchdog_ms = value;
    }
    else if (n == "band_slack" && value >= 1) t.band_slack = value;
    else if (n == "cell_form") {
        if (value != -1 && value != 1 && value != 2) { set_last_error("cell_form must be -1, 1 or 2"); return ANYSEQ_ERR_BAD_ARG; }
        t.cell_form = value;
    }
    else if (n == "packed_cells" && value >= -1 && value <= 1) t.packed_cells = value;
    else if (n == "force_generic") t.force_generic = value != 0;
    else if (n == "force_affine") t.force_affine = value != 0;
    else if (n == "local_end_cell") t.local_end_cell = value != 0;
    else if (n == "batch_chunk_bytes" && value >= (1 << 16)) t.batch_chunk_bytes = value;
    else if (n == "batch_chunk_pairs" && value >= 1) t.batch_chunk_pairs = value;
    else if (n == "batch_copy_threads" && value >= 1) t.batch_copy_threads = value;
    else if (n == "batch_packed") t.batch_packed = value != 0;
    else if (n == "batch_quad") t.batch_quad = value != 0;
    else if (n == "align_with_score") t.align_with_score = value != 0;
    else if (n == "small_model") t.small_model = value != 0;
    else {
        set_last_error("unknown option " + n);
        return ANYSEQ_ERR_BAD_ARG;
    }
    return ANYSEQ_OK;
}

int anyseq_score(anyseq_ctx* ctx, const anyseq_scoring* sc, const char* query, int lenq,
                 const char* subject, int lens, anyseq_result* out)
{
    if (!ctx || !sc || !out) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.score_host(*sc, query, lenq, subject, lens, out);
}

int anyseq_score_device(anyseq_ctx* ctx, const anyseq_scoring* sc, const void* d_query, int lenq,
                        const void* d_subject, int lens, anyseq_result* out)
{
    if (!ctx || !sc || !out) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.score_device(*sc, static_cast<const uint8_t*>(d_query), lenq,
                                 static_cast<const uint8_t*>(d_subject), lens, out);
}

int anyseq_align(anyseq_ctx* ctx, const anyseq_scoring* sc, const char* query, int lenq,
                 const char* subject, int lens, char* alQuery, char* alSubject, anyseq_result* out)
{
    if (!ctx || !sc || !out || !alQuery || !alSubject) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.align_host(*sc, query, lenq, subject, lens, alQuery, alSubject, out);
}

int anyseq_align_full(anyseq_ctx* ctx, const anyseq_scoring* sc, const char* query, int lenq,
                      const char* subject, int lens, char* alQuery, char* alSubject, anyseq_result* out, int32_t* start)
{
    if (!ctx || !sc || !out || !alQuery || !alSubject) return ANYSEQ_ERR_BAD_ARG;
    int st[2] = {0, 0};
    const int rc = ctx->eng.align_full_host(*sc, query, lenq, subject, lens, alQuery, alSubject, out, st);
    if (start) { start[0] = st[0]; start[1] = st[1]; }
    return rc;
}

int anyseq_align_batch(anyseq_ctx* ctx, const anyseq_scoring* sc, const char* queries, const int64_t* q_off,
                       const char* subjects, const int64_t* s_off, int64_t npairs, int32_t* scores,
                       int32_t* ends, int32_t* starts, char* alQuery, char* alSubject, anyseq_result* out)
{
    if (!ctx || !sc) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.align_batch_host(*sc, queries, q_off, subjects, s_off, npairs, scores, ends, starts, alQuery,
                                     alSubject, out);
}

int anyseq_align_batch_device(anyseq_ctx* ctx, const anyseq_scoring* sc, const void* d_queries,
                              const int64_t* d_q_off, const void* d_subjects, const int64_t* d_s_off,
                              int64_t npairs, int32_t* d_scores, int32_t* d_ends, int32_t* d_starts,
                              char* d_alQuery, char* d_alSubject, anyseq_result* out)
{
    if (!ctx || !sc || npairs < 0 || (npairs > 0 && (!d_q_off || !d_s_off || !d_scores || !d_alQuery || !d_alSubject)))
        return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.align_batch_device(*sc, static_cast<const uint8_t*>(d_queries), d_q_off,
                                       static_cast<const uint8_t*>(d_subjects), d_s_off, npairs, d_scores, d_ends,
                                       d_starts, d_alQuery, d_alSubject, out);
}

int anyseq_last_splits(anyseq_ctx* ctx, int32_t* out, int cap)
{
    if (!ctx) return ANYSEQ_ERR_BAD_ARG;
    const std::vector<int>& v = ctx->eng.last_splits();
    const int n = (int)v.size();
    if (out) for (int i = 0; i < n && i < cap; ++i) out[i] = v[i];
    return n;
}

int anyseq_last_split_types(anyseq_ctx* ctx, int32_t* out, int cap)
{
    if (!ctx) return ANYSEQ_ERR_BAD_ARG;
    const std::vector<int>& v = ctx->eng.last_types();
    const int n = (int)v.size();
    if (out) for (int i = 0; i < n && i < cap; ++i) out[i] = v[i];
    return n;
}

int64_t anyseq_cigar(const char* aq, const char* as, int64_t len, char* out, int64_t cap)
{
    // derived view (SURVEY.md 8b "Output format"): '=' equal symbols, 'X'
    // different symbols, 'I' gap in the query row, 'D' gap in the subject row
    std::string cg;
    char cur = 0;
    int64_t run = 0;
    auto emit = [&]() {
        if (run > 0) { cg += std::to_string(run); cg += cur; }
    };
    for (int64_t k = 0; k < len; ++k) {
        const char a = aq[k], b = as[k];
        if (a == ' ' && b == ' ') continue;
        char op;
        if (a == '_') op = 'I';
        else if (b == '_') op = 'D';
        else op = (a == b) ? '=' : 'X';
        if (op != cur) { emit(); cur = op; run = 0; }
        ++run;
    }
    emit();
    const int64_t need = (int64_t)cg.size();
    if (!out || cap < need + 1) return -(need + 1);
    std::memcpy(out, cg.c_str(), (size_t)need + 1);
    return need;
}

int anyseq_score_batch(anyseq_ctx* ctx, const anyseq_scoring* sc, const char* queries,
                       const int64_t* q_off, const char* subjects, const int64_t* s_off,
                       int64_t npairs, int32_t* scores, anyseq_result* out)
{
    if (!ctx || !sc || !q_off || !s_off || !scores || npairs < 0) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.score_batch_host(*sc, queries, q_off, subjects, s_off, npairs, scores, out);
}

int anyseq_score_batch_device(anyseq_ctx* ctx, const anyseq_scoring* sc, const void* d_queries,
                              const int64_t* d_q_off, const void* d_subjects, const int64_t* d_s_off,
                              int64_t npairs, int32_t* d_scores, anyseq_result* out)
{
    if (!ctx || !sc || !d_q_off || !d_s_off || !d_scores || npairs < 0) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.score_batch_device(*sc, static_cast<const uint8_t*>(d_queries), d_q_off,
                                       static_cast<const uint8_t*>(d_subjects), d_s_off, npairs,
                                       d_scores, out);
}

int anyseq_score_batch_ends(anyseq_ctx* ctx, const anyseq_scoring* sc, const char* queries, const int64_t* q_off,
                            const char* subjects, const int64_t* s_off, int64_t npairs, int32_t* scores, int32_t* ends,
                            anyseq_result* out)
{
    if (!ctx || !sc || !q_off || !s_off || !scores || !ends || npairs < 0) {
        anyseq::set_last_error("batch end cells: null argument");
        return ANYSEQ_ERR_BAD_ARG;
    }
    return ctx->eng.score_batch_host(*sc, queries, q_off, subjects, s_off, npairs, scores, out, ends);
}

int anyseq_score_batch_ends_device(anyseq_ctx* ctx, const anyseq_scoring* sc, const void* d_queries,
                                   const int64_t* d_q_off, const void* d_subjects, const int64_t* d_s_off,
                                   int64_t npairs, int32_t* d_scores, int32_t* d_ends, anyseq_result* out)
{
    if (!ctx || !sc || !d_q_off || !d_s_off || !d_scores || !d_ends || npairs < 0) {
        anyseq::set_last_error("batch end cells: null argument");
        return ANYSEQ_ERR_BAD_ARG;
    }
    return ctx->eng.score_batch_device(*sc, static_cast<const uint8_t*>(d_queries), d_q_off,
                                       static_cast<const uint8_t*>(d_subjects), d_s_off, npairs, d_scores, out, d_ends);
}

int anyseq_strip_inbox_create(anyseq_ctx* ctx, int rows, anyseq_inbox** out, void* ipc_handle_64B)
{
    if (!ctx || !out || rows < 1) return ANYSEQ_ERR_BAD_ARG;
    anyseq::Inbox* b = nullptr;
    int rc = ctx->eng.inbox_create(rows, &b, ipc_handle_64B);
    if (rc) return rc;
    anyseq_inbox* box = new anyseq_inbox();
    box->box = *b;
    delete b;
    *out = box;
    return ANYSEQ_OK;
}

int anyseq_strip_inbox_open(anyseq_ctx* ctx, const void* ipc_handle_64B, int rows, anyseq_inbox** out)
{
    if (!ctx || !out || !ipc_handle_64B || rows < 1) return ANYSEQ_ERR_BAD_ARG;
    anyseq::Inbox* b = nullptr;
    int rc = ctx->eng.inbox_open(ipc_handle_64B, rows, &b);
    if (rc) return rc;
    anyseq_inbox* box = new anyseq_inbox();
    box->box = *b;
    delete b;
    *out = box;
    return ANYSEQ_OK;
}

int anyseq_strip_inbox_reset(anyseq_ctx* ctx, anyseq_inbox* box)
{
    if (!ctx || !box) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.inbox_reset(&box->box);
}

void anyseq_strip_inbox_destroy(anyseq_ctx* ctx, anyseq_inbox* box)
{
    if (!ctx || !box) return;
    ctx->eng.inbox_destroy(&box->box);
    delete box;
}

int anyseq_score_strip_device(anyseq_ctx* ctx, const anyseq_scoring* sc, const void* d_query, int lenq,
                              const void* d_subject_slice, int col_begin, int col_end, int lens_total,
                              anyseq_inbox* inbox, anyseq_inbox* next_inbox, anyseq_strip_partial* out)
{
    if (!ctx || !sc || !out) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.score_strip_device(*sc, static_cast<const uint8_t*>(d_query), lenq,
                                       static_cast<const uint8_t*>(d_subject_slice), col_begin, col_end,
                                       lens_total, inbox ? &inbox->box : nullptr,
                                       next_inbox ? &next_inbox->box : nullptr, out);
}

int anyseq_score_strip(anyseq_ctx* ctx, const anyseq_scoring* sc, const char* query, int lenq,
                       const char* subject_slice, int col_begin, int col_end, int lens_total,
                       anyseq_inbox* inbox, anyseq_inbox* next_inbox, anyseq_strip_partial* out)
{
    if (!ctx || !sc || !out) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.score_strip_host(*sc, query, lenq, subject_slice, col_begin, col_end, lens_total,
                                     inbox ? &inbox->box : nullptr, next_inbox ? &next_inbox->box : nullptr, out);
}

int anyseq_score_strip_device_multi(anyseq_ctx* ctx, const anyseq_scoring* sc, int npairs, const void* const* d_query,
                                    int lenq, const void* const* d_subject_slice, int col_begin, int col_end,
                                    int lens_total, anyseq_inbox* const* inbox, anyseq_inbox* const* next_inbox,
                                    anyseq_strip_partial* out)
{
    if (!ctx || !sc || !out || npairs < 1 || npairs > 8 || !d_query || !d_subject_slice) return ANYSEQ_ERR_BAD_ARG;
    const uint8_t* q[8];
    const uint8_t* s[8];
    anyseq::Inbox* in[8];
    anyseq::Inbox* nx[8];
    bool any_in = false, any_nx = false;
    for (int p = 0; p < npairs; ++p) {
        q[p] = static_cast<const uint8_t*>(d_query[p]);
        s[p] = static_cast<const uint8_t*>(d_subject_slice[p]);
        in[p] = (inbox && inbox[p]) ? &inbox[p]->box : nullptr;
        nx[p] = (next_inbox && next_inbox[p]) ? &next_inbox[p]->box : nullptr;
        any_in |= in[p] != nullptr;
        any_nx |= nx[p] != nullptr;
    }
    return ctx->eng.score_strip_device_multi(*sc, npairs, q, lenq, s, col_begin, col_end, lens_total,
                                             any_in ? in : nullptr, any_nx ? nx : nullptr, out);
}

// Combine per-rank partial results exactly as a single-GPU run would
// (src/scoring.impala:29-137): global = H(m-1,n-1) of the last rank;
// semiglobal = last-row maximum first (lowest column, the -1 candidate with
// value 0 included), then the last column only if strictly greater; local =
// maximum over ranks.
int anyseq_strip_combine(const anyseq_scoring* sc, const anyseq_strip_partial* parts, int nranks,
                         anyseq_result* out)
{
    if (!sc || !parts || nranks < 1 || !out) return ANYSEQ_ERR_BAD_ARG;
    std::memset(out, 0, sizeof(*out));
    out->end_i = -1;
    out->end_j = -1;
    float ms = 0.f;
    int launches = 0;
    for (int r = 0; r < nranks; ++r) {
        ms = parts[r].kernel_ms > ms ? parts[r].kernel_ms : ms;
        launches += parts[r].kernel_launches;
    }
    out->kernel_ms = ms;
    out->kernel_launches = launches;
    // end cells as finish_score_kernel reports them on one GPU (get_score_pos, src/scoring.impala:29-77)
    const int m = parts[nranks - 1].lenq, n = parts[nranks - 1].lens_total;
    if (sc->mode == ANYSEQ_GLOBAL) {
        out->score = parts[nranks - 1].corner;
        out->end_i = m - 1;
        out->end_j = n - 1;
    } else if (sc->mode == ANYSEQ_SEMIGLOBAL) {
        int rs = 0, rj = -1;                       // candidate H(m-1,-1) = 0
        for (int r = 0; r < nranks; ++r)
            if (parts[r].row_best > rs) { rs = parts[r].row_best; rj = parts[r].row_best_j; }
        int cs = 0, ci = -1;
        if (parts[nranks - 1].col_best > cs) { cs = parts[nranks - 1].col_best; ci = parts[nranks - 1].col_best_i; }
        int64_t score = rs;
        out->end_i = m - 1;
        out->end_j = rj;
        if (cs > rs) { score = cs; out->end_i = ci; out->end_j = n - 1; }
        out->score = score;
    } else {
        int best = anyseq::kScoreMin;
        for (int r = 0; r < nranks; ++r) best = parts[r].local_best > best ? parts[r].local_best : best;
        out->score = best;
    }
    return ANYSEQ_OK;
}

int anyseq_align_sharded(anyseq_ctx* ctx, const anyseq_scoring* sc, const char* query, int lenq, const char* subject, int lens,
                         int rank, int world, anyseq_bcast_fn bcast, void* user, char* alQuery, char* alSubject,
                         int64_t* out_lo, int64_t* out_hi, anyseq_result* out)
{
    if (!ctx || !sc || !out || !alQuery || !alSubject || !out_lo || !out_hi) return ANYSEQ_ERR_BAD_ARG;
    anyseq::TracebackShard sh;
    sh.rank = rank;
    sh.world = world;
    sh.bcast = bcast;
    sh.user = user;
    const int rc = ctx->eng.align_host_sharded(*sc, query, lenq, subject, lens, alQuery, alSubject, out, &sh);
    *out_lo = sh.out_lo;
    *out_hi = sh.out_hi;
    return rc;
}

int anyseq_measure_int_peak(anyseq_ctx* ctx, int kind, double* ops_per_s, float* sm_mhz_est)
{
    if (!ctx) return ANYSEQ_ERR_BAD_ARG;
    return ctx->eng.measure_int_peak(kind, ops_per_s, sm_mhz_est);
}

int anyseq_plan_launch_scheme(int sm_count, const anyseq_scoring* sc, int lenq, int lens, int chained, anyseq_launch_plan* out)
{
    anyseq::ScoreParams sp;
    bool affine = false;
    if (!sc) return ANYSEQ_ERR_BAD_ARG;
    int rc = anyseq::make_score_params(*sc, &sp, &affine);
    if (rc) return rc;
    // the launch would be refused: so is its plan (a device-free way to ask whether a problem is in range)
    if ((rc = anyseq::check_score_range(*sc, lenq, lens))) return rc;
    anyseq::Engine planner;          // never init()ed: no device, no buffers -- only the planning members are used
    return planner.plan_launch(sm_count, sc->mode, affine, lenq, lens, chained != 0, sp, out);
}

int anyseq_plan_launch(int sm_count, int mode, int affine, int lenq, int lens, int chained, anyseq_launch_plan* out)
{
    // the scheme of the whole-genome benchmark, (2, -1, -2, -1); gap_init = 0 for a linear-gap plan
    const anyseq_scoring sc = {mode, 2, -1, affine ? -2 : 0, -1};
    return anyseq_plan_launch_scheme(sm_count, &sc, lenq, lens, chained, out);
}

int anyseq_device_info(anyseq_ctx* ctx, int* sm_count, int* resident_warps, char* name64)
{
    if (!ctx) return ANYSEQ_ERR_BAD_ARG;
    if (sm_count) *sm_count = ctx->eng.sm_count;
    if (resident_warps) *resident_warps = ctx->eng.resident_warps(32, false, true);
    if (name64) std::memcpy(name64, ctx->eng.name, 64);
    return ANYSEQ_OK;
}

// ---------------------------------------------------------------------------
// Legacy symbols (src/import.h:14-41): process-wide default engine on the
// current CUDA device, reference scoring linear_scoring_scheme(2,-1,-1).
// No error channel exists in the reference interface: failures print to stderr
// and abort() (SURVEY.md 8b "Errors").
// ---------------------------------------------------------------------------
static anyseq_ctx* default_ctx()
{
    static anyseq_ctx* ctx = nullptr;
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    if (!ctx) {
        int rc = anyseq_ctx_create(-1, &ctx);
        if (rc) {
            std::fprintf(stderr, "anyseq_b200: cannot create CUDA engine (%d): %s\n", rc, anyseq_last_error());
            std::abort();
        }
    }
    return ctx;
}

static score_t legacy_score(int mode, const char* q, int lenq, const char* s, int lens)
{
    anyseq_scoring sc = {mode, 2, -1, 0, -1};
    anyseq_result res;
    int rc = anyseq_score(default_ctx(), &sc, q, lenq, s, lens, &res);
    if (rc) {
        std::fprintf(stderr, "anyseq_b200: score failed (%d): %s\n", rc, anyseq_last_error());
        std::abort();
    }
    return (score_t)res.score;   // sign-extended (the reference leaves the upper half undefined, quirk Q5)
}

static score_t legacy_align(int mode, const char* q, int lenq, const char* s, int lens, char* alq, char* als)
{
    anyseq_scoring sc = {mode, 2, -1, 0, -1};
    anyseq_result res;
    int rc = anyseq_align(default_ctx(), &sc, q, lenq, s, lens, alq, als, &res);
    if (rc) {
        std::fprintf(stderr, "anyseq_b200: alignment failed (%d): %s\n", rc, anyseq_last_error());
        std::abort();
    }
    const char* env = std::getenv("ANYSEQ_TRUE_SCORE");
    if (env && env[0] == '1') return (score_t)res.score;
    // quirk Q1: value of the never-relaxed scoring object (src/align.impala:244,264)
    if (mode == ANYSEQ_GLOBAL) return (score_t)lenq * -1;
    if (mode == ANYSEQ_SEMIGLOBAL) return 0;
    return (score_t)anyseq::kScoreMin;
}

// traceback_full exports (src/export.impala:38,94,151): the scoring object has been relaxed there, so these
// return the real score
static score_t legacy_align_full(int mode, const char* q, int lenq, const char* s, int lens, char* alq, char* als)
{
    anyseq_scoring sc = {mode, 2, -1, 0, -1};
    anyseq_result res;
    int rc = anyseq_align_full(default_ctx(), &sc, q, lenq, s, lens, alq, als, &res, nullptr);
    if (rc) {
        std::fprintf(stderr, "anyseq_b200: full-matrix alignment failed (%d): %s\n", rc, anyseq_last_error());
        std::abort();
    }
    return (score_t)res.score;
}
score_t construct_global_alignment_fulltb(const char* q, int lenq, const char* s, int lens, char* alq, char* als) { return legacy_align_full(ANYSEQ_GLOBAL, q, lenq, s, lens, alq, als); }
score_t construct_semiglobal_alignment_fulltb(const char* q, int lenq, const char* s, int lens, char* alq, char* als) { return legacy_align_full(ANYSEQ_SEMIGLOBAL, q, lenq, s, lens, alq, als); }
score_t construct_local_alignment_fulltb(const char* q, int lenq, const char* s, int lens, char* alq, char* als) { return legacy_align_full(ANYSEQ_LOCAL, q, lenq, s, lens, alq, als); }

score_t global_alignment_score(const char* q, int lenq, const char* s, int lens) { return legacy_score(ANYSEQ_GLOBAL, q, lenq, s, lens); }
score_t semiglobal_alignment_score(const char* q, int lenq, const char* s, int lens) { return legacy_score(ANYSEQ_SEMIGLOBAL, q, lenq, s, lens); }
score_t local_alignment_score(const char* q, int lenq, const char* s, int lens) { return legacy_score(ANYSEQ_LOCAL, q, lenq, s, lens); }

score_t construct_global_alignment(const char* q, int lenq, const char* s, int lens, char* alq, char* als) { return legacy_align(ANYSEQ_GLOBAL, q, lenq, s, lens, alq, als); }
score_t construct_semiglobal_alignment(const char* q, int lenq, const char* s, int lens, char* alq, char* als) { return legacy_align(ANYSEQ_SEMIGLOBAL, q, lenq, s, lens, alq, als); }
score_t construct_local_alignment(const char* q, int lenq, const char* s, int lens, char* alq, char* als) { return legacy_align(ANYSEQ_LOCAL, q, lenq, s, lens, alq, als); }

}  // extern "C"
