// nph_api.cu — the C ABI of libnph.so (include/nph.h): context, uploads, scheduling, fetches.
// All device work is launched from here; there is no CPU implementation of any entry point.
#include "nph_internal.cuh"
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <chrono>
#include <cstdlib>
#include <new>

int nph_set_cuda_error(nph_ctx* ctx, cudaError_t e, const char* what)
{
    if (ctx) {
        ctx->last_error = std::string(what) + ": " + cudaGetErrorString(e);
    }
    if (e == cudaErrorMemoryAllocation) return NPH_ERR_NOMEM;
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return NPH_ERR_NO_DEVICE;
    return NPH_ERR_CUDA;
}

extern "C" int nph_destroy(nph_ctx* ctx);

namespace {

// clip-penalty table (see np_oracle.c:npo_flank_table for the derivation; ref profile_hmm_r9.inl:200-260)
int ensure_flank(nph_ctx* ctx, size_t n)
{
    if (ctx->h_flank.size() >= n && ctx->d_flank.p) return NPH_OK;
    size_t want = std::max<size_t>(n + n / 2, 4096);
    std::vector<float>& f = ctx->h_flank;
    f.resize(want);
    const double start_to_clip = 0.5, clip_self = 0.9;
    const float bg = -3.0f;
    f[0] = (float)log(1 - start_to_clip);
    f[1] = (float)(log(start_to_clip) + bg + log(1 - clip_self));
    for (size_t i = 2; i < want; ++i) f[i] = (float)(log(clip_self) + bg + f[i - 1]);
    NPH_TRY(nph_reserve(ctx, ctx->d_flank, want));
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_flank.p, f.data(), want * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    return NPH_OK;
}

// calculate_transitions (ref: profile_hmm_r9.inl:17-76).  The reference evaluates log() on float
// probabilities in C++, i.e. std::log(float) == logf of the host libm; we call the same function so
// the values are the ones the reference would use on this machine.
void const_transitions(HmmConsts& c)
{
    float p_skip = 0.0025;
    float p_bad = 0.001;
    float p_bad_self = p_bad;
    float p_skip_self = 0.3;
    float p_third = (1.0f - p_bad_self) / 3;
    float p_km = 1.0f - p_skip_self;
    c.lp_mk = logf(p_skip);
    c.lp_mb = logf(p_bad);
    c.lp_bb = logf(p_bad_self);
    c.lp_bk = logf(p_third);
    c.lp_bm_next = logf(p_third);
    c.lp_bm_self = logf(p_third);
    c.lp_kk = logf(p_skip_self);
    c.lp_km = logf(p_km);
    c.log_inv_sqrt_2pi = (float)log(0.3989422804014327);
}

inline float2 read_transitions(double events_per_base, double indel_bias)
{
    double epb = events_per_base * indel_bias;
    epb = std::max(1.25, epb);
    float p_stay = (float)(1 - (1 / epb));
    float p_skip = 0.0025;
    float p_bad = 0.001;
    float p_mm_next = 1.0f - p_stay - p_skip - p_bad;
    return make_float2(logf(p_stay), logf(p_mm_next));
}

int create_common(nph_ctx** out, int device, bool own_stream, cudaStream_t stream)
{
    if (!out) return NPH_ERR_INVALID;
    *out = nullptr;
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev <= 0) return NPH_ERR_NO_DEVICE;
    if (device < 0 || device >= n_dev) return NPH_ERR_INVALID;
    nph_ctx* ctx = new (std::nothrow) nph_ctx();
    if (!ctx) return NPH_ERR_NOMEM;
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return NPH_ERR_NO_DEVICE; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return NPH_ERR_CUDA; }
    ctx->sm_count = prop.multiProcessorCount;
    if (own_stream) {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { ctx->stream = nullptr; delete ctx; return NPH_ERR_CUDA; }
        ctx->own_stream = true;
    } else {
        ctx->stream = stream;
    }
    // every allocation below is checked; a failure releases what exists so far through nph_destroy
    auto fail = [&](int rc) { nph_destroy(ctx); return rc; };
    if (cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_reset, cudaEventDisableTiming) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->cstream, cudaStreamNonBlocking) != cudaSuccess) return fail(NPH_ERR_CUDA);
    if (nph_reserve(ctx, ctx->d_progress, 1) != NPH_OK) return fail(NPH_ERR_NOMEM);
    if (cudaMallocHost((void**)&ctx->h_progress_vals, sizeof(uint32_t) * (nph_ctx::kLevelChunks + 1)) != cudaSuccess) {
        ctx->h_progress_vals = nullptr;
        return fail(NPH_ERR_NOMEM);
    }
    for (int i = 0; i <= nph_ctx::kLevelChunks; ++i) ctx->h_progress_vals[i] = (uint32_t)(i + 1);
    for (int i = 0; i < nph_ctx::kSideStreams; ++i) {
        if (cudaStreamCreateWithFlags(&ctx->side[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming) != cudaSuccess) return fail(NPH_ERR_CUDA);
    }

    // quantised log-sum table, built exactly like p7_FLogsumInit (ref: src/common/logsum.cpp:57-69)
    std::vector<float> tbl(NPH_TBL_SMEM);
    for (int i = 0; i < NPH_LOGSUM_CUT; ++i) tbl[i] = (float)log(1. + exp((double)-i / 1000.f));
    tbl[NPH_LOGSUM_CUT] = 0.0f;
    if (nph_reserve(ctx, ctx->d_logsum, NPH_TBL_SMEM) != NPH_OK) return fail(NPH_ERR_NOMEM);
    if (cudaMemcpy(ctx->d_logsum.p, tbl.data(), sizeof(float) * NPH_TBL_SMEM, cudaMemcpyHostToDevice) != cudaSuccess) return fail(NPH_ERR_CUDA);
    const_transitions(ctx->consts);
    if (nph_reserve(ctx, ctx->d_counters, NPH_NUM_COUNTERS) != NPH_OK) return fail(NPH_ERR_NOMEM);
    if (ensure_flank(ctx, 4096) != NPH_OK) return fail(NPH_ERR_CUDA);
    *out = ctx;
    return NPH_OK;
}

} // namespace

int nph_upload_read_transitions(nph_ctx* ctx, double indel_bias)
{
    std::vector<float2>& trans = ctx->h_stage_trans;
    trans.resize(ctx->n_reads);
    for (size_t i = 0; i < ctx->n_reads; ++i) trans[i] = read_transitions(ctx->h_events_per_base[i], indel_bias);
    NPH_TRY(nph_reserve(ctx, ctx->d_trans, ctx->n_reads));
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_trans.p, trans.data(), sizeof(float2) * ctx->n_reads, cudaMemcpyHostToDevice, ctx->stream));
    return NPH_OK;
}

extern "C" {

int nph_version(void) { return NPH_VERSION_MAJOR * 1000 + NPH_VERSION_MINOR; }

const char* nph_strerror(int status)
{
    switch (status) {
        case NPH_OK: return "ok";
        case NPH_ERR_NO_DEVICE: return "no usable CUDA device (libnph has no CPU path)";
        case NPH_ERR_CUDA: return "CUDA runtime error (see nph_last_error)";
        case NPH_ERR_INVALID: return "invalid argument";
        case NPH_ERR_NOMEM: return "out of memory";
        case NPH_ERR_STATE: return "call sequence error";
        case NPH_ERR_UNSUPPORTED: return "unsupported shape";
    }
    return "unknown status";
}

const char* nph_last_error(const nph_ctx* ctx) { return ctx ? ctx->last_error.c_str() : ""; }

int nph_create(nph_ctx** ctx_out, int device) { return create_common(ctx_out, device, true, nullptr); }
int nph_create_on_stream(nph_ctx** ctx_out, int device, void* cuda_stream)
{
    return create_common(ctx_out, device, false, (cudaStream_t)cuda_stream);
}

int nph_destroy(nph_ctx* ctx)
{
    if (!ctx) return NPH_ERR_INVALID;
    cudaSetDevice(ctx->device);
    if (ctx->stream || !ctx->own_stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_reset) cudaEventDestroy(ctx->ev_reset);
    if (ctx->cstream) { cudaStreamSynchronize(ctx->cstream); cudaStreamDestroy(ctx->cstream); }
    if (ctx->h_progress_vals) cudaFreeHost(ctx->h_progress_vals);
    for (int i = 0; i < nph_ctx::kSideStreams; ++i) { if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]); if (ctx->side[i]) cudaStreamDestroy(ctx->side[i]); }
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;                      // the device buffers free themselves
    return NPH_OK;
}

int nph_sync(nph_ctx* ctx)
{
    if (!ctx) return NPH_ERR_INVALID;
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NPH_OK;
}

void* nph_stream(nph_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int nph_model_upload(nph_ctx* ctx, const double* level_mean, const double* level_stdv,
                     const double* level_log_stdv, uint32_t n_states, uint32_t k,
                     uint32_t alphabet_size, uint32_t* model_id_out)
{
    if (!ctx || !level_mean || !level_stdv || !level_log_stdv || !model_id_out || n_states == 0) return NPH_ERR_INVALID;
    uint64_t expect = 1;
    for (uint32_t i = 0; i < k; ++i) expect *= alphabet_size;
    if (expect != n_states || k == 0 || k > 16 || alphabet_size == 0 || alphabet_size > 255) return NPH_ERR_INVALID;   // ref asserts states.size() == alphabet^k (profile_hmm_r9.inl:305)
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    DevModel m;
    const size_t bytes = sizeof(double) * n_states;
    NPH_TRY(nph_reserve(ctx, m.mean, n_states));
    NPH_TRY(nph_reserve(ctx, m.stdv, n_states));
    NPH_TRY(nph_reserve(ctx, m.log_stdv, n_states));
    NPH_CUDA(ctx, cudaMemcpyAsync(m.mean.p, level_mean, bytes, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(m.stdv.p, level_stdv, bytes, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(m.log_stdv.p, level_log_stdv, bytes, cudaMemcpyHostToDevice, ctx->stream));
    m.n_states = n_states; m.k = k; m.alphabet_size = alphabet_size;
    ctx->models.push_back(std::move(m));
    std::vector<DevModelView> views(ctx->models.size());
    for (size_t i = 0; i < views.size(); ++i)
        views[i] = DevModelView{ctx->models[i].mean.p, ctx->models[i].stdv.p, ctx->models[i].log_stdv.p, ctx->models[i].n_states,
                                (uint16_t)ctx->models[i].k, (uint16_t)ctx->models[i].alphabet_size};
    NPH_TRY(nph_reserve(ctx, ctx->d_models, views.size()));
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_models.p, views.data(), sizeof(DevModelView) * views.size(), cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *model_id_out = (uint32_t)ctx->models.size() - 1;
    return NPH_OK;
}

// Shared by the staged call (pipelined = false: everything on the context's stream, synchronous) and by the
// one-shot call (pipelined = true: read records on the main stream, event levels in chunks on the copy stream,
// each chunk followed by a progress word the forward kernel polls — so scoring starts while levels still arrive).
int nph_reads_load_impl(nph_ctx* ctx, const nph_read* reads, size_t n_reads,
                           const float* ev_mean, const double* ev_start_time, size_t n_events_total, bool pipelined)
{
    if (!ctx || !reads || !ev_mean || n_reads == 0) return NPH_ERR_INVALID;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    std::vector<DevRead>& hr = ctx->h_stage_reads;
    std::vector<double>& hd = ctx->h_stage_drift;
    hr.resize(n_reads);
    hd.resize(n_reads);
    ctx->h_events_per_base.resize(n_reads);
    ctx->h_read_n_events.resize(n_reads);
    bool any_drift = false;
    for (size_t i = 0; i < n_reads; ++i) {
        const nph_read& r = reads[i];
        if (r.n_events == 0 || r.n_events > n_events_total || r.event_off > n_events_total - r.n_events) return NPH_ERR_INVALID;
        hr[i].event_off = r.event_off; hr[i].n_events = r.n_events; hr[i].pad = 0;
        hr[i].scale = r.scale; hr[i].shift = r.shift; hr[i].var = r.var; hr[i].log_var = r.log_var;
        hd[i] = r.drift;
        any_drift |= (r.drift != 0.0);
        ctx->h_events_per_base[i] = r.events_per_base;
        ctx->h_read_n_events[i] = r.n_events;
    }
    if (any_drift && !ev_start_time) return NPH_ERR_INVALID;
    NPH_TRY(nph_reserve(ctx, ctx->d_reads, n_reads));
    NPH_TRY(nph_reserve(ctx, ctx->d_drift, n_reads));
    NPH_TRY(nph_reserve(ctx, ctx->d_level, n_events_total));
    ctx->n_reads = n_reads;
    ctx->n_events_total = n_events_total;
    ctx->level_chunk_events = 0;
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_reads.p, hr.data(), sizeof(DevRead) * n_reads, cudaMemcpyHostToDevice, ctx->stream));
    if (pipelined && !any_drift && n_events_total >= (size_t)1 << 20) {
        // drift == 0 everywhere: the drift-scaled level IS the event mean (level - time*0.0 narrows back exactly),
        // so levels go straight from the caller's buffer into d_level, chunk by chunk, behind progress words.
        size_t chunk = (n_events_total + nph_ctx::kLevelChunks - 1) / nph_ctx::kLevelChunks;
        chunk = (chunk + 31) / 32 * 32;                       // 128-byte lines never straddle two chunks
        ctx->level_chunk_events = chunk;
        NPH_CUDA(ctx, cudaMemsetAsync(ctx->d_progress.p, 0, sizeof(uint32_t), ctx->cstream));
        NPH_CUDA(ctx, cudaEventRecord(ctx->ev_reset, ctx->cstream));
        NPH_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_reset, 0));
        ctx->levels_inflight = true;
        ctx->ev_mean_resident = false;                        // only d_level is filled on this path
        return NPH_OK;                                         // chunks are queued by upload_level_chunks()
    }
    NPH_TRY(nph_reserve(ctx, ctx->d_ev_mean, n_events_total));
    ctx->ev_mean_resident = true;
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_drift.p, hd.data(), sizeof(double) * n_reads, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_ev_mean.p, ev_mean, sizeof(float) * n_events_total, cudaMemcpyHostToDevice, ctx->stream));
    if (any_drift) {
        NPH_TRY(nph_reserve(ctx, ctx->d_ev_time, n_events_total));
        NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_ev_time.p, ev_start_time, sizeof(double) * n_events_total, cudaMemcpyHostToDevice, ctx->stream));
        NPH_TRY(nph_launch_read_prologue(ctx));
    } else {
        // drift == 0 for every read: level - time*0.0 narrows back to level exactly, so the
        // drift-scaled level IS the event mean and the start times need not cross PCIe at all.
        NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_level.p, ctx->d_ev_mean.p, sizeof(float) * n_events_total, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NPH_OK;
}

int nph_upload_level_chunks(nph_ctx* ctx, const float* ev_mean)
{
    const size_t chunk = ctx->level_chunk_events, total = ctx->n_events_total;
    uint32_t c = 0;
    for (size_t off = 0; off < total; off += chunk, ++c) {
        const size_t n = std::min(chunk, total - off);
        NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_level.p + off, ev_mean + off, sizeof(float) * n, cudaMemcpyHostToDevice, ctx->cstream));
        NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_progress.p, ctx->h_progress_vals + c, sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->cstream));
    }
    return NPH_OK;
}

void nph_finish_level_upload(nph_ctx* ctx)
{
    if (!ctx->levels_inflight) return;
    cudaStreamSynchronize(ctx->cstream);
    ctx->levels_inflight = false;
    ctx->level_chunk_events = 0;
}

int nph_reads_load(nph_ctx* ctx, const nph_read* reads, size_t n_reads,
                   const float* ev_mean, const double* ev_start_time, size_t n_events_total)
{
    NPH_TRY(nph_reads_load_impl(ctx, reads, n_reads, ev_mean, ev_start_time, n_events_total, false));
    ctx->reads_loaded = true;
    ctx->jobs_loaded = false;
    ctx->abea_loaded = false;
    return NPH_OK;
}

// kmer_ranks != nullptr: ranks (uint32 per k-mer); else seq_codes (uint8 per base) — n_total counts whichever it is
static int jobs_upload_async(nph_ctx* ctx, const uint32_t* kmer_ranks, const uint8_t* seq_codes, size_t n_ranks_total,
                             const nph_hmm_job* jobs, size_t n_jobs, double indel_bias)
{
    if ((!kmer_ranks && !seq_codes) || !jobs) return NPH_ERR_INVALID;
    ctx->codes_mode = kmer_ranks == nullptr;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));

    if (ctx->codes_mode) NPH_TRY(nph_reserve(ctx, ctx->d_codes, n_ranks_total + 16));
    else NPH_TRY(nph_reserve(ctx, ctx->d_ranks, n_ranks_total));
    NPH_TRY(nph_reserve(ctx, ctx->d_jobs, n_jobs));
    NPH_TRY(nph_reserve(ctx, ctx->d_order, n_jobs));
    NPH_TRY(nph_reserve(ctx, ctx->d_scores, n_jobs));
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_jobs.p, jobs, sizeof(nph_hmm_job) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    if (ctx->codes_mode) NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_codes.p, seq_codes, n_ranks_total, cudaMemcpyHostToDevice, ctx->stream));
    else NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_ranks.p, kmer_ranks, sizeof(uint32_t) * n_ranks_total, cudaMemcpyHostToDevice, ctx->stream));
    return nph_upload_read_transitions(ctx, indel_bias);
}

int nph_jobs_schedule(nph_ctx* ctx, size_t n_jobs, size_t n_ranks_total)
{
    // validate + classify + schedule on the device (hmm_schedule.cu); synchronises the stream once
    uint32_t max_E = 1;
    NPH_TRY(nph_schedule_hmm_jobs(ctx, n_jobs, n_ranks_total, &max_E));
    NPH_TRY(ensure_flank(ctx, (size_t)max_E + 2));
    NPH_TRY(nph_reserve(ctx, ctx->d_scratch, nph_hmm_scratch_bytes(ctx)));
    ctx->n_jobs = n_jobs;
    ctx->n_ranks = n_ranks_total;
    ctx->jobs_loaded = true;
    return NPH_OK;
}

int nph_hmm_jobs_load(nph_ctx* ctx, const uint32_t* kmer_ranks, size_t n_ranks_total,
                      const nph_hmm_job* jobs, size_t n_jobs, double indel_bias)
{
    if (!ctx) return NPH_ERR_INVALID;
    if (n_jobs == 0) { ctx->n_jobs = 0; ctx->classes.clear(); ctx->jobs_loaded = true; return NPH_OK; }   // empty batch: nothing to score
    if (!ctx->reads_loaded) return NPH_ERR_STATE;
    NPH_TRY(jobs_upload_async(ctx, kmer_ranks, nullptr, n_ranks_total, jobs, n_jobs, indel_bias));
    return nph_jobs_schedule(ctx, n_jobs, n_ranks_total);
}

int nph_hmm_jobs_load_seq(nph_ctx* ctx, const uint8_t* seq_codes, size_t n_codes_total,
                          const nph_hmm_job* jobs, size_t n_jobs, double indel_bias)
{
    if (!ctx) return NPH_ERR_INVALID;
    if (n_jobs == 0) { ctx->n_jobs = 0; ctx->classes.clear(); ctx->jobs_loaded = true; return NPH_OK; }
    if (!ctx->reads_loaded) return NPH_ERR_STATE;
    if (!seq_codes) return NPH_ERR_INVALID;
    NPH_TRY(jobs_upload_async(ctx, nullptr, seq_codes, n_codes_total, jobs, n_jobs, indel_bias));
    return nph_jobs_schedule(ctx, n_jobs, n_codes_total);
}

int nph_hmm_score(nph_ctx* ctx, float* scores_dev)
{
    if (!ctx) return NPH_ERR_INVALID;
    if (!ctx->jobs_loaded) return NPH_ERR_STATE;
    if (ctx->n_jobs == 0) return NPH_OK;
    if (!ctx->reads_loaded) return NPH_ERR_STATE;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    return nph_launch_hmm_forward(ctx, scores_dev);
}

int nph_hmm_scores_fetch(nph_ctx* ctx, float* scores_out, size_t n_jobs)
{
    if (!ctx) return NPH_ERR_INVALID;
    if (n_jobs == 0) return NPH_OK;
    if (!scores_out) return NPH_ERR_INVALID;
    if (!ctx->jobs_loaded || n_jobs > ctx->n_jobs) return NPH_ERR_STATE;
    NPH_CUDA(ctx, cudaMemcpyAsync(scores_out, ctx->d_scores.p, sizeof(float) * n_jobs, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NPH_OK;
}

static int hmm_score_batch_impl(nph_ctx* ctx,
                                const nph_read* reads, size_t n_reads,
                                const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                                const uint32_t* kmer_ranks, const uint8_t* seq_codes, size_t n_ranks_total,
                                const nph_hmm_job* jobs, size_t n_jobs,
                                double indel_bias, float* scores_out)
{
    static const bool timing = getenv("NPH_TIMING") != nullptr;   // development aid: per-phase host wall time on stderr
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = now();
    if (!ctx) return NPH_ERR_INVALID;
    if (n_jobs == 0) return NPH_OK;                              // empty batch
    // Order of issue matters: small read records + jobs + ranks first (the scheduler needs only those), then the
    // event levels in chunks on the copy stream; the forward kernels start as soon as the schedule exists and wait
    // per job on the progress word of the chunk that holds their read (hmm_forward_kernel.cuh).
    ctx->levels_inflight = false;
    int rc = nph_reads_load_impl(ctx, reads, n_reads, ev_mean, ev_start_time, n_events_total, true);
    if (rc == NPH_OK) { ctx->reads_loaded = true; ctx->jobs_loaded = false; ctx->abea_loaded = false; }
    const double t1 = now();
    if (rc == NPH_OK) rc = jobs_upload_async(ctx, kmer_ranks, seq_codes, n_ranks_total, jobs, n_jobs, indel_bias);
    if (rc == NPH_OK && ctx->levels_inflight) rc = nph_upload_level_chunks(ctx, ev_mean);
    if (rc == NPH_OK) rc = nph_jobs_schedule(ctx, n_jobs, n_ranks_total);
    const double t2 = now();
    if (rc == NPH_OK) rc = nph_hmm_score(ctx, nullptr);
    if (rc == NPH_OK) rc = nph_hmm_scores_fetch(ctx, scores_out, n_jobs);
    nph_finish_level_upload(ctx);                                // also on error paths: never leave copies in flight
    const double t3 = now();
    if (timing) fprintf(stderr, "[nph] reads %.2f ms  jobs+schedule %.2f ms  score+fetch %.2f ms\n", t1 - t0, t2 - t1, t3 - t2);
    return rc;
}

int nph_hmm_score_batch(nph_ctx* ctx,
                        const nph_read* reads, size_t n_reads,
                        const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                        const uint32_t* kmer_ranks, size_t n_ranks_total,
                        const nph_hmm_job* jobs, size_t n_jobs,
                        double indel_bias, float* scores_out)
{
    if (n_jobs && !kmer_ranks) return NPH_ERR_INVALID;
    return hmm_score_batch_impl(ctx, reads, n_reads, ev_mean, ev_start_time, n_events_total, kmer_ranks, nullptr, n_ranks_total, jobs, n_jobs, indel_bias, scores_out);
}

int nph_hmm_score_batch_seq(nph_ctx* ctx,
                            const nph_read* reads, size_t n_reads,
                            const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                            const uint8_t* seq_codes, size_t n_codes_total,
                            const nph_hmm_job* jobs, size_t n_jobs,
                            double indel_bias, float* scores_out)
{
    if (n_jobs && !seq_codes) return NPH_ERR_INVALID;
    return hmm_score_batch_impl(ctx, reads, n_reads, ev_mean, ev_start_time, n_events_total, nullptr, seq_codes, n_codes_total, jobs, n_jobs, indel_bias, scores_out);
}

// profile_hmm_score_set's combination step (ref: src/hmm/nanopolish_profile_hmm.cpp:32-56): host
// arithmetic on already-computed scores, in double through the quantised table logsum.
int nph_score_set_combine(const float* scores, size_t n_groups, uint32_t n_alt, float* out)
{
    if (!scores || !out || n_alt == 0) return NPH_ERR_INVALID;
    // C++11 function-local static: initialised exactly once even when OpenMP threads race into the first call
    struct Table {
        float v[NPH_LOGSUM_TBL];
        Table() { for (int i = 0; i < NPH_LOGSUM_TBL; ++i) v[i] = (float)log(1. + exp((double)-i / 1000.f)); }
    };
    static const Table table;
    const float* tbl = table.v;
    const double pen = log((double)n_alt);
    for (size_t g = 0; g < n_groups; ++g) {
        double score = scores[g * n_alt] - pen;
        for (uint32_t i = 1; i < n_alt; ++i) {
            const double alt = scores[g * n_alt + i] - pen;
            const float a = (float)score, b = (float)alt;
            const float mx = a > b ? a : b, mn = a < b ? a : b;
            // !(d < 15.7f) also catches NaN / inf differences (a NaN or +inf score): no out-of-range table index, like the device path's clamp
            const float d = mx - mn;
            score = (mn == -INFINITY || !(d < 15.7f)) ? mx : mx + tbl[(int)(d * 1000.f)];
        }
        out[g] = (float)score;
    }
    return NPH_OK;
}

int nph_last_kernel_ms(nph_ctx* ctx, float* ms_out, int* launches_out)
{
    if (!ctx || !ms_out) return NPH_ERR_INVALID;
    if (!ctx->timing_valid) return NPH_ERR_STATE;
    if (ctx->timing_valid == 2) *ms_out = ctx->staged_ms;
    else {
        NPH_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
        NPH_CUDA(ctx, cudaEventElapsedTime(ms_out, ctx->ev0, ctx->ev1));
    }
    if (launches_out) *launches_out = ctx->last_launches;
    return NPH_OK;
}

int nph_host_alloc(void** ptr_out, size_t bytes)
{
    if (!ptr_out) return NPH_ERR_INVALID;
    cudaError_t e = cudaMallocHost(ptr_out, bytes);
    if (e != cudaSuccess) return e == cudaErrorMemoryAllocation ? NPH_ERR_NOMEM : NPH_ERR_NO_DEVICE;
    return NPH_OK;
}

int nph_host_free(void* ptr)
{
    return cudaFreeHost(ptr) == cudaSuccess ? NPH_OK : NPH_ERR_CUDA;
}

} // extern "C"
