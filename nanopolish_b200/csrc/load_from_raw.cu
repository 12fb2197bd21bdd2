// load_from_raw.cu — SURVEY.md section 8(f) row N4: the whole read prologue of SquiggleRead::load_from_raw
// (src/nanopolish_squiggle_read.cpp:226-336) for a batch of raw reads in ONE call, chained on the device:
//
//   raw samples --trim_kernel--> ranges --ed_* kernels--> events --convert_kernel--> SquiggleEvent arrays (compact)
//      --mom_kernel--> shift/scale --abea_kernel--> aligned pairs --recalibrate_kernel--> base_to_event_map, scalings, QC
//
// The raw samples cross PCIe once and the events never leave the device between the steps; what comes back is what a
// SquiggleRead keeps (event mean/stdv/start_time/duration, the event map, the scalings and the QC verdict).  The host
// takes part twice, with a few bytes per read: after the trim (which reads survive) and after event detection (the
// event counts size the compact layout, ABEA's band storage and — through host libm, like the reference — ABEA's
// per-read transition log-probabilities).
#include "nph_internal.cuh"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

namespace {

constexpr int kConvWarps = 8;

struct ConvParams {
    const nph_event* events;         // capacity layout: read t at cap_off[t]
    const uint64_t* cap_off;
    const uint64_t* out_off;         // compact layout
    const uint32_t* n_events;
    const double* sample_rate;
    uint32_t n_reads;
    int reverse;                     // direct RNA: event i lands at n-1-i (std::reverse, squiggle_read.cpp:262-265)
    float* mean; float* stdv; float* duration; float* level;
    double* start_time;
    DevRead* reads;
};

// events -> SquiggleEvent fields (squiggle_read.cpp:243-250): duration = (float)(length / sample_rate), start_time the
// running FP64 sum of the float durations (folded in event order by one lane), and the device read record ABEA uses
// (scalings of a fresh read: scale 1, shift 0, var 1; drift 0 makes the drift-scaled level the mean itself).
__global__ void __launch_bounds__(kConvWarps * 32) convert_kernel(const ConvParams p)
{
    __shared__ float s_d[kConvWarps][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    for (uint32_t t = blockIdx.x * kConvWarps + wib; t < p.n_reads; t += gridDim.x * kConvWarps) {
        const nph_event* ev = p.events + p.cap_off[t];
        const uint64_t o = p.out_off[t];
        const uint32_t n = p.n_events[t];
        const double rate = p.sample_rate[t];
        double acc = 0.0;
        for (uint32_t i0 = 0; i0 < n; i0 += 32) {
            const uint32_t i = i0 + lane;
            const uint64_t oi = o + (p.reverse ? n - 1 - i : i);
            float d = 0.0f;
            if (i < n) {
                const nph_event e = ev[i];
                d = (float)__ddiv_rn((double)e.length, rate);
                p.mean[oi] = e.mean; p.level[oi] = e.mean; p.stdv[oi] = e.stdv; p.duration[oi] = d;
            }
            s_d[wib][lane] = d;
            __syncwarp();
            // every lane folds the same 32 values in order (identical rounding in all lanes), keeping its own prefix
            double mine = acc;
            const int cnt = (int)min(32u, n - i0);
            for (int j = 0; j < cnt; ++j) {
                if (j == lane) mine = acc;
                acc = __dadd_rn(acc, (double)s_d[wib][j]);
            }
            if (i < n) p.start_time[oi] = mine;
            __syncwarp();
        }
        if (lane == 0) {
            DevRead r;
            r.event_off = o; r.n_events = n; r.pad = 0; r.scale = 1.0; r.shift = 0.0; r.var = 1.0; r.log_var = 0.0;
            p.reads[t] = r;
        }
    }
}

// MoM estimate into the device read records (set4(shift, scale, 0, 1)) and the nph_read view the calibration reads
__global__ void apply_mom_kernel(const double* mom, DevRead* reads, nph_read* views, uint32_t n)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    DevRead r = reads[t];
    r.shift = mom[2 * t]; r.scale = mom[2 * t + 1];
    reads[t] = r;
    nph_read v;
    v.event_off = r.event_off; v.n_events = r.n_events; v.reserved = 0;
    v.scale = r.scale; v.shift = r.shift; v.drift = 0.0; v.var = 1.0; v.log_var = 0.0; v.events_per_base = 0.0;
    views[t] = v;
}

} // namespace

extern "C" int nph_load_from_raw_batch(nph_ctx* ctx, const float* raw, size_t n_samples_total,
                                       const uint32_t* kmer_ranks, size_t n_ranks_total,
                                       const nph_raw_job* jobs, size_t n_jobs, uint32_t model_id, const nph_event_params* params,
                                       uint64_t* event_off_out, float* ev_mean_out, float* ev_stdv_out, double* ev_start_time_out,
                                       float* ev_duration_out, size_t events_cap,
                                       nph_event_range* base_to_event_out, nph_calibration* calibrations_out)
{
    if (!ctx || !params) return NPH_ERR_INVALID;
    if (n_jobs == 0) return NPH_OK;
    if (!raw || !kmer_ranks || !jobs || !event_off_out || !ev_mean_out || !ev_stdv_out || !ev_start_time_out || !ev_duration_out || !calibrations_out)
        return NPH_ERR_INVALID;
    if (model_id >= ctx->models.size()) return NPH_ERR_INVALID;
    const uint32_t n_states = ctx->models[model_id].n_states;
    for (size_t j = 0; j < n_jobs; ++j) {
        const nph_raw_job& jb = jobs[j];
        if (jb.sample_off + jb.n_samples > n_samples_total || jb.n_kmers == 0 || jb.rank_off + jb.n_kmers > n_ranks_total || !(jb.sample_rate > 0.0))
            return NPH_ERR_INVALID;
    }
    uint32_t max_rank = 0;
    for (size_t i = 0; i < n_ranks_total; ++i) max_rank = std::max(max_rank, kmer_ranks[i]);     // branch-free: vectorises
    if (max_rank >= n_states) return NPH_ERR_INVALID;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    ctx->reads_loaded = false; ctx->jobs_loaded = false; ctx->abea_loaded = false;    // resident batches are replaced

    // ---- 1. raw samples up once; trim (defaults hard-coded at the reference's call site) ----
    std::vector<nph_raw_read> rr(n_jobs);
    size_t cap_total = 0;
    for (size_t j = 0; j < n_jobs; ++j) { rr[j] = nph_raw_read{jobs[j].sample_off, 0, jobs[j].n_samples, 0}; cap_total += jobs[j].n_samples / 2 + 8; }
    // the arena holds the trim's scratch, then (from its start again) the detector's and the conversion's per-read arrays;
    // it is reserved for the larger of the two, the latter as if every read survived the trim whole
    TrimScratch ts;
    EdScratch es;
    struct { uint64_t *cap_off, *out_off; double* rate; } conv{};
    auto trim_layout = [&](NphCarve& a) { ts = nph_trim_layout(a, rr.data(), n_jobs, 100); };
    auto ed_layout = [&](NphCarve& a, size_t n_reads, size_t events_total) {
        es = nph_ed_layout(a, n_reads, events_total);
        conv.cap_off = a.take<uint64_t>(n_reads);
        conv.out_off = a.take<uint64_t>(n_reads);
        conv.rate = a.take<double>(n_reads);
    };
    // the samples get a buffer of their own so that they outlive the call (nph_polya_after_load reads them)
    nph_ctx::LoadedRaw& kept = ctx->loaded_raw;
    kept.valid = false;
    NPH_TRY(nph_reserve(ctx, kept.d_raw, std::max<size_t>(nph_align256(sizeof(float) * n_samples_total) / sizeof(float), 1)));
    const size_t arena_bytes = std::max(nph_measure(trim_layout), nph_measure([&](NphCarve& a) { ed_layout(a, n_jobs, cap_total); }));
    NPH_TRY(nph_borrow_arena(ctx, [&](NphCarve& a) { a.take<uint8_t>(arena_bytes); }));
    NPH_TRY(nph_carve(ctx, ctx->d_arena, trim_layout));
    float* d_raw = kept.d_raw.p;
    NPH_CUDA(ctx, cudaMemcpyAsync(d_raw, raw, sizeof(float) * n_samples_total, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    int launches = 0;
    float staged_ms = 0.0f, ms = 0.0f;          // device time of the stages, summed (each stage ends in a sync)
    std::vector<nph_raw_range> range(n_jobs);
    NPH_TRY(nph_trim_device(ctx, d_raw, n_samples_total, rr.data(), n_jobs, 200, 10, 100, 0.0f, ts, range.data())); ++launches;
    ctx->h_last_trim = range;                   // for nph_last_trim_ranges (SRF_LOAD_RAW_SAMPLES keeps rt.raw[rt.start .. rt.end))
    NPH_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1)); staged_ms += ms;
    const bool verbose = getenv("NPH_TIMING") != nullptr;
    if (verbose) fprintf(stderr, "[nph] load_from_raw: trim %.2f ms", ms);

    // outputs of the reads that do not get as far as alignment
    for (size_t j = 0; j < n_jobs; ++j) {
        nph_calibration c{};
        c.shift = 0.0; c.scale = 1.0; c.drift = 0.0; c.var = 1.0; c.events_per_base = 0.0; c.n_used = 0;
        c.status = NPH_CAL_EMPTY_AFTER_TRIM | NPH_CAL_NOT_ALIGNED;
        calibrations_out[j] = c;
    }
    std::vector<uint32_t> live;
    for (size_t j = 0; j < n_jobs; ++j) if (range[j].end > range[j].start) live.push_back((uint32_t)j);
    kept.jobs.assign(jobs, jobs + n_jobs);
    kept.live_index.assign(n_jobs, -1);
    for (size_t t = 0; t < live.size(); ++t) kept.live_index[live[t]] = (int64_t)t;
    kept.n_samples_total = n_samples_total; kept.n_ranks_total = n_ranks_total;
    kept.d_duration = nullptr; kept.d_b2e = nullptr; kept.d_cal = nullptr;
    if (live.empty()) {
        if (base_to_event_out) for (size_t i = 0; i < n_ranks_total; ++i) base_to_event_out[i] = nph_event_range{-1, -1};
        for (size_t j = 0; j <= n_jobs; ++j) event_off_out[j] = 0;
        kept.event_off.assign(n_jobs + 1, 0);
        kept.valid = true;
        ctx->last_launches = launches; ctx->staged_ms = staged_ms; ctx->timing_valid = 2;
        return NPH_OK;
    }
    const size_t nl = live.size();

    // ---- 2. event detection over the surviving ranges (events stay on the device) ----
    std::vector<nph_raw_read> tr(nl);
    std::vector<uint64_t> cap_off(nl);
    uint64_t room = 0;
    for (size_t t = 0; t < nl; ++t) {
        const uint32_t j = live[t], ns = range[j].end - range[j].start;
        cap_off[t] = room;
        tr[t] = nph_raw_read{jobs[j].sample_off + range[j].start, room, ns, ns / 2 + 8};   // >= 3 samples between boundaries
        room += ns / 2 + 8;
    }
    NPH_TRY(nph_carve(ctx, ctx->d_arena, [&](NphCarve& a) { ed_layout(a, nl, room); }));
    std::vector<uint32_t> counts;
    int ed_launches = 0;
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    NPH_TRY(nph_detect_events_device(ctx, d_raw, n_samples_total, tr.data(), nl, params, es, room, counts, &ed_launches));
    launches += ed_launches;
    NPH_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1)); staged_ms += ms;
    if (verbose) fprintf(stderr, "  events %.2f ms", ms);

    // ---- 3. compact layout, SquiggleEvent conversion, outputs of the event arrays ----
    std::vector<uint64_t> out_off(nl + 1, 0);
    for (size_t t = 0; t < nl; ++t) out_off[t + 1] = out_off[t] + counts[t];
    const uint64_t n_events_total = out_off[nl];
    {
        uint64_t acc = 0;
        size_t t = 0;
        for (size_t j = 0; j < n_jobs; ++j) {
            event_off_out[j] = acc;
            if (t < nl && live[t] == j) { acc += counts[t]; ++t; }
        }
        event_off_out[n_jobs] = acc;
    }
    if (n_events_total > events_cap) { ctx->last_error = "nph_load_from_raw_batch: events_cap too small (n_samples_total / 3 always suffices)"; return NPH_ERR_UNSUPPORTED; }
    uint64_t n_live_ranks = 0, pairs_total = 0;
    std::vector<nph_abea_job> aj(nl);
    for (size_t t = 0; t < nl; ++t) {
        const nph_raw_job& jb = jobs[live[t]];
        aj[t] = nph_abea_job{jb.rank_off, pairs_total, (uint32_t)t, jb.n_kmers, counts[t] + jb.n_kmers, 0};
        pairs_total += aj[t].pairs_cap;
        n_live_ranks += jb.n_kmers;
    }
    (void)n_live_ranks;
    NPH_TRY(nph_reserve(ctx, ctx->d_ev_mean, n_events_total));
    ctx->ev_mean_resident = true;
    NPH_TRY(nph_reserve(ctx, ctx->d_ev_time, n_events_total));
    NPH_TRY(nph_reserve(ctx, ctx->d_level, n_events_total));
    NPH_TRY(nph_reserve(ctx, ctx->d_reads, nl));
    struct { float *stdv, *dur; double* mom; nph_read* views; nph_event_range* b2e; nph_calibration* cal; int* bad; } d{};
    auto prep_layout = [&](NphCarve& a) {
        d.stdv = a.take<float>(n_events_total);
        d.dur = a.take<float>(n_events_total);
        d.mom = a.take<double>(2 * nl);
        d.views = a.take<nph_read>(nl);
        d.b2e = a.take<nph_event_range>(n_ranks_total);
        d.cal = a.take<nph_calibration>(nl);
        d.bad = a.take<int>(1);
    };
    NPH_TRY(nph_lay_out(ctx, ctx->d_prep, prep_layout));
    {
        std::vector<double> rate(nl);
        for (size_t t = 0; t < nl; ++t) rate[t] = jobs[live[t]].sample_rate;
        NPH_CUDA(ctx, cudaMemcpyAsync(conv.cap_off, cap_off.data(), sizeof(uint64_t) * nl, cudaMemcpyHostToDevice, ctx->stream));
        NPH_CUDA(ctx, cudaMemcpyAsync(conv.out_off, out_off.data(), sizeof(uint64_t) * nl, cudaMemcpyHostToDevice, ctx->stream));
        NPH_CUDA(ctx, cudaMemcpyAsync(conv.rate, rate.data(), sizeof(double) * nl, cudaMemcpyHostToDevice, ctx->stream));
        ConvParams cp{};
        cp.events = es.events; cp.cap_off = conv.cap_off; cp.out_off = conv.out_off; cp.n_events = es.n_events; cp.sample_rate = conv.rate; cp.n_reads = (uint32_t)nl; cp.reverse = params->reverse_events ? 1 : 0;
        cp.mean = ctx->d_ev_mean.p; cp.stdv = d.stdv; cp.duration = d.dur; cp.level = ctx->d_level.p; cp.start_time = ctx->d_ev_time.p; cp.reads = ctx->d_reads.p;
        NPH_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
        convert_kernel<<<(unsigned)std::min<size_t>((nl + kConvWarps - 1) / kConvWarps, (size_t)ctx->sm_count * 8), kConvWarps * 32, 0, ctx->stream>>>(cp); ++launches;
        NPH_CUDA(ctx, cudaGetLastError());
        NPH_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        // rate[] etc. must outlive the copies: the stream is synchronised below before they go out of scope
        NPH_CUDA(ctx, cudaMemcpyAsync(ev_mean_out, ctx->d_ev_mean.p, sizeof(float) * n_events_total, cudaMemcpyDeviceToHost, ctx->stream));
        NPH_CUDA(ctx, cudaMemcpyAsync(ev_stdv_out, d.stdv, sizeof(float) * n_events_total, cudaMemcpyDeviceToHost, ctx->stream));
        NPH_CUDA(ctx, cudaMemcpyAsync(ev_start_time_out, ctx->d_ev_time.p, sizeof(double) * n_events_total, cudaMemcpyDeviceToHost, ctx->stream));
        NPH_CUDA(ctx, cudaMemcpyAsync(ev_duration_out, d.dur, sizeof(float) * n_events_total, cudaMemcpyDeviceToHost, ctx->stream));
        NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        NPH_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1)); staged_ms += ms;
        if (verbose) fprintf(stderr, "  convert %.2f ms", ms);
    }

    // ---- 4. MoM scalings and event alignment (the arena becomes ABEA's band storage) ----
    ctx->n_reads = nl;
    ctx->n_events_total = n_events_total;
    ctx->h_read_n_events.assign(counts.begin(), counts.end());
    ctx->reads_loaded = true;                      // for the staged ABEA calls below; cleared again before returning
    int rc = nph_abea_jobs_load(ctx, kmer_ranks, n_ranks_total, aj.data(), nl, model_id, pairs_total);
    if (rc == NPH_OK) rc = nph_launch_mom(ctx, d.mom, params->reverse_events != 0);
    if (rc == NPH_OK) {
        apply_mom_kernel<<<(unsigned)((nl + 127) / 128), 128, 0, ctx->stream>>>(d.mom, ctx->d_reads.p, d.views, (uint32_t)nl);
        launches += 2;
        if (cudaGetLastError() != cudaSuccess) rc = NPH_ERR_CUDA;
    }
    if (rc == NPH_OK) { rc = nph_launch_abea(ctx); ++launches; }
    ctx->reads_loaded = false;
    ctx->abea_loaded = false;
    if (rc != NPH_OK) return rc;

    // ---- 5. base_to_event_map, events_per_base, recalibration, QC ----
    NPH_CUDA(ctx, cudaMemsetAsync(d.b2e, 0xff, sizeof(nph_event_range) * n_ranks_total, ctx->stream));
    NphCalArgs ca{};
    ca.ev_mean = ctx->d_ev_mean.p; ca.reads = d.views; ca.ranks = ctx->d_abea_ranks.p; ca.jobs = ctx->d_abea_jobs.p;
    ca.results = ctx->d_abea_res.p; ca.pairs = ctx->d_pairs.p; ca.n_jobs = (uint32_t)nl; ca.model_id = model_id;
    ca.b2e = d.b2e; ca.out = d.cal; ca.bad_input = d.bad;
    NPH_TRY(nph_launch_recalibrate(ctx, ca)); ++launches;
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    std::vector<nph_calibration> cal(nl);
    NPH_CUDA(ctx, cudaMemcpyAsync(cal.data(), d.cal, sizeof(nph_calibration) * nl, cudaMemcpyDeviceToHost, ctx->stream));
    if (base_to_event_out)
        NPH_CUDA(ctx, cudaMemcpyAsync(base_to_event_out, d.b2e, sizeof(nph_event_range) * n_ranks_total, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (size_t t = 0; t < nl; ++t) calibrations_out[live[t]] = cal[t];
    kept.event_off.assign(event_off_out, event_off_out + n_jobs + 1);
    kept.d_duration = d.dur; kept.d_b2e = d.b2e; kept.d_cal = d.cal;
    kept.valid = true;
    NPH_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1)); staged_ms += ms;     // ev0 was recorded at the ABEA launch
    if (verbose) fprintf(stderr, "  abea+calibration %.2f ms  (total %.2f ms, %zu of %zu reads aligned)\n", ms, staged_ms, nl, n_jobs);
    ctx->last_launches = launches;
    ctx->staged_ms = staged_ms;
    ctx->timing_valid = 2;
    return NPH_OK;
}

extern "C" int nph_last_trim_ranges(nph_ctx* ctx, nph_raw_range* ranges_out, size_t n_jobs)
{
    if (!ctx || !ranges_out) return NPH_ERR_INVALID;
    if (n_jobs != ctx->h_last_trim.size()) return NPH_ERR_STATE;
    std::copy(ctx->h_last_trim.begin(), ctx->h_last_trim.end(), ranges_out);
    return NPH_OK;
}
