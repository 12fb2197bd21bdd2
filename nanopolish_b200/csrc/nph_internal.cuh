// nph_internal.cuh — shared declarations of libnph.so (not installed; the public surface is include/nph.h)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <string>
#include <vector>
#include <algorithm>
#include "../../include/nph.h"

#define NPH_LOGSUM_TBL 16000        // ref: p7_LOGSUM_TBL, src/common/logsum.h:20
#define NPH_LOGSUM_CUT 15700        // (max-min) >= 15.7f returns max: entries >= 15700 are never read
#define NPH_TBL_SMEM   (NPH_LOGSUM_CUT + 1)   // +1: a zero entry that the clamped index lands on
#define NPH_NUM_COUNTERS 64          // work-queue counters: one per forward class (<= 40) + ABEA (last)

// Per-read record on the device (what the kernels need of nph_read after the prologue).
struct DevRead {
    uint64_t event_off;
    uint32_t n_events;
    uint32_t pad;
    double scale, shift, var, log_var;
};

// The eight read-independent transition log-probabilities + Gaussian constant, computed on the host
// with libm exactly as the reference does (logf of float probabilities).
struct HmmConsts {
    float lp_mk, lp_mb, lp_bb, lp_bk, lp_bm_next, lp_bm_self, lp_kk, lp_km;
    float log_inv_sqrt_2pi;
};

struct DevModel {
    double* mean = nullptr;
    double* stdv = nullptr;
    double* log_stdv = nullptr;
    uint32_t n_states = 0, k = 0, alphabet_size = 0;
};

// Device-side view of the models for kernels (array of pointers)
struct DevModelView { const double* mean; const double* stdv; const double* log_stdv; uint32_t n_states; uint16_t k; uint16_t alphabet_size; };

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;   // elements
};

struct nph_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 0;
    std::string last_error;

    // constant tables
    float* d_logsum = nullptr;       // NPH_TBL_SMEM floats
    DevBuf<float> d_flank;           // clip-penalty table, grown on demand
    std::vector<float> h_flank;
    HmmConsts consts;

    // models
    std::vector<DevModel> models;
    DevBuf<DevModelView> d_models;

    // resident reads
    size_t n_reads = 0, n_events_total = 0;
    DevBuf<DevRead> d_reads;
    DevBuf<float> d_ev_mean;
    DevBuf<double> d_ev_time;
    DevBuf<float> d_level;           // drift-scaled levels
    DevBuf<double> d_drift;          // per read SquiggleScalings::drift (consumed by the read prologue)
    std::vector<double> h_events_per_base;
    std::vector<uint32_t> h_read_n_events;
    bool reads_loaded = false;
    bool ev_mean_resident = false;   // d_ev_mean holds this batch's raw event means (false after the pipelined one-shot score, which fills d_level only)

    // resident HMM jobs
    size_t n_jobs = 0, n_ranks = 0;
    DevBuf<uint32_t> d_ranks;
    DevBuf<uint8_t> d_codes;         // jobs loaded through the *_seq calls: base codes instead of k-mer ranks (jobs' rank_off index this)
    bool codes_mode = false;
    bool jobs_trusted = false;       // the resident jobs and their ranks were written by a kernel of ours (methylation.cu, variants.cu): the
                                     // scheduler validates the jobs' read / event ranges but does not walk their ranks again
    DevBuf<uint64_t> d_rank_base;    // base-code jobs: where each job's ranks start in d_ranks (hmm_schedule.cu)
    DevBuf<nph_hmm_job> d_jobs;
    DevBuf<float2> d_trans;          // per read: (lp_mm_self, lp_mm_next)
    DevBuf<uint32_t> d_order;        // job indices grouped by kernel class, heavy first
    DevBuf<float> d_scores;
    DevBuf<unsigned int> d_counters;
    DevBuf<uint8_t> d_sched_cls;     // per job: kernel class
    DevBuf<uint16_t> d_sched_bkt;    // per job: schedule key bucket
    DevBuf<unsigned int> d_sched_hist;   // histogram + offsets + summary
    DevBuf<uint8_t> d_scratch;
    struct ClassLaunch { int cols_per_lane; int group_width; bool chained; size_t first; size_t count; double cost; };
    std::vector<ClassLaunch> classes;
    uint32_t max_kpad = 0, max_period = 0;
    bool jobs_loaded = false;

    // resident ABEA jobs
    size_t n_abea_jobs = 0, abea_pairs_total = 0;
    uint32_t abea_model = 0;
    DevBuf<nph_abea_job> d_abea_jobs;
    DevBuf<uint32_t> d_abea_ranks;
    DevBuf<nph_aligned_pair> d_pairs;
    DevBuf<nph_abea_result> d_abea_res;
    DevBuf<uint8_t> d_abea_scratch;
    DevBuf<uint32_t> d_abea_order;
    DevBuf<double> d_abea_consts;    // per job (lp_stay, lp_step); also the MoM output buffer
    DevBuf<uint8_t> d_prep;          // load_from_raw: event SoA staging, MoM output, calibration buffers
    uint32_t abea_kmax = 0;
    uint64_t abea_trace_stride = 0;
    bool abea_loaded = false;

    // resident call-methylation batch (methylation.cu)
    struct MethState {
        bool loaded = false, ran = false;
        size_t n_records = 0, n_ref = 0, n_pairs = 0, prov_total = 0;
        nph_meth_params params{};
        double indel_bias = 1.0;
        uint64_t n_sites = 0, n_ranks = 0, n_scored_events = 0;
        DevBuf<uint8_t> d_ref;
        DevBuf<nph_aligned_pair> d_pairs;
        bool compact = false;              // event alignments came as int16 deltas per reference base (nph_methylation_load_compact)
        DevBuf<uint16_t> d_deltas;         // int16 deltas, n_ref entries
        DevBuf<uint32_t> d_dense;          // int32 event index per reference base after the prefix sum (INT32_MIN: no pair), then per record: first_event, first valid offset
        DevBuf<nph_meth_record> d_records;
        DevBuf<uint64_t> d_prov_off;       // n_records + 1: where each record's provisional group rows start
        DevBuf<uint8_t> d_prov;            // provisional group rows (MethGroup)
        DevBuf<uint64_t> d_counts;         // per record: groups, ranks (2 x n_records), then the prefix arrays and the summary
        DevBuf<nph_meth_site> d_sites;
        DevBuf<uint8_t> d_tsv_in;          // nph_methylation_tsv: contig, read names, name offsets, strand flags
        DevBuf<uint64_t> d_tsv_off;        // bytes of each record's rows, then their exclusive prefix (n_records + 1) and the flags word
        DevBuf<uint8_t> d_tsv;             // the rows
        std::vector<uint64_t> h_prov_off;
    } meth;

    // resident variant-screening batch (variants.cu)
    struct ScreenState {
        bool loaded = false, ran = false;
        nph_screen_params params{};
        double indel_bias = 1.0;
        size_t n_pos = 0, n_records = 0, n_ref = 0, n_deltas = 0;
        uint32_t n_rounds = 0;
        uint64_t n_jobs = 0, n_scored_events = 0, n_jobs_no_exit = 0, n_reference_events = 0;
        DevBuf<uint8_t> d_ref;
        DevBuf<uint16_t> d_deltas;
        DevBuf<uint32_t> d_dense;          // event index per reference base of every record, then first_event, first valid
        DevBuf<nph_meth_record> d_records;
        DevBuf<uint64_t> d_pos_off;        // n_pos + 1: where each position's bounded reads start
        DevBuf<uint8_t> d_pos_reads;       // {record, e1, e2} per bounded read
        DevBuf<uint8_t> d_state;           // per position: totals (9 doubles), alive mask, reads done, valid mask
        DevBuf<uint64_t> d_job_off;        // per position: first job of the round (+ totals)
    } screen;

    // measurement
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // side streams so that the tail of one forward class overlaps the head of the next (fork/join by events)
    static const int kSideStreams = 4;
    cudaStream_t side[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[4] = {nullptr, nullptr, nullptr, nullptr};
    int last_launches = 0;
    int timing_valid = 0;            // 0 none, 1 = ev0..ev1, 2 = staged_ms (a call with host round trips between its kernels)
    float staged_ms = 0.0f;

    // pipelined level upload of the one-shot call: copy stream, progress word polled by the forward kernel
    static const int kLevelChunks = 8;
    cudaStream_t cstream = nullptr;
    cudaEvent_t ev_reset = nullptr;
    uint32_t* d_progress = nullptr;          // number of level chunks that have landed
    uint32_t* h_progress_vals = nullptr;     // pinned {1, 2, ...}: sources of the progress writes
    size_t level_chunk_events = 0;           // 0 = levels fully resident, kernels do not poll
    bool levels_inflight = false;
    std::vector<DevRead> h_stage_reads;      // host staging that must outlive async copies
    std::vector<double> h_stage_drift;
    std::vector<float2> h_stage_trans;
    std::vector<nph_raw_range> h_last_trim;  // surviving sample range per job of the last nph_load_from_raw_batch

    // what the last nph_load_from_raw_batch leaves for nph_polya_after_load (polya.cu): the raw samples in their own buffer,
    // the compact event durations, the event map and the calibrations in d_prep (valid until d_prep is reused)
    struct LoadedRaw {
        bool valid = false;
        DevBuf<float> d_raw;                 // every raw sample of the call, as uploaded
        const float* d_duration = nullptr;   // compact job order over the live reads
        const nph_event_range* d_b2e = nullptr;
        const nph_calibration* d_cal = nullptr;   // live-read order
        std::vector<nph_raw_job> jobs;
        std::vector<int64_t> live_index;     // per job: index among the live reads, -1 if nothing survived the trim
        std::vector<uint64_t> event_off;     // per job: first event in the compact layout (n_jobs + 1)
        size_t n_samples_total = 0, n_ranks_total = 0;
    } loaded_raw;
    DevBuf<uint8_t> d_polya;                 // polya.cu: jobs, results, backpointers, per-k-mer durations (+ inputs of the one-shot call)

};

int nph_set_cuda_error(nph_ctx* ctx, cudaError_t e, const char* what);
#define NPH_CUDA(ctx, call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return nph_set_cuda_error((ctx), e__, #call); } while (0)

template <typename T>
int nph_reserve(nph_ctx* ctx, DevBuf<T>& b, size_t n);

// kernels (defined in hmm_forward.cu / abea.cu)
int nph_launch_read_prologue(nph_ctx* ctx);
int nph_launch_hmm_forward(nph_ctx* ctx, float* scores_dev);
size_t nph_hmm_scratch_bytes(const nph_ctx* ctx, int* warps_total_out);
int nph_launch_abea(nph_ctx* ctx);
int nph_schedule_hmm_jobs(nph_ctx* ctx, size_t n_jobs, size_t n_ranks_total, uint32_t* max_E_out);
// per-read (lp_mm_self, lp_mm_next) of the resident reads into ctx->d_trans (host libm, like calculate_transitions)
int nph_upload_read_transitions(nph_ctx* ctx, double indel_bias);
// compact event alignments -> event index per reference base (methylation.cu): dense[ref_off + o] (INT32_MIN: no entry), first_valid[record]
int nph_expand_event_maps(nph_ctx* ctx, const int16_t* d_deltas, const int32_t* d_first_event, const nph_meth_record* d_records, uint32_t n_records,
                          int32_t* d_dense, int32_t* d_first_valid);
extern "C" {   // defined inside nph_api.cu's extern "C" block (internal all the same: not in include/nph.h)
// validate + classify + schedule the n_jobs jobs already sitting in ctx->d_jobs / d_ranks (one stream sync), size the scratch
int nph_jobs_schedule(nph_ctx* ctx, size_t n_jobs, size_t n_ranks_total);
// nph_reads_load's body; pipelined = true (one-shot calls) leaves the event levels to nph_upload_level_chunks, which queues them
// on the copy stream behind progress words the forward kernel polls (ctx->levels_inflight says whether that path was taken)
int nph_reads_load_impl(nph_ctx* ctx, const nph_read* reads, size_t n_reads, const float* ev_mean, const double* ev_start_time, size_t n_events_total, bool pipelined);
int nph_upload_level_chunks(nph_ctx* ctx, const float* ev_mean);
// after a one-shot call: wait for the copy stream and leave the pipelined mode
void nph_finish_level_upload(nph_ctx* ctx);
}

// ---- device-level pieces of the raw-read prologue (event_detect.cu, squiggle_prep.cu, abea.cu), chained by
// load_from_raw.cu without leaving the device.  Inputs named d_* are device pointers; everything runs on ctx->stream.
size_t nph_ed_scratch_bytes(size_t n_samples_total, size_t n_reads, size_t events_total);
int nph_detect_events_device(nph_ctx* ctx, const float* d_raw, size_t n_samples_total, const nph_raw_read* reads, size_t n_reads,
                             const nph_event_params* params, uint8_t* scratch, size_t events_total,
                             nph_event** d_events_out, uint32_t** d_n_events_out, std::vector<uint32_t>& h_n_events, int* launches_out);
size_t nph_trim_scratch_bytes(const nph_raw_read* reads, size_t n_reads, int32_t varseg_chunk);
int nph_trim_device(nph_ctx* ctx, const float* d_raw, size_t n_samples_total, const nph_raw_read* reads, size_t n_reads,
                    int32_t trim_start, int32_t trim_end, int32_t varseg_chunk, float varseg_thresh, uint8_t* scratch,
                    nph_raw_range* ranges_out /* host */);
struct NphCalArgs {
    const float* ev_mean;
    const nph_read* reads;
    const uint32_t* ranks;
    const nph_abea_job* jobs;
    const nph_abea_result* results;
    const nph_aligned_pair* pairs;
    uint32_t n_jobs, model_id;
    nph_event_range* b2e;        // n_kmers entries per job at rank_off
    nph_calibration* out;
    int* bad_input;
};
int nph_launch_recalibrate(nph_ctx* ctx, const NphCalArgs& args);
int nph_launch_mom(nph_ctx* ctx, double* d_shift_scale_out, bool reversed = false);     // over the loaded ABEA jobs: 2 doubles per job
