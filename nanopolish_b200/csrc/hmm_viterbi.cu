// hmm_viterbi.cu — K3: Viterbi alignment of events to the k-mers of a sequence (SURVEY.md section 8f, row N1).
//
// Replaces, for a batch of (sequence, HMMInputData, flags) jobs:
//   profile_hmm_align_r9          ref: src/hmm/nanopolish_profile_hmm_r9.cpp:73-204
//   ProfileHMMViterbiOutputR9     ref: src/hmm/nanopolish_profile_hmm_r9.inl:130-197
//   (the fill itself is profile_hmm_fill_generic_r9, .inl:265-433, shared with the forward score)
//
// Same systolic mapping as the forward kernel (hmm_forward_kernel.cuh): a warp per job, lane j owns C
// k-mer columns, strips of 32*C columns chained.  Differences:
//   * (+) is max with the reference's argmax rule — a compare chain over the six movement types in
//     index order where a LATER index wins ties (`from = max == x[i] ? i : from`), so an all -inf cell
//     records FROM_SOFT like the reference does;
//   * each block-cell stores its three 3-bit movement codes (9 bits in a uint16) to a per-warp trace
//     laid out by systolic step, so the 32 lanes of a step write one contiguous line;
//   * the reference keeps the whole float matrix only to report l_fm along the path; we keep no
//     values: after the backtrack the path is replayed forwards, and l_fm of each state is recomputed
//     from its predecessor with the very float operations the fill used (transition + value, + emission),
//     which reproduces the stored matrix entries bit for bit;
//   * the backtrack starts at (last event, MATCH of the last k-mer) and stops at FROM_SOFT, as the
//     reference does; where the reference would trip an assert (fewer than 2 events, path entering a
//     -inf cell) the job returns zero states.
#include "hmm_viterbi_kernel.cuh"
#include <algorithm>
#include <string>
#include <vector>

namespace {

constexpr int kWarps = 16;
constexpr int kThreads = kWarps * 32;
using namespace nph_vit;

struct VitParams {
    const float* level;
    const DevRead* reads;
    const float2* trans;
    const DevModelView* models;
    const uint32_t* ranks;
    const nph_hmm_job* jobs;
    const uint64_t* states_off;      // n_jobs + 1
    const uint32_t* order;
    uint32_t n_jobs;
    unsigned int* counter;
    const float* flank;
    nph_align_state* states;
    uint32_t* n_states;
    float* scores;
    float4* scratch_params;
    float* scratch_edge;
    uint16_t* scratch_trace;
    uint32_t kpad_stride, edge_stride;
    uint64_t trace_stride;           // uint16 elements per warp
    HmmConsts c;
};

template <int C>
__global__ void __launch_bounds__(kThreads, 1) hmm_viterbi_kernel(const VitParams p)
{
    constexpr int STRIP = 32 * C;
    const int lane = threadIdx.x & 31;
    const int warp_global = blockIdx.x * kWarps + (threadIdx.x >> 5);
    __shared__ uint16_t s_tile[kWarps][32 * 32];
    VitScratch sc;
    sc.tile = s_tile[threadIdx.x >> 5];
    sc.params = p.scratch_params + (size_t)warp_global * p.kpad_stride;
    sc.edge_m = p.scratch_edge + (size_t)warp_global * 3 * p.edge_stride;
    sc.edge_b = sc.edge_m + p.edge_stride;
    sc.edge_k = sc.edge_b + p.edge_stride;
    sc.trace = p.scratch_trace + (size_t)warp_global * p.trace_stride;
    const float NEG = -CUDART_INF_F;
    (void)STRIP;

    for (;;) {
        uint32_t slot = 0;
        if (lane == 0) slot = atomicAdd(p.counter, 1u);
        slot = __shfl_sync(kFull, slot, 0);
        if (slot >= p.n_jobs) break;
        const uint32_t job_idx = p.order[slot];
        const nph_hmm_job job = p.jobs[job_idx];
        VitJob j;
        j.rd = p.reads[job.read];
        j.tr = p.trans[job.read];
        j.mv = p.models[job.model_id];
        j.lv = p.level + j.rd.event_off;
        j.rk = p.ranks + job.rank_off;
        j.K = (int)job.n_kmers;
        j.E = (int)(job.event_stop > job.event_start ? job.event_stop - job.event_start : job.event_start - job.event_stop) + 1;
        j.stride = job.stride;
        j.e_first = (long long)job.event_start;
        j.pre_clip = (job.flags & NPH_HAF_ALLOW_PRE_CLIP) != 0;
        nph_align_state* const out = p.states + p.states_off[job_idx];
        const int cap = (int)(p.states_off[job_idx + 1] - p.states_off[job_idx]);

        if (j.E < 2) {                   // the reference asserts n_events >= 2 (profile_hmm_r9.cpp:88)
            if (lane == 0) { p.n_states[job_idx] = 0; if (p.scores) p.scores[job_idx] = NEG; }
            continue;
        }
        float last_v = NEG;
        const int n = viterbi_align<C>(p.c, p.flank, j, sc, out, cap, &last_v, lane);
        if (lane == 0) {
            p.n_states[job_idx] = (uint32_t)n;
            if (p.scores) p.scores[job_idx] = n ? last_v : NEG;
        }
        __syncwarp();
    }
}

template <int C>
int launch_vit(nph_ctx* ctx, const VitParams& base, const uint32_t* order, size_t count, unsigned int* counter, int max_ctas)
{
    VitParams p = base;
    p.order = order; p.n_jobs = (uint32_t)count; p.counter = counter;
    int grid = std::min(ctx->sm_count, max_ctas);
    if ((size_t)grid * kWarps > count) grid = (int)((count + kWarps - 1) / kWarps);
    if (grid < 1) grid = 1;
    hmm_viterbi_kernel<C><<<grid, kThreads, 0, ctx->stream>>>(p);
    NPH_CUDA(ctx, cudaGetLastError());
    return NPH_OK;
}

const int kVitCols[] = {1, 2, 3, 4, 6, 8};
const int kNumVit = 6;

inline uint32_t vit_steps(uint32_t K, uint32_t E, int C)
{
    const uint32_t strip = 32u * C, n_strips = (K + strip - 1) / strip;
    const uint32_t P = n_strips > 1 ? std::max<uint32_t>(E, kMinPeriod) : E;
    return (n_strips - 1) * P + E + ((K - (n_strips - 1) * strip) - 1) / C;
}

} // namespace

extern "C" int nph_hmm_align_batch(nph_ctx* ctx,
                                   const nph_read* reads, size_t n_reads,
                                   const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                                   const uint32_t* kmer_ranks, size_t n_ranks_total,
                                   const nph_hmm_job* jobs, size_t n_jobs, double indel_bias,
                                   nph_align_state* states_out, const uint64_t* states_off,
                                   uint32_t* n_states_out, float* scores_out)
{
    if (!ctx || !jobs || !states_out || !states_off || !n_states_out || n_jobs == 0) return NPH_ERR_INVALID;
    NPH_TRY(nph_reads_load(ctx, reads, n_reads, ev_mean, ev_start_time, n_events_total));
    return nph_hmm_align(ctx, kmer_ranks, n_ranks_total, jobs, n_jobs, indel_bias, states_out, states_off, n_states_out, scores_out);
}

extern "C" int nph_hmm_align(nph_ctx* ctx,
                             const uint32_t* kmer_ranks, size_t n_ranks_total,
                             const nph_hmm_job* jobs, size_t n_jobs, double indel_bias,
                             nph_align_state* states_out, const uint64_t* states_off,
                             uint32_t* n_states_out, float* scores_out)
{
    if (!ctx || !jobs || !states_out || !states_off || !n_states_out || n_jobs == 0) return NPH_ERR_INVALID;
    if (!ctx->reads_loaded) return NPH_ERR_STATE;
    // jobs, ranks, transitions and validation go through the forward path's loader (same job semantics)
    NPH_TRY(nph_hmm_jobs_load(ctx, kmer_ranks, n_ranks_total, jobs, n_jobs, indel_bias));

    // class per job (columns per lane) and schedule, longest first
    std::vector<std::vector<uint32_t>> steps(kNumVit), jobs_of(kNumVit);
    uint32_t max_kpad = 32, max_period = kMinPeriod;
    uint64_t max_trace = 1;
    for (size_t j = 0; j < n_jobs; ++j) {
        const nph_hmm_job& jb = jobs[j];
        const uint32_t E = (jb.event_stop > jb.event_start ? jb.event_stop - jb.event_start : jb.event_start - jb.event_stop) + 1;
        const uint32_t K = jb.n_kmers;
        if (states_off[j + 1] < states_off[j]) return NPH_ERR_INVALID;
        double best = 1e300; int bi = 0; uint32_t bsteps = 0;
        for (int i = 0; i < kNumVit; ++i) {
            const uint32_t st = vit_steps(K, E, kVitCols[i]);
            const double cost = (double)st * (120.0 + 70.0 * kVitCols[i]);
            if (cost < best) { best = cost; bi = i; bsteps = st; }
        }
        steps[bi].push_back(bsteps);
        jobs_of[bi].push_back((uint32_t)j);
        const uint32_t strip = 32u * kVitCols[bi], n_strips = (K + strip - 1) / strip;
        max_kpad = std::max(max_kpad, n_strips * strip);
        max_period = std::max(max_period, std::max<uint32_t>(E, kMinPeriod));
        max_trace = std::max<uint64_t>(max_trace, (uint64_t)(bsteps + 1) * strip);
    }
    std::vector<uint32_t> order;
    order.reserve(n_jobs);
    size_t first[kNumVit + 1];
    for (int i = 0; i < kNumVit; ++i) {
        first[i] = order.size();
        for (uint32_t t : longest_first(steps[i])) order.push_back(jobs_of[i][t]);
    }
    first[kNumVit] = order.size();

    // The movement trace is per resident warp and sized by the batch's largest job ((steps + 1) x strip uint16 entries),
    // so one long window must not multiply by every warp of the chip: the number of resident CTAs is capped so that
    // the trace arena stays within kTraceBudget, and a job whose trace does not fit a single CTA's 16 warps within
    // that budget is refused with NPH_ERR_UNSUPPORTED (documented in include/nph.h) instead of a NOMEM surprise.
    const size_t trace_stride = ((max_trace + 63) / 64) * 64;
    const uint64_t kTraceBudget = 16ull << 30;
    const uint64_t per_cta = (uint64_t)sizeof(uint16_t) * trace_stride * kWarps;
    if (per_cta > kTraceBudget) {
        ctx->last_error = "profile_hmm_align window too large: its movement trace needs " + std::to_string(per_cta >> 20) + " MiB per CTA (limit 16 GiB)";
        return NPH_ERR_UNSUPPORTED;
    }
    const int max_ctas = (int)std::min<uint64_t>((uint64_t)ctx->sm_count, std::max<uint64_t>(1, kTraceBudget / per_cta));
    const int warps = max_ctas * kWarps;
    const size_t total_states = (size_t)states_off[n_jobs];
    VitParams p{};
    uint64_t* d_off = nullptr;
    uint32_t* d_order = nullptr;
    auto layout = [&](NphCarve& a) {
        p.scratch_params = a.take<float4>((size_t)max_kpad * warps);
        p.scratch_edge = a.take<float>(3 * ((size_t)max_period + 8) * warps);
        p.scratch_trace = a.take<uint16_t>(trace_stride * warps);
        p.states = a.take<nph_align_state>(total_states);
        p.states_off = d_off = a.take<uint64_t>(n_jobs + 1);
        p.n_states = a.take<uint32_t>(n_jobs);
        d_order = a.take<uint32_t>(n_jobs);
    };
    NPH_TRY(nph_borrow_arena(ctx, layout));
    p.level = ctx->d_level.p; p.reads = ctx->d_reads.p; p.trans = ctx->d_trans.p; p.models = ctx->d_models.p;
    p.ranks = ctx->d_ranks.p; p.jobs = ctx->d_jobs.p; p.flank = ctx->d_flank.p; p.scores = ctx->d_scores.p;
    p.kpad_stride = max_kpad; p.edge_stride = max_period + 8; p.trace_stride = trace_stride; p.c = ctx->consts;
    NPH_CUDA(ctx, cudaMemcpyAsync(d_off, states_off, sizeof(uint64_t) * (n_jobs + 1), cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d_order, order.data(), sizeof(uint32_t) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemsetAsync(ctx->d_counters.p, 0, sizeof(unsigned int) * NPH_NUM_COUNTERS, ctx->stream));
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    int launches = 0;
    for (int i = 0; i < kNumVit; ++i) {
        const size_t count = first[i + 1] - first[i];
        if (!count) continue;
        int rc = NPH_ERR_STATE;
        switch (kVitCols[i]) {
            case 1: rc = launch_vit<1>(ctx, p, d_order + first[i], count, ctx->d_counters.p + i, max_ctas); break;
            case 2: rc = launch_vit<2>(ctx, p, d_order + first[i], count, ctx->d_counters.p + i, max_ctas); break;
            case 3: rc = launch_vit<3>(ctx, p, d_order + first[i], count, ctx->d_counters.p + i, max_ctas); break;
            case 4: rc = launch_vit<4>(ctx, p, d_order + first[i], count, ctx->d_counters.p + i, max_ctas); break;
            case 6: rc = launch_vit<6>(ctx, p, d_order + first[i], count, ctx->d_counters.p + i, max_ctas); break;
            case 8: rc = launch_vit<8>(ctx, p, d_order + first[i], count, ctx->d_counters.p + i, max_ctas); break;
        }
        if (rc != NPH_OK) return rc;
        ++launches;
    }
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->last_launches = launches;
    ctx->timing_valid = true;
    NPH_CUDA(ctx, cudaMemcpyAsync(states_out, p.states, sizeof(nph_align_state) * total_states, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(n_states_out, p.n_states, sizeof(uint32_t) * n_jobs, cudaMemcpyDeviceToHost, ctx->stream));
    if (scores_out) NPH_CUDA(ctx, cudaMemcpyAsync(scores_out, ctx->d_scores.p, sizeof(float) * n_jobs, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NPH_OK;
}
