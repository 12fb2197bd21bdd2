// hmm_forward.cu — K1 dispatcher: per-read prologue kernel, scratch sizing and the per-class launches of
// the forward kernel template (hmm_forward_kernel.cuh; one translation unit per group width).
#include "hmm_forward_kernel.cuh"
#include <algorithm>
#include <cmath>
#include <vector>

using namespace nph_fwd;

namespace {

// ---- per-read device prologue: drift-scaled level of every event ----
// x = (float)( (double)mean - (double)(float)(t - t0) * drift )   (squiggle_read.h:149-154, 168-171)
__global__ void read_prologue_kernel(const DevRead* __restrict__ reads, const double* __restrict__ drift,
                                     const float* __restrict__ ev_mean, const double* __restrict__ ev_time,
                                     float* __restrict__ level, uint32_t n_reads)
{
    for (uint32_t r = blockIdx.x; r < n_reads; r += gridDim.x) {
        const DevRead rd = reads[r];
        const double dr = drift[r];
        const float* m = ev_mean + rd.event_off;
        const double* t = ev_time + rd.event_off;
        float* out = level + rd.event_off;
        const double t0 = t[0];
        for (uint32_t i = threadIdx.x; i < rd.n_events; i += blockDim.x) {
            const float time = (float)__dsub_rn(t[i], t0);
            out[i] = (float)__dsub_rn((double)m[i], __dmul_rn((double)time, dr));
        }
    }
}

} // namespace

// One pair of scratch slices per side stream: classes running concurrently on different SMs index their per-warp
// scratch by (block, warp) and must not share it.
struct FwdScratch { float4* params; float* edge; };

static void fwd_layout(NphCarve& a, const nph_ctx* ctx, FwdScratch (&s)[nph_ctx::kSideStreams])
{
    const size_t warps = (size_t)ctx->sm_count * kMaxWarpsPerCta;
    for (FwdScratch& x : s) {
        x.params = a.take<float4>((size_t)ctx->max_kpad * warps);
        x.edge = a.take<float>(3 * ((size_t)ctx->max_period + 8) * warps);
    }
}

size_t nph_hmm_scratch_bytes(const nph_ctx* ctx)
{
    FwdScratch s[nph_ctx::kSideStreams];
    return nph_measure([&](NphCarve& a) { fwd_layout(a, ctx, s); });
}

int nph_launch_read_prologue(nph_ctx* ctx)
{
    const uint32_t n = (uint32_t)ctx->n_reads;
    if (n == 0) return NPH_OK;
    int grid = (int)std::min<size_t>(n, (size_t)ctx->sm_count * 16);
    read_prologue_kernel<<<grid, 256, 0, ctx->stream>>>(ctx->d_reads.p, ctx->d_drift.p, ctx->d_ev_mean.p,
                                                        ctx->d_ev_time.p, ctx->d_level.p, n);
    NPH_CUDA(ctx, cudaGetLastError());
    return NPH_OK;
}

int nph_launch_hmm_forward(nph_ctx* ctx, float* scores_dev)
{
    FwdParams p{};
    p.level = ctx->d_level.p;
    p.reads = ctx->d_reads.p;
    p.trans = ctx->d_trans.p;
    p.models = ctx->d_models.p;
    p.ranks = ctx->d_ranks.p;
    p.jobs = ctx->d_jobs.p;
    p.logsum_g = ctx->d_logsum.p;
    p.flank = ctx->d_flank.p;
    p.scores = scores_dev ? scores_dev : ctx->d_scores.p;
    p.kpad_stride = ctx->max_kpad;
    p.edge_stride = ctx->max_period + 8;
    p.c = ctx->consts;
    p.lsum_bias = NPH_LOGSUM_ADDR_BIAS;
    p.lsum_scale = 4u;
    p.neg_zero = -0.0f;
    p.progress = (ctx->levels_inflight && ctx->level_chunk_events) ? ctx->d_progress.p : nullptr;
    p.chunk_events = (uint32_t)ctx->level_chunk_events;
    FwdScratch scratch[nph_ctx::kSideStreams];
    NPH_TRY(nph_carve(ctx, ctx->d_scratch, [&](NphCarve& a) { fwd_layout(a, ctx, scratch); }));

    NPH_CUDA(ctx, cudaMemsetAsync(ctx->d_counters.p, 0, sizeof(unsigned int) * NPH_NUM_COUNTERS, ctx->stream));
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    // fork: the classes run on side streams so that the tail of one overlaps the head of the next
    // (a CTA takes a whole SM, so kernels overlap SM by SM as CTAs retire); heaviest class first.
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));
    std::vector<size_t> idx;
    for (size_t ci = 0; ci < ctx->classes.size(); ++ci) if (ctx->classes[ci].count) idx.push_back(ci);
    std::sort(idx.begin(), idx.end(), [&](size_t a, size_t b) { return ctx->classes[a].cost > ctx->classes[b].cost; });
    bool used[nph_ctx::kSideStreams] = {false, false, false, false};
    int launches = 0;
    for (size_t t = 0; t < idx.size(); ++t) {
        const size_t ci = idx[t];
        const auto& cl = ctx->classes[ci];
        const int si = (int)(t % nph_ctx::kSideStreams);
        cudaStream_t st = ctx->side[si];
        if (!used[si]) { NPH_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_fork, 0)); used[si] = true; }
        p.scratch_params = scratch[si].params;
        p.scratch_edge = scratch[si].edge;
        int rc = NPH_ERR_STATE;
        switch (cl.group_width) {
            case 4: rc = launch_width<4, false>(ctx, p, cl, (int)ci, st); break;
            case 8: rc = launch_width<8, false>(ctx, p, cl, (int)ci, st); break;
            case 16: rc = launch_width<16, false>(ctx, p, cl, (int)ci, st); break;
            case 32: rc = cl.chained ? launch_width<32, true>(ctx, p, cl, (int)ci, st) : launch_width<32, false>(ctx, p, cl, (int)ci, st); break;
        }
        if (rc != NPH_OK) return rc;
        ++launches;
    }
    for (int si = 0; si < nph_ctx::kSideStreams; ++si) {
        if (!used[si]) continue;
        NPH_CUDA(ctx, cudaEventRecord(ctx->ev_join[si], ctx->side[si]));
        NPH_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join[si], 0));
    }
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->last_launches = launches;
    ctx->timing_valid = true;
    return NPH_OK;
}
