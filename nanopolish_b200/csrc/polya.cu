// polya.cu — SURVEY.md section 8(f) row N5: `nanopolish polya` (src/nanopolish_polya_estimator.cpp) for a batch of reads.
//
// One warp per read, persistent CTAs handing out reads longest first.  Per read:
//   1. Viterbi over every trimmed raw sample (SegmentationHMM::viterbi, :372-463).  The 32 lanes evaluate the six emissions
//      of the next 32 samples (the expensive part: five expf and three logf each, csrc/polya_math.cuh), lane 0 then runs the
//      max-plus recurrence over them serially in the reference's operation order (a parallel max-plus scan would regroup the
//      float sums and change them) and the warp writes the 6-bit backpointers of the 32 steps to global memory as 32 bytes.
//   2. Backtrack (:447-458) by lane 0 over the backpointers staged into shared memory 1 KB at a time, collecting what
//      segment_squiggle (:466-508) keeps: the last S->L, L->A, A->P and P->T transitions and the count of C samples.
//   3. Read rate (estimate_unaligned_duration_profile, :564-599): per-k-mer duration sums in event order, then the element
//      of rank size/2 by an 8-pass radix select over the order-preserving bit patterns (no sort: only the order statistic
//      matters).
//   4. estimate_polya_length (:638-662), post_segmentation_qc (:688-702), post_estimation_qc (:707-722).
// Every float and double operation is spelled with its rounding; the library is built with -fmad=false.
#include "nph_internal.cuh"
#include "polya_math.cuh"

#include <cmath>
#include <vector>

namespace {

using namespace nph_polya_math;

constexpr int kWarps = 8;                 // warps per CTA
constexpr int kStage = 1024;              // backpointer bytes staged per backtrack round

enum { S_ = 0, L_ = 1, A_ = 2, P_ = 3, C_ = 4, T_ = 5 };

struct PolyaArgs {
    const float* samples;
    const float* durations;
    const nph_event_range* map;
    const nph_polya_job* jobs;
    const uint32_t* order;                // jobs, longest first
    uint32_t n_jobs;
    uint64_t n_samples_total, n_events_total, n_map_total;
    uint8_t* bptr;                        // per warp slot: one byte per sample of the read it holds (bp_stride bytes)
    double* kmer_dur;                     // per warp slot: one double per map entry (kd_stride doubles)
    uint64_t bp_stride, kd_stride;
    nph_polya_result* results;
    unsigned int* next;                   // work counter
    int* bad;                             // 1 + index of an invalid job
};

struct Gauss { float mean, stdv, log_stdv; };

// SegmentationHMM's constructor (:327-353): mean = shift + scale * mean, stdv = var * stdv, log_stdv = logf(stdv)
__device__ __forceinline__ Gauss scaled(float mean, float stdv, float scale, float shift, float var)
{
    Gauss g;
    g.mean = __fadd_rn(shift, __fmul_rn(scale, mean));
    g.stdv = __fmul_rn(var, stdv);
    g.log_stdv = logf_glibc(g.stdv);
    return g;
}

struct Hmm { Gauss s, l, a0, a1, p, t0, t1; float log_inv_sqrt_2pi; };

// normal_pdf / log_normal_pdf (src/hmm/nanopolish_emissions.h:19-24, :51-55) with inv_sqrt_2pi = (float)0.3989422804014327
__device__ __forceinline__ float normal_pdf(float x, const Gauss& g)
{
    const float a = __fdiv_rn(__fsub_rn(x, g.mean), g.stdv);
    return __fmul_rn(__fdiv_rn(0.3989422804014327f, g.stdv), expf_glibc(__fmul_rn(__fmul_rn(-0.5f, a), a)));
}
__device__ __forceinline__ float log_normal_pdf(float x, const Gauss& g, float log_inv_sqrt_2pi)
{
    const float a = __fdiv_rn(__fsub_rn(x, g.mean), g.stdv);
    return __fadd_rn(__fsub_rn(log_inv_sqrt_2pi, g.log_stdv), __fmul_rn(__fmul_rn(-0.5f, a), a));
}

// SegmentationHMM::emit_log_proba (:259-306) for all six states
__device__ __forceinline__ void emissions(float x, const Hmm& h, float e[6])
{
    const float xx = (x > 200.0f || x < 40.0f) ? 100.0f : x;
    e[S_] = logf_glibc(__fadd_rn(__fmul_rn(0.50f, normal_pdf(xx, h.s)), __fmul_rn(0.50f, 0.00476f)));
    e[L_] = log_normal_pdf(xx, h.l, h.log_inv_sqrt_2pi);
    e[A_] = logf_glibc(__fadd_rn(__fmul_rn(0.874f, normal_pdf(xx, h.a0)), __fmul_rn(0.126f, normal_pdf(xx, h.a1))));
    e[P_] = log_normal_pdf(xx, h.p, h.log_inv_sqrt_2pi);
    e[C_] = (xx > 70.0f && xx < 140.0f) ? -4.2485f : -INFINITY;
    e[T_] = logf_glibc(__fadd_rn(__fmul_rn(0.346f, normal_pdf(xx, h.t0)), __fmul_rn(0.654f, normal_pdf(xx, h.t1))));
}

__device__ __forceinline__ float fmax_ref(float a, float b) { return (a < b) ? b : a; }   // std::max

// regions[j] = bptrs[j][regions[j+1]] from the packed byte of sample j
__device__ __forceinline__ int predecessor(uint32_t b, int next)
{
    switch (next) {
        case L_: return (b & 1u) ? L_ : S_;
        case A_: return (b & 2u) ? A_ : L_;
        case P_: { const uint32_t c = (b >> 2) & 3u; return c == 0 ? P_ : (c == 1 ? A_ : C_); }
        case C_: return (b & 16u) ? C_ : P_;
        case T_: return (b & 32u) ? T_ : P_;
        default: return S_;
    }
}

__device__ __forceinline__ uint64_t order_key(double v)
{
    const uint64_t u = (uint64_t)__double_as_longlong(v);
    return (u >> 63) ? ~u : (u | (1ull << 63));
}
__device__ __forceinline__ double key_value(uint64_t k)
{
    return __longlong_as_double((long long)((k >> 63) ? (k & ~(1ull << 63)) : ~k));
}

// validation: exactly where the reference would read out of bounds, assert, or (n_samples < 2) index before the samples
__global__ void polya_validate_kernel(const PolyaArgs a)
{
    const int lane = threadIdx.x & 31;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < a.n_jobs; t += warps) {
        const nph_polya_job jb = a.jobs[t];
        if (jb.n_events == 0) continue;                               // READ_FAILED_LOAD: nothing else is read
        bool ok = jb.n_samples >= 2 && jb.n_kmers >= 1 && jb.sample_off <= a.n_samples_total && jb.n_samples <= a.n_samples_total - jb.sample_off
                  && jb.event_off <= a.n_events_total && jb.n_events <= a.n_events_total - jb.event_off
                  && jb.map_off <= a.n_map_total && jb.n_kmers <= a.n_map_total - jb.map_off;
        if (ok)
            for (uint32_t i = lane; i < jb.n_kmers; i += 32) {
                const nph_event_range r = a.map[jb.map_off + i];
                if (r.start == -1) continue;
                if (r.start < 0 || r.stop < r.start || (uint32_t)r.stop >= jb.n_events) ok = false;
            }
        ok = __all_sync(0xffffffffu, ok);
        if (!ok && lane == 0) atomicCAS(a.bad, 0, (int)t + 1);
    }
}

__global__ void __launch_bounds__(kWarps * 32) polya_kernel(const PolyaArgs a)
{
    __shared__ float s_em[kWarps][6][32];
    __shared__ uint8_t s_bp[kWarps][32];
    __shared__ uint8_t s_tr[kWarps][kStage];
    __shared__ unsigned int s_hist[kWarps][256];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t slot_w = blockIdx.x * kWarps + w;

    // transition log-probabilities (:313-326): logf of the float table, -inf for zero entries
    const float tSS = logf_glibc(0.10f), tSL = logf_glibc(0.90f), tLL = logf_glibc(0.90f), tLA = logf_glibc(0.10f);
    const float tAA = logf_glibc(0.95f), tAP = logf_glibc(0.05f), tPP = logf_glibc(0.89f), tPC = logf_glibc(0.01f);
    const float tPT = logf_glibc(0.10f), tCP = logf_glibc(0.99f), tCC = logf_glibc(0.01f), tTT = logf_glibc(1.00f);
    const float lsS = logf_glibc(1.00f);

    for (;;) {
        unsigned int slot = 0;
        if (lane == 0) slot = atomicAdd(a.next, 1u);
        slot = __shfl_sync(0xffffffffu, slot, 0);
        if (slot >= a.n_jobs) return;
        const uint32_t t = a.order[slot];
        const nph_polya_job jb = a.jobs[t];
        nph_polya_result res{};
        if (jb.n_events == 0) {
            if (lane == 0) { res.qc = NPH_POLYA_FAILED_LOAD; a.results[t] = res; }
            continue;
        }
        const float scale = __double2float_rn(jb.scale), shift = __double2float_rn(jb.shift), var = __double2float_rn(jb.var);
        Hmm h;
        h.s = scaled(70.2737f, 3.7743f, scale, shift, var);
        h.l = scaled(110.973f, 5.237f, scale, shift, var);
        h.a0 = scaled(79.347f, 8.3702f, scale, shift, var);
        h.a1 = scaled(63.3126f, 2.7464f, scale, shift, var);
        h.p = scaled(108.883f, 3.257f, scale, shift, var);
        h.t0 = scaled(79.679f, 6.966f, scale, shift, var);
        h.t1 = scaled(105.784f, 16.022f, scale, shift, var);
        h.log_inv_sqrt_2pi = -0x1.d67f1cp-1f;                     // log_inv_sqrt_2pi = (float)log(0.3989422804014327)
        const uint32_t n = jb.n_samples;
        const float* x = a.samples + jb.sample_off;
        uint8_t* bp = a.bptr + (uint64_t)slot_w * a.bp_stride;     // this warp's scratch: jobs may share samples or map entries

        // ---- 1. forward Viterbi ----
        float vS = 0.f, vL = 0.f, vA = 0.f, vP = 0.f, vC = 0.f, vT = 0.f;     // lane 0's scores of the last step
        for (uint32_t i0 = 0; i0 < n; i0 += 32) {
            const uint32_t i = i0 + lane;
            if (i < n) {
                float e[6];
                emissions(x[i == 0 ? n - 1 : i], h, e);          // step 0 reads samples[n-1] (:385-386)
                #pragma unroll
                for (int k = 0; k < 6; ++k) s_em[w][k][lane] = e[k];
            }
            __syncwarp();
            if (lane == 0) {
                const uint32_t cnt = min(32u, n - i0);
                uint32_t j = 0;
                if (i0 == 0) {
                    vS = __fadd_rn(lsS, s_em[w][S_][0]);
                    vL = __fadd_rn(-INFINITY, s_em[w][L_][0]);   // log_start_probs[L] + emission, as the reference adds them
                    vA = vP = vC = vT = -INFINITY;
                    s_bp[w][0] = 0;
                    j = 1;
                }
                for (; j < cnt; ++j) {
                    const float s_to_s = __fadd_rn(vS, tSS), s_to_l = __fadd_rn(vS, tSL);
                    const float l_to_l = __fadd_rn(vL, tLL), l_to_a = __fadd_rn(vL, tLA);
                    const float a_to_a = __fadd_rn(vA, tAA), a_to_p = __fadd_rn(vA, tAP);
                    const float p_to_p = __fadd_rn(vP, tPP), p_to_c = __fadd_rn(vP, tPC), p_to_t = __fadd_rn(vP, tPT);
                    const float c_to_c = __fadd_rn(vC, tCC), c_to_p = __fadd_rn(vC, tCP);
                    const float t_to_t = __fadd_rn(vT, tTT);
                    vS = __fadd_rn(s_to_s, s_em[w][S_][j]);
                    vL = __fadd_rn(fmax_ref(l_to_l, s_to_l), s_em[w][L_][j]);
                    vA = __fadd_rn(fmax_ref(a_to_a, l_to_a), s_em[w][A_][j]);
                    vP = __fadd_rn(fmax_ref(p_to_p, fmax_ref(a_to_p, c_to_p)), s_em[w][P_][j]);
                    vC = __fadd_rn(fmax_ref(c_to_c, p_to_c), s_em[w][C_][j]);
                    vT = __fadd_rn(fmax_ref(p_to_t, t_to_t), s_em[w][T_][j]);
                    uint32_t b = 0;
                    b |= (s_to_l < l_to_l) ? 1u : 0u;                                        // L: L (1) or S (0)
                    b |= (l_to_a < a_to_a) ? 2u : 0u;                                        // A: A (1) or L (0)
                    const uint32_t pc = (a_to_p < p_to_p && c_to_p < p_to_p) ? 0u : ((p_to_p < a_to_p && c_to_p < a_to_p) ? 1u : 2u);
                    b |= pc << 2;                                                            // P: P (0), A (1), C (2)
                    b |= (p_to_c < c_to_c) ? 16u : 0u;                                       // C: C (1) or P (0)
                    b |= (p_to_t < t_to_t) ? 32u : 0u;                                       // T: T (1) or P (0)
                    s_bp[w][j] = (uint8_t)b;
                }
            }
            __syncwarp();
            if (i < n) bp[i] = s_bp[w][lane];
            __syncwarp();
        }
        res.end_score = vT;

        // ---- 2. backtrack + segment_squiggle ----
        uint64_t seg_start = 0, seg_leader = 1, seg_adapter = 2, seg_polya = 3, cliffs = 0;
        bool f_s = false, f_l = false, f_a = false, f_p = false;
        int cur = T_;                                             // regions[n-1]
        // j runs n-2 .. 1; staged in windows [lo, hi] of kStage bytes, highest first
        for (int64_t hi = (int64_t)n - 2; hi >= 1; hi -= kStage) {
            const int64_t lo = max((int64_t)1, hi - kStage + 1);
            for (int64_t q = lo + lane; q <= hi; q += 32) s_tr[w][q - lo] = bp[q];
            __syncwarp();
            if (lane == 0) {
                for (int64_t j = hi; j >= lo; --j) {
                    const int r = predecessor(s_tr[w][j - lo], cur);
                    if (!f_s && r == S_ && cur == L_) { f_s = true; seg_start = (uint64_t)j; }
                    if (!f_l && r == L_ && cur == A_) { f_l = true; seg_leader = (uint64_t)j; }
                    if (!f_a && r == A_ && cur == P_) { f_a = true; seg_adapter = (uint64_t)j; }
                    if (!f_p && r == P_ && cur == T_) { f_p = true; seg_polya = (uint64_t)j; }
                    if (r == C_) ++cliffs;
                    cur = r;
                }
            }
            cur = __shfl_sync(0xffffffffu, cur, 0);
            __syncwarp();
        }
        if (lane == 0) {
            if (!f_s && cur == L_) seg_start = 0;                 // regions[0] is S
            if (seg_leader == 1 || seg_adapter == 2 || seg_polya == 3) {
                seg_leader = (uint64_t)n - 3; seg_adapter = (uint64_t)n - 2; seg_polya = (uint64_t)n - 1;
            }
        }

        // ---- 3. read rate: per-k-mer durations, then the element of rank size/2 ----
        const uint32_t m = jb.n_kmers;
        double* kd = a.kmer_dur + (uint64_t)slot_w * a.kd_stride;
        const float* dur = a.durations + jb.event_off;
        for (uint32_t i = lane; i < m; i += 32) {
            const nph_event_range r = a.map[jb.map_off + i];
            double acc = 0.0;
            if (r.start != -1)
                for (int32_t j = r.start; j <= r.stop; ++j) acc = __dadd_rn(acc, (double)dur[j]);
            kd[i] = acc;
        }
        __syncwarp();
        uint64_t prefix = 0;
        uint32_t rank = m / 2;
        for (int pass = 7; pass >= 0; --pass) {
            for (int b = lane; b < 256; b += 32) s_hist[w][b] = 0;
            __syncwarp();
            const int sh = pass * 8;
            const uint64_t hmask = (pass == 7) ? 0ull : (~0ull << (sh + 8));
            for (uint32_t i = lane; i < m; i += 32) {
                const uint64_t k = order_key(kd[i]);
                if ((k & hmask) == prefix) atomicAdd(&s_hist[w][(k >> sh) & 255u], 1u);
            }
            __syncwarp();
            if (lane == 0) {
                uint32_t b = 0;
                while (rank >= s_hist[w][b]) { rank -= s_hist[w][b]; ++b; }
                prefix |= (uint64_t)b << sh;
            }
            prefix = __shfl_sync(0xffffffffu, prefix, 0);
            rank = __shfl_sync(0xffffffffu, rank, 0);
            __syncwarp();
        }

        // ---- 4. length and QC ----
        if (lane == 0) {
            const double median = key_value(prefix);
            const double read_rate = __ddiv_rn(1.0, median);
            const double sr = jb.sample_rate;
            const double polya_duration = __ddiv_rn(__ull2double_rn(seg_polya - (seg_adapter + 1)), sr);
            double polya_length = __dadd_rn(__dmul_rn(polya_duration, read_rate), -5.0);
            polya_length = (0.0 < polya_length) ? polya_length : 0.0;                 // std::max(0.0, .)
            const double n_adapter = __ull2double_rn((seg_adapter + 1) - seg_leader);
            const double n_polya = __ull2double_rn(seg_polya - (seg_adapter + 1));
            const double adapter_length = __dmul_rn(__ddiv_rn(__ull2double_rn(seg_adapter - (seg_leader - 1)), sr), read_rate);
            uint32_t qc = 0;
            if (n_adapter < 200.0 || n_polya < 200.0) qc |= NPH_POLYA_NOREGION;
            if (adapter_length > 300.0) qc |= NPH_POLYA_ADAPTER;
            res.start = seg_start; res.leader = seg_leader; res.adapter = seg_adapter; res.polya = seg_polya; res.cliffs = cliffs;
            res.read_rate = read_rate; res.polya_length = polya_length; res.qc = qc;
            a.results[t] = res;
        }
        __syncwarp();
    }
}

// resident form: jobs of the last load_from_raw batch from its device outputs
struct AfterLoadArgs {
    const nph_raw_job* raw_jobs;
    const nph_raw_range* trim;
    const int64_t* live_index;
    const uint64_t* event_off;            // n_jobs + 1, compact
    const nph_calibration* cal;           // live order
    uint32_t n_jobs;
    nph_polya_job* jobs_out;
};

__global__ void after_load_jobs_kernel(const AfterLoadArgs a)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.n_jobs) return;
    const nph_raw_job rj = a.raw_jobs[j];
    nph_polya_job pj{};
    const int64_t li = a.live_index[j];
    pj.sample_off = rj.sample_off + a.trim[j].start;
    pj.n_samples = a.trim[j].end - a.trim[j].start;
    pj.map_off = rj.rank_off;
    pj.n_kmers = rj.n_kmers;
    pj.sample_rate = rj.sample_rate;
    pj.event_off = a.event_off[j];
    pj.n_events = 0;                                  // failed load unless calibrated
    if (li >= 0) {
        const nph_calibration c = a.cal[li];
        if (c.status == 0) {
            pj.n_events = (uint32_t)(a.event_off[j + 1] - a.event_off[j]);
            pj.shift = c.shift; pj.scale = c.scale; pj.var = c.var;
        }
    }
    a.jobs_out[j] = pj;
}

// Per-warp scratch: backpointers (1 B per sample) and per-k-mer durations (8 B per map entry) of the read a warp holds,
// sized from the batch's longest read.  The grid is the resident warps (at most one per job), fewer if that scratch would
// exceed the larger of the batch's own footprint and 1 GiB.
struct ScratchPlan { unsigned blocks = 1; uint64_t bp_stride = 256, kd_stride = 32; };

int plan_scratch(nph_ctx* ctx, const std::vector<nph_polya_job>& jobs, ScratchPlan* plan)
{
    uint64_t max_n = 1, max_k = 1, sum = 0;
    for (const nph_polya_job& j : jobs) {
        if (!j.n_events) continue;
        max_n = std::max<uint64_t>(max_n, j.n_samples); max_k = std::max<uint64_t>(max_k, j.n_kmers);
        sum += j.n_samples + 8ull * j.n_kmers;
    }
    int per_sm = 0;
    NPH_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, polya_kernel, kWarps * 32, 0));
    ScratchPlan p;
    p.bp_stride = nph_align256(max_n);
    p.kd_stride = nph_align256(8 * max_k) / 8;
    const uint64_t per_block = kWarps * (p.bp_stride + 8 * p.kd_stride);
    const uint64_t budget = std::max<uint64_t>(sum, 1ull << 30);
    size_t blocks = std::min<size_t>((jobs.size() + kWarps - 1) / kWarps, (size_t)ctx->sm_count * std::max(per_sm, 1));
    blocks = std::max<size_t>(1, std::min<size_t>(blocks, budget / per_block));
    p.blocks = (unsigned)blocks;
    *plan = p;
    return NPH_OK;
}

struct PolyaControl { unsigned int next; int bad; };      // work counter, 1 + index of an invalid job

// run_polya's slices, behind the inputs of its caller
struct RunScratch { uint32_t* order; nph_polya_result* results; PolyaControl* ctl; double* kmer_dur; uint8_t* bptr; };

RunScratch run_layout(NphCarve& a, size_t n_jobs, const ScratchPlan& plan)
{
    RunScratch s;
    s.order = a.take<uint32_t>(n_jobs);
    s.results = a.take<nph_polya_result>(n_jobs);
    s.ctl = a.take<PolyaControl>(1);
    s.kmer_dur = a.take<double>((size_t)plan.blocks * kWarps * plan.kd_stride);
    s.bptr = a.take<uint8_t>((size_t)plan.blocks * kWarps * plan.bp_stride);
    return s;
}

// validate, schedule and run the jobs already at d_jobs; samples / durations / map are device pointers
int run_polya(nph_ctx* ctx, const float* d_samples, size_t n_samples_total, const float* d_dur, size_t n_events_total,
              const nph_event_range* d_map, size_t n_map_total, nph_polya_job* d_jobs, const std::vector<nph_polya_job>& jobs,
              const ScratchPlan& plan, const RunScratch& s, nph_polya_result* results_out)
{
    const size_t n_jobs = jobs.size();
    std::vector<uint32_t> length(n_jobs);
    for (size_t i = 0; i < n_jobs; ++i) length[i] = jobs[i].n_events ? jobs[i].n_samples : 0u;
    const std::vector<uint32_t> order = longest_first(length);
    NPH_CUDA(ctx, cudaMemcpyAsync(s.order, order.data(), sizeof(uint32_t) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemsetAsync(s.ctl, 0, nph_align256(sizeof(PolyaControl)), ctx->stream));     // the slice's whole extent

    PolyaArgs pa{};
    pa.samples = d_samples; pa.durations = d_dur; pa.map = d_map; pa.jobs = d_jobs; pa.order = s.order; pa.n_jobs = (uint32_t)n_jobs;
    pa.n_samples_total = n_samples_total; pa.n_events_total = n_events_total; pa.n_map_total = n_map_total;
    pa.bptr = s.bptr; pa.kmer_dur = s.kmer_dur; pa.bp_stride = plan.bp_stride; pa.kd_stride = plan.kd_stride;
    pa.results = s.results; pa.next = &s.ctl->next; pa.bad = &s.ctl->bad;
    const unsigned vblocks = (unsigned)std::min<size_t>((n_jobs + kWarps - 1) / kWarps, (size_t)ctx->sm_count * 8);
    polya_validate_kernel<<<vblocks, kWarps * 32, 0, ctx->stream>>>(pa);
    NPH_CUDA(ctx, cudaGetLastError());
    int bad = 0;
    NPH_CUDA(ctx, cudaMemcpyAsync(&bad, pa.bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (bad) {
        ctx->last_error = "nph_polya: invalid job " + std::to_string(bad - 1);
        return NPH_ERR_INVALID;
    }
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    polya_kernel<<<plan.blocks, kWarps * 32, 0, ctx->stream>>>(pa);
    NPH_CUDA(ctx, cudaGetLastError());
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(results_out, s.results, sizeof(nph_polya_result) * n_jobs, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->last_launches = 2;
    ctx->timing_valid = 1;
    return NPH_OK;
}

} // namespace

extern "C" int nph_polya_batch(nph_ctx* ctx, const float* samples, size_t n_samples_total, const float* durations, size_t n_events_total,
                               const nph_event_range* map, size_t n_map_total, const nph_polya_job* jobs, size_t n_jobs,
                               nph_polya_result* results_out)
{
    if (!ctx) return NPH_ERR_INVALID;
    if (n_jobs == 0) return NPH_OK;
    if (!jobs || !results_out || (n_samples_total && !samples) || (n_events_total && !durations) || (n_map_total && !map)) return NPH_ERR_INVALID;
    if (n_jobs > 0xffffffffu) return NPH_ERR_UNSUPPORTED;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    std::vector<nph_polya_job> hj(jobs, jobs + n_jobs);
    ScratchPlan plan;
    NPH_TRY(plan_scratch(ctx, hj, &plan));
    struct { float *samples, *durations; nph_event_range* map; nph_polya_job* jobs; } d{};
    RunScratch rs;
    auto layout = [&](NphCarve& a) {
        d.samples = a.take<float>(std::max<size_t>(n_samples_total, 1));
        d.durations = a.take<float>(std::max<size_t>(n_events_total, 1));
        d.map = a.take<nph_event_range>(std::max<size_t>(n_map_total, 1));
        d.jobs = a.take<nph_polya_job>(n_jobs);
        rs = run_layout(a, n_jobs, plan);
    };
    NPH_TRY(nph_lay_out(ctx, ctx->d_polya, layout));
    if (n_samples_total) NPH_CUDA(ctx, cudaMemcpyAsync(d.samples, samples, sizeof(float) * n_samples_total, cudaMemcpyHostToDevice, ctx->stream));
    if (n_events_total) NPH_CUDA(ctx, cudaMemcpyAsync(d.durations, durations, sizeof(float) * n_events_total, cudaMemcpyHostToDevice, ctx->stream));
    if (n_map_total) NPH_CUDA(ctx, cudaMemcpyAsync(d.map, map, sizeof(nph_event_range) * n_map_total, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.jobs, jobs, sizeof(nph_polya_job) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    return run_polya(ctx, d.samples, n_samples_total, d.durations, n_events_total, d.map, n_map_total, d.jobs, hj, plan, rs, results_out);
}

extern "C" int nph_polya_after_load(nph_ctx* ctx, nph_polya_result* results_out, size_t n_jobs)
{
    if (!ctx || !results_out) return NPH_ERR_INVALID;
    const nph_ctx::LoadedRaw& k = ctx->loaded_raw;
    if (!k.valid || n_jobs != k.jobs.size()) return NPH_ERR_STATE;
    if (n_jobs == 0) return NPH_OK;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n_events_total = k.event_off.back();
    // the host needs the job lengths for the schedule and the scratch: the same values the kernel writes, from the host copies
    std::vector<nph_polya_job> hj(n_jobs);
    for (size_t j = 0; j < n_jobs; ++j) {
        nph_polya_job& pj = hj[j];
        pj = nph_polya_job{};
        pj.n_samples = ctx->h_last_trim[j].end - ctx->h_last_trim[j].start;
        pj.n_kmers = k.jobs[j].n_kmers;
        pj.n_events = k.live_index[j] >= 0 ? (uint32_t)(k.event_off[j + 1] - k.event_off[j]) : 0u;
    }
    ScratchPlan plan;
    NPH_TRY(plan_scratch(ctx, hj, &plan));
    struct { nph_raw_job* raw_jobs; nph_raw_range* trim; int64_t* live_index; uint64_t* event_off; nph_polya_job* jobs; } d{};
    RunScratch rs;
    auto layout = [&](NphCarve& a) {
        d.raw_jobs = a.take<nph_raw_job>(n_jobs);
        d.trim = a.take<nph_raw_range>(n_jobs);
        d.live_index = a.take<int64_t>(n_jobs);
        d.event_off = a.take<uint64_t>(n_jobs + 1);
        d.jobs = a.take<nph_polya_job>(n_jobs);
        rs = run_layout(a, n_jobs, plan);
    };
    NPH_TRY(nph_lay_out(ctx, ctx->d_polya, layout));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.raw_jobs, k.jobs.data(), sizeof(nph_raw_job) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.trim, ctx->h_last_trim.data(), sizeof(nph_raw_range) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.live_index, k.live_index.data(), sizeof(int64_t) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.event_off, k.event_off.data(), sizeof(uint64_t) * (n_jobs + 1), cudaMemcpyHostToDevice, ctx->stream));
    AfterLoadArgs al{};
    al.raw_jobs = d.raw_jobs; al.trim = d.trim; al.live_index = d.live_index; al.event_off = d.event_off; al.cal = k.d_cal; al.n_jobs = (uint32_t)n_jobs; al.jobs_out = d.jobs;
    after_load_jobs_kernel<<<(unsigned)((n_jobs + 127) / 128), 128, 0, ctx->stream>>>(al);
    NPH_CUDA(ctx, cudaGetLastError());
    return run_polya(ctx, k.d_raw.p, k.n_samples_total, k.d_duration, n_events_total, k.d_b2e, k.n_ranks_total, d.jobs, hj, plan, rs, results_out);
}
