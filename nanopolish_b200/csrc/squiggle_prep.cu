// squiggle_prep.cu — the two remaining device steps of SquiggleRead::load_from_raw around event detection and ABEA
// (SURVEY.md section 8f, row N4):
//
//   trim_kernel          trim_and_segment_raw -> trim_raw_by_mad          ref: src/thirdparty/scrappie/scrappie_common.c:9-190
//                        (call site src/nanopolish_squiggle_read.cpp:226-233: trim_start 200, trim_end 10, chunk 100, perc 0.0)
//   recalibrate_kernel   base_to_event_map + events_per_base              ref: src/nanopolish_squiggle_read.cpp:273-302
//                        get_eventalignment_for_1d_basecalls              ref: src/nanopolish_squiggle_read.cpp:340-391
//                        recalibrate_model(scale_var=true, scale_drift=false)   ref: src/nanopolish_methyltrain.cpp:204-307
//
// Both are bit-exact restatements: medians are order statistics (only values at sorted positions are read, so no sort
// order among equal samples can matter),
// interpolated with the reference's float/double mix; the normal equations are summed in k-mer order by one lane
// (FP64, no contraction), and the 2x2 solve is Eigen's full-pivot LU written out.
#include "nph_internal.cuh"

#include <cstdlib>
#include <cstring>

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kTrimThreads = 256;
constexpr int kTrimWarps = kTrimThreads / 32;
constexpr int kMaxChunk = 128;           // samples per MAD chunk a warp holds in registers (reference uses 100)
constexpr int kCalWarps = 8;

// ------------------------------------------------------------------------------------------------------------
// quantilef's interpolation (scrappie_common.c:57-66) given the two order statistics it reads.
//   idx  = (size_t)(p * (nx - 1));  remf = p * (nx - 1) - idx          (float arithmetic)
//   out  = (1.0 - remf) * space[idx] + remf * space[idx + 1]           (double product + float product, narrowed)
// ------------------------------------------------------------------------------------------------------------
struct QuantilePos { uint32_t idx; float remf; bool interp; };

__host__ __device__ inline QuantilePos quantile_pos(float p, uint32_t nx)
{
    QuantilePos q;
    const float pos = p * (float)(nx - 1);
    q.idx = (uint32_t)pos;
    q.remf = pos - (float)q.idx;
    q.interp = q.idx < nx - 1;
    return q;
}

__device__ __forceinline__ float quantile_mix(const QuantilePos q, float lo, float hi)
{
    if (!q.interp) return lo;
    const double a = __dmul_rn(__dsub_rn(1.0, (double)q.remf), (double)lo);
    const double b = (double)__fmul_rn(q.remf, hi);
    return __double2float_rn(__dadd_rn(a, b));
}

__device__ __forceinline__ float sel_slot(const float (&v)[4], int s)
{
    float r = v[0];
    r = (s == 1) ? v[1] : r;
    r = (s == 2) ? v[2] : r;
    r = (s == 3) ? v[3] : r;
    return r;
}

// Order statistics q.idx and q.idx+1 of the n (<= 128) values a warp holds four per lane (slot s of lane l is element
// l + 32 s; slots past n must hold +inf).  A bitonic sorting network over the 128 slots: partners 1..16 apart sit in
// another lane (shuffle), partners 32 or 64 apart in another slot of the same lane.  Only VALUES at sorted positions are
// read, so how equal elements are ordered cannot matter (the reference's qsort comparator never reports equality
// either).  ~300 instructions per sort instead of ~1500 for rank counting.
__device__ __forceinline__ void warp_sort128(float (&v)[4], int lane)
{
#pragma unroll
    for (int k = 2; k <= 128; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j >= 1; j >>= 1) {
            if (j >= 32) {
                const int js = j >> 5;                         // partner slot distance: 1 or 2
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    if ((s & js) == 0) {
                        const bool up = (((s << 5) & k) == 0);   // k is 64 or 128 here: direction depends on the slot only
                        const float lo = fminf(v[s], v[s | js]), hi = fmaxf(v[s], v[s | js]);
                        v[s] = up ? lo : hi;
                        v[s | js] = up ? hi : lo;
                    }
                }
            } else {
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const float o = __shfl_xor_sync(kFull, v[s], j);
                    const int i = (s << 5) | lane;
                    const bool up = ((i & k) == 0);
                    const bool take_min = (((lane & j) == 0) == up);
                    v[s] = take_min ? fminf(v[s], o) : fmaxf(v[s], o);
                }
            }
        }
    }
}

__device__ __forceinline__ void warp_order_stats(float (&v)[4], const QuantilePos q, int lane, float& lo, float& hi)
{
    warp_sort128(v, lane);
    const int p0 = (int)q.idx, p1 = min((int)q.idx + 1, 127);
    lo = __shfl_sync(kFull, sel_slot(v, p0 >> 5), p0 & 31);
    hi = __shfl_sync(kFull, sel_slot(v, p1 >> 5), p1 & 31);
}

struct TrimParams {
    const float* raw;
    const nph_raw_read* reads;
    uint32_t n_reads;
    int32_t trim_start, trim_end, chunk;
    float perc;
    float* mad;                  // scratch: one float per chunk, read r at mad_off[r]
    const uint64_t* mad_off;
    nph_raw_range* out;
};

__global__ void __launch_bounds__(kTrimThreads) trim_kernel(const TrimParams p)
{
    __shared__ float s_stat[2];
    __shared__ int s_first, s_last;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const QuantilePos qc = quantile_pos(0.5f, (uint32_t)p.chunk);
    for (uint32_t r = blockIdx.x; r < p.n_reads; r += gridDim.x) {
        const nph_raw_read rd = p.reads[r];
        const float* __restrict__ x = p.raw + rd.sample_off;
        const uint32_t nchunk = rd.n_samples / (uint32_t)p.chunk;
        float* mad = p.mad + p.mad_off[r];
        if (nchunk == 0) {                      // the reference reads past an empty array and then asserts
            if (threadIdx.x == 0) p.out[r] = nph_raw_range{0u, 0u};
            continue;
        }
        // madf of every chunk (scrappie_common.c:98-119): median, absolute deviations, median again, * 1.4826f
        for (uint32_t c = wib; c < nchunk; c += kTrimWarps) {
            const float* xc = x + (size_t)c * p.chunk;
            const float inf = __int_as_float(0x7f800000);
            float x4[4], v[4];
#pragma unroll
            for (int s = 0; s < 4; ++s) { x4[s] = (lane + 32 * s < p.chunk) ? xc[lane + 32 * s] : inf; v[s] = x4[s]; }
            float lo, hi;
            warp_order_stats(v, qc, lane, lo, hi);
            const float med = quantile_mix(qc, lo, hi);
#pragma unroll
            for (int s = 0; s < 4; ++s) v[s] = (lane + 32 * s < p.chunk) ? fabsf(__fsub_rn(x4[s], med)) : inf;
            warp_order_stats(v, qc, lane, lo, hi);
            if (lane == 0) mad[c] = __fmul_rn(quantile_mix(qc, lo, hi), 1.4826f);
        }
        if (threadIdx.x == 0) { s_first = (int)nchunk; s_last = -1; }
        __syncthreads();
        // threshold = quantilef(madarr, perc): order statistics by rank counting over the whole array
        const QuantilePos qm = quantile_pos(p.perc, nchunk);
        for (uint32_t i = threadIdx.x; i < nchunk; i += kTrimThreads) {
            const float me = mad[i];
            uint32_t rank = 0;
            for (uint32_t j = 0; j < nchunk; ++j) { const float o = mad[j]; rank += (o < me || (o == me && j < i)) ? 1u : 0u; }
            if (rank == qm.idx) s_stat[0] = me;
            if (rank == qm.idx + 1) s_stat[1] = me;
        }
        __syncthreads();
        const float thresh = quantile_mix(qm, s_stat[0], qm.interp ? s_stat[1] : 0.0f);
        for (uint32_t i = threadIdx.x; i < nchunk; i += kTrimThreads) {
            if (mad[i] > thresh) { atomicMin(&s_first, (int)i); atomicMax(&s_last, (int)i); }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            // leading chunks at or below the threshold are dropped, same from the end; then the fixed trims
            long long start = (long long)s_first * p.chunk;
            long long end = (long long)(s_last + 1) * p.chunk;
            nph_raw_range o{0u, 0u};
            if (end > start) {                  // the reference asserts this
                start += p.trim_start;
                end -= p.trim_end;
                if (start < end) { o.start = (uint32_t)start; o.end = (uint32_t)end; }
            }
            p.out[r] = o;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------------------
// recalibration
// ------------------------------------------------------------------------------------------------------------
struct CalParams {
    NphCalArgs a;
    const DevModelView* models;
};

// A.fullPivLu().solve(b) for the symmetric 2x2 system, the way Eigen 3.3 computes it: largest |entry| (column-major
// scan, first wins) to the top-left by a row and a column swap, one elimination step, rank decided against
// epsilon * 2 * max pivot, unit-lower then upper substitution, columns permuted back.
__host__ __device__ inline void full_piv_lu_solve_2x2(double a00, double a01, double a11, double b0, double b1, double& x0, double& x1)
{
    double m[2][2] = {{a00, a01}, {a01, a11}};
    double b[2] = {b0, b1};
    int pr = 0, pc = 0;
    double big = fabs(m[0][0]);
    if (fabs(m[1][0]) > big) { big = fabs(m[1][0]); pr = 1; pc = 0; }
    if (fabs(m[0][1]) > big) { big = fabs(m[0][1]); pr = 0; pc = 1; }
    if (fabs(m[1][1]) > big) { big = fabs(m[1][1]); pr = 1; pc = 1; }
    x0 = 0.0; x1 = 0.0;
    if (big == 0.0) return;
    if (pr == 1) { double t; t = m[0][0]; m[0][0] = m[1][0]; m[1][0] = t; t = m[0][1]; m[0][1] = m[1][1]; m[1][1] = t; t = b[0]; b[0] = b[1]; b[1] = t; }
    if (pc == 1) { double t; t = m[0][0]; m[0][0] = m[0][1]; m[0][1] = t; t = m[1][0]; m[1][0] = m[1][1]; m[1][1] = t; }
#ifdef __CUDA_ARCH__
    const double l = __ddiv_rn(m[1][0], m[0][0]);
    const double u11 = __dsub_rn(m[1][1], __dmul_rn(l, m[0][1]));
    const double c1 = __dsub_rn(b[1], __dmul_rn(l, b[0]));
#else
    const double l = m[1][0] / m[0][0];
    const double u11 = m[1][1] - l * m[0][1];
    const double c1 = b[1] - l * b[0];
#endif
    double maxpivot = big;
    if (fabs(u11) > maxpivot) maxpivot = fabs(u11);
    const double thr = 2.220446049250313e-16 * 2.0 * maxpivot;
    double y0, y1;
    if (fabs(u11) > thr) {
#ifdef __CUDA_ARCH__
        y1 = __ddiv_rn(c1, u11);
        y0 = __ddiv_rn(__dsub_rn(b[0], __dmul_rn(y1, m[0][1])), m[0][0]);
#else
        y1 = c1 / u11;
        y0 = (b[0] - y1 * m[0][1]) / m[0][0];
#endif
    } else {                                    // rank 1: the dependent unknown is set to zero
        y1 = 0.0;
#ifdef __CUDA_ARCH__
        y0 = __ddiv_rn(b[0], m[0][0]);
#else
        y0 = b[0] / m[0][0];
#endif
    }
    if (pc == 1) { x0 = y1; x1 = y0; } else { x0 = y0; x1 = y1; }
}

__global__ void __launch_bounds__(kCalWarps * 32) recalibrate_kernel(const CalParams p)
{
    __shared__ double s_e[kCalWarps][32], s_mu[kCalWarps][32], s_sd[kCalWarps][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const DevModelView mv = p.models[p.a.model_id];
    for (uint32_t j = blockIdx.x * kCalWarps + wib; j < p.a.n_jobs; j += gridDim.x * kCalWarps) {
        const nph_abea_job job = p.a.jobs[j];
        const nph_read rd = p.a.reads[job.read];
        const uint32_t np = p.a.results[j].n_pairs;
        const nph_aligned_pair* __restrict__ pr = p.a.pairs + job.pairs_off;
        const uint32_t* __restrict__ rk = p.a.ranks + job.rank_off;
        nph_event_range* b2e = p.a.b2e + job.rank_off;
        const int nk = (int)job.n_kmers;
        nph_calibration cal;
        cal.shift = rd.shift; cal.scale = rd.scale; cal.drift = rd.drift; cal.var = rd.var;
        cal.events_per_base = 0.0; cal.n_used = 0; cal.status = 0;

        // base_to_event_map (squiggle_read.cpp:273-300).  A pair counts when its event differs from the previous
        // pair's; per k-mer keep the first and the last such pair (by position in the list, like the loop does).
        for (int ki = lane; ki < nk; ki += 32) b2e[ki] = nph_event_range{0x7fffffff, -1};
        __syncwarp();
        int ev_min = 0x7fffffff, ev_max = -1;
        bool bad = false;
        for (uint32_t i = lane; i < np; i += 32) {
            const nph_aligned_pair a = pr[i];
            if (a.ref_pos < 0 || a.ref_pos >= nk || a.read_pos < 0 || (uint32_t)a.read_pos >= rd.n_events) { bad = true; continue; }
            ev_min = min(ev_min, a.read_pos); ev_max = max(ev_max, a.read_pos);
            const int prev = i > 0 ? pr[i - 1].read_pos : -1;
            if (a.read_pos != prev) { atomicMin(&b2e[a.ref_pos].start, (int)i); atomicMax(&b2e[a.ref_pos].stop, (int)i); }
        }
        bad = __any_sync(kFull, bad);
        __syncwarp();
        for (int ki = lane; ki < nk; ki += 32) {
            const nph_event_range rg = b2e[ki];
            b2e[ki] = rg.stop < 0 ? nph_event_range{-1, -1} : nph_event_range{pr[rg.start].read_pos, pr[rg.stop].read_pos};
        }
        __syncwarp();
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { ev_min = min(ev_min, __shfl_xor_sync(kFull, ev_min, o)); ev_max = max(ev_max, __shfl_xor_sync(kFull, ev_max, o)); }
        if (bad) { if (lane == 0) { *p.a.bad_input = 1; cal.status = NPH_CAL_NOT_ALIGNED; p.a.out[j] = cal; } continue; }
        if (np == 0) { if (lane == 0) { cal.status = NPH_CAL_NOT_ALIGNED; p.a.out[j] = cal; } continue; }
        cal.events_per_base = __ddiv_rn((double)(unsigned long long)(ev_max - ev_min), (double)(unsigned long long)nk);

        // get_eventalignment_for_1d_basecalls + the extraction loop of recalibrate_model: walking k-mers in order, the
        // first event of a k-mer that has events is state 'M' unless the k-mer emitted just before has the same rank.
        double A00 = 0.0, A01 = 0.0, A11 = 0.0, B0 = 0.0, B1 = 0.0;
        uint32_t carry_rank = 0xffffffffu, n_used = 0;
        for (int k0 = 0; k0 < nk; k0 += 32) {
            const int ki = k0 + lane;
            nph_event_range rg{-1, -1};
            uint32_t rank = 0;
            if (ki < nk) { rg = b2e[ki]; rank = rk[ki]; }
            const bool has = rg.start != -1 && rg.start <= rg.stop;
            const unsigned hm = __ballot_sync(kFull, has);
            const unsigned below = hm & ((1u << lane) - 1u);
            const int src = below ? 31 - __clz(below) : 0;
            const uint32_t nb = __shfl_sync(kFull, rank, src);
            const uint32_t prev_rank = below ? nb : carry_rank;
            const bool is_m = has && prev_rank != rank;
            if (hm) carry_rank = __shfl_sync(kFull, rank, 31 - __clz(hm));
            const unsigned mm = __ballot_sync(kFull, is_m);
            if (mm == 0) continue;
            s_e[wib][lane] = is_m ? (double)p.a.ev_mean[rd.event_off + (uint32_t)rg.start] : 0.0;
            s_mu[wib][lane] = is_m ? mv.mean[rank] : 0.0;
            s_sd[wib][lane] = is_m ? mv.stdv[rank] : 1.0;
            __syncwarp();
            if (lane == 0) {
                for (unsigned rest = mm; rest; rest &= rest - 1) {
                    const int t = __ffs(rest) - 1;
                    const double sd = s_sd[wib][t], mu = s_mu[wib][t], e = s_e[wib][t];
                    const double inv_var = __ddiv_rn(1.0, __dmul_rn(sd, sd));
                    A00 = __dadd_rn(A00, inv_var);
                    A01 = __dadd_rn(A01, __dmul_rn(mu, inv_var));
                    A11 = __dadd_rn(A11, __dmul_rn(__dmul_rn(mu, mu), inv_var));
                    B0 = __dadd_rn(B0, __dmul_rn(e, inv_var));
                    B1 = __dadd_rn(B1, __dmul_rn(__dmul_rn(mu, e), inv_var));
                }
            }
            n_used += __popc(mm);
            __syncwarp();
        }
        cal.n_used = n_used;
        if (n_used < 200) {                      // minNumEventsToRescale: scalings stay as they were, read fails QC
            if (lane == 0) { cal.status = NPH_CAL_TOO_FEW_EVENTS; p.a.out[j] = cal; }
            continue;
        }
        double shift = 0.0, scale = 0.0;
        if (lane == 0) full_piv_lu_solve_2x2(A00, A01, A11, B0, B1, shift, scale);
        shift = __shfl_sync(kFull, shift, 0);
        scale = __shfl_sync(kFull, scale, 0);
        // scale_var: var = sqrt(mean of squared standardised residuals), second pass in the same order
        double var = 0.0;
        carry_rank = 0xffffffffu;
        for (int k0 = 0; k0 < nk; k0 += 32) {
            const int ki = k0 + lane;
            nph_event_range rg{-1, -1};
            uint32_t rank = 0;
            if (ki < nk) { rg = b2e[ki]; rank = rk[ki]; }
            const bool has = rg.start != -1 && rg.start <= rg.stop;
            const unsigned hm = __ballot_sync(kFull, has);
            const unsigned below = hm & ((1u << lane) - 1u);
            const int src = below ? 31 - __clz(below) : 0;
            const uint32_t nb = __shfl_sync(kFull, rank, src);
            const uint32_t prev_rank = below ? nb : carry_rank;
            const bool is_m = has && prev_rank != rank;
            if (hm) carry_rank = __shfl_sync(kFull, rank, 31 - __clz(hm));
            const unsigned mm = __ballot_sync(kFull, is_m);
            if (mm == 0) continue;
            double term = 0.0;
            if (is_m) {
                const double e = (double)p.a.ev_mean[rd.event_off + (uint32_t)rg.start], mu = mv.mean[rank], sd = mv.stdv[rank];
                const double yi = __dsub_rn(__dsub_rn(e, shift), __dmul_rn(scale, mu));
                term = __ddiv_rn(__dmul_rn(yi, yi), __dmul_rn(sd, sd));
            }
            s_e[wib][lane] = term;
            __syncwarp();
            if (lane == 0) for (unsigned rest = mm; rest; rest &= rest - 1) var = __dadd_rn(var, s_e[wib][__ffs(rest) - 1]);
            __syncwarp();
        }
        if (lane == 0) {
            var = __dsqrt_rn(__ddiv_rn(var, (double)(unsigned long long)n_used));
            cal.shift = shift; cal.scale = scale; cal.drift = 0.0; cal.var = var;
            if (var > 2.5) cal.status |= NPH_CAL_HIGH_VAR;                              // MIN_CALIBRATION_VAR
            else if (cal.events_per_base > 5.0) cal.status |= NPH_CAL_TOO_MANY_STAYS;   // squiggle_read.cpp:331-336
            p.a.out[j] = cal;
        }
    }
}

} // namespace

TrimScratch nph_trim_layout(NphCarve& a, const nph_raw_read* reads, size_t n_reads, int32_t varseg_chunk)
{
    uint64_t n_chunks = 0;
    for (size_t i = 0; i < n_reads; ++i) n_chunks += reads[i].n_samples / (uint32_t)varseg_chunk;
    TrimScratch s;
    s.reads = a.take<nph_raw_read>(n_reads);
    s.mad_off = a.take<uint64_t>(n_reads);
    s.mad = a.take<float>(n_chunks + 1);
    s.out = a.take<nph_raw_range>(n_reads);
    return s;
}

// trim_and_segment_raw over reads whose samples are on the device, in the scratch of nph_trim_layout; the ranges come
// back to the host (one sync).
int nph_trim_device(nph_ctx* ctx, const float* d_raw, size_t n_samples_total, const nph_raw_read* reads, size_t n_reads,
                    int32_t trim_start, int32_t trim_end, int32_t varseg_chunk, float varseg_thresh, const TrimScratch& s,
                    nph_raw_range* ranges_out)
{
    if (varseg_chunk < 2 || !(varseg_thresh >= 0.0f && varseg_thresh <= 1.0f) || trim_start < 0 || trim_end < 0) return NPH_ERR_INVALID;   // reference asserts
    if (varseg_chunk > kMaxChunk) return NPH_ERR_UNSUPPORTED;
    std::vector<uint64_t> mad_off(n_reads);
    uint64_t n_chunks = 0;
    for (size_t i = 0; i < n_reads; ++i) {
        if (reads[i].sample_off + reads[i].n_samples > n_samples_total) return NPH_ERR_INVALID;
        mad_off[i] = n_chunks;
        n_chunks += reads[i].n_samples / (uint32_t)varseg_chunk;
    }
    TrimParams p{};
    p.mad = s.mad; p.out = s.out;
    p.raw = d_raw; p.reads = s.reads; p.mad_off = s.mad_off; p.n_reads = (uint32_t)n_reads;
    p.trim_start = trim_start; p.trim_end = trim_end; p.chunk = varseg_chunk; p.perc = varseg_thresh;
    NPH_CUDA(ctx, cudaMemcpyAsync(s.reads, reads, sizeof(nph_raw_read) * n_reads, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(s.mad_off, mad_off.data(), sizeof(uint64_t) * n_reads, cudaMemcpyHostToDevice, ctx->stream));
    trim_kernel<<<(unsigned)std::min<size_t>(n_reads, (size_t)ctx->sm_count * 8), kTrimThreads, 0, ctx->stream>>>(p);
    NPH_CUDA(ctx, cudaGetLastError());
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(ranges_out, p.out, sizeof(nph_raw_range) * n_reads, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NPH_OK;
}

int nph_launch_recalibrate(nph_ctx* ctx, const NphCalArgs& args)
{
    CalParams p{};
    p.a = args;
    p.models = ctx->d_models.p;
    NPH_CUDA(ctx, cudaMemsetAsync(args.bad_input, 0, sizeof(int), ctx->stream));
    const int grid = (int)std::min<size_t>((args.n_jobs + kCalWarps - 1) / kCalWarps, (size_t)ctx->sm_count * 8);
    recalibrate_kernel<<<grid, kCalWarps * 32, 0, ctx->stream>>>(p);
    NPH_CUDA(ctx, cudaGetLastError());
    return NPH_OK;
}

extern "C" int nph_trim_raw_batch(nph_ctx* ctx, const float* raw, size_t n_samples_total, const nph_raw_read* reads, size_t n_reads,
                                  int32_t trim_start, int32_t trim_end, int32_t varseg_chunk, float varseg_thresh,
                                  nph_raw_range* ranges_out)
{
    if (!ctx) return NPH_ERR_INVALID;
    if (n_reads == 0) return NPH_OK;
    if (!raw || !reads || !ranges_out) return NPH_ERR_INVALID;
    if (varseg_chunk < 2) return NPH_ERR_INVALID;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    float* d_raw = nullptr;
    TrimScratch ts;
    auto layout = [&](NphCarve& a) { d_raw = a.take<float>(n_samples_total); ts = nph_trim_layout(a, reads, n_reads, varseg_chunk); };
    NPH_TRY(nph_borrow_arena(ctx, layout));
    NPH_CUDA(ctx, cudaMemcpyAsync(d_raw, raw, sizeof(float) * n_samples_total, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    NPH_TRY(nph_trim_device(ctx, d_raw, n_samples_total, reads, n_reads, trim_start, trim_end, varseg_chunk, varseg_thresh, ts, ranges_out));
    ctx->last_launches = 1;
    ctx->timing_valid = true;
    return NPH_OK;
}

extern "C" int nph_recalibrate_batch(nph_ctx* ctx, const nph_read* reads, size_t n_reads, const float* ev_mean, size_t n_events_total,
                                     const uint32_t* kmer_ranks, size_t n_ranks_total, const nph_abea_job* jobs, size_t n_jobs,
                                     uint32_t model_id, const nph_aligned_pair* pairs, size_t pairs_total,
                                     const nph_abea_result* results, nph_event_range* base_to_event_out, nph_calibration* calibrations_out)
{
    if (!ctx) return NPH_ERR_INVALID;
    if (n_jobs == 0) return NPH_OK;
    if (!reads || !ev_mean || !kmer_ranks || !jobs || !results || !calibrations_out || (!pairs && pairs_total)) return NPH_ERR_INVALID;
    if (model_id >= ctx->models.size()) return NPH_ERR_INVALID;
    const uint32_t n_states = ctx->models[model_id].n_states;
    for (size_t i = 0; i < n_reads; ++i)
        if (reads[i].event_off + reads[i].n_events > n_events_total) return NPH_ERR_INVALID;
    for (size_t j = 0; j < n_jobs; ++j) {
        const nph_abea_job& jb = jobs[j];
        if (jb.read >= n_reads || jb.n_kmers == 0 || jb.rank_off + jb.n_kmers > n_ranks_total) return NPH_ERR_INVALID;
        if (results[j].n_pairs > jb.pairs_cap || jb.pairs_off + results[j].n_pairs > pairs_total) return NPH_ERR_INVALID;
    }
    for (size_t i = 0; i < n_ranks_total; ++i)
        if (kmer_ranks[i] >= n_states) return NPH_ERR_INVALID;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    NphCalArgs a{};
    struct { float* ev; nph_read* reads; uint32_t* rk; nph_abea_job* jobs; nph_abea_result* res; nph_aligned_pair* pairs; } d{};
    auto layout = [&](NphCarve& c) {
        d.ev = c.take<float>(n_events_total);
        d.reads = c.take<nph_read>(n_reads);
        d.rk = c.take<uint32_t>(n_ranks_total);
        d.jobs = c.take<nph_abea_job>(n_jobs);
        d.res = c.take<nph_abea_result>(n_jobs);
        d.pairs = c.take<nph_aligned_pair>(pairs_total + 1);
        a.b2e = c.take<nph_event_range>(n_ranks_total);
        a.out = c.take<nph_calibration>(n_jobs);
        a.bad_input = c.take<int>(1);
    };
    NPH_TRY(nph_borrow_arena(ctx, layout));
    a.ev_mean = d.ev; a.reads = d.reads; a.model_id = model_id; a.ranks = d.rk; a.jobs = d.jobs;
    a.results = d.res; a.pairs = d.pairs; a.n_jobs = (uint32_t)n_jobs;
    NPH_CUDA(ctx, cudaMemcpyAsync(d.ev, ev_mean, sizeof(float) * n_events_total, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.reads, reads, sizeof(nph_read) * n_reads, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.rk, kmer_ranks, sizeof(uint32_t) * n_ranks_total, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.jobs, jobs, sizeof(nph_abea_job) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.res, results, sizeof(nph_abea_result) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    if (pairs_total) NPH_CUDA(ctx, cudaMemcpyAsync(d.pairs, pairs, sizeof(nph_aligned_pair) * pairs_total, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    NPH_TRY(nph_launch_recalibrate(ctx, a));
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->last_launches = 1;
    ctx->timing_valid = true;
    int bad = 0;
    NPH_CUDA(ctx, cudaMemcpyAsync(calibrations_out, a.out, sizeof(nph_calibration) * n_jobs, cudaMemcpyDeviceToHost, ctx->stream));
    if (base_to_event_out)
        NPH_CUDA(ctx, cudaMemcpyAsync(base_to_event_out, a.b2e, sizeof(nph_event_range) * n_ranks_total, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(&bad, a.bad_input, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (bad) { ctx->last_error = "nph_recalibrate_batch: an aligned pair lies outside its read or sequence"; return NPH_ERR_INVALID; }
    return NPH_OK;
}
