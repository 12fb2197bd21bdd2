// abea.cu — K2: adaptive banded event-to-sequence alignment on sm_100a, and the method-of-moments
// scaling estimate that prepares its input.
//
// Replaces, for a batch of reads:
//   adaptive_banded_simple_event_align   ref: src/nanopolish_raw_loader.cpp:77-379
//   estimate_scalings_using_mom          ref: src/nanopolish_raw_loader.cpp:17-60
//
// Design (DESIGN.md has the long form):
//   * one warp per read.  The reference keeps an (E+K+2) x 100 float band matrix plus a byte trace
//     per read (5 MB + 1.2 MB at 8k events) that it mallocs and fills with -inf on every call.  Here
//     the two live bands sit in registers: lane L owns the DP columns c = k+1 with c == L (mod 32)
//     through a 128-column circular window (4 register slots per lane), so a k-mer's Gaussian stays
//     in registers for the ~100+ bands it spends inside the band, "up" is the lane's own register,
//     "left"/"diag" arrive from lane L-1 by one shuffle per slot, and the event of every column
//     simply advances by one per band.
//   * Suzuki's move rule needs the two end cells of the previous band: two register-select +
//     shuffle broadcasts.
//   * the trace is 2 bits per cell, 32 B per band, written coalesced to a per-warp scratch that
//     stays L2 resident; the backtrack reads it back in 2 KB blocks through shared memory.
//   * scores follow the reference's mixed precision exactly: float band cells, transition terms added
//     in FP64 (lp_step/lp_stay/lp_skip are doubles there) and narrowed once; ties are broken by the
//     same compare chain (D, then U, then L wins on equality); so paths are identical.
#include "nph_internal.cuh"
#include "exact_math.cuh"
#include <math_constants.h>
#include <algorithm>
#include <cmath>
#include <vector>

namespace {

#ifndef NPH_ABEA_WARPS
#define NPH_ABEA_WARPS 20
#endif
constexpr int kWarps = NPH_ABEA_WARPS;
constexpr int kThreads = kWarps * 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kBW = 100;                 // ALN_BANDWIDTH (raw_loader.cpp:72)
#ifndef NPH_ABEA_TRACE_ROWS
#define NPH_ABEA_TRACE_ROWS 64
#endif
constexpr int kTraceBlockRows = NPH_ABEA_TRACE_ROWS;      // band rows fetched per backtrack block
constexpr int kFromD = 0, kFromU = 1, kFromL = 2;

struct AbeaJobConsts { double lp_stay; double lp_step; };

struct AbeaParams {
    const float* level;
    const DevRead* reads;
    const DevModelView* models;
    uint32_t model_id;
    const uint32_t* ranks;
    const nph_abea_job* jobs;
    const AbeaJobConsts* consts;
    const uint32_t* order;
    uint32_t n_jobs;
    unsigned int* counter;
    nph_aligned_pair* pairs;
    nph_abea_result* results;
    float4* scratch_params;     // per warp: kmax_stride float4 {mu', sigma', log(1/sqrt 2pi) - log sigma', RN(1/sigma')}
    uint8_t* scratch_trace;     // per warp: trace_stride bytes (32 per band)
    uint32_t kmax_stride;
    uint64_t trace_stride;
    double lp_skip, lp_trim;
    float log_inv_sqrt_2pi;
    int active_warps;            // warps per CTA that take jobs (small batches are spread over all SMs)
};

__device__ __forceinline__ float sel4(const float (&v)[4], int s)
{
    float r = v[0];
    r = (s == 1) ? v[1] : r;
    r = (s == 2) ? v[2] : r;
    r = (s == 3) ? v[3] : r;
    return r;
}

__global__ void __launch_bounds__(kThreads, 1) abea_kernel(const AbeaParams p)
{
    __shared__ __align__(16) uint8_t s_trace[kWarps][kTraceBlockRows * 32];
    __shared__ float s_em[kWarps][32];

    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    if (wib >= p.active_warps) return;        // warps are independent: no block-level barrier below
    const int warp_global = blockIdx.x * kWarps + wib;
    float4* const prm = p.scratch_params + (size_t)warp_global * p.kmax_stride;
    uint8_t* const trace = p.scratch_trace + (size_t)warp_global * p.trace_stride;
    const float NEG = -CUDART_INF_F;
    const DevModelView mv = p.models[p.model_id];

    for (;;) {
        uint32_t slot_idx = 0;
        if (lane == 0) slot_idx = atomicAdd(p.counter, 1u);
        slot_idx = __shfl_sync(kFull, slot_idx, 0);
        if (slot_idx >= p.n_jobs) break;
        const uint32_t job_idx = p.order[slot_idx];
        const nph_abea_job job = p.jobs[job_idx];
        const DevRead rd = p.reads[job.read];
        const AbeaJobConsts jc = p.consts[job_idx];
        const int E = (int)rd.n_events;
        const int K = (int)job.n_kmers;
        const float* lv = p.level + rd.event_off;
        const double lp_step = jc.lp_step, lp_stay = jc.lp_stay, lp_skip = p.lp_skip, lp_trim = p.lp_trim;

        // ---- prologue: read-scaled Gaussian of every k-mer (FP64 like the reference, then narrowed)
        {
            const uint32_t* rk = p.ranks + job.rank_off;
            for (int i = lane; i < K; i += 32) {
                const uint32_t r = rk[i];
                const float mu = (float)__dadd_rn(__dmul_rn(rd.scale, mv.mean[r]), rd.shift);
                const float sd = (float)__dmul_rn(mv.stdv[r], rd.var);
                const float lsd = (float)__dadd_rn(mv.log_stdv[r], rd.log_var);
                prm[i] = make_float4(mu, sd, __fsub_rn(p.log_inv_sqrt_2pi, lsd), __frcp_rn(sd));
            }
        }
        __syncwarp();

        // ---- band state.  Column c = k+1 (c == 0 is the trim column k == -1).  Band bi holds the columns
        // [lo, lo+99] with lo = band_lower_left[bi].kmer_idx + 1, and the event of column c is bi-1-c.
        // Band 1 (the state we start from): lo = -50, only cell (event 0, trim column) = lp_trim.
        int lo = -kBW / 2;                       // band 1: kmer_idx = -1 - 50
        int cs[4];                               // column currently held by each register slot
        float b1[4];                             // own column in band bi-1
        double b1d[4], dgd[4];                   // the same widened (every band value enters three sums as a double: widen it once) ; left column in band bi-2
        float mu[4], sd[4], cc[4], ry[4], xn[4];
        {
            const int ulo = lo + 128;
            const int base = ulo + ((lane - ulo) & 31);
            const int s0 = (base >> 5) & 3;
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                cs[s] = base + 32 * ((s - s0) & 3) - 128;
                b1[s] = (cs[s] == 0) ? (float)lp_trim : NEG;      // band 1, trim cell of event 0
                b1d[s] = (double)b1[s];
                dgd[s] = (cs[s] == 1) ? 0.0 : (double)NEG;        // band 0: start cell (-1,-1) = 0 is left-diag of column 1
                mu[s] = 0.f; sd[s] = 1.f; cc[s] = 0.f; ry[s] = 1.f; xn[s] = 0.f;
                if (cs[s] >= 1 && cs[s] <= K) {
                    const float4 g = prm[cs[s] - 1];
                    mu[s] = g.x; sd[s] = g.y; cc[s] = g.z; ry[s] = g.w;
                }
                const int e2 = 2 - 1 - cs[s];                      // event of this column in band 2
                if (e2 >= 0 && e2 < E) xn[s] = lv[e2];
            }
        }
        float best = NEG;
        int best_e = -1;
        const int n_bands = E + K + 2;
        const int uK = K + 128;
        const int laneK = uK & 31, slotK = (uK >> 5) & 3;

        float4 g_next = (lo + 128 <= K) ? prm[lo + 128 - 1] : make_float4(0.f, 1.f, 0.f, 1.f);   // Gaussian of the next column to enter a slot
        float x_down = lv[min(max(1 - lo, 0), E - 1)];       // level the lowest column meets in band 2 (already loaded above: a down move rewrites the same value)
        for (int bi = 2; bi < n_bands; ++bi) {
            // Suzuki's rule on the two ends of band bi-1 (offset 0 = column lo, offset 99 = column lo+99)
            bool right;
            {
                const int u0 = lo + 128, u1 = lo + 128 + (kBW - 1);
                const float ll = __shfl_sync(kFull, sel4(b1, (u0 >> 5) & 3), u0 & 31);
                const float ur = __shfl_sync(kFull, sel4(b1, (u1 >> 5) & 3), u1 & 31);
                right = (ll == NEG && ur == NEG) ? ((bi & 1) == 1) : (ll < ur);
            }
            // left neighbour column in band bi-1 (lane 0's neighbour lives in lane 31, previous slot)
            double lfd[4];
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const double send = (lane == 31) ? b1d[(s + 3) & 3] : b1d[s];
                lfd[s] = __shfl_sync(kFull, send, (lane + 31) & 31);
            }
            if (right) {
                // column `lo` leaves the band for good: exactly one (lane, slot) owns it; that slot now follows
                // column lo+128 (not yet in band: everything about it is -inf until the band reaches it)
                // (its Gaussian was fetched at the previous right move, so no load sits on this band's critical path; the
                // slot's event level is refreshed below like every other slot's and is not used before the band arrives)
                const int u = lo + 128;
                const bool own = lane == (u & 31);
                const int cn = lo + 128;
                const float4 g = g_next;
                // the slot is the same for the whole warp: branch on it once instead of predicating the four slots' copies
#define NPH_ABEA_NEW_COLUMN(S) if (own) { cs[S] = cn; b1[S] = NEG; b1d[S] = (double)NEG; dgd[S] = (double)NEG; lfd[S] = (double)NEG; \
                                          mu[S] = g.x; sd[S] = g.y; cc[S] = g.z; ry[S] = g.w; }
                switch ((u >> 5) & 3) {
                    case 0: NPH_ABEA_NEW_COLUMN(0) break;
                    case 1: NPH_ABEA_NEW_COLUMN(1) break;
                    case 2: NPH_ABEA_NEW_COLUMN(2) break;
                    default: NPH_ABEA_NEW_COLUMN(3) break;
                }
#undef NPH_ABEA_NEW_COLUMN
                lo += 1;
                g_next = (lo + 128 <= K) ? prm[lo + 128 - 1] : make_float4(0.f, 1.f, 0.f, 1.f);
            } else {
                // the band moved down: its lowest column meets a new event (fetched one band ahead); every other column's event
                // level came from its left neighbour, and after a right move the column that entered the window got its own that way
                const int u = lo + 128;
                const bool own = lane == (u & 31);
                switch ((u >> 5) & 3) {
                    case 0: if (own) xn[0] = x_down; break;
                    case 1: if (own) xn[1] = x_down; break;
                    case 2: if (own) xn[2] = x_down; break;
                    default: if (own) xn[3] = x_down; break;
                }
            }
            uint32_t tbyte = 0;
            const int hi = lo + (kBW - 1);
            const unsigned col_lim = (unsigned)min(hi, K);     // a real cell needs 1 <= c <= min(hi, K)
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const int c = cs[s];
                const int e = bi - 1 - c;
                const bool cell = ((unsigned)e < (unsigned)E) && ((unsigned)(c - 1) < col_lim);
                const float x = xn[s];
                // emission (emissions.h:51-55) — computed for every slot, used where the cell exists
                const float a = div_by_cached_rcp(__fsub_rn(x, mu[s]), sd[s], ry[s]);
                const float em = __fadd_rn(cc[s], __fmul_rn(__fmul_rn(-0.5f, a), a));
                const double emd = (double)em;
                const float score_d = (float)__dadd_rn(__dadd_rn(dgd[s], lp_step), emd);
                const float score_u = (float)__dadd_rn(__dadd_rn(b1d[s], lp_stay), emd);
                const float score_l = (float)__dadd_rn(lfd[s], lp_skip);
                float mx = score_d;
                int from = kFromD;
                mx = score_u > mx ? score_u : mx;
                from = (mx == score_u) ? kFromU : from;
                mx = score_l > mx ? score_l : mx;
                from = (mx == score_l) ? kFromL : from;
                dgd[s] = lfd[s];
                b1[s] = cell ? mx : NEG;
                b1d[s] = (double)b1[s];
                tbyte |= (uint32_t)(cell ? from : 0) << (2 * s);
            }
            // next band's event levels: column c meets event bi - c, which column c - 1 met in this band — shift the levels one
            // column up (lane 0's neighbour lives in lane 31, previous slot) instead of four clamped loads; the level the lowest
            // column would meet after a down move is fetched now (one broadcast load), a band ahead of its use
            {
                float xs[4];
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const float send = (lane == 31) ? xn[(s + 3) & 3] : xn[s];
                    xs[s] = __shfl_sync(kFull, send, (lane + 31) & 31);
                }
#pragma unroll
                for (int s = 0; s < 4; ++s) xn[s] = xs[s];
                x_down = lv[min(max(bi - lo, 0), E - 1)];
            }
            if (lo <= 0) {
                // the trim column (c == 0, k-mer -1) is still inside the band: lp_trim * (event + 1), from = U (:206-216)
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const int e = bi - 1;
                    if (cs[s] == 0 && e < E) { b1[s] = (float)__dmul_rn(lp_trim, (double)(e + 1)); b1d[s] = (double)b1[s]; tbyte |= (uint32_t)kFromU << (2 * s); }
                }
            }
            trace[(size_t)bi * 32 + lane] = (uint8_t)tbyte;

            // best end cell: last k-mer (column K) against any event, remaining events trimmed (:309-324).
            // Bands visit that column's events in increasing order, so a strict '>' keeps the first maximum.
            if (hi >= K && lane == laneK) {
                const int c = (slotK == 0) ? cs[0] : (slotK == 1) ? cs[1] : (slotK == 2) ? cs[2] : cs[3];
                const int e = bi - 1 - c;
                if (c == K && e >= 0 && e < E) {
                    const float v = sel4(b1, slotK);
                    const float sc = (float)__dadd_rn((double)v, __dmul_rn((double)(unsigned long long)(E - e), lp_trim));
                    if (sc > best) { best = sc; best_e = e; }
                }
            }
        }
        __syncwarp();
        best_e = __shfl_sync(kFull, best_e, laneK);
        int status = 0;
        if (best_e < 0) { status |= NPH_ABEA_NO_END_CELL; }

        // ---- backtrack (:332-361): every lane walks the same path out of the shared trace block; lane 0 records it
        nph_aligned_pair* const out = p.pairs + job.pairs_off;
        const int cap = (int)job.pairs_cap;
        int n_out = 0, max_gap = 0, last_k = -1;
        if (!status) {
            int cur_e = best_e, cur_k = K - 1, cur_gap = 0;
            int blk_lo = 1 << 30;
            while (cur_k >= 0 && cur_e >= 0) {
                const int bi = cur_e + cur_k + 2;
                if (bi < blk_lo) {
                    __syncwarp();
                    blk_lo = max(0, bi - (kTraceBlockRows - 1));
                    const uint4* src = reinterpret_cast<const uint4*>(trace + (size_t)blk_lo * 32);
                    uint4* dst = reinterpret_cast<uint4*>(s_trace[wib]);
#pragma unroll
                    for (int i = 0; i < (kTraceBlockRows * 32) / (16 * 32); ++i) dst[lane + 32 * i] = __ldcg(src + lane + 32 * i);
                    __syncwarp();
                }
                const int u = cur_k + 1 + 128;
                const uint32_t byte = s_trace[wib][(bi - blk_lo) * 32 + (u & 31)];
                const int from = (byte >> (2 * ((u >> 5) & 3))) & 3;
                if (n_out < cap) { if (lane == 0) out[cap - 1 - n_out] = nph_aligned_pair{cur_k, cur_e}; }
                else status |= NPH_ABEA_PAIRS_OVERFLOW;
                ++n_out;
                last_k = cur_k;
                if (from == kFromD) { cur_k -= 1; cur_e -= 1; cur_gap = 0; }
                else if (from == kFromU) { cur_e -= 1; cur_gap = 0; }
                else { cur_k -= 1; cur_gap += 1; max_gap = max(max_gap, cur_gap); }
            }
        }
        __syncwarp();

        // ---- QC (:365-372): mean emission over the path, summed in path order in FP64 like the reference
        double sum_emission = 0.0;
        if (!status) {
            for (int i0 = 0; i0 < n_out; i0 += 32) {
                const int i = i0 + lane;
                float em = 0.f;
                if (i < n_out) {
                    const unsigned long long raw = __ldcg(reinterpret_cast<const unsigned long long*>(out + (cap - 1 - i)));
                    const int pk = (int)(uint32_t)(raw & 0xffffffffull), pe = (int)(uint32_t)(raw >> 32);   // {ref_pos, read_pos}
                    const float4 g = prm[pk];
                    const float a = div_by_cached_rcp(__fsub_rn(lv[pe], g.x), g.y, g.w);
                    em = __fadd_rn(g.z, __fmul_rn(__fmul_rn(-0.5f, a), a));
                }
                s_em[wib][lane] = em;
                __syncwarp();
                if (lane == 0) {
                    const int cnt = min(32, n_out - i0);
                    for (int j = 0; j < cnt; ++j) sum_emission = __dadd_rn(sum_emission, (double)s_em[wib][j]);
                }
                __syncwarp();
            }
        }
        sum_emission = __shfl_sync(kFull, sum_emission, 0);
        const double avg = sum_emission / (double)n_out;
        if (!status) {
            if (avg < -5.0) status |= NPH_ABEA_LOW_EMISSION;
            if (!(last_k == 0)) status |= NPH_ABEA_NOT_SPANNED;     // path starts at K-1 by construction
            if (max_gap > 50) status |= NPH_ABEA_MAX_GAP;
        }
        // ---- pairs were written back to front at the end of the slot: move them to its start, ascending
        if (!status && n_out < cap) {
            const int shift = cap - n_out;
            for (int i0 = 0; i0 < n_out; i0 += 32) {
                const int i = i0 + lane;
                unsigned long long v = 0;
                if (i < n_out) v = __ldcg(reinterpret_cast<const unsigned long long*>(out + shift + i));
                __syncwarp();
                if (i < n_out) reinterpret_cast<unsigned long long*>(out)[i] = v;
                __syncwarp();
            }
        }
        if (lane == 0) {
            nph_abea_result r;
            r.n_pairs = status ? 0u : (uint32_t)n_out;
            r.status = status;
            r.max_gap = max_gap;
            r.n_aligned = (uint32_t)n_out;
            r.avg_log_emission = status & (NPH_ABEA_NO_END_CELL | NPH_ABEA_PAIRS_OVERFLOW) ? 0.0 : avg;
            p.results[job_idx] = r;
        }
        __syncwarp();
    }
}

// ---- method of moments (raw_loader.cpp:17-60): strictly sequential FP64 sums, one warp per read:
// lanes stage 32 values at a time, lane 0 folds them in index order so the rounding sequence is the reference's.
struct MomParams {
    const float* ev_mean;
    const DevRead* reads;
    const DevModelView* models;
    uint32_t model_id;
    const uint32_t* ranks;
    const nph_abea_job* jobs;
    uint32_t n_jobs;
    double* out;     // 2 per job: shift, scale
    int reversed;    // 1: the event array is stored back to front (direct RNA after load_from_raw's reversal); the sums
                     // still run in acquisition order, the order the reference's MoM sees (squiggle_read.cpp:237-239)
};

__global__ void __launch_bounds__(kThreads) mom_kernel(const MomParams p)
{
    __shared__ double s_buf[kWarps][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const DevModelView mv = p.models[p.model_id];
    for (uint32_t j = blockIdx.x * kWarps + wib; j < p.n_jobs; j += gridDim.x * kWarps) {
        const nph_abea_job job = p.jobs[j];
        const DevRead rd = p.reads[job.read];
        const float* m = p.ev_mean + rd.event_off;
        const uint32_t* rk = p.ranks + job.rank_off;
        const int n = (int)rd.n_events, nk = (int)job.n_kmers;
        double ev_sum = 0.0, k_sum = 0.0, k_sq = 0.0, ev_sq = 0.0;
        for (int i0 = 0; i0 < n; i0 += 32) {
            s_buf[wib][lane] = (i0 + lane < n) ? (double)m[p.reversed ? n - 1 - (i0 + lane) : i0 + lane] : 0.0;
            __syncwarp();
            if (lane == 0) { const int cnt = min(32, n - i0); for (int t = 0; t < cnt; ++t) ev_sum = __dadd_rn(ev_sum, s_buf[wib][t]); }
            __syncwarp();
        }
        for (int i0 = 0; i0 < nk; i0 += 32) {
            s_buf[wib][lane] = (i0 + lane < nk) ? mv.mean[rk[i0 + lane]] : 0.0;
            __syncwarp();
            if (lane == 0) {
                const int cnt = min(32, nk - i0);
                for (int t = 0; t < cnt; ++t) { const double l = s_buf[wib][t]; k_sum = __dadd_rn(k_sum, l); k_sq = __dadd_rn(k_sq, __dmul_rn(l, l)); }
            }
            __syncwarp();
        }
        double shift = 0.0;
        if (lane == 0) shift = __dsub_rn(__ddiv_rn(ev_sum, (double)n), __ddiv_rn(k_sum, (double)nk));
        shift = __shfl_sync(kFull, shift, 0);
        for (int i0 = 0; i0 < n; i0 += 32) {
            double d = 0.0;
            if (i0 + lane < n) { d = __dsub_rn((double)m[p.reversed ? n - 1 - (i0 + lane) : i0 + lane], shift); d = __dmul_rn(d, d); }
            s_buf[wib][lane] = d;
            __syncwarp();
            if (lane == 0) { const int cnt = min(32, n - i0); for (int t = 0; t < cnt; ++t) ev_sq = __dadd_rn(ev_sq, s_buf[wib][t]); }
            __syncwarp();
        }
        if (lane == 0) {
            p.out[2 * (size_t)j] = shift;
            p.out[2 * (size_t)j + 1] = __ddiv_rn(__ddiv_rn(ev_sq, (double)n), __ddiv_rn(k_sq, (double)nk));
        }
    }
}

int validate_abea_jobs(nph_ctx* ctx, const nph_abea_job* jobs, size_t n_jobs, size_t n_ranks_total, uint32_t model_id,
                       size_t pairs_total)
{
    if (model_id >= ctx->models.size()) return NPH_ERR_INVALID;
    for (size_t j = 0; j < n_jobs; ++j) {
        const nph_abea_job& jb = jobs[j];
        if (jb.read >= ctx->n_reads || jb.n_kmers == 0) return NPH_ERR_INVALID;
        if (jb.n_kmers > n_ranks_total || jb.rank_off > n_ranks_total - jb.n_kmers) return NPH_ERR_INVALID;      // overflow-safe
        if (jb.pairs_cap > pairs_total || jb.pairs_off > pairs_total - jb.pairs_cap) return NPH_ERR_INVALID;
    }
    return NPH_OK;
}

// ABEA's band storage in ctx->d_arena: per warp, the k-mer parameters and the trace
void abea_layout(NphCarve& a, const nph_ctx* ctx, AbeaParams& p)
{
    const size_t warps = (size_t)ctx->sm_count * kWarps;
    p.scratch_params = a.take<float4>((size_t)ctx->abea_kmax * warps);
    p.scratch_trace = a.take<uint8_t>(ctx->abea_trace_stride * warps);
}

} // namespace

int nph_launch_abea(nph_ctx* ctx)
{
    AbeaParams p{};
    p.level = ctx->d_level.p;
    p.reads = ctx->d_reads.p;
    p.models = ctx->d_models.p;
    p.model_id = ctx->abea_model;
    p.ranks = ctx->d_abea_ranks.p;
    p.jobs = ctx->d_abea_jobs.p;
    p.order = ctx->d_abea_order.p;
    p.n_jobs = (uint32_t)ctx->n_abea_jobs;
    p.counter = ctx->d_counters.p + (NPH_NUM_COUNTERS - 1);
    p.pairs = ctx->d_pairs.p;
    p.results = ctx->d_abea_res.p;
    p.kmax_stride = ctx->abea_kmax;
    p.trace_stride = ctx->abea_trace_stride;
    NPH_TRY(nph_carve(ctx, ctx->d_arena, [&](NphCarve& a) { abea_layout(a, ctx, p); }));
    p.consts = reinterpret_cast<const AbeaJobConsts*>(ctx->d_abea_consts.p);
    p.lp_skip = log(1e-10);
    p.lp_trim = log(0.01);
    p.log_inv_sqrt_2pi = ctx->consts.log_inv_sqrt_2pi;
    NPH_CUDA(ctx, cudaMemsetAsync(ctx->d_counters.p + (NPH_NUM_COUNTERS - 1), 0, sizeof(unsigned int), ctx->stream));
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    // A read is one warp's sequential walk over ~E+K bands, so a BamProcessor-sized batch (512 reads) is latency
    // bound: give every warp its own scheduler slot across all SMs before stacking warps on one SM.
    const int grid = (int)std::min<size_t>((size_t)ctx->sm_count, ctx->n_abea_jobs);
    p.active_warps = (int)std::min<size_t>((size_t)kWarps, (ctx->n_abea_jobs + grid - 1) / grid);
    abea_kernel<<<grid, kThreads, 0, ctx->stream>>>(p);
    NPH_CUDA(ctx, cudaGetLastError());
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->last_launches = 1;
    ctx->timing_valid = true;
    return NPH_OK;
}

// estimate_scalings_using_mom over the loaded ABEA jobs (reads, ranks and jobs already on the device)
int nph_launch_mom(nph_ctx* ctx, double* d_shift_scale_out, bool reversed)
{
    if (!ctx->ev_mean_resident) return NPH_ERR_STATE;      // the pipelined one-shot score leaves only d_level behind
    MomParams p{};
    p.reversed = reversed ? 1 : 0;
    p.ev_mean = ctx->d_ev_mean.p; p.reads = ctx->d_reads.p; p.models = ctx->d_models.p; p.model_id = ctx->abea_model;
    p.ranks = ctx->d_abea_ranks.p; p.jobs = ctx->d_abea_jobs.p; p.n_jobs = (uint32_t)ctx->n_abea_jobs; p.out = d_shift_scale_out;
    const int grid = (int)std::min<size_t>((ctx->n_abea_jobs + kWarps - 1) / kWarps, (size_t)ctx->sm_count * 4);
    mom_kernel<<<grid, kThreads, 0, ctx->stream>>>(p);
    NPH_CUDA(ctx, cudaGetLastError());
    return NPH_OK;
}

extern "C" {

int nph_abea_jobs_load(nph_ctx* ctx, const uint32_t* kmer_ranks, size_t n_ranks_total,
                       const nph_abea_job* jobs, size_t n_jobs, uint32_t model_id, size_t pairs_total)
{
    if (!ctx || !kmer_ranks || !jobs || n_jobs == 0) return NPH_ERR_INVALID;
    if (!ctx->reads_loaded) return NPH_ERR_STATE;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    NPH_TRY(validate_abea_jobs(ctx, jobs, n_jobs, n_ranks_total, model_id, pairs_total));

    // per-job transition penalties, evaluated with the host libm in FP64 exactly as raw_loader.cpp:95-108
    std::vector<AbeaJobConsts> consts(n_jobs);
    std::vector<uint64_t> bands(n_jobs);
    uint32_t kmax = 1;
    uint64_t max_bands = 4;
    const double lp_skip = log(1e-10);
    for (size_t j = 0; j < n_jobs; ++j) {
        const double n_events = (double)ctx->h_read_n_events[jobs[j].read];
        const double events_per_kmer = n_events / jobs[j].n_kmers;
        const double p_stay = 1 - (1 / (events_per_kmer + 1));
        consts[j].lp_stay = log(p_stay);
        consts[j].lp_step = log(1.0 - exp(lp_skip) - exp(consts[j].lp_stay));
        bands[j] = (uint64_t)ctx->h_read_n_events[jobs[j].read] + jobs[j].n_kmers + 2;
        kmax = std::max(kmax, jobs[j].n_kmers);
        max_bands = std::max(max_bands, bands[j]);
    }
    const std::vector<uint32_t> order = longest_first(bands);   // longest reads first

    ctx->abea_kmax = kmax;
    ctx->abea_trace_stride = 32 * (max_bands + kTraceBlockRows);
    // ABEA owns the arena (this load sets abea_loaded below); the pointers abea_layout writes into p are not needed here
    AbeaParams p{};
    NPH_TRY(nph_reserve(ctx, ctx->d_arena, nph_measure([&](NphCarve& a) { abea_layout(a, ctx, p); })));
    NPH_TRY(nph_reserve(ctx, ctx->d_abea_jobs, n_jobs));
    NPH_TRY(nph_reserve(ctx, ctx->d_abea_ranks, n_ranks_total));
    NPH_TRY(nph_reserve(ctx, ctx->d_abea_order, n_jobs));
    NPH_TRY(nph_reserve(ctx, ctx->d_abea_consts, 2 * n_jobs));
    NPH_TRY(nph_reserve(ctx, ctx->d_pairs, pairs_total));
    NPH_TRY(nph_reserve(ctx, ctx->d_abea_res, n_jobs));
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_abea_jobs.p, jobs, sizeof(nph_abea_job) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_abea_ranks.p, kmer_ranks, sizeof(uint32_t) * n_ranks_total, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_abea_order.p, order.data(), sizeof(uint32_t) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_abea_consts.p, consts.data(), sizeof(AbeaJobConsts) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->n_abea_jobs = n_jobs;
    ctx->abea_pairs_total = pairs_total;
    ctx->abea_model = model_id;
    ctx->abea_loaded = true;
    return NPH_OK;
}

int nph_abea_run(nph_ctx* ctx)
{
    if (!ctx) return NPH_ERR_INVALID;
    if (!ctx->reads_loaded || !ctx->abea_loaded) return NPH_ERR_STATE;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    return nph_launch_abea(ctx);
}

int nph_abea_fetch(nph_ctx* ctx, nph_aligned_pair* pairs_out, size_t pairs_total, nph_abea_result* results, size_t n_jobs)
{
    if (!ctx || !pairs_out || !results) return NPH_ERR_INVALID;
    if (!ctx->abea_loaded || n_jobs > ctx->n_abea_jobs || pairs_total > ctx->abea_pairs_total) return NPH_ERR_STATE;
    NPH_CUDA(ctx, cudaMemcpyAsync(pairs_out, ctx->d_pairs.p, sizeof(nph_aligned_pair) * pairs_total, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(results, ctx->d_abea_res.p, sizeof(nph_abea_result) * n_jobs, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NPH_OK;
}

int nph_abea_batch(nph_ctx* ctx,
                   const nph_read* reads, size_t n_reads,
                   const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                   const uint32_t* kmer_ranks, size_t n_ranks_total,
                   const nph_abea_job* jobs, size_t n_jobs, uint32_t model_id,
                   nph_aligned_pair* pairs_out, size_t pairs_total, nph_abea_result* results)
{
    if (n_jobs == 0) return ctx ? NPH_OK : NPH_ERR_INVALID;      // empty batch
    NPH_TRY(nph_reads_load(ctx, reads, n_reads, ev_mean, ev_start_time, n_events_total));
    NPH_TRY(nph_abea_jobs_load(ctx, kmer_ranks, n_ranks_total, jobs, n_jobs, model_id, pairs_total));
    NPH_TRY(nph_abea_run(ctx));
    return nph_abea_fetch(ctx, pairs_out, pairs_total, results, n_jobs);
}

int nph_mom_batch(nph_ctx* ctx, const nph_read* reads, size_t n_reads,
                  const float* ev_mean, size_t n_events_total,
                  const uint32_t* kmer_ranks, size_t n_ranks_total,
                  const nph_abea_job* jobs, size_t n_jobs, uint32_t model_id, double* shift_scale_out)
{
    if (!ctx || !reads || !ev_mean || !kmer_ranks || !jobs || !shift_scale_out || n_jobs == 0) return NPH_ERR_INVALID;
    // scalings are what this call estimates: load the reads with whatever the caller has (only events are used)
    NPH_TRY(nph_reads_load(ctx, reads, n_reads, ev_mean, nullptr, n_events_total));
    if (model_id >= ctx->models.size()) return NPH_ERR_INVALID;
    for (size_t j = 0; j < n_jobs; ++j) {
        if (jobs[j].read >= n_reads || jobs[j].n_kmers == 0 || jobs[j].n_kmers > n_ranks_total || jobs[j].rank_off > n_ranks_total - jobs[j].n_kmers) return NPH_ERR_INVALID;
    }
    NPH_TRY(nph_reserve(ctx, ctx->d_abea_jobs, n_jobs));
    NPH_TRY(nph_reserve(ctx, ctx->d_abea_ranks, n_ranks_total));
    NPH_TRY(nph_reserve(ctx, ctx->d_abea_consts, 2 * n_jobs));
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_abea_jobs.p, jobs, sizeof(nph_abea_job) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(ctx->d_abea_ranks.p, kmer_ranks, sizeof(uint32_t) * n_ranks_total, cudaMemcpyHostToDevice, ctx->stream));
    MomParams p{};
    p.ev_mean = ctx->d_ev_mean.p; p.reads = ctx->d_reads.p; p.models = ctx->d_models.p; p.model_id = model_id;
    p.ranks = ctx->d_abea_ranks.p; p.jobs = ctx->d_abea_jobs.p; p.n_jobs = (uint32_t)n_jobs; p.out = ctx->d_abea_consts.p;
    int grid = (int)std::min<size_t>((n_jobs + kWarps - 1) / kWarps, (size_t)ctx->sm_count * 4);
    mom_kernel<<<grid, kThreads, 0, ctx->stream>>>(p);
    NPH_CUDA(ctx, cudaGetLastError());
    NPH_CUDA(ctx, cudaMemcpyAsync(shift_scale_out, ctx->d_abea_consts.p, sizeof(double) * 2 * n_jobs, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->abea_loaded = false;
    return NPH_OK;
}

} // extern "C"
