// event_detect.cu — SURVEY.md section 8(f) row N4: scrappie's event detector, the step in front of MoM and ABEA.
//
// Replaces, for a batch of raw reads:
//   detect_events            ref: src/thirdparty/scrappie/event_detection.c:268-319
//   compute_sum_sumsq        ref: :35-49      compute_tstat   ref: :62-118
//   short_long_peak_detector ref: :122-201    create_event(s) ref: :216-266
// as called by SquiggleRead::load_from_raw (src/nanopolish_squiggle_read.cpp:229-235; the trimmed raw_table is
// discarded there, so the whole signal is segmented).
//
// The reference makes five passes over each read and mallocs five arrays (two FP64 prefix sums, two t-statistic
// vectors, a peak list).  The prefix sums are strictly sequential FP64 accumulations, so the result is only
// reproducible by walking each read in order; parallelism is across reads.  One thread streams one read in a single
// pass: the running sums live in registers, a (2*w2+1)-deep ring of the last prefix values per thread lives in shared
// memory (the two t-statistics at position i only need sums at i-w..i+w), the short/long peak detector is a register
// state machine, and each boundary emits its event from the sums captured when the peak was set.  HBM traffic is the
// algorithmic minimum: 4 B per sample in, 24 B per event out.  Every float/double operation mirrors the C source's
// promotions (float products, double quotient, double sqrt) so boundaries, means and stdvs are bit-identical.
#include "nph_internal.cuh"
#include "exact_math.cuh"
#include <cfloat>
#include <algorithm>
#include <vector>
#include <cstdlib>

namespace {

constexpr int kThreads = 128;
constexpr int kMaxW2 = 16;

struct DetParams {
    const float* raw;
    const nph_raw_read* reads;
    const uint32_t* order;
    uint32_t n_reads;
    nph_event* events;
    uint32_t* n_events;
    int* overflow;
    uint32_t w1, w2;
    float t1, t2, peak_height;
    uint32_t ring;         // 2*w2 + 1
};

struct Detector {
    float threshold;
    unsigned long long window_length;
    unsigned long long masked_to;
    long long peak_pos;
    float peak_value;
    bool valid_peak;
    double s_at_peak, q_at_peak;      // prefix sums at peak_pos, captured when the peak is set
};

// t-statistic at position i from prefix values (compute_tstat's loop body, same promotions)
__device__ __forceinline__ float tstat_at(double s_lo, double q_lo, double s_mid, double q_mid, double s_hi, double q_hi, float wf)
{
    const double sum1 = __dsub_rn(s_mid, s_lo);
    const double sumsq1 = __dsub_rn(q_mid, q_lo);
    const float sum2 = (float)__dsub_rn(s_hi, s_mid);
    const float sumsq2 = (float)__dsub_rn(q_hi, q_mid);
    const float mean1 = (float)__ddiv_rn(sum1, (double)wf);
    const float mean2 = __fdiv_rn(sum2, wf);
    double cv = __dsub_rn(__ddiv_rn(sumsq1, (double)wf), (double)__fmul_rn(mean1, mean1));
    cv = __dadd_rn(cv, (double)__fdiv_rn(sumsq2, wf));
    cv = __dsub_rn(cv, (double)__fmul_rn(mean2, mean2));
    float combined_var = fmaxf((float)cv, FLT_MIN);
    const float delta_mean = __fsub_rn(mean2, mean1);
    return (float)__ddiv_rn(fabs((double)delta_mean), __dsqrt_rn((double)__fdiv_rn(combined_var, wf)));
}

__device__ __forceinline__ void emit_event(nph_event* out, uint32_t& count, uint32_t cap, unsigned long long start, unsigned long long end,
                                           double s0, double q0, double s1, double q1)
{
    if (count < cap) {
        nph_event e;
        e.start = start;
        e.length = (float)(end - start);                             // size_t difference, as in create_event
        e.mean = __fdiv_rn((float)__dsub_rn(s1, s0), e.length);
        const float deltasqr = (float)__dsub_rn(q1, q0);
        const float var = __fsub_rn(__fdiv_rn(deltasqr, e.length), __fmul_rn(e.mean, e.mean));
        e.stdv = __fsqrt_rn(fmaxf(var, 0.0f));
        e.reserved = 0;
        out[count] = e;
    }
    ++count;
}

// Fallback for reads whose prefix sums are not provably exact (the guard of ed_fused_kernel): one thread streams one read.
__global__ void __launch_bounds__(kThreads) detect_events_stream_kernel(const DetParams p)
{
    extern __shared__ double s_ring[];                                // [2][ring][kThreads]: S then Q
    const uint32_t slot_idx = blockIdx.x * kThreads + threadIdx.x;
    if (slot_idx >= p.n_reads) return;
    const uint32_t ridx = p.order[slot_idx];
    const nph_raw_read rd = p.reads[ridx];
    const float* __restrict__ raw = p.raw + rd.sample_off;
    const unsigned long long n = rd.n_samples;
    nph_event* out = p.events + rd.event_off;
    const uint32_t R = p.ring;
    double* ringS = s_ring + threadIdx.x;
    double* ringQ = s_ring + (size_t)R * kThreads + threadIdx.x;
#define RS(slot) ringS[(size_t)(slot) * kThreads]
#define RQ(slot) ringQ[(size_t)(slot) * kThreads]

    const uint32_t w1 = p.w1, w2 = p.w2;
    const float wf1 = (float)w1, wf2 = (float)w2;
    const bool on1 = !(n < 2ull * w1 || w1 < 2), on2 = !(n < 2ull * w2 || w2 < 2);
    Detector d0{p.t1, w1, 0ull, -1, FLT_MAX, false, 0.0, 0.0};
    Detector d1{p.t2, w2, 0ull, -1, FLT_MAX, false, 0.0, 0.0};

    double S = 0.0, Q = 0.0;
    unsigned long long consumed = 0;          // prefix index available: S == prefix[consumed]
    RS(0) = 0.0; RQ(0) = 0.0;                 // prefix[0]
    uint32_t slot_w = 0;                      // ring slot of prefix[consumed]
    // ring slots of prefix[i - w2], [i - w1], [i], [i + w1], [i + w2]; negative indices are never read
    int sl_m2 = -(int)w2, sl_m1 = -(int)w1, sl_0 = 0, sl_p1 = (int)w1, sl_p2 = (int)w2;
    sl_p1 %= (int)R; sl_p2 %= (int)R;

    uint32_t count = 0;
    unsigned long long prev_pos = 0;
    double prev_s = 0.0, prev_q = 0.0;

    for (unsigned long long i = 0; i < n; ++i) {
        // make prefix[min(n, i + w2)] available
        const unsigned long long need = (i + w2 < n) ? i + w2 : n;
        while (consumed < need) {
            const float x = raw[consumed];
            S = __dadd_rn(S, (double)x);
            Q = __dadd_rn(Q, (double)__fmul_rn(x, x));
            ++consumed;
            slot_w = (slot_w + 1 == R) ? 0 : slot_w + 1;
            RS(slot_w) = S; RQ(slot_w) = Q;
        }
        const double s_mid = RS(sl_0), q_mid = RQ(sl_0);
        float ts1 = 0.0f, ts2 = 0.0f;
        if (on1 && i >= w1 && i <= n - w1) ts1 = tstat_at(RS(sl_m1), RQ(sl_m1), s_mid, q_mid, RS(sl_p1), RQ(sl_p1), wf1);
        if (on2 && i >= w2 && i <= n - w2) ts2 = tstat_at(RS(sl_m2), RQ(sl_m2), s_mid, q_mid, RS(sl_p2), RQ(sl_p2), wf2);

        // short_long_peak_detector, iteration i: short detector first, then long
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            Detector& d = k == 0 ? d0 : d1;
            if (d.masked_to >= i) continue;
            const float cur = k == 0 ? ts1 : ts2;
            if (d.peak_pos == -1) {
                if (cur < d.peak_value) {
                    d.peak_value = cur;
                } else if (__fsub_rn(cur, d.peak_value) > p.peak_height) {
                    d.peak_value = cur; d.peak_pos = (long long)i; d.s_at_peak = s_mid; d.q_at_peak = q_mid;
                }
            } else {
                if (cur > d.peak_value) { d.peak_value = cur; d.peak_pos = (long long)i; d.s_at_peak = s_mid; d.q_at_peak = q_mid; }
                if (k == 0 && d.peak_value > d.threshold) {
                    d1.masked_to = (unsigned long long)d.peak_pos + d.window_length;
                    d1.peak_pos = -1; d1.peak_value = FLT_MAX; d1.valid_peak = false;
                }
                if (__fsub_rn(d.peak_value, cur) > p.peak_height && d.peak_value > d.threshold) d.valid_peak = true;
                if (d.valid_peak && (i - (unsigned long long)d.peak_pos) > d.window_length / 2) {
                    const unsigned long long pk = (unsigned long long)d.peak_pos;
                    emit_event(out, count, rd.event_cap, prev_pos, pk, prev_s, prev_q, d.s_at_peak, d.q_at_peak);
                    prev_pos = pk; prev_s = d.s_at_peak; prev_q = d.q_at_peak;
                    d.peak_pos = -1; d.peak_value = cur; d.valid_peak = false;
                }
            }
        }
        // advance the five ring cursors
        sl_m2 = (sl_m2 + 1 == (int)R) ? 0 : sl_m2 + 1;
        sl_m1 = (sl_m1 + 1 == (int)R) ? 0 : sl_m1 + 1;
        sl_0 = (sl_0 + 1 == (int)R) ? 0 : sl_0 + 1;
        sl_p1 = (sl_p1 + 1 == (int)R) ? 0 : sl_p1 + 1;
        sl_p2 = (sl_p2 + 1 == (int)R) ? 0 : sl_p2 + 1;
    }
    // last event: previous boundary to the end of the signal (a signal without peaks is one event)
    emit_event(out, count, rd.event_cap, prev_pos, n, prev_s, prev_q, S, Q);
    if (count > rd.event_cap) { *p.overflow = 1; p.n_events[ridx] = 0; }
    else p.n_events[ridx] = count;
#undef RS
#undef RQ
}


// =============================================================================================================
// Fast path.  The reference accumulates FP64 prefix sums of the samples (and of their float squares) sequentially,
// which no parallel algorithm reproduces in general.  But when every partial sum is EXACTLY representable nothing
// is ever rounded, so any summation order gives the same doubles, and every quantity the detector derives from
// the prefix arrays (window sums of the t-statistics, segment sums of the events) equals the exact sum of the
// samples involved.  The guard proves that per read: all samples are integer multiples of 2^L (L = smallest ulp
// exponent present) and |partial sum| <= n * max|x| < 2^(ceil(log2 n) + Emax + 1); if that span fits 53 bits (and
// likewise for the float squares) the read takes the parallel path, otherwise the streaming fallback above.
// Real traces (40-200 pA) pass with ~10 bits to spare.
//   ed_fused_kernel : guard + both t-statistics + the short/long peak detector in ONE pass over the samples
//   ed_events_kernel: thread per event, exact FP64 segment sums -> start / length / mean / stdv
// =============================================================================================================
struct FastParams {
    const float* raw;
    const nph_raw_read* reads;
    const uint32_t* order;       // reads sorted by length (desc)
    uint32_t n_reads;
    uint32_t* peaks;             // per read at event_off, event_cap entries
    uint32_t* n_peaks;           // per read
    uint8_t* exact;              // per read: 1 = fast path
    nph_event* events;
    uint32_t* n_events;
    int* overflow;
    uint32_t* stats;             // [0] repair walks, [1] reads sent to the streaming fallback (diagnostics: $NPH_EVENTS_STATS)
    uint32_t w1, w2;
    float t1, t2, peak_height;
    uint32_t warm;
};

// ---- peak detector -------------------------------------------------------------------------------------------
// short_long_peak_detector (event_detection.c:122-201) is a sequential state machine over the two t-statistic
// vectors, ~36 000 dependent steps per read.  Its state is tiny and re-synchronises quickly (both detectors reset at
// every boundary they emit, about every 9 samples), so a read is walked as 32 (or 64, 128) segments in parallel: each
// lane warms up on the samples before its segment from a fresh state, snapshots the state at its segment start and
// runs the segment recording boundaries; then every lane's snapshot is compared with its left neighbour's final
// state.  If all comparisons agree bit for bit, each lane provably started from the true sequential state (induction
// from lane 0, which starts at sample 0).  A lane whose comparison fails re-walks its segment from the neighbour's
// final state, and the check repeats — exact either way.
struct PeakState {
    uint32_t m0, m1;         // masked_to
    int pp0, pp1;            // peak_pos (-1 = none yet)
    float pv0, pv1;          // peak_value
    int v0, v1;              // valid_peak
};

__device__ __forceinline__ PeakState fresh_state() { return PeakState{0u, 0u, -1, -1, FLT_MAX, FLT_MAX, 0, 0}; }

__device__ __forceinline__ bool same_state(const PeakState& a, const PeakState& b)
{
    return a.m0 == b.m0 && a.m1 == b.m1 && a.pp0 == b.pp0 && a.pp1 == b.pp1 && __float_as_uint(a.pv0) == __float_as_uint(b.pv0) &&
           __float_as_uint(a.pv1) == __float_as_uint(b.pv1) && a.v0 == b.v0 && a.v1 == b.v1;
}

struct PeakConsts { float thr0, thr1, ph; uint32_t w0, half0, half1; };

// one step at position i; returns the boundaries emitted (0, 1 or 2) in e0 (short detector) / e1 (long detector)
__device__ __forceinline__ void peak_step(PeakState& st, const PeakConsts& k, uint32_t i, float ts1, float ts2, int& e0, int& e1)
{
    e0 = -1; e1 = -1;
    {   // short detector
        const bool act = !(st.m0 >= i);
        const float cur = ts1;
        const bool nopeak = st.pp0 < 0;
        const bool lower = cur < st.pv0;
        const bool rise = !lower && (__fsub_rn(cur, st.pv0) > k.ph);
        const bool upd = cur > st.pv0;
        const float npv = nopeak ? ((lower || rise) ? cur : st.pv0) : (upd ? cur : st.pv0);
        const int npp = nopeak ? (rise ? (int)i : -1) : (upd ? (int)i : st.pp0);
        const bool in2 = act && !nopeak;
        const bool over = npv > k.thr0;
        const bool dominate = in2 && over;                  // the short detector will fire: silence the long one
        const bool nvalid = st.v0 || (in2 && over && (__fsub_rn(npv, cur) > k.ph));
        const bool emit = in2 && nvalid && ((i - (uint32_t)npp) > k.half0);
        if (emit) e0 = npp;
        if (dominate) { st.m1 = (uint32_t)npp + k.w0; st.pp1 = -1; st.pv1 = FLT_MAX; st.v1 = 0; }
        if (act) { st.pv0 = emit ? cur : npv; st.pp0 = emit ? -1 : npp; st.v0 = emit ? 0 : (nvalid ? 1 : 0); }
    }
    {   // long detector
        const bool act = !(st.m1 >= i);
        const float cur = ts2;
        const bool nopeak = st.pp1 < 0;
        const bool lower = cur < st.pv1;
        const bool rise = !lower && (__fsub_rn(cur, st.pv1) > k.ph);
        const bool upd = cur > st.pv1;
        const float npv = nopeak ? ((lower || rise) ? cur : st.pv1) : (upd ? cur : st.pv1);
        const int npp = nopeak ? (rise ? (int)i : -1) : (upd ? (int)i : st.pp1);
        const bool in2 = act && !nopeak;
        const bool nvalid = st.v1 || (in2 && (npv > k.thr1) && (__fsub_rn(npv, cur) > k.ph));
        const bool emit = in2 && nvalid && ((i - (uint32_t)npp) > k.half1);
        if (emit) e1 = npp;
        if (act) { st.pv1 = emit ? cur : npv; st.pp1 = emit ? -1 : npp; st.v1 = emit ? 0 : (nvalid ? 1 : 0); }
    }
}

constexpr int kPeakWarps = 4;
#ifndef NPH_ED_CTAS
#define NPH_ED_CTAS 5          // resident CTAs per SM the fused kernel is compiled for (registers <= 65536 / (128 * NPH_ED_CTAS)); six fit the
                              // shared memory but cost spills: 4.46 ms against 4.37 ms for 4 096 reads x 36 000 samples
#endif

// =============================================================================================================
// ed_fused_kernel: guard + t-statistics + peaks in ONE pass over the samples; only the boundaries are written.
// The warp(s) that own a read walk it as 32 (64, 128) segments; the 32x32 tile of t-statistics the lanes consume is
// COMPUTED by the warp from the raw samples (row rr = the next 32 positions of lane rr's range, one lane per position:
// the row and its 2*w2 halo are loaded coalesced one row ahead, widened ONCE and staged in shared memory), and the
// exactness guard rides along on the samples the warp touches anyway.
//   * what bounds it is not HBM but the float<->double conversion unit: compute_tstat needs >= 10 conversions per
//     window and position however it is arranged (float sums, float means, float variance, double quotient), and a
//     conversion costs 8.5 clk per warp instruction (scripts/ubench_cvt.cu, profiles/r02_ubench_cvt.txt)
//   * divisions by the window length are Markstein divisions by a cached reciprocal (exact_math.cuh); the final
//     |delta| / sqrt(v) is D * rsqrt(v) in FP64 (<= 2 ulp) rounded to float, accepted only when that FP64 value is
//     more than 2^10 ulps away from a float rounding boundary (so the correctly rounded chain dsqrt -> ddiv -> float
//     provably rounds to the same float); otherwise that position takes the reference's operations one by one
//   * boundaries are recorded during the walk into a per-lane slice of the read's peak array and compacted afterwards
//   * a segment whose warm-up did not reach the true state is re-walked from its left neighbour's final state until
//     the chain verifies (induction from lane 0)
// A read that fails the guard (or overflows a lane's slice) is flagged for the streaming fallback.
// =============================================================================================================
struct TsConsts {
    uint32_t w1, w2;
    float w1f, w2f, r1f, r2f;        // window lengths as float, RN(1/w) in float
    double w1d, w2d, r1d, r2d;       // ... and in double
};

struct GuardAcc { uint32_t vmin, vmax, qmin, qmax; };     // min / max of |x| and |x*x| bit patterns over nonzero values

__device__ __forceinline__ double ddiv_by_cached_rcp(double a, double b, double y)
{
    const double q0 = __dmul_rn(a, y);
    const double r0 = __fma_rn(-q0, b, a);
    const double q1 = __fma_rn(r0, y, q0);
    const double r1 = __fma_rn(-q1, b, a);
    return __fma_rn(r1, y, q1);
}

// compute_tstat's loop body (event_detection.c:91-112) for one window, from the exact left/right window sums.
// Branch-free fast form: returns the candidate and whether it is proven (see the header); the caller runs
// tstat_windows_exact for the rare unproven position.  Straight-line so the two windows of a position interleave.
struct TsCand { float t; float combined_var, delta_mean; bool proven; };

__device__ __forceinline__ TsCand tstat_windows(double sl, double ql, double sr, double qr, float wf, float rf, double wd, double rd)
{
    const float sum2 = (float)sr, sumsq2 = (float)qr;
    const float mean1 = (float)ddiv_by_cached_rcp(sl, wd, rd);
    const float mean2 = div_by_cached_rcp(sum2, wf, rf);
    double cv = __dsub_rn(ddiv_by_cached_rcp(ql, wd, rd), (double)__fmul_rn(mean1, mean1));
    cv = __dadd_rn(cv, (double)div_by_cached_rcp(sumsq2, wf, rf));
    cv = __dsub_rn(cv, (double)__fmul_rn(mean2, mean2));
    TsCand c;
    c.combined_var = fmaxf((float)cv, FLT_MIN);
    c.delta_mean = __fsub_rn(mean2, mean1);
    const bool in_range = c.combined_var >= 8.6736174e-19f /*2^-60*/ && c.combined_var <= 1.1529215e18f /*2^60*/;
    const float v = div_by_cached_rcp(c.combined_var, wf, rf);
    const double y = __dmul_rn(fabs((double)c.delta_mean), rsqrt((double)v));
    const unsigned long long bits = (unsigned long long)__double_as_longlong(y);
    const uint32_t lo = (uint32_t)bits & 0x1FFFFFFFu, ex = (uint32_t)(bits >> 52);
    // a zero difference of means is exactly 0 (v > 0); otherwise y must be a normal float well away from a rounding boundary
    c.proven = in_range && (c.delta_mean == 0.0f || ((lo - 0x10000000u + 1024u) >= 2048u && (ex - 923u) < 200u));
    c.t = (float)y;
    return c;
}

__device__ __noinline__ float tstat_windows_exact(float combined_var, float delta_mean, float wf)
{
    return (float)__ddiv_rn(fabs((double)delta_mean), __dsqrt_rn((double)__fdiv_rn(combined_var, wf)));
}

// A row of the tile: the 32 positions [p0 + w2, p0 + w2 + 32) of one lane's range.  The warp first stages the row and its
// halo (32 + 2*w2 samples from p0; zeros outside the read) in shared memory as doubles — x and the float product x*x,
// each sample converted ONCE (the float->double conversion is the scarce resource here: 8.5 clk per warp instruction,
// profiles/r02_ubench_cvt.txt) — and feeds the exactness guard with the samples it touches.
constexpr int kFusedMaxW2 = 14;                   // scrappie: 6 (DNA), 14 (RNA); wider windows take the streaming kernel
constexpr int kRowBuf = 32 + 2 * kFusedMaxW2;

struct RowRegs { float v0, v1; };          // the two samples of a row this lane stages: slots lane and lane + 32

// issue the global loads of a row (p0 = first staged position; it may have wrapped below 0: such positions fail p < n)
__device__ __forceinline__ RowRegs load_row(const float* __restrict__ x, uint32_t n, uint32_t p0, uint32_t w2, int lane)
{
    RowRegs r{0.0f, 0.0f};
    const uint32_t pa = p0 + (uint32_t)lane, pb = pa + 32u;
    if (pa < n) r.v0 = x[pa];
    if ((uint32_t)lane < 2u * w2 && pb < n) r.v1 = x[pb];
    return r;
}

__device__ __forceinline__ void stage_row(const RowRegs& r, uint32_t w2, double* __restrict__ sdx, double* __restrict__ sdq, GuardAcc& ga, int lane)
{
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const uint32_t s = (uint32_t)lane + 32u * h;
        if (h == 1 && s >= 32u + 2u * w2) break;
        const float v = h ? r.v1 : r.v0;
        const float q = __fmul_rn(v, v);
        const uint32_t vb = __float_as_uint(v) & 0x7fffffffu, qb = __float_as_uint(q);
        ga.vmax = max(ga.vmax, vb); ga.qmax = max(ga.qmax, qb);
        ga.vmin = min(ga.vmin, vb ? vb : 0xffffffffu); ga.qmin = min(ga.qmin, qb ? qb : 0xffffffffu);
        sdx[s] = (double)v; sdq[s] = (double)q;
    }
}

// both t-statistics at position pos (staged slot lane + w2) of a read; 0 where compute_tstat leaves its zeros
template <int W1, int W2>
__device__ __forceinline__ void tstat_pair(const double* __restrict__ sdx, const double* __restrict__ sdq, uint32_t n, uint32_t pos,
                                           const TsConsts& tc, int lane, float& a, float& b)
{
    const uint32_t w1 = W1 ? (uint32_t)W1 : tc.w1, w2 = W2 ? (uint32_t)W2 : tc.w2;
    // compute_tstat leaves zeros when the signal is shorter than two windows or the window shorter than 2 (:73-:76), and at the ends
    const bool v1 = w1 >= 2 && n >= 2 * w1 && pos >= w1 && pos <= n - w1, v2 = w2 >= 2 && n >= 2 * w2 && pos >= w2 && pos <= n - w2;
    a = 0.0f; b = 0.0f;
    if (!(v1 || v2)) return;
    const double* cx = sdx + lane + w2;                                  // cx[0] = x[pos]; cx[-1-j] left window, cx[j] right window
    const double* cq = sdq + lane + w2;
    // both windows unconditionally (the staged row has the halo; a window that does not apply is discarded below)
    double sl = 0.0, ql = 0.0, sr = 0.0, qr = 0.0;
#pragma unroll
    for (int j = 0; j < (int)w1; ++j) {
        sl = __dadd_rn(sl, cx[-1 - j]); ql = __dadd_rn(ql, cq[-1 - j]);
        sr = __dadd_rn(sr, cx[j]); qr = __dadd_rn(qr, cq[j]);
    }
    const TsCand ca = tstat_windows(sl, ql, sr, qr, tc.w1f, tc.r1f, tc.w1d, tc.r1d);
#pragma unroll
    for (int j = (int)w1; j < (int)w2; ++j) {
        sl = __dadd_rn(sl, cx[-1 - j]); ql = __dadd_rn(ql, cq[-1 - j]);
        sr = __dadd_rn(sr, cx[j]); qr = __dadd_rn(qr, cq[j]);
    }
    const TsCand cb = tstat_windows(sl, ql, sr, qr, tc.w2f, tc.r2f, tc.w2d, tc.r2d);
    a = ca.t; b = cb.t;
    if (v1 && !ca.proven) a = tstat_windows_exact(ca.combined_var, ca.delta_mean, tc.w1f);
    if (v2 && !cb.proven) b = tstat_windows_exact(cb.combined_var, cb.delta_mean, tc.w2f);
    if (!v1) a = 0.0f;
    if (!v2) b = 0.0f;
}

struct FusedSmem {                       // per warp, 9 216 bytes: six CTAs of four warps fit an SM
    float a[32][32], b[32][32];          // the tile of t-statistics: row = lane that will consume it, column XOR row (bank-conflict free
                                         // for the row-wise producer and the column-wise consumer without padding); after the walks
                                         // the first 32 words of `a` carry the lanes' boundary counts to the read's first warp
    double dx[kRowBuf];                  // one staged row: the samples, widened
    PeakState last;                      // final state of the warp's lane 31 (for the next warp of the same read)
    double dq[kRowBuf];                  // ... and their float squares, widened
    GuardAcc guard;                      // the warp's guard extrema
    uint32_t flag, over, pad[2];         // chain verified / some slice overflowed
};
static_assert(sizeof(FusedSmem) == 9216, "FusedSmem layout");

// One cooperative walk: lane l walks [from_l, from_l + len_l), the first wlen_l steps being warm-up (state only); at
// step wlen_l the state is snapshotted and from there boundaries are counted and recorded into region[0..R).
template <int W1, int W2>
__device__ __forceinline__ uint32_t fused_walk(PeakState& st, PeakState& snap, const TsConsts& tc, const PeakConsts& k,
                                               const float* __restrict__ x, uint32_t n, uint32_t from, uint32_t len, uint32_t wlen,
                                               uint32_t* __restrict__ region, uint32_t R, GuardAcc& ga, FusedSmem& sm, int lane)
{
    const uint32_t w2 = W2 ? (uint32_t)W2 : tc.w2;
    uint32_t maxlen = len;
    for (int o = 16; o; o >>= 1) maxlen = max(maxlen, __shfl_xor_sync(0xffffffffu, maxlen, o));
    uint32_t cnt = 0;
    for (uint32_t c = 0; c < maxlen; c += 32) {
        // rows are software-pipelined: the samples of the next row are in flight while this row's statistics are computed.
        // The loop starts one row early (rr = -1 only loads) so that `cur` is never the direct target of a load: a load into it
        // on the entry path would make ptxas encode a scoreboard wait at its first use that, inside the loop, also waits for
        // the prefetch just issued (measured: 24 % of all stall samples sat on that one instruction).
        if (c + 32 < len) asm volatile("prefetch.global.L2 [%0];" :: "l"(x + from + c + 32 + w2));     // my next tile's line
        uint32_t fr = 0, ln = 0;
        RowRegs cur{0.0f, 0.0f};
#pragma unroll 1
        for (int rr = -1; rr < 32; ++rr) {
            const uint32_t fr_n = __shfl_sync(0xffffffffu, from, (rr + 1) & 31), ln_n = __shfl_sync(0xffffffffu, len, (rr + 1) & 31);
            RowRegs nxt{0.0f, 0.0f};
            if (rr < 31 && c < ln_n) nxt = load_row(x, n, fr_n + c - w2, w2, lane);
            if (rr >= 0 && c < ln) {                                     // warp-uniform
                stage_row(cur, w2, sm.dx, sm.dq, ga, lane);
                __syncwarp();
                float a = 0.0f, b = 0.0f;
                if (c + lane < ln) tstat_pair<W1, W2>(sm.dx, sm.dq, n, fr + c + lane, tc, lane, a, b);
                sm.a[rr][lane ^ rr] = a; sm.b[rr][lane ^ rr] = b;
                __syncwarp();
            }
            cur = nxt; fr = fr_n; ln = ln_n;
        }
        if (c == wlen) snap = st;
        const bool rec = c >= wlen;
        const uint32_t steps = len > c ? min(32u, len - c) : 0u;
        for (uint32_t t = 0; t < steps; ++t) {
            int e0, e1;
            peak_step(st, k, from + c + t, sm.a[lane][t ^ lane], sm.b[lane][t ^ lane], e0, e1);
            if (rec && e0 >= 0) { if (cnt < R) region[cnt] = (uint32_t)e0; ++cnt; }
            if (rec && e1 >= 0) { if (cnt < R) region[cnt] = (uint32_t)e1; ++cnt; }
        }
        __syncwarp();
    }
    return cnt;
}

constexpr uint32_t kFusedWarm = 128;      // multiple of 32; $NPH_EVENTS_WARMUP overrides (rounded up to 32)

__device__ __forceinline__ void read_barrier(int id, int threads) { asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(threads) : "memory"); }

// WPR warps walk one read as 32*WPR segments (a CTA of kPeakWarps warps holds kPeakWarps / WPR reads): small batches
// and the tail of a large one get WPR times the parallelism for warm / segment more work.
template <int W1, int W2, int WPR>
__global__ void __launch_bounds__(kPeakWarps * 32, NPH_ED_CTAS) ed_fused_kernel(const FastParams p, const TsConsts tc)
{
    constexpr int LANES = 32 * WPR;
    __shared__ FusedSmem s_mem[kPeakWarps];
    const int wib = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int rslot = wib / WPR, part = wib % WPR, w0 = rslot * WPR;          // this warp's read within the CTA, its part of it
    const uint32_t slot = blockIdx.x * (kPeakWarps / WPR) + rslot;
    if (slot >= p.n_reads) return;
    const int bar_id = 1 + rslot;                                          // named barrier of the read's WPR warps
    const uint32_t ridx = p.order[slot];
    const nph_raw_read rd = p.reads[ridx];
    const uint32_t n = rd.n_samples;
    const float* __restrict__ x = p.raw + rd.sample_off;
    uint32_t* peaks = p.peaks + rd.event_off;
    const uint32_t cap_peaks = rd.event_cap ? rd.event_cap - 1 : 0;       // events = boundaries + 1
    const uint32_t R = cap_peaks / LANES;                                 // a lane's slice of the peak array
    const uint32_t gl = (uint32_t)part * 32u + (uint32_t)lane;             // lane within the read
    uint32_t* region = peaks + (size_t)gl * R;
    const PeakConsts k{p.t1, p.t2, p.peak_height, p.w1, p.w1 / 2, p.w2 / 2};

    const uint32_t seg = ((n + LANES - 1) / LANES + 31) / 32 * 32;         // segment length, multiple of 32
    const uint32_t b0 = (unsigned long long)gl * seg < n ? gl * seg : n, b1 = min(n, b0 + seg);
    const bool mine = b0 < n;                                              // lanes past the end of the read own nothing
    const uint32_t a0 = b0 > p.warm ? b0 - p.warm : 0;                     // b0, warm multiples of 32: so is the warm-up length
    GuardAcc ga{0xffffffffu, 0u, 0xffffffffu, 0u};
    PeakState st = fresh_state(), snap = st;
    uint32_t cnt = fused_walk<W1, W2>(st, snap, tc, k, x, n, mine ? a0 : 0u, mine ? b1 - a0 : 0u, mine ? b0 - a0 : 0u, region, R, ga,
                                      s_mem[wib], lane);
    // ---- the guard (the exactness test of the header, plus the operand range the cached-reciprocal divisions are proven for) ----
    for (int o = 16; o; o >>= 1) {
        ga.vmin = min(ga.vmin, __shfl_xor_sync(0xffffffffu, ga.vmin, o)); ga.vmax = max(ga.vmax, __shfl_xor_sync(0xffffffffu, ga.vmax, o));
        ga.qmin = min(ga.qmin, __shfl_xor_sync(0xffffffffu, ga.qmin, o)); ga.qmax = max(ga.qmax, __shfl_xor_sync(0xffffffffu, ga.qmax, o));
    }
    if (WPR > 1) {
        if (lane == 0) s_mem[wib].guard = ga;
        read_barrier(bar_id, LANES);
        for (int w = 0; w < WPR; ++w) {
            const GuardAcc g = s_mem[w0 + w].guard;
            ga.vmin = min(ga.vmin, g.vmin); ga.vmax = max(ga.vmax, g.vmax); ga.qmin = min(ga.qmin, g.qmin); ga.qmax = max(ga.qmax, g.qmax);
        }
    }
    bool exact;
    {
        int lg = 0;
        while ((1ull << lg) < (unsigned long long)n + 1) ++lg;             // ceil(log2(n + 1))
        // biased exponents; ulp exponent = e - 150, top = e - 127: span = lg + (emax - 127) + 1 - (emin - 150)
        const int evx = (int)(ga.vmax >> 23), evn = (int)(ga.vmin >> 23), eqx = (int)(ga.qmax >> 23), eqn = (int)(ga.qmin >> 23);
        const bool okx = ga.vmax == 0u || (evn >= 97 && evx <= 157 && lg + evx + 24 - evn <= 53);       // |x| in [2^-30, 2^31)
        const bool okq = ga.qmax == 0u || (eqn >= 66 && eqx <= 188 && lg + eqx + 24 - eqn <= 53);       // x*x in [2^-61, 2^62)
        exact = okx && okq;                                                // the same in every warp of the read
    }
    // ---- verification and repair: my snapshot must equal the final state of the lane to my left ----
    uint32_t repairs = 0;
    for (int round = 0; exact && round < LANES; ++round) {
        if (WPR > 1) {
            if (lane == 31) s_mem[wib].last = st;
            read_barrier(bar_id, LANES);
        }
        PeakState left;
        left.m0 = __shfl_up_sync(0xffffffffu, st.m0, 1); left.m1 = __shfl_up_sync(0xffffffffu, st.m1, 1);
        left.pp0 = __shfl_up_sync(0xffffffffu, st.pp0, 1); left.pp1 = __shfl_up_sync(0xffffffffu, st.pp1, 1);
        left.pv0 = __shfl_up_sync(0xffffffffu, st.pv0, 1); left.pv1 = __shfl_up_sync(0xffffffffu, st.pv1, 1);
        left.v0 = __shfl_up_sync(0xffffffffu, st.v0, 1); left.v1 = __shfl_up_sync(0xffffffffu, st.v1, 1);
        if (WPR > 1 && lane == 0 && part > 0) left = s_mem[wib - 1].last;
        const bool ok = !mine || gl == 0 || same_state(snap, left);
        bool all_ok = __all_sync(0xffffffffu, ok);
        if (WPR > 1) {
            if (lane == 0) s_mem[wib].flag = all_ok ? 1u : 0u;
            read_barrier(bar_id, LANES);
            all_ok = true;
            for (int w = 0; w < WPR; ++w) all_ok = all_ok && s_mem[w0 + w].flag != 0u;
        }
        if (all_ok) break;
        // re-walk the segments that started from a wrong state, now from the neighbour's final state (lanes 0..round are right)
        PeakState s2 = ok ? st : left, sn2 = s2;
        GuardAcc g2{0xffffffffu, 0u, 0xffffffffu, 0u};
        const uint32_t c2 = fused_walk<W1, W2>(s2, sn2, tc, k, x, n, ok ? 0u : b0, ok ? 0u : b1 - b0, 0u, region, R, g2, s_mem[wib], lane);
        if (!ok) { st = s2; snap = left; cnt = c2; }
        ++repairs;
    }
    // ---- counts of all the read's lanes, then its first warp compacts the slices ----
    const bool over = __any_sync(0xffffffffu, cnt > R);                    // a lane's slice was too small: streaming fallback
    __syncwarp();                                                          // the tile is free now
    reinterpret_cast<uint32_t*>(&s_mem[wib].a[0][0])[lane] = cnt;
    if (lane == 0) s_mem[wib].over = over ? 1u : 0u;
    if (WPR > 1) read_barrier(bar_id, LANES); else __syncwarp();
    if (part != 0) return;
    for (int w = 0; w < WPR; ++w) if (s_mem[w0 + w].over) exact = false;
    auto cnt_of = [&](int s) { return reinterpret_cast<const uint32_t*>(&s_mem[w0 + (s >> 5)].a[0][0])[s & 31]; };
    uint32_t total = 0;
    for (int s = 0; s < LANES; ++s) total += cnt_of(s);
    if (exact && total <= cap_peaks) {
        // slice 0 is in place; destinations never pass their sources, slices and chunks go left to right
        uint32_t ds = cnt_of(0);
        for (int s = 1; s < LANES; ++s) {
            const uint32_t cs = cnt_of(s);
            const uint32_t* src = peaks + (size_t)s * R;
            if (ds != (uint32_t)s * R) {
                for (uint32_t q = 0; q < cs; q += 32) {
                    uint32_t v = 0;
                    if (q + lane < cs) v = src[q + lane];
                    __syncwarp();
                    if (q + lane < cs) peaks[ds + q + lane] = v;
                    __syncwarp();
                }
            }
            ds += cs;
        }
    }
    if (lane == 0) {
        p.exact[ridx] = exact ? 1 : 0;
        if (repairs) atomicAdd(&p.stats[0], repairs);
        if (!exact) atomicAdd(&p.stats[1], 1u);
        if (exact) {
            if (total > cap_peaks) { *p.overflow = 1; p.n_peaks[ridx] = 0; p.n_events[ridx] = 0; }
            else { p.n_peaks[ridx] = total; p.n_events[ridx] = total + 1; }
        }
    }
}

template <int WPR>
static void launch_fused(const FastParams& f, const TsConsts& tc, size_t n_reads, cudaStream_t stream)
{
    const unsigned blocks = (unsigned)((n_reads + kPeakWarps / WPR - 1) / (kPeakWarps / WPR));
    void (*kern)(const FastParams, const TsConsts) = ed_fused_kernel<0, 0, WPR>;
    if (f.w1 == 3 && f.w2 == 6) kern = ed_fused_kernel<3, 6, WPR>;
    else if (f.w1 == 7 && f.w2 == 14) kern = ed_fused_kernel<7, 14, WPR>;
    // five CTAs per SM need the large shared-memory carve-out (static shared memory alone does not ask for it)
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    kern<<<blocks, kPeakWarps * 32, 0, stream>>>(f, tc);
}

// block per read, thread per event
__global__ void __launch_bounds__(256) ed_events_kernel(const FastParams p)
{
    for (uint32_t r = blockIdx.x; r < p.n_reads; r += gridDim.x) {
        if (!p.exact[r]) continue;
        const nph_raw_read rd = p.reads[r];
        const uint32_t ne = p.n_events[r];
        if (ne == 0) continue;
        const float* __restrict__ x = p.raw + rd.sample_off;
        const uint32_t* peaks = p.peaks + rd.event_off;
        nph_event* out = p.events + rd.event_off;
        const unsigned long long n = rd.n_samples;
        for (uint32_t ev = threadIdx.x; ev < ne; ev += blockDim.x) {
            const unsigned long long start = ev == 0 ? 0ull : peaks[ev - 1];
            const unsigned long long end = ev == ne - 1 ? n : peaks[ev];
            // exact segment sums; boundaries emitted out of order give a negative sum, like sums[end] - sums[start]
            const unsigned long long lo = start < end ? start : end, hi = start < end ? end : start;
            double s = 0.0, q = 0.0;
            for (unsigned long long j = lo; j < hi; ++j) { const float v = x[j]; s = __dadd_rn(s, (double)v); q = __dadd_rn(q, (double)__fmul_rn(v, v)); }
            if (end < start) { s = -s; q = -q; }
            nph_event e;
            e.start = start;
            e.length = (float)(end - start);
            e.mean = __fdiv_rn((float)s, e.length);
            const float var = __fsub_rn(__fdiv_rn((float)q, e.length), __fmul_rn(e.mean, e.mean));
            e.stdv = __fsqrt_rn(fmaxf(var, 0.0f));
            e.reserved = 0;
            out[ev] = e;
        }
    }
}

} // namespace

EdScratch nph_ed_layout(NphCarve& a, size_t n_reads, size_t events_total)
{
    EdScratch s;
    s.reads = a.take<nph_raw_read>(n_reads);
    s.order = a.take<uint32_t>(n_reads);
    s.events = a.take<nph_event>(events_total);
    s.n_events = a.take<uint32_t>(n_reads);
    s.ctl = a.take<EdControl>(1);
    s.peaks = a.take<uint32_t>(events_total);
    s.n_peaks = a.take<uint32_t>(n_reads);
    s.exact = a.take<uint8_t>(n_reads);
    return s;
}

// Event detection over reads whose samples are already on the device, in the scratch of nph_ed_layout.  Returns the
// counts on the host too.  Synchronises the stream (twice: the list of reads that need the sequential fallback, then the
// counts).
int nph_detect_events_device(nph_ctx* ctx, const float* d_raw, size_t n_samples_total, const nph_raw_read* reads, size_t n_reads,
                             const nph_event_params* params, const EdScratch& s, size_t events_total,
                             std::vector<uint32_t>& h_n_events, int* launches_out)
{
    if (params->window_length2 > kMaxW2 || params->window_length1 > params->window_length2 || params->window_length1 == 0) return NPH_ERR_UNSUPPORTED;
    std::vector<uint32_t> n_samples(n_reads);
    for (size_t i = 0; i < n_reads; ++i) {
        const nph_raw_read& r = reads[i];
        if (r.n_samples == 0 || r.sample_off + r.n_samples > n_samples_total || r.event_off + r.event_cap > events_total || r.event_cap == 0)
            return NPH_ERR_INVALID;
        if (r.n_samples > 0xFFFFFF00u) return NPH_ERR_UNSUPPORTED;      // position arithmetic is 32-bit with a 2*w2 halo
        n_samples[i] = r.n_samples;
    }
    // threads of a warp walk reads of similar length: longest first
    const std::vector<uint32_t> order = longest_first(n_samples);

    DetParams p{};
    p.events = s.events; p.n_events = s.n_events; p.overflow = &s.ctl->overflow;
    p.raw = d_raw; p.reads = s.reads; p.order = s.order; p.n_reads = (uint32_t)n_reads;
    p.w1 = params->window_length1; p.w2 = params->window_length2;
    p.t1 = params->threshold1; p.t2 = params->threshold2; p.peak_height = params->peak_height;
    p.ring = 2 * p.w2 + 1;
    NPH_CUDA(ctx, cudaMemcpyAsync(s.reads, reads, sizeof(nph_raw_read) * n_reads, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(s.order, order.data(), sizeof(uint32_t) * n_reads, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemsetAsync(s.ctl, 0, nph_align256(sizeof(EdControl)), ctx->stream));     // the slice's whole extent
    // fast path first (fused guard + t-statistics + peaks, then events); reads that fail the exactness guard take the stream kernel
    FastParams f{};
    f.raw = d_raw; f.reads = s.reads; f.order = s.order; f.n_reads = (uint32_t)n_reads;
    f.peaks = s.peaks; f.n_peaks = s.n_peaks; f.exact = s.exact;
    f.events = p.events; f.n_events = p.n_events; f.overflow = p.overflow;
    f.stats = s.ctl->stats;
    f.w1 = p.w1; f.w2 = p.w2; f.t1 = p.t1; f.t2 = p.t2; f.peak_height = p.peak_height;
    int launches = 0;
    if (p.w2 > (uint32_t)kFusedMaxW2) {
        NPH_CUDA(ctx, cudaMemsetAsync(s.exact, 0, n_reads, ctx->stream));   // windows wider than the staged row: every read streams
    } else {
        // one pass over the samples: guard + t-statistics + peaks (ed_fused_kernel)
        TsConsts tc{};
        tc.w1 = p.w1; tc.w2 = p.w2;
        tc.w1f = (float)p.w1; tc.w2f = (float)p.w2; tc.r1f = 1.0f / tc.w1f; tc.r2f = 1.0f / tc.w2f;
        tc.w1d = (double)p.w1; tc.w2d = (double)p.w2; tc.r1d = 1.0 / tc.w1d; tc.r2d = 1.0 / tc.w2d;
        f.warm = getenv("NPH_EVENTS_WARMUP") ? ((uint32_t)atoi(getenv("NPH_EVENTS_WARMUP")) + 31u) / 32u * 32u : kFusedWarm;
        // warps per read: one when the batch alone fills the machine (20 resident warps per SM; measured 4 096 reads: 4.3 / 4.8 / 5.0 ms
        // with 1 / 2 / 4), more for small batches (512 reads: 1.46 / 1.02 / 0.86 ms) as long as a segment stays >= 2 warm-ups long
        int wpr = 1;
        const size_t want = (size_t)ctx->sm_count * 20;
        while (wpr < 4 && n_reads * wpr < want && n_samples[order[0]] / (64u * wpr) >= 2 * f.warm) wpr *= 2;
        if (getenv("NPH_EVENTS_WPR")) wpr = atoi(getenv("NPH_EVENTS_WPR"));
        if (wpr >= 4) launch_fused<4>(f, tc, n_reads, ctx->stream);
        else if (wpr == 2) launch_fused<2>(f, tc, n_reads, ctx->stream);
        else launch_fused<1>(f, tc, n_reads, ctx->stream);
        ++launches;
        NPH_CUDA(ctx, cudaGetLastError());
    }
    ed_events_kernel<<<(unsigned)std::min<size_t>(n_reads, (size_t)ctx->sm_count * 16), 256, 0, ctx->stream>>>(f); ++launches;
    NPH_CUDA(ctx, cudaGetLastError());
    // fallback list
    std::vector<uint8_t> exact(n_reads);
    NPH_CUDA(ctx, cudaMemcpyAsync(exact.data(), s.exact, n_reads, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    std::vector<uint32_t> slow;
    for (size_t t = 0; t < n_reads; ++t) if (!exact[order[t]] || getenv("NPH_EVENTS_FORCE_STREAM")) slow.push_back(order[t]);
    if (!slow.empty()) {
        NPH_CUDA(ctx, cudaMemcpyAsync(s.order, slow.data(), sizeof(uint32_t) * slow.size(), cudaMemcpyHostToDevice, ctx->stream));
        p.n_reads = (uint32_t)slow.size();
        const size_t smem = sizeof(double) * 2 * p.ring * kThreads;
        NPH_CUDA(ctx, cudaFuncSetAttribute(detect_events_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        detect_events_stream_kernel<<<(unsigned)((slow.size() + kThreads - 1) / kThreads), kThreads, smem, ctx->stream>>>(p); ++launches;
        NPH_CUDA(ctx, cudaGetLastError());
    }
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    int overflow = 0;
    h_n_events.resize(n_reads);
    NPH_CUDA(ctx, cudaMemcpyAsync(h_n_events.data(), p.n_events, sizeof(uint32_t) * n_reads, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(&overflow, p.overflow, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (getenv("NPH_EVENTS_STATS")) {
        uint32_t st[2] = {0, 0};
        cudaMemcpy(st, f.stats, sizeof(st), cudaMemcpyDeviceToHost);
        fprintf(stderr, "[nph events] reads %zu  repair walks %u  streaming fallback %zu (guard/slice %u)\n", n_reads, st[0], slow.size(), st[1]);
    }
    if (launches_out) *launches_out = launches;
    return overflow ? NPH_ERR_UNSUPPORTED : NPH_OK;
}

extern "C" int nph_detect_events_batch(nph_ctx* ctx, const float* raw, size_t n_samples_total, const nph_raw_read* reads, size_t n_reads,
                                       const nph_event_params* params, nph_event* events_out, size_t events_total, uint32_t* n_events_out)
{
    if (!ctx || !params) return NPH_ERR_INVALID;
    if (n_reads == 0) return NPH_OK;
    if (!raw || !reads || !events_out || !n_events_out) return NPH_ERR_INVALID;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    float* d_raw = nullptr;
    EdScratch es;
    auto layout = [&](NphCarve& a) { d_raw = a.take<float>(n_samples_total); es = nph_ed_layout(a, n_reads, events_total); };
    NPH_TRY(nph_borrow_arena(ctx, layout));
    NPH_CUDA(ctx, cudaMemcpyAsync(d_raw, raw, sizeof(float) * n_samples_total, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    std::vector<uint32_t> counts;
    int launches = 0;
    const int rc = nph_detect_events_device(ctx, d_raw, n_samples_total, reads, n_reads, params, es, events_total, counts, &launches);
    if (rc != NPH_OK && rc != NPH_ERR_UNSUPPORTED) return rc;
    if (!launches) return rc;                       // parameters refused before anything ran
    ctx->last_launches = launches;
    ctx->timing_valid = true;
    // only the events that exist cross PCIe: a read's room (n_samples / 2 in practice) is ~4.5 x what it fills, and the room of a
    // 4 096-read batch is 1.8 GB.  One copy per read when that saves more than the copies' launch cost, else the whole arena.
    size_t used = 0;
    for (size_t i = 0; i < n_reads; ++i) used += counts[i];
    if (used * 2 < events_total && n_reads <= 65536) {
        for (size_t i = 0; i < n_reads; ++i)
            if (counts[i])
                NPH_CUDA(ctx, cudaMemcpyAsync(events_out + reads[i].event_off, es.events + reads[i].event_off, sizeof(nph_event) * counts[i],
                                              cudaMemcpyDeviceToHost, ctx->stream));
    } else {
        NPH_CUDA(ctx, cudaMemcpyAsync(events_out, es.events, sizeof(nph_event) * events_total, cudaMemcpyDeviceToHost, ctx->stream));
    }
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    std::copy(counts.begin(), counts.end(), n_events_out);
    return rc;
}
