/* oracle/np_polya.c — TEST INFRASTRUCTURE ONLY: a plain-C restatement of `nanopolish polya`'s per-read computation
 * (src/nanopolish_polya_estimator.cpp:204-722), pinned to the compiled reference by tests/test_polya.py and used as the
 * checker of large device batches.  Same job / result layout as include/nph.h (nph_polya_job, nph_polya_result); the
 * emissions call the C library's expf / logf, as the reference does.  Build: gcc -std=c99 -ffp-contract=off (no FMA
 * contraction, so every float operation rounds where the reference's does).
 *
 *   npo_polya(samples, durations, map, jobs, n_jobs, results, threads)
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct { int32_t start, stop; } npo_event_range;
typedef struct {
    uint64_t sample_off, event_off, map_off;
    uint32_t n_samples, n_events, n_kmers, reserved;
    double sample_rate, shift, scale, var;
} npo_polya_job;
typedef struct {
    uint64_t start, leader, adapter, polya, cliffs;
    double read_rate, polya_length;
    float end_score;
    uint32_t qc;
} npo_polya_result;

enum { S_ = 0, L_ = 1, A_ = 2, P_ = 3, C_ = 4, T_ = 5 };
typedef struct { float mean, stdv, log_stdv; } gauss;

static gauss scaled(float mean, float stdv, float scale, float shift, float var)
{
    gauss g;
    g.mean = shift + scale * mean;
    g.stdv = var * stdv;
    g.log_stdv = logf(g.stdv);
    return g;
}

static const float inv_sqrt_2pi = 0.3989422804014327f;
static float normal_pdf(float x, gauss g)
{
    float a = (x - g.mean) / g.stdv;
    return inv_sqrt_2pi / g.stdv * expf(-0.5f * a * a);
}
static float log_normal_pdf(float x, gauss g, float lisp)
{
    float a = (x - g.mean) / g.stdv;
    return lisp - g.log_stdv + (-0.5f * a * a);
}

typedef struct { gauss s, l, a0, a1, p, t0, t1; float lisp; } hmm;

static void emit(float x, const hmm* h, float e[6])
{
    float xx = (x > 200.0f || x < 40.0f) ? 100.0f : x;
    e[S_] = logf(0.50f * normal_pdf(xx, h->s) + 0.50f * 0.00476f);
    e[L_] = log_normal_pdf(xx, h->l, h->lisp);
    e[A_] = logf((0.874f * normal_pdf(xx, h->a0)) + (0.126f * normal_pdf(xx, h->a1)));
    e[P_] = log_normal_pdf(xx, h->p, h->lisp);
    e[C_] = (xx > 70.0f && xx < 140.0f) ? -4.2485f : -INFINITY;
    e[T_] = logf((0.346f * normal_pdf(xx, h->t0)) + (0.654f * normal_pdf(xx, h->t1)));
}

static float fmax_ref(float a, float b) { return (a < b) ? b : a; }   /* std::max */

static int cmp_double(const void* x, const void* y)
{
    double a = *(const double*)x, b = *(const double*)y;
    return (a < b) ? -1 : (b < a) ? 1 : 0;
}

static void polya_one(const float* samples, const float* durations, const npo_event_range* map, const npo_polya_job* jb,
                      npo_polya_result* out)
{
    memset(out, 0, sizeof(*out));
    if (jb->n_events == 0) { out->qc = 4; return; }
    const float ls[6] = { logf(1.0f), -INFINITY, -INFINITY, -INFINITY, -INFINITY, -INFINITY };
    const float tSS = logf(0.10f), tSL = logf(0.90f), tLL = logf(0.90f), tLA = logf(0.10f), tAA = logf(0.95f), tAP = logf(0.05f);
    const float tPP = logf(0.89f), tPC = logf(0.01f), tPT = logf(0.10f), tCP = logf(0.99f), tCC = logf(0.01f), tTT = logf(1.00f);
    const float scale = (float)jb->scale, shift = (float)jb->shift, var = (float)jb->var;
    hmm h;
    h.s = scaled(70.2737f, 3.7743f, scale, shift, var);
    h.l = scaled(110.973f, 5.237f, scale, shift, var);
    h.a0 = scaled(79.347f, 8.3702f, scale, shift, var);
    h.a1 = scaled(63.3126f, 2.7464f, scale, shift, var);
    h.p = scaled(108.883f, 3.257f, scale, shift, var);
    h.t0 = scaled(79.679f, 6.966f, scale, shift, var);
    h.t1 = scaled(105.784f, 16.022f, scale, shift, var);
    h.lisp = (float)log(0.3989422804014327);
    const size_t n = jb->n_samples;
    const float* x = samples + jb->sample_off;
    uint8_t* bp = (uint8_t*)malloc(n);
    float e[6];
    emit(x[n - 1], &h, e);
    float v[6] = { ls[S_] + e[S_], ls[L_] + e[L_], -INFINITY, -INFINITY, -INFINITY, -INFINITY };
    for (size_t i = 1; i < n; ++i) {
        float s_to_s = v[S_] + tSS, s_to_l = v[S_] + tSL, l_to_l = v[L_] + tLL, l_to_a = v[L_] + tLA;
        float a_to_a = v[A_] + tAA, a_to_p = v[A_] + tAP, p_to_p = v[P_] + tPP, p_to_c = v[P_] + tPC, p_to_t = v[P_] + tPT;
        float c_to_c = v[C_] + tCC, c_to_p = v[C_] + tCP, t_to_t = v[T_] + tTT;
        emit(x[i], &h, e);
        v[S_] = s_to_s + e[S_];
        v[L_] = fmax_ref(l_to_l, s_to_l) + e[L_];
        v[A_] = fmax_ref(a_to_a, l_to_a) + e[A_];
        v[P_] = fmax_ref(p_to_p, fmax_ref(a_to_p, c_to_p)) + e[P_];
        v[C_] = fmax_ref(c_to_c, p_to_c) + e[C_];
        v[T_] = fmax_ref(p_to_t, t_to_t) + e[T_];
        uint8_t b = 0;
        if (s_to_l < l_to_l) b |= 1;
        if (l_to_a < a_to_a) b |= 2;
        if ((a_to_p < p_to_p) && (c_to_p < p_to_p)) b |= 0 << 2;
        else if ((p_to_p < a_to_p) && (c_to_p < a_to_p)) b |= 1 << 2;
        else b |= 2 << 2;
        if (p_to_c < c_to_c) b |= 16;
        if (p_to_t < t_to_t) b |= 32;
        bp[i] = b;
    }
    out->end_score = v[T_];
    /* backtrack into region labels, then segment_squiggle's forward scan */
    uint8_t* reg = (uint8_t*)malloc(n);
    memset(reg, S_, n);
    reg[n - 1] = T_;
    for (size_t j = n - 2; j > 0; --j) {
        const uint8_t b = bp[j];
        int r;
        switch (reg[j + 1]) {
            case L_: r = (b & 1) ? L_ : S_; break;
            case A_: r = (b & 2) ? A_ : L_; break;
            case P_: { int c = (b >> 2) & 3; r = c == 0 ? P_ : (c == 1 ? A_ : C_); break; }
            case C_: r = (b & 16) ? C_ : P_; break;
            case T_: r = (b & 32) ? T_ : P_; break;
            default: r = S_;
        }
        reg[j] = (uint8_t)r;
        if (j == 1) break;
    }
    uint64_t st = 0, le = 1, ad = 2, po = 3, cl = 0;
    for (size_t i = 0; i < n; ++i) {
        if (reg[i] == S_ && i + 1 < n && reg[i + 1] == L_) st = i;
        if (reg[i] == L_ && reg[i + 1] == A_) le = i;
        if (reg[i] == A_ && reg[i + 1] == P_) ad = i;
        if (reg[i] == P_ && reg[i + 1] == T_) po = i;
        if (reg[i] == C_) cl++;
    }
    if (le == 1 || ad == 2 || po == 3) { le = (uint64_t)n - 3; ad = (uint64_t)n - 2; po = (uint64_t)n - 1; }
    free(reg); free(bp);
    out->start = st; out->leader = le; out->adapter = ad; out->polya = po; out->cliffs = cl;
    /* read rate */
    const size_t m = jb->n_kmers;
    double* d = (double*)calloc(m, sizeof(double));
    for (size_t i = 0; i < m; ++i) {
        const npo_event_range r = map[jb->map_off + i];
        if (r.start == -1) continue;
        for (int32_t j = r.start; j <= r.stop; ++j) d[i] += durations[jb->event_off + j];
    }
    qsort(d, m, sizeof(double), cmp_double);
    const double read_rate = 1.0 / d[m / 2];
    free(d);
    const double sr = jb->sample_rate;
    double polya_length = (double)(po - (ad + 1)) / sr * read_rate + -5.0;
    polya_length = (0.0 < polya_length) ? polya_length : 0.0;
    const double n_adapter = (double)((ad + 1) - le), n_polya = (double)(po - (ad + 1));
    const double adapter_length = (double)(ad - (le - 1)) / sr * read_rate;
    uint32_t qc = 0;
    if (n_adapter < 200.0 || n_polya < 200.0) qc |= 1;
    if (adapter_length > (double)300.0f) qc |= 2;
    out->read_rate = read_rate; out->polya_length = polya_length; out->qc = qc;
}

void npo_polya(const float* samples, const float* durations, const npo_event_range* map, const npo_polya_job* jobs, size_t n_jobs,
               npo_polya_result* results, int threads)
{
    #pragma omp parallel for schedule(dynamic, 1) num_threads(threads > 0 ? threads : 1)
    for (long long t = 0; t < (long long)n_jobs; ++t)
        polya_one(samples, durations, map, &jobs[t], &results[t]);
}
