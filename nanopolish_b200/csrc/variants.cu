// variants.cu — candidate screening of `nanopolish variants` on the device (SURVEY.md section 8f row N2, BASELINE configs[4]).
//
// Replaces, for a whole reference region at once:
//   generate_candidate_single_base_edits      ref: src/nanopolish_call_variants.cpp:288-361
//   AlignmentDB::get_event_subsequences        ref: src/alignment/nanopolish_alignment_db.cpp:172-221
//   AlignmentDB::_find_by_ref_bounds           ref: src/alignment/nanopolish_alignment_db.cpp:688-731
//   score_variant_thresholded                  ref: src/common/nanopolish_variant.cpp:765-799
//   Haplotype::apply_variant on the 22-base test haplotype   ref: src/nanopolish_haplotype.cpp:30-85
// (profile_hmm_score_set with no methylation alternative is profile_hmm_score: K1, unchanged.)
//
// Kernels:
//   var_bounds_kernel   per position: the records whose event alignment bounds the window, in record order, with their
//                       event range (two passes: count, then fill behind a prefix sum)
//   var_ranks_kernel    per (position, sequence, strand): the k-mer ranks of the base window and of its nine edited versions
//                       (substitution / insertion per base, deletion), both strands — a fixed pool K1's jobs point into
//   var_emit_kernel     per round: the jobs of the next reads_per_round reads of every position that still has a live
//                       candidate (base + live candidates per read)
//   var_accumulate_kernel  per position: the sequential `if (fabs(total) < threshold) total += variant - base` over the
//                       round's reads in order; candidates inside the threshold stay live
// The host drives the rounds; per round one read-back (job count) plus the scheduler's summary.
#include "nph_internal.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

int nph_launch_hmm_forward(nph_ctx* ctx, float* scores_dev);

namespace {

constexpr int kNoEvent = INT32_MIN;
constexpr int kSeqs = NPH_SCREEN_SLOTS + 1;      // nine candidates + the base haplotype (slot 9)
constexpr int kBlock = 256;
constexpr int kListCap = 2048;                   // records overlapping one block of positions, kept in shared memory

struct PosRead { uint32_t record; int32_t e1, e2; };

struct PosState {
    double total[NPH_SCREEN_SLOTS];
    uint32_t valid;       // bit c: candidate c exists (bit 31: the position is screened at all)
    uint32_t alive;       // bit c: |total_c| < threshold so far
    uint32_t done;        // reads consumed
    uint32_t chunk;       // reads of the current round
    unsigned long long ref_rows;   // DP rows the reference's loop scores at this position (2 sequences per candidate and read until exit)
};

struct VarDev {
    int flank, region_start, n_pos, n_ref, k, rpr;
    uint32_t flags, threshold;
    int win;              // 2 * flank + 2
    int stride;           // rank slots per (position, sequence, strand): the insertion's win + 1 - k + 1 k-mers
};

// first offset >= from with an event-alignment entry (n: none)
__device__ __forceinline__ int first_valid_from(const int32_t* __restrict__ dense, int n, int from)
{
    for (int o = from < 0 ? 0 : from; o < n; ++o) if (dense[o] != kNoEvent) return o;
    return n;
}

// _find_by_ref_bounds + the event/bp ratio test of get_event_subsequences for one record and window [cs, ce]
__device__ __forceinline__ bool window_events(const nph_meth_record& R, const int32_t* __restrict__ dense, int fv, int cs, int ce, int& e1, int& e2)
{
    const int n = (int)R.ref_len;
    if (fv >= n) return false;                                   // aligned_events.empty()
    const int os = cs - R.ref_start_pos, oe = ce - R.ref_start_pos;
    if (oe >= n || os >= n) return false;                        // lower_bound(ref_stop) == end()
    const int is = first_valid_from(dense, n, os);
    if (is >= n) return false;
    const int ie = first_valid_from(dense, n, oe);
    if (ie >= n) return false;
    if (!(is <= os || is != fv)) return false;                   // left_bounded; right_bounded always holds for a lower_bound
    e1 = dense[is]; e2 = dense[ie];
    const double ratio = fabs((double)(e1 - e2)) / fabs((double)(ce - cs));
    return ratio < 20.0;                                         // MAX_EVENT_TO_BP_RATIO
}

// pass 0: counts per position; pass 1: fills pos_reads behind pos_off
template <bool FILL>
__global__ void __launch_bounds__(kBlock) var_bounds_kernel(const VarDev d, const nph_meth_record* __restrict__ records, uint32_t n_records,
                                                            const int32_t* __restrict__ dense, const int32_t* __restrict__ first_valid,
                                                            uint64_t* __restrict__ counts, const uint64_t* __restrict__ pos_off,
                                                            PosRead* __restrict__ pos_reads)
{
    __shared__ uint32_t s_list[kListCap];
    __shared__ uint32_t s_n, s_warp[kBlock / 32];
    const int p0 = blockIdx.x * kBlock;
    const int pi = p0 + threadIdx.x;
    // records that can bound a window of this block of positions: their extent meets [first window start, last window end]
    const int lo = d.region_start + p0 - d.flank, hi = d.region_start + min(p0 + kBlock - 1, d.n_pos - 1) + 1 + d.flank;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    bool overflow = false;
    for (uint32_t base = 0; base < n_records; base += kBlock) {
        const uint32_t r = base + threadIdx.x;
        bool take = false;
        if (r < n_records) {
            const nph_meth_record R = records[r];
            take = R.ref_len > 0 && R.ref_start_pos <= hi && R.ref_start_pos + (int)R.ref_len - 1 >= lo;
        }
        // ordered append: record order is the order the reference walks its event records in
        const unsigned m = __ballot_sync(0xffffffffu, take);
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        if (lane == 0) s_warp[w] = __popc(m);
        __syncthreads();
        uint32_t before = 0;
        for (int i = 0; i < w; ++i) before += s_warp[i];
        uint32_t tot = 0;
        for (int i = 0; i < kBlock / 32; ++i) tot += s_warp[i];
        const uint32_t at = s_n + before + __popc(m & ((1u << lane) - 1u));
        if (take) { if (at < kListCap) s_list[at] = r; else overflow = true; }
        __syncthreads();
        if (threadIdx.x == 0) s_n = min(s_n + tot, (uint32_t)kListCap + 1u);
        __syncthreads();
    }
    const bool use_list = !__syncthreads_or(overflow) && s_n <= kListCap;
    if (pi >= d.n_pos) return;
    const int i = d.region_start + pi;
    const int cs = i - d.flank, ce = i + 1 + d.flank;
    const bool pos_ok = cs >= d.region_start && ce <= d.region_start + d.n_ref - 1;       // are_coordinates_valid
    uint64_t cnt = 0;
    PosRead* out = FILL ? pos_reads + pos_off[pi] : nullptr;
    if (pos_ok) {
        const uint32_t n_it = use_list ? s_n : n_records;
        for (uint32_t t = 0; t < n_it; ++t) {
            const uint32_t r = use_list ? s_list[t] : t;
            const nph_meth_record R = records[r];
            int e1, e2;
            if (window_events(R, dense + R.ref_off, first_valid[r], cs, ce, e1, e2)) {
                if (FILL) out[cnt] = PosRead{r, e1, e2};
                ++cnt;
            }
        }
    }
    if (!FILL) counts[pi] = cnt;
}

// exclusive prefix over n values: out[i], out[n] = total.  Three small launches (per-block sums, a one-block scan of the
// sums, per-block scan with the block's base) instead of one block walking the whole array: 200 000 positions took 0.36 ms
// per call in the one-block form, ten calls per screening.
constexpr int kScanBlock = 1024;
__device__ __forceinline__ unsigned long long block_scan_incl(unsigned long long v, unsigned long long* s /* 32 */, int t)
{
    const int lane = t & 31, w = t >> 5;
    for (int o = 1; o < 32; o <<= 1) { const unsigned long long x = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += x; }
    if (lane == 31) s[w] = v;
    __syncthreads();
    if (w == 0) {
        unsigned long long x = s[lane];
        for (int o = 1; o < 32; o <<= 1) { const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
        s[lane] = x;
    }
    __syncthreads();
    if (w > 0) v += s[w - 1];
    __syncthreads();
    return v;
}
__global__ void __launch_bounds__(kScanBlock) prefix_sums_kernel(const uint64_t* __restrict__ in, uint32_t n, uint64_t* __restrict__ block_sum)
{
    __shared__ unsigned long long s[32];
    const uint32_t i = blockIdx.x * kScanBlock + threadIdx.x;
    const unsigned long long incl = block_scan_incl(i < n ? in[i] : 0ull, s, threadIdx.x);
    if (threadIdx.x == kScanBlock - 1) block_sum[blockIdx.x] = incl;
}
__global__ void __launch_bounds__(kScanBlock) prefix_top_kernel(uint64_t* __restrict__ block_sum, uint32_t n_blocks, uint64_t* __restrict__ total)
{
    __shared__ unsigned long long s[32];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_blocks; base += kScanBlock) {
        const uint32_t i = base + threadIdx.x;
        const unsigned long long v = i < n_blocks ? block_sum[i] : 0ull;
        const unsigned long long incl = block_scan_incl(v, s, threadIdx.x);
        if (i < n_blocks) block_sum[i] = carry + incl - v;
        __syncthreads();
        if (threadIdx.x == kScanBlock - 1) carry += incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}
__global__ void __launch_bounds__(kScanBlock) prefix_apply_kernel(const uint64_t* __restrict__ in, uint32_t n, const uint64_t* __restrict__ block_base,
                                                                  uint64_t* __restrict__ out)
{
    __shared__ unsigned long long s[32];
    const uint32_t i = blockIdx.x * kScanBlock + threadIdx.x;
    const unsigned long long v = i < n ? in[i] : 0ull;
    const unsigned long long incl = block_scan_incl(v, s, threadIdx.x);
    if (i < n) out[i] = block_base[blockIdx.x] + incl - v;
}
// scratch: (n + 1023) / 1024 entries
static int prefix_exclusive(nph_ctx* ctx, const uint64_t* in, uint32_t n, uint64_t* out, uint64_t* scratch, cudaStream_t st)
{
    const uint32_t nb = (n + kScanBlock - 1) / kScanBlock;
    prefix_sums_kernel<<<nb, kScanBlock, 0, st>>>(in, n, scratch);
    prefix_top_kernel<<<1, kScanBlock, 0, st>>>(scratch, nb, out + n);
    prefix_apply_kernel<<<nb, kScanBlock, 0, st>>>(in, n, scratch, out);
    if (cudaGetLastError() != cudaSuccess) { ctx->last_error = "prefix kernels failed to launch"; return NPH_ERR_CUDA; }
    return NPH_OK;
}

// the sequence of slot `seq` at a position: the window with the slot's edit applied (codes 0..3), length returned.
// slots 2j / 2j+1: substitution to / insertion of base j at window offset `flank`; slot 8: deletion of that base; slot 9: base.
__device__ __forceinline__ int edited_window(const uint8_t* __restrict__ w, int win, int flank, int seq, uint8_t* out)
{
    if (seq == NPH_SCREEN_SLOTS) { for (int t = 0; t < win; ++t) out[t] = w[t]; return win; }
    if (seq == 8) {                                              // ref_seq = bases i-1, i; alt = base i-1
        for (int t = 0; t < flank; ++t) out[t] = w[t];
        for (int t = flank + 1; t < win; ++t) out[t - 1] = w[t];
        return win - 1;
    }
    const int j = seq >> 1;
    if ((seq & 1) == 0) { for (int t = 0; t < win; ++t) out[t] = w[t]; out[flank] = (uint8_t)j; return win; }
    for (int t = 0; t <= flank; ++t) out[t] = w[t];              // alt = base i followed by j
    out[flank + 1] = (uint8_t)j;
    for (int t = flank + 1; t < win; ++t) out[t + 1] = w[t];
    return win + 1;
}

__device__ __forceinline__ uint8_t dna_code(uint8_t c) { return c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : 0; }   // Alphabet::rank: unknown -> 0

// thread per (position, sequence): ranks of both strands into the pool, candidate validity into the position state
__global__ void __launch_bounds__(kBlock) var_ranks_kernel(const VarDev d, const uint8_t* __restrict__ ref, uint32_t* __restrict__ pool,
                                                           PosState* __restrict__ state, const uint64_t* __restrict__ pos_off)
{
    const long long gid = (long long)blockIdx.x * kBlock + threadIdx.x;
    if (gid >= (long long)d.n_pos * kSeqs) return;
    const int pi = (int)(gid / kSeqs), seq = (int)(gid % kSeqs);
    const int i = d.region_start + pi;
    const int cs = i - d.flank, ce = i + 1 + d.flank;
    const bool pos_ok = cs >= d.region_start && ce <= d.region_start + d.n_ref - 1;
    if (seq == NPH_SCREEN_SLOTS) {
        // the base-haplotype thread also initialises the position's state
        PosState st;
        for (int c = 0; c < NPH_SCREEN_SLOTS; ++c) st.total[c] = 0.0;
        st.valid = 0; st.alive = 0; st.done = 0; st.chunk = 0; st.ref_rows = 0;
        if (pos_ok) {
            const uint8_t b = dna_code(ref[cs - d.region_start + d.flank]), bp = dna_code(ref[cs - d.region_start + d.flank - 1]);
            uint32_t v = 0x80000000u;
            for (int j = 0; j < 4; ++j) if (j != b) v |= (1u << (2 * j)) | (1u << (2 * j + 1));   // substitution != ref; insertion "A" -> "AA" is redundant
            if (bp != b) v |= 1u << 8;                                                           // deletion "AA" -> "A" is redundant
            st.valid = v;
            st.alive = (pos_off[pi + 1] > pos_off[pi]) ? (v & 0x1ffu) : 0u;                      // no event sequence: nothing to score, quality 0
        }
        state[pi] = st;
    }
    if (!pos_ok) return;
    uint8_t w[NPH_SCREEN_MAX_WINDOW], sq[NPH_SCREEN_MAX_WINDOW + 1];
    for (int t = 0; t < d.win; ++t) w[t] = dna_code(ref[cs - d.region_start + t]);
    const int L = edited_window(w, d.win, d.flank, seq, sq);
    const int nk = L - d.k + 1;
    uint32_t* fw = pool + ((size_t)pi * kSeqs + seq) * 2 * d.stride;
    uint32_t* rc = fw + d.stride;
    for (int q = 0; q < nk; ++q) {
        uint32_t rf = 0, rr = 0;
        for (int t = 0; t < d.k; ++t) {
            rf = rf * 4u + sq[q + t];
            rr = rr * 4u + (3u - sq[q + d.k - 1 - t]);          // HMMInputSequence::get_kmer_rank(q, k, true): rank of the k-mer's reverse complement
        }
        fw[q] = rf; rc[q] = rr;
    }
}

// round bookkeeping, thread per position: how many jobs the position contributes this round
__global__ void var_round_count_kernel(const VarDev d, PosState* __restrict__ state, const uint64_t* __restrict__ pos_off, uint64_t* __restrict__ job_cnt)
{
    const int pi = blockIdx.x * blockDim.x + threadIdx.x;
    if (pi >= d.n_pos) return;
    PosState& st = state[pi];
    const uint32_t n_reads = (uint32_t)(pos_off[pi + 1] - pos_off[pi]);
    uint32_t chunk = 0;
    if (st.alive && st.done < n_reads) chunk = min((uint32_t)d.rpr, n_reads - st.done);
    st.chunk = chunk;
    job_cnt[pi] = (uint64_t)chunk * (1u + __popc(st.alive));
}

__global__ void var_emit_kernel(const VarDev d, const PosState* __restrict__ state, const uint64_t* __restrict__ pos_off,
                                const PosRead* __restrict__ pos_reads, const nph_meth_record* __restrict__ records,
                                const uint64_t* __restrict__ job_off, nph_hmm_job* __restrict__ jobs, unsigned long long* __restrict__ events)
{
    const int pi = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long ev = 0;
    if (pi < d.n_pos) {
        const PosState st = state[pi];
        if (st.chunk) {
            const PosRead* rd = pos_reads + pos_off[pi] + st.done;
            nph_hmm_job* out = jobs + job_off[pi];
            for (uint32_t r = 0; r < st.chunk; ++r) {
                const PosRead pr = rd[r];
                const nph_meth_record R = records[pr.record];
                nph_hmm_job jb;
                jb.read = R.read; jb.model_id = R.model_id;
                jb.event_start = (uint32_t)pr.e1; jb.event_stop = (uint32_t)pr.e2;
                jb.stride = R.rc ? -1 : 1;                    // EventAlignmentRecord::stride agrees with rc for every read the HMM accepts (profile_hmm_r9.inl:275)
                jb.rc = R.rc; jb.flags = (uint8_t)d.flags; jb.reserved = 0;
                const unsigned long long E = (unsigned long long)(pr.e1 > pr.e2 ? pr.e1 - pr.e2 : pr.e2 - pr.e1) + 1ull;
                // the base haplotype first, then the live candidates in slot order
                for (int seq = NPH_SCREEN_SLOTS; ; ) {
                    const int L = seq == NPH_SCREEN_SLOTS ? d.win : (seq == 8 ? d.win - 1 : ((seq & 1) ? d.win + 1 : d.win));
                    jb.n_kmers = (uint32_t)(L - d.k + 1);
                    jb.rank_off = ((uint64_t)pi * kSeqs + (uint64_t)seq) * 2 * d.stride + (R.rc ? d.stride : 0);
                    *out++ = jb;
                    ev += E;
                    if (seq == NPH_SCREEN_SLOTS) seq = -1;
                    do { ++seq; } while (seq < NPH_SCREEN_SLOTS && !((st.alive >> seq) & 1u));
                    if (seq >= NPH_SCREEN_SLOTS) break;
                }
            }
        }
    }
    // scored events of the round
    for (int o = 16; o; o >>= 1) ev += __shfl_xor_sync(0xffffffffu, ev, o);
    if ((threadIdx.x & 31) == 0 && ev) atomicAdd(events, ev);
}

__global__ void var_accumulate_kernel(const VarDev d, PosState* __restrict__ state, const uint64_t* __restrict__ job_off,
                                      const float* __restrict__ scores, unsigned int* __restrict__ any_left, const uint64_t* __restrict__ pos_off,
                                      const PosRead* __restrict__ pos_reads, unsigned long long* __restrict__ ref_events)
{
    const int pi = blockIdx.x * blockDim.x + threadIdx.x;
    if (pi >= d.n_pos) return;
    PosState st = state[pi];
    if (!st.chunk) return;
    const float* s = scores + job_off[pi];
    const PosRead* rd = pos_reads + pos_off[pi] + st.done;
    const double thr = (double)d.threshold;
    unsigned long long ref_ev = 0;
    for (uint32_t r = 0; r < st.chunk; ++r) {
        const double base_score = (double)*s++;                 // double base_score = profile_hmm_score_set(...) (a float)
        const unsigned long long E = (unsigned long long)(rd[r].e1 > rd[r].e2 ? rd[r].e1 - rd[r].e2 : rd[r].e2 - rd[r].e1) + 1ull;
        for (int c = 0; c < NPH_SCREEN_SLOTS; ++c) {
            if (!((st.alive >> c) & 1u)) continue;
            const double variant_score = (double)*s++;
            if (fabs(st.total[c]) < thr) {
                st.total[c] = __dadd_rn(st.total[c], __dsub_rn(variant_score, base_score));
                ref_ev += 2ull * E;                              // what the reference's loop scores here: the base AND the variant sequence
            }
        }
    }
    if (ref_ev) atomicAdd(ref_events, ref_ev);
    st.ref_rows += ref_ev;
    st.done += st.chunk;
    uint32_t alive = 0;
    for (int c = 0; c < NPH_SCREEN_SLOTS; ++c) if (((st.alive >> c) & 1u) && fabs(st.total[c]) < thr) alive |= 1u << c;
    st.alive = alive;
    st.chunk = 0;
    state[pi] = st;
    if (alive && st.done < (uint32_t)(pos_off[pi + 1] - pos_off[pi])) atomicOr(any_left, 1u);
}

__global__ void var_output_kernel(const VarDev d, const PosState* __restrict__ state, const uint64_t* __restrict__ pos_off,
                                  double* __restrict__ qual, uint32_t* __restrict__ n_reads, unsigned long long* __restrict__ ref_rows)
{
    const int pi = blockIdx.x * blockDim.x + threadIdx.x;
    if (pi >= d.n_pos) return;
    const PosState st = state[pi];
    ref_rows[pi] = st.ref_rows;
    for (int c = 0; c < NPH_SCREEN_SLOTS; ++c)
        qual[(size_t)pi * NPH_SCREEN_SLOTS + c] = ((st.valid >> c) & 1u) ? st.total[c] : __longlong_as_double(0x7ff8000000000000ll);
    n_reads[pi] = (uint32_t)(pos_off[pi + 1] - pos_off[pi]);
}

int make_dev(nph_ctx* ctx, const nph_screen_params& p, size_t n_ref, VarDev& d)
{
    if (p.flank < 1 || 2 * p.flank + 3 > NPH_SCREEN_MAX_WINDOW) { ctx->last_error = "nph_screen_params: flank outside 1..30"; return NPH_ERR_UNSUPPORTED; }
    if (p.k < 1 || (int)p.k > 2 * p.flank + 1 || p.reads_per_round == 0 || n_ref < 2 || n_ref > 0x7fffffffu) return NPH_ERR_INVALID;
    d.flank = p.flank; d.region_start = p.region_start; d.n_ref = (int)n_ref; d.n_pos = (int)n_ref - 1;
    d.k = (int)p.k; d.rpr = (int)p.reads_per_round; d.flags = p.alignment_flags; d.threshold = p.score_threshold;
    d.win = 2 * p.flank + 2;
    d.stride = d.win + 1 - d.k + 1;
    return NPH_OK;
}

} // namespace

extern "C" int nph_screen_load(nph_ctx* ctx, const char* ref_bases, size_t n_ref_bases, const int16_t* event_deltas, size_t n_deltas_total,
                               const int32_t* first_event, const nph_meth_record* records, size_t n_records,
                               const nph_screen_params* params, double indel_bias)
{
    if (!ctx || !params || !ref_bases || (n_records && (!records || !first_event || (n_deltas_total && !event_deltas)))) return NPH_ERR_INVALID;
    nph_ctx::ScreenState& m = ctx->screen;
    m.loaded = false; m.ran = false;
    if (!ctx->reads_loaded) return NPH_ERR_STATE;
    VarDev d;
    NPH_TRY(make_dev(ctx, *params, n_ref_bases, d));
    for (size_t r = 0; r < n_records; ++r) {
        const nph_meth_record& R = records[r];
        const bool ok = R.read < ctx->n_reads && R.model_id < ctx->models.size() && R.ref_len <= n_deltas_total && R.ref_off <= n_deltas_total - R.ref_len &&
                        R.ref_len <= 0x3fffffffu;
        if (!ok) { ctx->last_error = "screening record " + std::to_string(r) + " is out of range (read, model or event-alignment slice)"; return NPH_ERR_INVALID; }
        const DevModel& mod = ctx->models[R.model_id];
        if (mod.k != params->k || mod.alphabet_size != 4) { ctx->last_error = "screening record " + std::to_string(r) + ": its model is not a nucleotide model of k = params.k"; return NPH_ERR_INVALID; }
    }
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    NPH_TRY(nph_reserve(ctx, m.d_ref, n_ref_bases + 16));
    NPH_TRY(nph_reserve(ctx, m.d_deltas, n_deltas_total + 16));
    NPH_TRY(nph_reserve(ctx, m.d_dense, n_deltas_total + 2 * n_records + 16));
    NPH_TRY(nph_reserve(ctx, m.d_records, n_records + 1));
    NPH_CUDA(ctx, cudaMemcpyAsync(m.d_ref.p, ref_bases, n_ref_bases, cudaMemcpyHostToDevice, ctx->stream));
    if (n_records) {
        NPH_CUDA(ctx, cudaMemcpyAsync(m.d_records.p, records, sizeof(nph_meth_record) * n_records, cudaMemcpyHostToDevice, ctx->stream));
        if (n_deltas_total) NPH_CUDA(ctx, cudaMemcpyAsync(m.d_deltas.p, event_deltas, sizeof(int16_t) * n_deltas_total, cudaMemcpyHostToDevice, ctx->stream));
        NPH_CUDA(ctx, cudaMemcpyAsync(m.d_dense.p + n_deltas_total, first_event, sizeof(int32_t) * n_records, cudaMemcpyHostToDevice, ctx->stream));
    }
    m.params = *params; m.indel_bias = indel_bias;
    m.n_pos = (size_t)d.n_pos; m.n_records = n_records; m.n_ref = n_ref_bases; m.n_deltas = n_deltas_total;
    m.loaded = true;
    return NPH_OK;
}

extern "C" int nph_screen_run(nph_ctx* ctx)
{
    if (!ctx) return NPH_ERR_INVALID;
    nph_ctx::ScreenState& m = ctx->screen;
    if (!m.loaded || !ctx->reads_loaded) return NPH_ERR_STATE;
    m.ran = false; m.n_rounds = 0; m.n_jobs = 0; m.n_scored_events = 0; m.n_jobs_no_exit = 0; m.n_reference_events = 0;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    VarDev d;
    NPH_TRY(make_dev(ctx, m.params, m.n_ref, d));
    const uint32_t n_pos = (uint32_t)m.n_pos, n_rec = (uint32_t)m.n_records;
    cudaStream_t st = ctx->stream;
    int32_t* dense = reinterpret_cast<int32_t*>(m.d_dense.p);
    int32_t* first_valid = dense + m.n_deltas + m.n_records;
    NPH_TRY(nph_expand_event_maps(ctx, reinterpret_cast<const int16_t*>(m.d_deltas.p), dense + m.n_deltas, m.d_records.p, n_rec, dense, first_valid));
    // per position: its event sequences
    NPH_TRY(nph_reserve(ctx, m.d_pos_off, (size_t)n_pos + 1));
    NPH_TRY(nph_reserve(ctx, m.d_job_off, 2 * ((size_t)n_pos + 1) + 8 + ((size_t)n_pos + 1023) / 1024 + 1));
    uint64_t* counts = m.d_job_off.p;                         // scratch: per-position counts, then per-round job counts / offsets
    uint64_t* job_off = m.d_job_off.p + (size_t)n_pos + 1;
    uint64_t* scan_scratch = job_off + (size_t)n_pos + 1 + 8;
    const int pgrid = (int)((n_pos + kBlock - 1) / kBlock);
    var_bounds_kernel<false><<<pgrid, kBlock, 0, st>>>(d, m.d_records.p, n_rec, dense, first_valid, counts, nullptr, nullptr);
    NPH_CUDA(ctx, cudaGetLastError());
    NPH_TRY(prefix_exclusive(ctx, counts, n_pos, m.d_pos_off.p, scan_scratch, st));
    uint64_t n_pos_reads = 0;
    NPH_CUDA(ctx, cudaMemcpyAsync(&n_pos_reads, m.d_pos_off.p + n_pos, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    NPH_CUDA(ctx, cudaStreamSynchronize(st));
    NPH_TRY(nph_reserve(ctx, m.d_pos_reads, sizeof(PosRead) * ((size_t)n_pos_reads + 1)));
    PosRead* pos_reads = reinterpret_cast<PosRead*>(m.d_pos_reads.p);
    var_bounds_kernel<true><<<pgrid, kBlock, 0, st>>>(d, m.d_records.p, n_rec, dense, first_valid, nullptr, m.d_pos_off.p, pos_reads);
    NPH_CUDA(ctx, cudaGetLastError());
    // rank pool (K1's d_ranks for this batch) and position state
    const size_t pool = (size_t)n_pos * kSeqs * 2 * (size_t)d.stride;
    NPH_TRY(nph_reserve(ctx, ctx->d_ranks, pool));
    NPH_TRY(nph_reserve(ctx, m.d_state, sizeof(PosState) * (size_t)n_pos + 64));      // + the counters: our DP rows, a flag, the reference's DP rows
    PosState* state = reinterpret_cast<PosState*>(m.d_state.p);
    NPH_CUDA(ctx, cudaMemsetAsync(ctx->d_ranks.p, 0, sizeof(uint32_t) * pool, st));
    const long long n_thr = (long long)n_pos * kSeqs;
    var_ranks_kernel<<<(unsigned)((n_thr + kBlock - 1) / kBlock), kBlock, 0, st>>>(d, m.d_ref.p, ctx->d_ranks.p, state, m.d_pos_off.p);
    NPH_CUDA(ctx, cudaGetLastError());
    NPH_TRY(nph_upload_read_transitions(ctx, m.indel_bias));
    ctx->codes_mode = false;
    // what the same screening costs without the early exit: every read of every candidate (+ the base per candidate, as the reference scores it)
    // counted on the host side from the totals: sum over positions of reads x (1 + candidates) — filled at the end from the state
    unsigned long long* d_events = reinterpret_cast<unsigned long long*>(m.d_state.p + sizeof(PosState) * (size_t)n_pos);
    unsigned int* d_any = reinterpret_cast<unsigned int*>(d_events + 1);
    NPH_CUDA(ctx, cudaMemsetAsync(d_events, 0, 24, st));
    float kernel_ms_total = 0.f;
    int launches_total = 0;
    for (;;) {
        var_round_count_kernel<<<pgrid, kBlock, 0, st>>>(d, state, m.d_pos_off.p, counts);
        NPH_CUDA(ctx, cudaGetLastError());
        NPH_TRY(prefix_exclusive(ctx, counts, n_pos, job_off, scan_scratch, st));
        NPH_CUDA(ctx, cudaGetLastError());
        uint64_t n_jobs = 0;
        NPH_CUDA(ctx, cudaMemcpyAsync(&n_jobs, job_off + n_pos, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        NPH_CUDA(ctx, cudaStreamSynchronize(st));                         // read-back: the round's job count
        if (n_jobs == 0) break;
        NPH_TRY(nph_reserve(ctx, ctx->d_jobs, (size_t)n_jobs));
        NPH_TRY(nph_reserve(ctx, ctx->d_order, (size_t)n_jobs));
        NPH_TRY(nph_reserve(ctx, ctx->d_scores, (size_t)n_jobs));
        var_emit_kernel<<<pgrid, kBlock, 0, st>>>(d, state, m.d_pos_off.p, pos_reads, m.d_records.p, job_off, ctx->d_jobs.p, d_events);
        NPH_CUDA(ctx, cudaGetLastError());
        ctx->jobs_loaded = false;
        ctx->jobs_trusted = true;                                         // var_ranks_kernel wrote the pool: the scheduler need not walk it every round
        const int rc_sched = nph_jobs_schedule(ctx, (size_t)n_jobs, pool); // validation + schedule (one more read-back)
        ctx->jobs_trusted = false;
        NPH_TRY(rc_sched);
        NPH_TRY(nph_launch_hmm_forward(ctx, nullptr));
        NPH_CUDA(ctx, cudaMemsetAsync(d_any, 0, sizeof(unsigned int), st));
        var_accumulate_kernel<<<pgrid, kBlock, 0, st>>>(d, state, job_off, ctx->d_scores.p, d_any, m.d_pos_off.p, pos_reads, d_events + 2);
        NPH_CUDA(ctx, cudaGetLastError());
        float ms = 0.f; int nl = 0;
        if (nph_last_kernel_ms(ctx, &ms, &nl) == NPH_OK) { kernel_ms_total += ms; launches_total += nl + 6; }
        m.n_rounds += 1;
        m.n_jobs += n_jobs;
    }
    unsigned long long ev[3] = {0, 0, 0};
    NPH_CUDA(ctx, cudaMemcpyAsync(ev, d_events, sizeof(ev), cudaMemcpyDeviceToHost, st));
    NPH_CUDA(ctx, cudaStreamSynchronize(st));
    m.n_scored_events = ev[0];
    m.n_reference_events = ev[2];
    ctx->staged_ms = kernel_ms_total; ctx->timing_valid = 2; ctx->last_launches = launches_total;
    m.ran = true;
    return NPH_OK;
}

extern "C" int nph_screen_counts(nph_ctx* ctx, uint32_t* n_rounds_out, uint64_t* n_jobs_out, uint64_t* n_scored_events_out, uint64_t* n_jobs_without_exit_out,
                                 uint64_t* n_reference_events_out)
{
    if (!ctx) return NPH_ERR_INVALID;
    nph_ctx::ScreenState& m = ctx->screen;
    if (!m.ran) return NPH_ERR_STATE;
    if (n_rounds_out) *n_rounds_out = m.n_rounds;
    if (n_jobs_out) *n_jobs_out = m.n_jobs;
    if (n_scored_events_out) *n_scored_events_out = m.n_scored_events;
    if (n_jobs_without_exit_out) *n_jobs_without_exit_out = m.n_jobs_no_exit;
    if (n_reference_events_out) *n_reference_events_out = m.n_reference_events;
    return NPH_OK;
}

extern "C" int nph_screen_fetch(nph_ctx* ctx, double* qualities_out, uint32_t* n_reads_out, uint64_t* reference_rows_out)
{
    if (!ctx || !qualities_out) return NPH_ERR_INVALID;
    nph_ctx::ScreenState& m = ctx->screen;
    if (!m.ran) return NPH_ERR_STATE;
    VarDev d;
    NPH_TRY(make_dev(ctx, m.params, m.n_ref, d));
    const uint32_t n_pos = (uint32_t)m.n_pos;
    // outputs staged in the (now idle) score buffer region: 9 doubles + 1 uint32 per position
    ctx->loaded_raw.valid = false;              // d_prep held the last load_from_raw batch's durations and map
    struct { double* q; unsigned long long* r; uint32_t* n; } out{};
    auto layout = [&](NphCarve& a) {
        out.q = a.take<double>((size_t)NPH_SCREEN_SLOTS * n_pos);
        out.r = a.take<unsigned long long>(n_pos);
        out.n = a.take<uint32_t>(n_pos);
    };
    NPH_TRY(nph_lay_out(ctx, ctx->d_prep, layout));
    const size_t b_q = sizeof(double) * NPH_SCREEN_SLOTS * (size_t)n_pos, b_n = sizeof(uint32_t) * (size_t)n_pos;
    const size_t b_r = sizeof(unsigned long long) * (size_t)n_pos;
    var_output_kernel<<<(n_pos + kBlock - 1) / kBlock, kBlock, 0, ctx->stream>>>(d, reinterpret_cast<const PosState*>(m.d_state.p), m.d_pos_off.p, out.q, out.n, out.r);
    NPH_CUDA(ctx, cudaGetLastError());
    NPH_CUDA(ctx, cudaMemcpyAsync(qualities_out, out.q, b_q, cudaMemcpyDeviceToHost, ctx->stream));
    std::vector<uint32_t> tmp;
    uint32_t* n_dst = n_reads_out;
    if (!n_dst) { tmp.resize(n_pos); n_dst = tmp.data(); }
    NPH_CUDA(ctx, cudaMemcpyAsync(n_dst, out.n, b_n, cudaMemcpyDeviceToHost, ctx->stream));
    if (reference_rows_out) NPH_CUDA(ctx, cudaMemcpyAsync(reference_rows_out, out.r, b_r, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    // jobs a screening without early exit would have run: per position reads x (1 + candidates)
    uint64_t full = 0;
    for (uint32_t p = 0; p < n_pos; ++p) {
        int cands = 0;
        for (int c = 0; c < NPH_SCREEN_SLOTS; ++c) cands += !std::isnan(qualities_out[(size_t)p * NPH_SCREEN_SLOTS + c]);
        if (cands) full += (uint64_t)n_dst[p] * (uint64_t)(1 + cands);
    }
    m.n_jobs_no_exit = full;
    return NPH_OK;
}

extern "C" int nph_screen_edits_batch(nph_ctx* ctx,
                                      const nph_read* reads, size_t n_reads,
                                      const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                                      const char* ref_bases, size_t n_ref_bases,
                                      const int16_t* event_deltas, size_t n_deltas_total, const int32_t* first_event,
                                      const nph_meth_record* records, size_t n_records,
                                      const nph_screen_params* params, double indel_bias,
                                      double* qualities_out, uint32_t* n_reads_out, uint64_t* n_scored_events_out)
{
    if (!ctx) return NPH_ERR_INVALID;
    NPH_TRY(nph_reads_load(ctx, reads, n_reads, ev_mean, ev_start_time, n_events_total));
    NPH_TRY(nph_screen_load(ctx, ref_bases, n_ref_bases, event_deltas, n_deltas_total, first_event, records, n_records, params, indel_bias));
    NPH_TRY(nph_screen_run(ctx));
    NPH_TRY(nph_screen_fetch(ctx, qualities_out, n_reads_out, nullptr));
    if (n_scored_events_out) *n_scored_events_out = ctx->screen.n_scored_events;
    return NPH_OK;
}
