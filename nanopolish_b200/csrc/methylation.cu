// methylation.cu — call-methylation's per-read enumeration on the device (SURVEY.md section 8f, row N3).
//
// Replaces, for a whole BamProcessor batch at once, the part of
//   calculate_methylation_for_read       ref: src/basemods/nanopolish_basemods.cpp:238-457
// between "Scan the sequence for motifs" (:301) and the two profile_hmm_score calls (:383-392):
//   Alphabet::is_motif_match             ref: src/common/nanopolish_alphabet.h:296-310 (complete recognition sites only)
//   the grouping loop                    ref: basemods.cpp:309-322
//   window / span / start-distance test  ref: basemods.cpp:329-338
//   AlignmentDB::_find_by_ref_bounds     ref: src/alignment/nanopolish_alignment_db.cpp:688-731
//   the event-span test and region filter   ref: basemods.cpp:359-365, 398-401
//   Alphabet::methylate / reverse_complement and HMMInputSequence::get_kmer_rank over the window
//                                        ref: nanopolish_alphabet.h:146-330, src/hmm/nanopolish_hmm_input_sequence.h:76-91
//
// Three small kernels around K1:
//   meth_scan_kernel   a warp per record: ballot scan for recognition sites 32 bases at a time, groups closed as the
//                      sites stream by, the two lower_bounds as 32-ary warp searches over the event alignment; writes a
//                      provisional row per surviving group and the record's group / k-mer-rank / scored-event counts
//   meth_prefix_kernel exclusive prefix sums of those counts over the records (site, job and rank offsets) + totals
//   meth_emit_kernel   a warp per record: per group, the window as alphabet ranks in shared memory (forward, or the
//                      reverse complement the way Alphabet::reverse_complement builds it), methylated copy with every
//                      complete recognition site replaced, rolling k-mer ranks by all lanes, two nph_hmm_job records and
//                      the site record — straight into the arrays K1's device-side scheduler reads
// then hmm_schedule.cu + the forward kernels run unchanged, and meth_fill_kernel copies the two scores of each group
// into its site record.  The host sees O(records) work only.
#include "nph_internal.cuh"
#include "tsv_format.cuh"
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

namespace {

constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr unsigned kFull = 0xffffffffu;

// a group that passed every test of the reference's loop, before its jobs exist
struct MethGroup {
    int32_t first, last;      // motif_sites[start_idx], motif_sites[end_idx - 1] (offsets into ref_seq)
    int32_t n_motif;
    int32_t e1, e2;           // _find_by_ref_bounds' event indices
    int32_t win_len;          // subseq.length(): sub_end - sub_start + 1, cut at the end of ref_seq like std::string::substr
};

struct MethSummary {
    unsigned long long n_sites, n_ranks, n_events;
    int error;                // 0, or 1 + index of a record with a window shorter than k
    int pad;
};

// the alphabet and site tables as the kernels use them (ranks, not characters)
struct MethDev {
    int32_t min_separation, min_flank, max_span, min_event_span, region_start, region_end;
    uint32_t k, asize, n_sites, site_len;
    uint8_t rank_of[256];                                              // Alphabet::rank (unknown symbols rank 0)
    uint8_t comp_rank_of[256];                                         // rank(complement(symbol))
    char    site[NPH_METH_MAX_SITES][NPH_METH_MAX_SITE_LEN];           // recognition sites, characters
    uint8_t site_m_rank[NPH_METH_MAX_SITES][NPH_METH_MAX_SITE_LEN];    // ranks of the methylated site
    uint8_t site_mrc_rank[NPH_METH_MAX_SITES][NPH_METH_MAX_SITE_LEN];  // ranks of what stands on the other strand: reverse(methylated complement)
};

// does a complete recognition site start at ref[i]?  (is_motif_match reports complete sites only; the partial
// matches match_to_site also knows — string end, string inside a site — never have the full length for len >= site_len)
__device__ __forceinline__ int site_at(const MethDev& d, const uint8_t* __restrict__ ref, int i, int n)
{
    if (i < 0 || i + (int)d.site_len > n) return -1;
    for (uint32_t s = 0; s < d.n_sites; ++s) {
        bool eq = true;
        for (uint32_t t = 0; t < d.site_len; ++t) eq = eq && (ref[i + t] == (uint8_t)d.site[s][t]);
        if (eq) return (int)s;
    }
    return -1;
}

// std::lower_bound(pairs, pairs + n, v, ref_pos < v) as a 32-ary search by the whole warp: every round the lanes probe
// 32 evenly spaced entries and the ballot tells which interval holds the boundary (3 rounds for a 4 000-event read
// instead of 12 dependent loads)
__device__ __forceinline__ int warp_lower_bound(const nph_aligned_pair* __restrict__ pairs, int n, int v, int lane)
{
    int lo = 0, hi = n;                       // the answer lies in [lo, hi]
    while (hi - lo > 32) {
        const int step = (hi - lo + 31) / 32;
        const int idx = lo + (lane + 1) * step - 1;
        const bool less = idx < hi && pairs[idx].ref_pos < v;
        const int c = __popc(__ballot_sync(kFull, less));      // probes 0..c-1 are < v (the probes are monotone)
        const int nlo = lo + c * step;
        const int nhi = min(hi, lo + (c + 1) * step - 1);       // probe c (if it exists) is >= v: the answer is at most its index
        lo = min(nlo, hi); hi = max(nhi, lo);
    }
    const int idx = lo + lane;
    const bool less = idx < hi && pairs[idx].ref_pos < v;
    return lo + __popc(__ballot_sync(kFull, less));
}

constexpr int kNoEvent = INT32_MIN;

// compact event alignments: per record, a prefix sum over its int16 deltas rebuilds the event index of every reference base that
// has an aligned_events entry (kNoEvent elsewhere) and notes the first such base
__global__ void __launch_bounds__(kThreads) meth_expand_kernel(const int16_t* __restrict__ deltas, const int32_t* __restrict__ first_event,
                                                               const nph_meth_record* __restrict__ records, uint32_t n_records,
                                                               int32_t* __restrict__ dense, int32_t* __restrict__ first_valid)
{
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * kWarps + (threadIdx.x >> 5);
    const uint32_t n_warps = gridDim.x * kWarps;
    for (uint32_t rec = warp; rec < n_records; rec += n_warps) {
        const nph_meth_record R = records[rec];
        const int16_t* dl = deltas + R.ref_off;
        int32_t* out = dense + R.ref_off;
        const int n = (int)R.ref_len;
        int running = first_event[rec];
        int fv = n;
        for (int base = 0; base < n; base += 32) {
            const int o = base + lane;
            const int dv = o < n ? (int)dl[o] : NPH_METH_NO_PAIR;
            const bool valid = dv != NPH_METH_NO_PAIR;
            int v = valid ? dv : 0;
#pragma unroll
            for (int sft = 1; sft < 32; sft <<= 1) { const int t = __shfl_up_sync(kFull, v, sft); if (lane >= sft) v += t; }
            if (o < n) out[o] = valid ? running + v : kNoEvent;
            running += __shfl_sync(kFull, v, 31);
            const unsigned m = __ballot_sync(kFull, valid);
            if (m && fv == n) fv = base + (__ffs(m) - 1);
        }
        if (lane == 0) first_valid[rec] = fv;
    }
}

// first offset >= from with an aligned_events entry (n: none): the dense counterpart of std::lower_bound on ref_pos
__device__ __forceinline__ int warp_first_valid(const int32_t* __restrict__ dense, int n, int from, int lane)
{
    for (int base = from < 0 ? 0 : from; base < n; base += 32) {
        const int o = base + lane;
        const unsigned m = __ballot_sync(kFull, o < n && dense[o] != kNoEvent);
        if (m) return base + (__ffs(m) - 1);
    }
    return n;
}

struct ScanArgs {
    const uint8_t* ref;
    const int32_t* dense;       // compact mode: event index per reference base (nullptr: pair lists)
    const int32_t* first_valid;
    const nph_aligned_pair* pairs;
    const nph_meth_record* records;
    const uint64_t* prov_off;
    MethGroup* prov;
    uint64_t* counts;          // [3 * n_records]: groups, ranks, scored events per record
    MethSummary* sum;
    uint32_t n_records;
};

__global__ void __launch_bounds__(kThreads) meth_scan_kernel(const ScanArgs a, const MethDev d)
{
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * kWarps + (threadIdx.x >> 5);
    const uint32_t n_warps = gridDim.x * kWarps;
    for (uint32_t rec = warp; rec < a.n_records; rec += n_warps) {
        const nph_meth_record R = a.records[rec];
        const uint8_t* ref = a.ref + R.ref_off;
        const nph_aligned_pair* pairs = a.pairs ? a.pairs + R.pair_off : nullptr;
        const int32_t* dense = a.dense ? a.dense + R.ref_off : nullptr;
        const int fv = a.dense ? a.first_valid[rec] : 0;
        const int n = (int)R.ref_len, np = a.dense ? 0 : (int)R.n_pairs;
        MethGroup* out = a.prov + a.prov_off[rec];
        unsigned long long n_groups = 0, n_ranks = 0, n_events = 0;
        int bad = 0;
        int g_first = 0, g_count = 0, last_site = 0;

        // closes the open group [g_first, last_site] of g_count sites: every test of basemods.cpp:329-365, 398-401 in order
        auto close_group = [&]() {
            const int sub_start = g_first - d.min_flank;
            const int sub_end = last_site + d.min_flank;
            const int span = last_site - g_first;
            if (sub_start <= d.min_separation || span > d.max_span) return;
            const int calling_start = sub_start + R.ref_start_pos, calling_end = sub_end + R.ref_start_pos;
            int e1, e2;
            if (dense) {
                // the two lower_bounds on the rebuilt list: first reference offset at or after the boundary that has an entry
                const int is = warp_first_valid(dense, n, sub_start, lane);
                const int ie = warp_first_valid(dense, n, sub_end, lane);
                if (is == n || ie == n) return;                                    // not bounded
                if (!(is <= sub_start || is != fv)) return;                        // left_bounded (see the pair form below)
                e1 = dense[is]; e2 = dense[ie];
            } else {
                const int is = warp_lower_bound(pairs, np, calling_start, lane);
                const int ie = warp_lower_bound(pairs, np, calling_end, lane);
                if (is == np || ie == np) return;                                  // not bounded
                // left_bounded: the entry at/after the boundary sits on it, or an earlier entry exists (it is < ref_start by
                // construction).  right_bounded: the lower_bound entry is >= ref_stop by construction.
                if (!(pairs[is].ref_pos <= calling_start || is != 0)) return;
                e1 = pairs[is].read_pos; e2 = pairs[ie].read_pos;
            }
            const int de = e2 > e1 ? e2 - e1 : e1 - e2;
            if (de <= d.min_event_span) return;
            // (the reference's event/bp ratio divides by calling_start - calling_end < 0 and so never exceeds its limit)
            const int start_position = g_first + R.ref_start_pos, end_position = last_site + R.ref_start_pos;
            if ((d.region_start != -1 && start_position < d.region_start) || (d.region_end != -1 && end_position >= d.region_end)) return;
            const int win_len = min(sub_end, n - 1) - sub_start + 1;               // std::string::substr cuts at the end
            if (win_len < (int)d.k) { bad = 1; return; }
            if (lane == 0) out[n_groups] = MethGroup{g_first, last_site, g_count, e1, e2, win_len};
            n_groups += 1;
            n_ranks += 2ull * (unsigned long long)(win_len - (int)d.k + 1);
            n_events += 2ull * (unsigned long long)(de + 1);
        };

        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            // the scan loop runs over i < ref_seq.size() - 1 (basemods.cpp:303)
            const bool hit = (i < n - 1) && site_at(d, ref, i, n) >= 0;
            unsigned mask = __ballot_sync(kFull, hit);
            while (mask) {
                const int pos = base + (__ffs(mask) - 1);
                mask &= mask - 1;
                if (g_count > 0 && pos - last_site > d.min_separation) { close_group(); g_count = 0; }
                if (g_count == 0) g_first = pos;
                g_count += 1;
                last_site = pos;
            }
        }
        if (g_count > 0) close_group();
        if (lane == 0) {
            a.counts[3 * (size_t)rec] = n_groups;
            a.counts[3 * (size_t)rec + 1] = n_ranks;
            a.counts[3 * (size_t)rec + 2] = n_events;
            if (bad) atomicCAS(&a.sum->error, 0, (int)(rec + 1));
        }
    }
}

// exclusive prefix sums over the records: site_off (n + 1 entries) and rank_off (n entries), plus the totals.
// One block; the record count of a batch is 10^3..10^6, i.e. at most ~1000 rounds of a 1024-wide scan.
__global__ void __launch_bounds__(1024) meth_prefix_kernel(const uint64_t* __restrict__ counts, uint32_t n_records,
                                                           uint64_t* __restrict__ site_off, uint64_t* __restrict__ rank_off,
                                                           MethSummary* __restrict__ sum)
{
    __shared__ unsigned long long s_a[1024], s_b[1024];
    __shared__ unsigned long long carry_a, carry_b, carry_e;
    const int t = threadIdx.x;
    if (t == 0) { carry_a = 0; carry_b = 0; carry_e = 0; }
    __syncthreads();
    unsigned long long ev = 0;
    for (uint32_t base = 0; base < n_records; base += 1024) {
        const uint32_t r = base + t;
        const unsigned long long va = r < n_records ? counts[3 * (size_t)r] : 0ull;
        const unsigned long long vb = r < n_records ? counts[3 * (size_t)r + 1] : 0ull;
        if (r < n_records) ev += counts[3 * (size_t)r + 2];
        s_a[t] = va; s_b[t] = vb;
        __syncthreads();
        for (int dlt = 1; dlt < 1024; dlt <<= 1) {
            const unsigned long long xa = t >= dlt ? s_a[t - dlt] : 0ull, xb = t >= dlt ? s_b[t - dlt] : 0ull;
            __syncthreads();
            s_a[t] += xa; s_b[t] += xb;
            __syncthreads();
        }
        if (r < n_records) { site_off[r] = carry_a + s_a[t] - va; rank_off[r] = carry_b + s_b[t] - vb; }
        __syncthreads();
        if (t == 1023) { carry_a += s_a[1023]; carry_b += s_b[1023]; }
        __syncthreads();
    }
    // scored events: plain block reduction
    s_a[t] = ev;
    __syncthreads();
    for (int dlt = 512; dlt > 0; dlt >>= 1) { if (t < dlt) s_a[t] += s_a[t + dlt]; __syncthreads(); }
    if (t == 0) {
        carry_e = s_a[0];
        site_off[n_records] = carry_a;
        sum->n_sites = carry_a; sum->n_ranks = carry_b; sum->n_events = carry_e;
    }
}

struct EmitArgs {
    const uint8_t* ref;
    const nph_meth_record* records;
    const uint64_t* prov_off;
    const MethGroup* prov;
    const uint64_t* counts;
    const uint64_t* site_off;
    const uint64_t* rank_off;
    nph_hmm_job* jobs;
    uint32_t* ranks;
    nph_meth_site* sites;
    uint32_t n_records;
};

__global__ void __launch_bounds__(kThreads) meth_emit_kernel(const EmitArgs a, const MethDev d)
{
    // per warp: the window over the methylation alphabet as ranks, unmethylated and methylated, in the orientation the
    // job's strand reads (HMMInputSequence's m_seq for rc == 0, its m_rc_seq for rc == 1)
    __shared__ uint8_t s_u[kWarps][NPH_METH_MAX_WINDOW];
    __shared__ uint8_t s_m[kWarps][NPH_METH_MAX_WINDOW];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint8_t* const su = s_u[w];
    uint8_t* const sm = s_m[w];
    const uint32_t warp = blockIdx.x * kWarps + w;
    const uint32_t n_warps = gridDim.x * kWarps;
    const int k = (int)d.k, rl = (int)d.site_len;
    for (uint32_t rec = warp; rec < a.n_records; rec += n_warps) {
        const nph_meth_record R = a.records[rec];
        const uint8_t* ref = a.ref + R.ref_off;
        const MethGroup* grp = a.prov + a.prov_off[rec];
        const int n_groups = (int)a.counts[3 * (size_t)rec];
        const uint64_t site0 = a.site_off[rec];
        uint64_t roff = a.rank_off[rec];
        for (int g = 0; g < n_groups; ++g) {
            const MethGroup G = grp[g];
            const int sub_start = G.first - d.min_flank;
            const int L = G.win_len;
            const uint8_t* win = ref + sub_start;
            // (1) plain ranks: forward, or the base-by-base reverse complement (no methylated symbol in the unmethylated string)
            for (int j = lane; j < L; j += 32) {
                const uint8_t r = R.rc ? d.comp_rank_of[win[L - 1 - j]] : d.rank_of[win[j]];
                su[j] = r; sm[j] = r;
            }
            __syncwarp();
            // (2) Alphabet::methylate: every complete recognition site of the window becomes its methylated form.  On the
            // other strand reverse_complement emits, for a methylated site at q, the methylated complement back to front
            // at [L - q - rl, L - q).
            for (int q = lane; q + rl <= L; q += 32) {
                const int s = site_at(d, win, q, L);
                if (s >= 0) {
                    if (!R.rc) { for (int t = 0; t < rl; ++t) sm[q + t] = d.site_m_rank[s][t]; }
                    else       { for (int t = 0; t < rl; ++t) sm[L - q - rl + t] = d.site_mrc_rank[s][t]; }
                }
            }
            __syncwarp();
            // (3) k-mer ranks: job k-mer i is the k-mer at i (rc == 0) or the one at L - i - k of the other strand's string
            const int nk = L - k + 1;
            uint32_t* ru = a.ranks + roff;
            uint32_t* rm = ru + nk;
            for (int i = lane; i < nk; i += 32) {
                const int p = R.rc ? L - i - k : i;
                uint32_t vu = 0, vm = 0;
                for (int j = 0; j < k; ++j) { vu = vu * d.asize + su[p + j]; vm = vm * d.asize + sm[p + j]; }
                ru[i] = vu; rm[i] = vm;
            }
            if (lane == 0) {
                const uint64_t site = site0 + (uint64_t)g;
                nph_hmm_job jb;
                jb.rank_off = roff; jb.read = R.read; jb.model_id = R.model_id;
                jb.event_start = (uint32_t)G.e1; jb.event_stop = (uint32_t)G.e2; jb.n_kmers = (uint32_t)nk;
                jb.stride = (uint32_t)G.e1 <= (uint32_t)G.e2 ? 1 : -1;       // compared as the uint32 members of HMMInputData
                jb.rc = R.rc; jb.flags = NPH_HAF_ALLOW_PRE_CLIP | NPH_HAF_ALLOW_POST_CLIP; jb.reserved = 0;
                a.jobs[2 * site] = jb;
                jb.rank_off = roff + (uint64_t)nk;
                a.jobs[2 * site + 1] = jb;
                a.sites[site] = nph_meth_site{G.first + R.ref_start_pos, G.last + R.ref_start_pos, (uint32_t)G.n_motif, rec, 0.f, 0.f};
            }
            roff += 2ull * (uint64_t)nk;
            __syncwarp();
        }
    }
}

__global__ void meth_fill_kernel(nph_meth_site* __restrict__ sites, const float* __restrict__ scores, uint64_t n_sites)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_sites; i += (uint64_t)gridDim.x * blockDim.x) {
        sites[i].ll_unmethylated = scores[2 * i];
        sites[i].ll_methylated = scores[2 * i + 1];
    }
}

int build_dev_params(nph_ctx* ctx, const nph_meth_params& p, MethDev& d)
{
    auto bad = [&](const char* what) { ctx->last_error = std::string("nph_meth_params: ") + what; return NPH_ERR_INVALID; };
    if (p.min_separation < 0 || p.min_flank < 0 || p.max_span < 0) return bad("negative window parameter");
    if (p.k == 0 || p.k > 12) return bad("k");
    if (p.alphabet_size == 0 || p.alphabet_size > 8) return bad("alphabet_size");
    if (p.n_sites == 0 || p.n_sites > NPH_METH_MAX_SITES) return bad("n_sites");
    if (p.site_len == 0 || p.site_len >= NPH_METH_MAX_SITE_LEN) return bad("site_len");
    if ((long long)p.max_span + 2ll * p.min_flank + 1 > NPH_METH_MAX_WINDOW) {
        ctx->last_error = "max_span + 2 * min_flank + 1 exceeds NPH_METH_MAX_WINDOW";
        return NPH_ERR_UNSUPPORTED;
    }
    std::memset(&d, 0, sizeof(d));
    d.min_separation = p.min_separation; d.min_flank = p.min_flank; d.max_span = p.max_span; d.min_event_span = p.min_event_span;
    d.region_start = p.region_start; d.region_end = p.region_end;
    d.k = p.k; d.asize = p.alphabet_size; d.n_sites = p.n_sites; d.site_len = p.site_len;
    int rank_of[256];
    for (int c = 0; c < 256; ++c) rank_of[c] = -1;
    for (uint32_t i = 0; i < p.alphabet_size; ++i) {
        if (!p.bases[i] || !p.complements[i]) return bad("bases / complements shorter than alphabet_size");
        rank_of[(unsigned char)p.bases[i]] = (int)i;
    }
    for (int c = 0; c < 256; ++c) d.rank_of[c] = (uint8_t)(rank_of[c] < 0 ? 0 : rank_of[c]);
    for (int c = 0; c < 256; ++c) d.comp_rank_of[c] = d.rank_of[c];            // overwritten for the alphabet's symbols below
    for (int c = 0; c < 256; ++c) {
        // Alphabet::complement(b) = m_complement[rank(b)]: an unknown symbol has rank 0 and complements like bases[0]
        const unsigned char comp = (unsigned char)p.complements[d.rank_of[c]];
        if (rank_of[comp] < 0) return bad("a complement is not a symbol of the alphabet");
        d.comp_rank_of[c] = (uint8_t)rank_of[comp];
    }
    for (uint32_t s = 0; s < p.n_sites; ++s) {
        for (uint32_t t = 0; t < p.site_len; ++t) {
            const unsigned char c0 = (unsigned char)p.sites[s][t], c1 = (unsigned char)p.sites_methylated[s][t],
                                c2 = (unsigned char)p.sites_methylated_complement[s][p.site_len - 1 - t];
            if (!c0 || rank_of[c0] < 0 || !c1 || rank_of[c1] < 0 || !c2 || rank_of[c2] < 0) return bad("a site symbol is not in the alphabet");
            d.site[s][t] = (char)c0;
            d.site_m_rank[s][t] = (uint8_t)rank_of[c1];
            d.site_mrc_rank[s][t] = (uint8_t)rank_of[c2];
        }
        // the device replaces every occurrence independently; the reference walks left to right and steps over a matched
        // site, which is the same thing as long as a site cannot overlap another occurrence (true of cpg, gpc, dam, dcm)
        for (uint32_t s2 = 0; s2 < p.n_sites; ++s2)
            for (uint32_t sh = 1; sh < p.site_len; ++sh)
                if (std::memcmp(p.sites[s] + sh, p.sites[s2], p.site_len - sh) == 0) {
                    ctx->last_error = "recognition sites that can overlap each other are not supported";
                    return NPH_ERR_UNSUPPORTED;
                }
    }
    return NPH_OK;
}

} // namespace

// event alignments either as pair lists (aligned_events) or in compact form (event_deltas + first_event)
static int meth_load(nph_ctx* ctx, const char* ref_bases, size_t n_ref_total,
                     const nph_aligned_pair* aligned_events, size_t n_pairs_total,
                     const int16_t* event_deltas, const int32_t* first_event,
                     const nph_meth_record* records, size_t n_records,
                     const nph_meth_params* params, double indel_bias)
{
    if (!ctx || !params) return NPH_ERR_INVALID;
    nph_ctx::MethState& m = ctx->meth;
    m.loaded = false; m.ran = false;
    const bool compact = event_deltas != nullptr;
    if (n_records == 0) { m.n_records = 0; m.loaded = true; return NPH_OK; }
    if (!ref_bases || !records || (!compact && !aligned_events && n_pairs_total) || (compact && !first_event)) return NPH_ERR_INVALID;
    if (!ctx->reads_loaded) return NPH_ERR_STATE;
    MethDev d;
    NPH_TRY(build_dev_params(ctx, *params, d));
    // O(records) validation and the provisional layout: a record has at most ref_len / (min_separation + 1) + 1 groups
    // (consecutive groups start more than min_separation bases apart)
    std::vector<uint64_t>& po = m.h_prov_off;
    po.resize(n_records + 1);
    uint64_t prov = 0;
    for (size_t r = 0; r < n_records; ++r) {
        const nph_meth_record& R = records[r];
        const bool ok = R.read < ctx->n_reads && R.model_id < ctx->models.size() && R.ref_len <= n_ref_total && R.ref_off <= n_ref_total - R.ref_len &&
                        R.ref_len <= 0x7fffffffu && (compact || (R.n_pairs <= n_pairs_total && R.pair_off <= n_pairs_total - R.n_pairs));
        if (!ok) { ctx->last_error = "methylation record " + std::to_string(r) + " is out of range (read, model, reference or event-alignment slice)"; return NPH_ERR_INVALID; }
        const DevModel& mod = ctx->models[R.model_id];
        if (mod.k != params->k || mod.alphabet_size != params->alphabet_size) {
            ctx->last_error = "methylation record " + std::to_string(r) + ": its model's k / alphabet differ from nph_meth_params";
            return NPH_ERR_INVALID;
        }
        po[r] = prov;
        prov += (uint64_t)R.ref_len / (uint64_t)(params->min_separation + 1) + 2;
    }
    po[n_records] = prov;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    NPH_TRY(nph_reserve(ctx, m.d_ref, n_ref_total + 16));
    if (compact) {
        NPH_TRY(nph_reserve(ctx, m.d_deltas, n_ref_total + 16));
        NPH_TRY(nph_reserve(ctx, m.d_dense, n_ref_total + 2 * n_records + 16));
    } else {
        NPH_TRY(nph_reserve(ctx, m.d_pairs, n_pairs_total + 1));
    }
    NPH_TRY(nph_reserve(ctx, m.d_records, n_records));
    NPH_TRY(nph_reserve(ctx, m.d_prov_off, n_records + 1));
    NPH_TRY(nph_reserve(ctx, m.d_prov, (size_t)prov * sizeof(MethGroup)));
    // counts (3 per record) | site_off (n + 1) | rank_off (n) | summary
    NPH_TRY(nph_reserve(ctx, m.d_counts, 5 * n_records + 1 + (sizeof(MethSummary) + 7) / 8 + 8));
    NPH_CUDA(ctx, cudaMemcpyAsync(m.d_records.p, records, sizeof(nph_meth_record) * n_records, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(m.d_prov_off.p, po.data(), sizeof(uint64_t) * (n_records + 1), cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(m.d_ref.p, ref_bases, n_ref_total, cudaMemcpyHostToDevice, ctx->stream));
    if (compact) {
        // first_event goes behind the dense array: [n_ref] event indices | [n_records] first_event | [n_records] first valid offset
        NPH_CUDA(ctx, cudaMemcpyAsync(m.d_deltas.p, event_deltas, sizeof(int16_t) * n_ref_total, cudaMemcpyHostToDevice, ctx->stream));
        NPH_CUDA(ctx, cudaMemcpyAsync(m.d_dense.p + n_ref_total, first_event, sizeof(int32_t) * n_records, cudaMemcpyHostToDevice, ctx->stream));
    } else if (n_pairs_total) {
        NPH_CUDA(ctx, cudaMemcpyAsync(m.d_pairs.p, aligned_events, sizeof(nph_aligned_pair) * n_pairs_total, cudaMemcpyHostToDevice, ctx->stream));
    }
    m.compact = compact;
    m.n_records = n_records; m.n_ref = n_ref_total; m.n_pairs = compact ? 0 : n_pairs_total; m.prov_total = (size_t)prov;
    m.params = *params; m.indel_bias = indel_bias;
    m.loaded = true;
    return NPH_OK;
}

int nph_expand_event_maps(nph_ctx* ctx, const int16_t* d_deltas, const int32_t* d_first_event, const nph_meth_record* d_records, uint32_t n_records,
                          int32_t* d_dense, int32_t* d_first_valid)
{
    if (n_records == 0) return NPH_OK;
    const int grid = (int)std::min<size_t>(((size_t)n_records + kWarps - 1) / kWarps, (size_t)ctx->sm_count * 8);
    meth_expand_kernel<<<grid, kThreads, 0, ctx->stream>>>(d_deltas, d_first_event, d_records, n_records, d_dense, d_first_valid);
    NPH_CUDA(ctx, cudaGetLastError());
    return NPH_OK;
}

extern "C" int nph_methylation_load(nph_ctx* ctx, const char* ref_bases, size_t n_ref_total,
                                    const nph_aligned_pair* aligned_events, size_t n_pairs_total,
                                    const nph_meth_record* records, size_t n_records,
                                    const nph_meth_params* params, double indel_bias)
{
    return meth_load(ctx, ref_bases, n_ref_total, aligned_events, n_pairs_total, nullptr, nullptr, records, n_records, params, indel_bias);
}

extern "C" int nph_methylation_load_compact(nph_ctx* ctx, const char* ref_bases, const int16_t* event_deltas, size_t n_ref_total,
                                            const int32_t* first_event, const nph_meth_record* records, size_t n_records,
                                            const nph_meth_params* params, double indel_bias)
{
    if (n_records && !event_deltas) return NPH_ERR_INVALID;
    return meth_load(ctx, ref_bases, n_ref_total, nullptr, 0, event_deltas, first_event, records, n_records, params, indel_bias);
}

extern "C" int nph_methylation_run(nph_ctx* ctx)
{
    if (!ctx) return NPH_ERR_INVALID;
    nph_ctx::MethState& m = ctx->meth;
    if (!m.loaded) return NPH_ERR_STATE;
    m.ran = false;
    m.n_sites = m.n_ranks = m.n_scored_events = 0;
    if (m.n_records == 0) { m.ran = true; return NPH_OK; }
    if (!ctx->reads_loaded) return NPH_ERR_STATE;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    MethDev d;
    NPH_TRY(build_dev_params(ctx, m.params, d));
    const uint32_t n = (uint32_t)m.n_records;
    uint64_t* counts = m.d_counts.p;
    uint64_t* site_off = counts + 3 * (size_t)n;
    uint64_t* rank_off = site_off + n + 1;
    MethSummary* d_sum = reinterpret_cast<MethSummary*>(rank_off + n);
    NPH_CUDA(ctx, cudaMemsetAsync(d_sum, 0, sizeof(MethSummary), ctx->stream));
    const int grid = (int)std::min<size_t>((m.n_records + kWarps - 1) / kWarps, (size_t)ctx->sm_count * 8);
    int32_t* dense = nullptr;
    int32_t* first_valid = nullptr;
    if (m.compact) {
        dense = reinterpret_cast<int32_t*>(m.d_dense.p);
        const int32_t* d_first_event = dense + m.n_ref;
        first_valid = dense + m.n_ref + m.n_records;
        meth_expand_kernel<<<grid, kThreads, 0, ctx->stream>>>(reinterpret_cast<const int16_t*>(m.d_deltas.p), d_first_event, m.d_records.p, n, dense, first_valid);
        NPH_CUDA(ctx, cudaGetLastError());
    }
    ScanArgs sa{m.d_ref.p, dense, first_valid, m.compact ? nullptr : m.d_pairs.p, m.d_records.p, m.d_prov_off.p,
                reinterpret_cast<MethGroup*>(m.d_prov.p), counts, d_sum, n};
    meth_scan_kernel<<<grid, kThreads, 0, ctx->stream>>>(sa, d);
    NPH_CUDA(ctx, cudaGetLastError());
    meth_prefix_kernel<<<1, 1024, 0, ctx->stream>>>(counts, n, site_off, rank_off, d_sum);
    NPH_CUDA(ctx, cudaGetLastError());
    MethSummary h{};
    NPH_CUDA(ctx, cudaMemcpyAsync(&h, d_sum, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));          // read-back 1 of 2: the counts that size the job arrays
    if (h.error) {
        ctx->last_error = "methylation record " + std::to_string(h.error - 1) + ": a window cut by the end of the reference is shorter than k";
        return NPH_ERR_INVALID;
    }
    m.n_sites = h.n_sites; m.n_ranks = h.n_ranks; m.n_scored_events = h.n_events;
    const size_t n_jobs = 2 * (size_t)h.n_sites;
    ctx->n_jobs = 0; ctx->jobs_loaded = false; ctx->codes_mode = false;       // the enumerator emits k-mer ranks
    if (n_jobs == 0) { ctx->classes.clear(); ctx->jobs_loaded = true; m.ran = true; return NPH_OK; }
    NPH_TRY(nph_reserve(ctx, ctx->d_ranks, (size_t)h.n_ranks));
    NPH_TRY(nph_reserve(ctx, ctx->d_jobs, n_jobs));
    NPH_TRY(nph_reserve(ctx, ctx->d_order, n_jobs));
    NPH_TRY(nph_reserve(ctx, ctx->d_scores, n_jobs));
    NPH_TRY(nph_reserve(ctx, m.d_sites, (size_t)h.n_sites));
    NPH_TRY(nph_upload_read_transitions(ctx, m.indel_bias));
    EmitArgs ea{m.d_ref.p, m.d_records.p, m.d_prov_off.p, reinterpret_cast<const MethGroup*>(m.d_prov.p), counts, site_off, rank_off,
                ctx->d_jobs.p, ctx->d_ranks.p, m.d_sites.p, n};
    meth_emit_kernel<<<grid, kThreads, 0, ctx->stream>>>(ea, d);
    NPH_CUDA(ctx, cudaGetLastError());
    ctx->jobs_trusted = true;                                     // meth_emit_kernel wrote these ranks: the scheduler need not walk them
    const int rc_sched = nph_jobs_schedule(ctx, n_jobs, (size_t)h.n_ranks);   // read-back 2 of 2: validation + schedule summary
    ctx->jobs_trusted = false;
    NPH_TRY(rc_sched);
    NPH_TRY(nph_launch_hmm_forward(ctx, nullptr));
    const int fgrid = (int)std::min<size_t>(((size_t)h.n_sites + 255) / 256, (size_t)ctx->sm_count * 8);
    meth_fill_kernel<<<fgrid, 256, 0, ctx->stream>>>(m.d_sites.p, ctx->d_scores.p, h.n_sites);
    NPH_CUDA(ctx, cudaGetLastError());
    ctx->last_launches += 6;                                     // scan, prefix, emit, classify/scan/scatter are counted with the forward classes' launches: 3 + 3
    m.ran = true;
    return NPH_OK;
}

// ---- methylation_calls.tsv on the device -------------------------------------------------------------------------
// One row per site record of a record that is its read's only scored strand (1D reads: every read of a call-methylation
// run today), the fields of the reference's writer (src/nanopolish_call_methylation.cpp:113-140 and the ScoredSite it
// prints, basemods.cpp:403-425): chromosome, strand, start, end, read_name, log_lik_ratio, log_lik_methylated,
// log_lik_unmethylated ("%.2lf" of the strand sums; the other strand's entries stay 0), num_calling_strands (1),
// num_motifs, sequence (the group with k - 1 bases of context before it and k after it, cut at the end of the record's
// reference).  The host's part of call-methylation was the formatting of these rows (6-9 ms per 10 000 reads on the box's
// 16-CPU quota, as long as the PCIe transfer); here a warp formats a record's rows straight from the site records.
namespace {

struct TsvArgs {
    const nph_meth_site* sites;
    const uint64_t* site_off;          // n_records + 1
    const nph_meth_record* records;
    const uint8_t* ref;
    const char* contig; uint32_t contig_len;
    const char* names; const uint32_t* name_off;       // n_records + 1
    const uint8_t* is_reverse;
    uint32_t k, n_records;
    uint64_t* rec_bytes;               // per record: bytes of its rows (len pass), then exclusive prefix in rec_off
    const uint64_t* rec_off;
    char* out;
    int* refused;                      // set when a value needs the C library (non-finite, |v| >= 2^52)
};

struct RowNums { nph_tsv::Fixed2 diff, m, u; uint32_t seq_b, seq_len; bool seq_ok; };

__device__ __forceinline__ RowNums row_numbers(const nph_meth_site& ms, const nph_meth_record& R, uint32_t k)
{
    RowNums r;
    // ScoredSite: ll_*[strand] = the float score, the other strand 0.0; the writer sums the two strands in double
    const double sum_m = __dadd_rn((double)ms.ll_methylated, 0.0), sum_u = __dadd_rn((double)ms.ll_unmethylated, 0.0);
    r.diff = nph_tsv::fixed2_of(__dsub_rn(sum_m, sum_u));
    r.m = nph_tsv::fixed2_of(sum_m);
    r.u = nph_tsv::fixed2_of(sum_u);
    // the sequence column starts k - 1 bases before the first site: a window parameter set that lets a group start closer to the
    // beginning of the record's reference than that makes the reference's substr throw; here the call is refused
    const int bs = (ms.start_position - R.ref_start_pos) - (int)k + 1;
    const uint32_t e = min((uint32_t)(ms.end_position - R.ref_start_pos) + k, R.ref_len);
    r.seq_ok = bs >= 0 && (uint32_t)bs <= e;
    r.seq_b = r.seq_ok ? (uint32_t)bs : 0u; r.seq_len = r.seq_ok ? e - (uint32_t)bs : 0u;
    return r;
}

__device__ __forceinline__ uint32_t row_len(const TsvArgs& a, const nph_meth_site& ms, const RowNums& r, uint32_t name_len)
{
    return a.contig_len + 3u + (uint32_t)nph_tsv::int_len(ms.start_position) + 1u + (uint32_t)nph_tsv::int_len(ms.end_position) + 1u + name_len + 1u +
           (uint32_t)nph_tsv::fixed2_len(r.diff) + 1u + (uint32_t)nph_tsv::fixed2_len(r.m) + 1u + (uint32_t)nph_tsv::fixed2_len(r.u) + 1u + 2u +
           (uint32_t)nph_tsv::ndigits(ms.n_motif) + 1u + r.seq_len + 1u;
}

// pass 1 (WRITE = false): bytes per record; pass 2 (WRITE = true): the rows at rec_off[record]
template <bool WRITE>
__global__ void __launch_bounds__(kThreads) meth_tsv_kernel(const TsvArgs a)
{
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * kWarps + (threadIdx.x >> 5);
    const uint32_t n_warps = gridDim.x * kWarps;
    for (uint32_t rec = warp; rec < a.n_records; rec += n_warps) {
        const uint64_t s0 = a.site_off[rec], s1 = a.site_off[rec + 1];
        if (s0 == s1) { if (!WRITE && lane == 0) a.rec_bytes[rec] = 0; continue; }
        const nph_meth_record R = a.records[rec];
        const uint32_t nb = a.name_off[rec], name_len = a.name_off[rec + 1] - nb;
        unsigned long long run = WRITE ? a.rec_off[rec] : 0ull;        // WRITE: where the next chunk of rows starts
        for (uint64_t base = s0; base < s1; base += 32) {
            const uint64_t s = base + lane;
            const bool have = s < s1;
            nph_meth_site ms{};
            RowNums r{};
            uint32_t len = 0;
            if (have) {
                ms = a.sites[s];
                r = row_numbers(ms, R, a.k);
                if (!(r.diff.ok && r.m.ok && r.u.ok)) atomicMax(a.refused, 1);
                if (!r.seq_ok) atomicMax(a.refused, 2);
                len = row_len(a, ms, r, name_len);
            }
            uint32_t incl = len;
            for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(kFull, incl, o); if (lane >= o) incl += v; }
            if (WRITE && have) {
                char* o = a.out + run + (incl - len);
                for (uint32_t i = 0; i < a.contig_len; ++i) *o++ = a.contig[i];
                *o++ = '\t'; *o++ = a.is_reverse[rec] ? '-' : '+'; *o++ = '\t';
                o = nph_tsv::put_int(o, ms.start_position); *o++ = '\t';
                o = nph_tsv::put_int(o, ms.end_position); *o++ = '\t';
                for (uint32_t i = 0; i < name_len; ++i) *o++ = a.names[nb + i];
                *o++ = '\t';
                o = nph_tsv::put_fixed2(o, r.diff); *o++ = '\t';
                o = nph_tsv::put_fixed2(o, r.m); *o++ = '\t';
                o = nph_tsv::put_fixed2(o, r.u); *o++ = '\t';
                *o++ = '1'; *o++ = '\t';
                o = nph_tsv::put_u64(o, ms.n_motif); *o++ = '\t';
                const uint8_t* sq = a.ref + R.ref_off + r.seq_b;
                for (uint32_t i = 0; i < r.seq_len; ++i) *o++ = (char)sq[i];
                *o++ = '\n';
            }
            run += __shfl_sync(kFull, incl, 31);
        }
        if (!WRITE && lane == 0) a.rec_bytes[rec] = run;
    }
}

// exclusive prefix of the per-record byte counts (one block; n + 1 entries out)
__global__ void __launch_bounds__(1024) meth_tsv_prefix_kernel(const uint64_t* __restrict__ bytes, uint32_t n, uint64_t* __restrict__ off)
{
    __shared__ unsigned long long s_a[1024];
    __shared__ unsigned long long carry;
    const int t = threadIdx.x;
    if (t == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t r = base + t;
        const unsigned long long v = r < n ? bytes[r] : 0ull;
        s_a[t] = v;
        __syncthreads();
        for (int dlt = 1; dlt < 1024; dlt <<= 1) {
            const unsigned long long x = t >= dlt ? s_a[t - dlt] : 0ull;
            __syncthreads();
            s_a[t] += x;
            __syncthreads();
        }
        if (r < n) off[r] = carry + s_a[t] - v;
        __syncthreads();
        if (t == 1023) carry += s_a[1023];
        __syncthreads();
    }
    if (t == 0) off[n] = carry;
}

} // namespace

extern "C" int nph_methylation_tsv(nph_ctx* ctx, const char* contig, const char* read_names, const uint32_t* name_off,
                                   const uint8_t* is_reverse, char* tsv_out, size_t cap, uint64_t* n_bytes_out)
{
    if (!ctx || !n_bytes_out) return NPH_ERR_INVALID;
    nph_ctx::MethState& m = ctx->meth;
    if (!m.ran) return NPH_ERR_STATE;
    *n_bytes_out = 0;
    if (m.n_records == 0 || m.n_sites == 0) return NPH_OK;
    if (!contig || !read_names || !name_off || !is_reverse) return NPH_ERR_INVALID;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = m.n_records, contig_len = std::strlen(contig), names_len = name_off[n];
    for (size_t r = 0; r < n; ++r) if (name_off[r] > name_off[r + 1]) { ctx->last_error = "name_off must ascend"; return NPH_ERR_INVALID; }
    // one staging block: contig | names | name offsets | strand flags
    struct { char *contig, *names; uint32_t* noff; uint8_t* rev; } d{};
    auto layout = [&](NphCarve& a) {
        d.contig = a.take<char>(contig_len + 1);
        d.names = a.take<char>(names_len + 1);
        d.noff = a.take<uint32_t>(n + 1);
        d.rev = a.take<uint8_t>(n);
    };
    NPH_TRY(nph_lay_out(ctx, m.d_tsv_in, layout));
    NPH_TRY(nph_reserve(ctx, m.d_tsv_off, 2 * n + 4));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.contig, contig, contig_len, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.names, read_names, names_len, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.noff, name_off, sizeof(uint32_t) * (n + 1), cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.rev, is_reverse, n, cudaMemcpyHostToDevice, ctx->stream));
    uint64_t* rec_bytes = m.d_tsv_off.p;
    uint64_t* rec_off = rec_bytes + n;                                  // n + 1 entries
    int* d_refused = reinterpret_cast<int*>(rec_off + n + 1);
    NPH_CUDA(ctx, cudaMemsetAsync(d_refused, 0, sizeof(int), ctx->stream));
    TsvArgs a{m.d_sites.p, m.d_counts.p + 3 * n, m.d_records.p, m.d_ref.p, d.contig, (uint32_t)contig_len,
              d.names, d.noff, d.rev, m.params.k, (uint32_t)n,
              rec_bytes, rec_off, nullptr, d_refused};
    const int grid = (int)std::min<size_t>((n + kWarps - 1) / kWarps, (size_t)ctx->sm_count * 8);
    meth_tsv_kernel<false><<<grid, kThreads, 0, ctx->stream>>>(a);
    NPH_CUDA(ctx, cudaGetLastError());
    meth_tsv_prefix_kernel<<<1, 1024, 0, ctx->stream>>>(rec_bytes, (uint32_t)n, rec_off);
    NPH_CUDA(ctx, cudaGetLastError());
    uint64_t total = 0;
    int refused = 0;
    NPH_CUDA(ctx, cudaMemcpyAsync(&total, rec_off + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(&refused, d_refused, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (refused == 2) {
        ctx->last_error = "a group starts fewer than k - 1 bases into its record's reference: the sequence column of its row is undefined (min_flank too small for k)";
        return NPH_ERR_INVALID;
    }
    if (refused) {
        ctx->last_error = "a log-likelihood is not finite or beyond 2^52: these rows need the C library's formatting (nph_methylation_fetch + host formatter)";
        return NPH_ERR_UNSUPPORTED;
    }
    *n_bytes_out = total;
    if (total > cap || !tsv_out) {
        ctx->last_error = "tsv_out too small: " + std::to_string(total) + " bytes";
        return NPH_ERR_INVALID;
    }
    NPH_TRY(nph_reserve(ctx, m.d_tsv, (size_t)total));
    a.out = reinterpret_cast<char*>(m.d_tsv.p);
    meth_tsv_kernel<true><<<grid, kThreads, 0, ctx->stream>>>(a);
    NPH_CUDA(ctx, cudaGetLastError());
    NPH_CUDA(ctx, cudaMemcpyAsync(tsv_out, m.d_tsv.p, (size_t)total, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->last_launches += 3;
    return NPH_OK;
}

extern "C" int nph_methylation_counts(nph_ctx* ctx, uint64_t* n_sites_out, uint64_t* n_jobs_out, uint64_t* n_scored_events_out)
{
    if (!ctx) return NPH_ERR_INVALID;
    if (!ctx->meth.ran) return NPH_ERR_STATE;
    if (n_sites_out) *n_sites_out = ctx->meth.n_sites;
    if (n_jobs_out) *n_jobs_out = 2 * ctx->meth.n_sites;
    if (n_scored_events_out) *n_scored_events_out = ctx->meth.n_scored_events;
    return NPH_OK;
}

extern "C" int nph_methylation_sites_dev(nph_ctx* ctx, const nph_meth_site** sites_dev_out, uint64_t* n_sites_out)
{
    if (!ctx || !sites_dev_out || !n_sites_out) return NPH_ERR_INVALID;
    if (!ctx->meth.ran) return NPH_ERR_STATE;
    *sites_dev_out = ctx->meth.n_sites ? ctx->meth.d_sites.p : nullptr;
    *n_sites_out = ctx->meth.n_sites;
    return NPH_OK;
}

extern "C" int nph_methylation_fetch(nph_ctx* ctx, uint64_t* site_off_out, nph_meth_site* sites_out, size_t sites_cap)
{
    if (!ctx || !site_off_out) return NPH_ERR_INVALID;
    nph_ctx::MethState& m = ctx->meth;
    if (!m.ran) return NPH_ERR_STATE;
    if (m.n_records == 0) { site_off_out[0] = 0; return NPH_OK; }
    if (m.n_sites > sites_cap) {
        ctx->last_error = "sites_cap too small: " + std::to_string(m.n_sites) + " site records";
        return NPH_ERR_INVALID;
    }
    if (m.n_sites && !sites_out) return NPH_ERR_INVALID;
    const uint64_t* site_off = m.d_counts.p + 3 * m.n_records;
    NPH_CUDA(ctx, cudaMemcpyAsync(site_off_out, site_off, sizeof(uint64_t) * (m.n_records + 1), cudaMemcpyDeviceToHost, ctx->stream));
    if (m.n_sites)
        NPH_CUDA(ctx, cudaMemcpyAsync(sites_out, m.d_sites.p, sizeof(nph_meth_site) * (size_t)m.n_sites, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NPH_OK;
}

extern "C" int nph_methylation_batch_compact(nph_ctx* ctx,
                                             const nph_read* reads, size_t n_reads,
                                             const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                                             const char* ref_bases, const int16_t* event_deltas, size_t n_ref_total,
                                             const int32_t* first_event,
                                             const nph_meth_record* records, size_t n_records,
                                             const nph_meth_params* params, double indel_bias,
                                             uint64_t* site_off_out, nph_meth_site* sites_out, size_t sites_cap,
                                             uint64_t* n_scored_events_out)
{
    if (!ctx || !site_off_out) return NPH_ERR_INVALID;
    if (n_records == 0) { site_off_out[0] = 0; if (n_scored_events_out) *n_scored_events_out = 0; return NPH_OK; }
    ctx->levels_inflight = false;
    int rc = nph_reads_load_impl(ctx, reads, n_reads, ev_mean, ev_start_time, n_events_total, true);
    if (rc == NPH_OK) { ctx->reads_loaded = true; ctx->jobs_loaded = false; ctx->abea_loaded = false; }
    if (rc == NPH_OK) rc = nph_methylation_load_compact(ctx, ref_bases, event_deltas, n_ref_total, first_event, records, n_records, params, indel_bias);
    if (rc == NPH_OK && ctx->levels_inflight) rc = nph_upload_level_chunks(ctx, ev_mean);
    if (rc == NPH_OK) rc = nph_methylation_run(ctx);
    if (rc == NPH_OK) rc = nph_methylation_fetch(ctx, site_off_out, sites_out, sites_cap);
    nph_finish_level_upload(ctx);
    if (rc == NPH_OK && n_scored_events_out) *n_scored_events_out = ctx->meth.n_scored_events;
    return rc;
}

extern "C" int nph_methylation_batch_compact_tsv(nph_ctx* ctx,
                                                 const nph_read* reads, size_t n_reads,
                                                 const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                                                 const char* ref_bases, const int16_t* event_deltas, size_t n_ref_total,
                                                 const int32_t* first_event,
                                                 const nph_meth_record* records, size_t n_records,
                                                 const nph_meth_params* params, double indel_bias,
                                                 const char* contig, const char* read_names, const uint32_t* name_off, const uint8_t* is_reverse,
                                                 char* tsv_out, size_t cap, uint64_t* n_bytes_out,
                                                 uint64_t* n_sites_out, uint64_t* n_scored_events_out)
{
    if (!ctx || !n_bytes_out) return NPH_ERR_INVALID;
    *n_bytes_out = 0;
    if (n_sites_out) *n_sites_out = 0;
    if (n_scored_events_out) *n_scored_events_out = 0;
    if (n_records == 0) return NPH_OK;
    ctx->levels_inflight = false;
    int rc = nph_reads_load_impl(ctx, reads, n_reads, ev_mean, ev_start_time, n_events_total, true);
    if (rc == NPH_OK) { ctx->reads_loaded = true; ctx->jobs_loaded = false; ctx->abea_loaded = false; }
    if (rc == NPH_OK) rc = nph_methylation_load_compact(ctx, ref_bases, event_deltas, n_ref_total, first_event, records, n_records, params, indel_bias);
    if (rc == NPH_OK && ctx->levels_inflight) rc = nph_upload_level_chunks(ctx, ev_mean);
    if (rc == NPH_OK) rc = nph_methylation_run(ctx);
    if (rc == NPH_OK) rc = nph_methylation_tsv(ctx, contig, read_names, name_off, is_reverse, tsv_out, cap, n_bytes_out);
    nph_finish_level_upload(ctx);
    if (n_sites_out) *n_sites_out = ctx->meth.n_sites;
    if (n_scored_events_out) *n_scored_events_out = ctx->meth.n_scored_events;
    return rc;
}

extern "C" int nph_methylation_batch(nph_ctx* ctx,
                                     const nph_read* reads, size_t n_reads,
                                     const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                                     const char* ref_bases, size_t n_ref_total,
                                     const nph_aligned_pair* aligned_events, size_t n_pairs_total,
                                     const nph_meth_record* records, size_t n_records,
                                     const nph_meth_params* params, double indel_bias,
                                     uint64_t* site_off_out, nph_meth_site* sites_out, size_t sites_cap,
                                     uint64_t* n_scored_events_out)
{
    if (!ctx || !site_off_out) return NPH_ERR_INVALID;
    if (n_records == 0) { site_off_out[0] = 0; if (n_scored_events_out) *n_scored_events_out = 0; return NPH_OK; }
    // Order of issue: read records first (small), then the reference bases / event alignments / records the enumeration
    // needs, then the event levels in chunks on the copy stream — the enumeration and the scheduler run while the levels
    // are still crossing PCIe, and the forward kernels wait per job on the chunk that holds their read.
    ctx->levels_inflight = false;
    int rc = nph_reads_load_impl(ctx, reads, n_reads, ev_mean, ev_start_time, n_events_total, true);
    if (rc == NPH_OK) { ctx->reads_loaded = true; ctx->jobs_loaded = false; ctx->abea_loaded = false; }
    if (rc == NPH_OK) rc = nph_methylation_load(ctx, ref_bases, n_ref_total, aligned_events, n_pairs_total, records, n_records, params, indel_bias);
    if (rc == NPH_OK && ctx->levels_inflight) rc = nph_upload_level_chunks(ctx, ev_mean);
    if (rc == NPH_OK) rc = nph_methylation_run(ctx);
    if (rc == NPH_OK) rc = nph_methylation_fetch(ctx, site_off_out, sites_out, sites_cap);
    nph_finish_level_upload(ctx);
    if (rc == NPH_OK && n_scored_events_out) *n_scored_events_out = ctx->meth.n_scored_events;
    return rc;
}
