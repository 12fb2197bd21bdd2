// eventalign_chain.cu — K4: a read's whole eventalign segment chain on the device (SURVEY.md section 8f, row N1).
//
// Replaces, for a batch of (read strand, BAM segment) chains, the per-segment loop body of
//   align_read_to_ref                          ref: src/alignment/nanopolish_eventalign.cpp:654-823
// with its helpers
//   get_end_pair                               ref: src/alignment/nanopolish_eventalign.cpp:196-207
//   SquiggleRead::get_closest_event_to         ref: src/nanopolish_squiggle_read.cpp:160-186
//   SquiggleRead::flip_k_strand                ref: src/nanopolish_squiggle_read.h:229-233
//   profile_hmm_align                          (viterbi_align, hmm_viterbi_kernel.cuh)
//
// The reference's loop is sequential per read: every window starts at the event where the previous window's output
// stopped.  Driving it from the host costs one launch and one round trip per window (≈ E/55 per read).  Here one
// warp owns one chain from its first window to its last: the cursor lives in registers, the window's k-mer ranks are
// read straight out of a per-record rank table of the reference (no per-window sequence is ever built), the Viterbi
// fill/backtrack is the same warp-level function the batch kernel uses, and the emission loop (≤ 50 event alignments
// per window, all of them in the last section) appends 12-byte records.  A batch of reads is ONE launch; chains are
// handed out longest first through an atomic counter to persistent CTAs (one per SM).
#include "hmm_viterbi_kernel.cuh"
#include <algorithm>
#include <vector>

namespace {

using namespace nph_vit;

constexpr int kWarps = 16;
constexpr int kThreads = kWarps * 32;
constexpr int kAlignStride = 100;    // reference bases per window (eventalign.cpp:666)
constexpr int kOutputStride = 50;    // event alignments emitted per window unless it is the last section (:667)

struct ChainParams {
    const float* level;
    const DevRead* reads;
    const float2* trans;
    const DevModelView* models;
    const float* flank;
    const nph_aligned_pair* pairs;
    const int32_t* map_start;
    const uint32_t* ranks_fwd;
    const uint32_t* ranks_rc;
    const nph_ea_chain* chains;
    const uint32_t* order;
    uint32_t n_chains;
    unsigned int* counter;
    nph_ea_record* records;
    nph_ea_result* results;
    float4* scratch_params;          // 32*C per warp
    uint16_t* scratch_trace;         // trace_stride per warp
    nph_align_state* scratch_states; // states_stride per warp
    uint64_t trace_stride;
    uint32_t states_stride;
    int e_cap;                       // most events a window may span
    HmmConsts c;
};

// get_end_pair: index of the pair with the highest ref_pos not above ref_pos_max, searching from pair_idx; the warp
// looks at 32 pairs at a time
__device__ __forceinline__ int warp_get_end_pair(const nph_aligned_pair* pairs, int n_pairs, int ref_pos_max, int pair_idx, int lane)
{
    for (int base = pair_idx < 0 ? 0 : pair_idx; base < n_pairs; base += 32) {
        const int idx = base + lane;
        const bool above = idx < n_pairs && pairs[idx].ref_pos > ref_pos_max;
        const unsigned m = __ballot_sync(kFull, above);
        if (m) return base + __ffs(m) - 2;
    }
    return n_pairs - 1;
}

// get_next_event / get_closest_event_to: the first event of the nearest k-mer that has one, looking backwards first
// (stop index excluded, like the reference).  Uniform across the warp: every lane walks the same few entries.
__device__ __forceinline__ int next_event(const int32_t* map, int start, int stop, int stride)
{
    for (; start != stop; start += stride) {
        const int ei = map[start];
        if (ei != -1) return ei;
    }
    return -1;
}
__device__ __forceinline__ int closest_event(const int32_t* map, int map_len, int k_idx)
{
    const int stop_before = max(0, k_idx - 1000);
    const int stop_after = min(k_idx + 1000, map_len - 1);
    const int before = next_event(map, k_idx, stop_before, -1);
    const int after = next_event(map, k_idx, stop_after, 1);
    return before == -1 ? after : before;
}

template <int C>
__global__ void __launch_bounds__(kThreads, 1) eventalign_chain_kernel(const ChainParams p)
{
    constexpr int STRIP = 32 * C;
    const int lane = threadIdx.x & 31;
    const int warp_global = blockIdx.x * kWarps + (threadIdx.x >> 5);
    __shared__ uint16_t s_tile[kWarps][32 * 32];
    VitScratch sc;
    sc.tile = s_tile[threadIdx.x >> 5];
    sc.params = p.scratch_params + (size_t)warp_global * STRIP;
    sc.edge_m = nullptr; sc.edge_b = nullptr; sc.edge_k = nullptr;       // single strip: never touched
    sc.trace = p.scratch_trace + (size_t)warp_global * p.trace_stride;
    nph_align_state* const states = p.scratch_states + (size_t)warp_global * p.states_stride;

    for (;;) {
        uint32_t slot = 0;
        if (lane == 0) slot = atomicAdd(p.counter, 1u);
        slot = __shfl_sync(kFull, slot, 0);
        if (slot >= p.n_chains) break;
        const uint32_t chain_idx = p.order[slot];
        const nph_ea_chain ch = p.chains[chain_idx];
        const nph_aligned_pair* pairs = p.pairs + ch.pair_off;
        const int n_pairs = (int)ch.n_pairs;
        const int32_t* map = p.map_start + ch.map_off;
        const int map_len = (int)ch.map_len;
        const uint32_t* rank_base = (ch.rc ? p.ranks_rc : p.ranks_fwd) + ch.rank_off;
        nph_ea_record* const rec = p.records + ch.out_off;
        const int k = (int)ch.k;

        VitJob j;
        j.rd = p.reads[ch.read];
        j.tr = p.trans[ch.read];
        j.mv = p.models[ch.model_id];
        j.lv = p.level + j.rd.event_off;
        j.pre_clip = false;                                  // align_read_to_ref calls profile_hmm_align with flags 0

        const int last_event = ch.last_event;
        const bool forward = ch.first_event < last_event;
        int curr_start_event = ch.first_event;
        int curr_start_ref = n_pairs > 0 ? pairs[0].ref_pos : 0;
        int curr_pair_idx = 0;
        uint32_t n_rec = 0, n_windows = 0;
        int status = NPH_EA_OK;

        while (n_pairs > 0 && ((forward && curr_start_event < last_event) || (!forward && curr_start_event > last_event))) {
            // the aligned pair approximately kAlignStride reference bases ahead
            const int end_pair_idx = warp_get_end_pair(pairs, n_pairs, curr_start_ref + kAlignStride, curr_pair_idx, lane);
            if (end_pair_idx < 0) break;                     // (the reference would index aligned_pairs[-1])
            const nph_aligned_pair end_pair = pairs[end_pair_idx];
            const int curr_end_ref = end_pair.ref_pos;
            int curr_end_read = end_pair.read_pos;
            if (ch.do_base_rc) curr_end_read = (int)ch.read_seq_len - curr_end_read - k;
            const int s = curr_start_ref - ch.ref_offset;
            const int l = curr_end_ref - curr_start_ref + 1;
            if (curr_end_read < 0 || curr_end_read >= map_len || s < 0 || l < 0 || s + l > (int)ch.ref_len) break;   // (substr / map access out of range)
            if (l < 2 * k) break;                            // require a minimum amount of sequence to align to
            const int event_stop = closest_event(map, map_len, curr_end_read);
            if (event_stop < 0 || curr_start_event < 0) break;
            const int span = curr_start_event > event_stop ? curr_start_event - event_stop : event_stop - curr_start_event;
            if (span < 2) break;                             // very few alignable events (large deletions)
            const int stride = curr_start_event < event_stop ? 1 : -1;
            if ((ch.rc != 0) != (stride == -1)) { status |= NPH_EA_RC_STRIDE; break; }
            if ((uint32_t)curr_start_event >= j.rd.n_events || (uint32_t)event_stop >= j.rd.n_events) { status |= NPH_EA_BAD_EVENT; break; }
            j.K = l - k + 1;
            j.E = span + 1;
            if (j.K > STRIP || j.E > p.e_cap) { status |= NPH_EA_WINDOW_TOO_LARGE; break; }
            j.rk = rank_base + s;
            j.stride = stride;
            j.e_first = (long long)curr_start_event;

            float last_v;
            const int n = viterbi_align<C, false>(p.c, p.flank, j, sc, states, (int)p.states_stride, &last_v, lane);
            n_windows += 1;

            // emission (eventalign.cpp:752-806): the first kOutputStride states (all of them in the last section) that are
            // not k-mer skips and not on the window's start event, 32 states at a time by ballot + prefix count
            const bool last_section = end_pair_idx == n_pairs - 1;
            const int limit = last_section ? 0x7fffffff : kOutputStride;
            const nph_align_state* const path = states + ((int)p.states_stride - n);       // ascending event order
            int num_output = 0, last_event_output = 0, last_ref_kmer_output = 0, overflow = 0;
            for (int base = 0; base < n && num_output < limit; base += 32) {
                const int idx = base + lane;
                int ev_idx = 0, ref_position = 0;
                char state = 'K';
                if (idx < n) {
                    const nph_align_state as = path[idx];
                    ev_idx = (int)as.event_idx; ref_position = curr_start_ref + (int)as.kmer_idx; state = as.state;
                }
                const bool emit = idx < n && state != 'K' && ev_idx != curr_start_event;
                const unsigned m = __ballot_sync(kFull, emit);
                const int pos = num_output + __popc(m & ((1u << lane) - 1u));
                const bool take = emit && pos < limit;
                const bool fits = n_rec + (uint32_t)pos < ch.out_cap;
                if (take && fits) {
                    nph_ea_record r;
                    r.ref_position = ref_position;
                    r.event_idx = ev_idx;
                    r.hmm_state = (uint8_t)state;
                    r.reserved[0] = 0; r.reserved[1] = 0; r.reserved[2] = 0;
                    rec[n_rec + pos] = r;
                }
                const unsigned mt = __ballot_sync(kFull, take);
                overflow |= __ballot_sync(kFull, take && !fits) != 0u;
                if (mt) {
                    const int last_lane = 31 - __clz(mt);
                    last_event_output = __shfl_sync(kFull, ev_idx, last_lane);
                    last_ref_kmer_output = __shfl_sync(kFull, ref_position, last_lane);
                    num_output += __popc(mt);
                }
            }
            n_rec += (uint32_t)num_output;
            if (overflow) { status |= NPH_EA_OUT_OVERFLOW; break; }
            // advance the cursor to where the output stopped
            curr_start_event = last_event_output;
            curr_start_ref = last_ref_kmer_output;
            if (num_output == 0) break;
            curr_pair_idx = warp_get_end_pair(pairs, n_pairs, curr_start_ref, curr_pair_idx, lane);
            __syncwarp();                                    // states[] is rewritten by the next window
        }
        if (lane == 0) {
            nph_ea_result res;
            res.n_records = n_rec; res.n_windows = n_windows; res.status = status; res.reserved = 0;
            p.results[chain_idx] = res;
        }
        __syncwarp();
    }
}

template <int C>
void launch_chain(const ChainParams& p, int grid, cudaStream_t stream)
{
    eventalign_chain_kernel<C><<<grid, kThreads, 0, stream>>>(p);
}

} // namespace

extern "C" int nph_eventalign_chain(nph_ctx* ctx,
                                    const nph_aligned_pair* pairs, size_t n_pairs_total,
                                    const int32_t* event_map_start, size_t n_map_total,
                                    const uint32_t* ref_ranks_fwd, const uint32_t* ref_ranks_rc, size_t n_ranks_total,
                                    const nph_ea_chain* chains, size_t n_chains, double indel_bias,
                                    nph_ea_record* records_out, size_t records_total, nph_ea_result* results_out)
{
    if (!ctx || !chains || !results_out || n_chains == 0) return NPH_ERR_INVALID;
    if (!pairs || !event_map_start || !ref_ranks_fwd || !ref_ranks_rc || (!records_out && records_total)) return NPH_ERR_INVALID;
    if (!ctx->reads_loaded) return NPH_ERR_STATE;
    NPH_CUDA(ctx, cudaSetDevice(ctx->device));

    // validate what the kernel indexes with, and pick the columns per lane: windows span at most kAlignStride + 1
    // reference bases, i.e. kAlignStride + 2 - k k-mers (96 for 6-mers: three columns per lane, every lane busy)
    uint32_t k_min = 255;
    std::vector<uint32_t> n_pairs(n_chains);
    for (size_t i = 0; i < n_chains; ++i) {
        const nph_ea_chain& c = chains[i];
        if (c.read >= ctx->n_reads || c.model_id >= ctx->models.size() || c.k == 0 || c.k != ctx->models[c.model_id].k) return NPH_ERR_INVALID;
        if (c.pair_off + c.n_pairs > n_pairs_total || c.map_off + c.map_len > n_map_total) return NPH_ERR_INVALID;
        const size_t n_ref_kmers = c.ref_len >= c.k ? (size_t)c.ref_len - c.k + 1 : 0;
        if (c.rank_off + n_ref_kmers > n_ranks_total || c.out_off + c.out_cap > records_total) return NPH_ERR_INVALID;
        k_min = std::min<uint32_t>(k_min, c.k);
        n_pairs[i] = c.n_pairs;
    }
    const std::vector<uint32_t> order = longest_first(n_pairs);     // longest chains first
    const int cols = (kAlignStride + 2 - (int)k_min) <= 96 ? 3 : 4;

    NPH_TRY(nph_upload_read_transitions(ctx, indel_bias));

    int grid = ctx->sm_count;
    if ((size_t)grid * kWarps > n_chains) grid = (int)((n_chains + kWarps - 1) / kWarps);
    const size_t warps = (size_t)grid * kWarps;
    // a window's events: typically ~1.7 per base of a 100-base window; the scratch takes 1024 (override for tests)
    int e_cap = 1024;
    if (const char* s = getenv("NPH_EA_EVENT_CAP")) e_cap = std::max(2, atoi(s));
    const size_t strip = 32 * (size_t)cols;
    const size_t trace_stride = ((size_t)(e_cap + 40) * strip + 63) / 64 * 64;
    const uint32_t states_stride = (uint32_t)(e_cap + strip + 8);

    struct {
        nph_aligned_pair* pairs; int32_t* map; uint32_t *rf, *rr; nph_ea_chain* chains; uint32_t* order; nph_ea_record* rec; nph_ea_result* res;
    } d{};
    ChainParams p{};
    auto layout = [&](NphCarve& a) {
        d.pairs = a.take<nph_aligned_pair>(n_pairs_total);
        d.map = a.take<int32_t>(n_map_total);
        d.rf = a.take<uint32_t>(n_ranks_total);
        d.rr = a.take<uint32_t>(n_ranks_total);
        d.chains = a.take<nph_ea_chain>(n_chains);
        d.order = a.take<uint32_t>(n_chains);
        d.rec = a.take<nph_ea_record>(records_total);
        d.res = a.take<nph_ea_result>(n_chains);
        p.scratch_params = a.take<float4>(strip * warps);
        p.scratch_trace = a.take<uint16_t>(trace_stride * warps);
        p.scratch_states = a.take<nph_align_state>(states_stride * warps);
    };
    NPH_TRY(nph_borrow_arena(ctx, layout));
    p.trace_stride = trace_stride; p.states_stride = states_stride; p.e_cap = e_cap;
    p.level = ctx->d_level.p; p.reads = ctx->d_reads.p; p.trans = ctx->d_trans.p; p.models = ctx->d_models.p; p.flank = ctx->d_flank.p;
    p.pairs = d.pairs; p.map_start = d.map; p.ranks_fwd = d.rf; p.ranks_rc = d.rr; p.chains = d.chains; p.order = d.order;
    p.n_chains = (uint32_t)n_chains; p.counter = ctx->d_counters.p; p.records = d.rec; p.results = d.res; p.c = ctx->consts;

    if (n_pairs_total) NPH_CUDA(ctx, cudaMemcpyAsync(d.pairs, pairs, sizeof(nph_aligned_pair) * n_pairs_total, cudaMemcpyHostToDevice, ctx->stream));
    if (n_map_total) NPH_CUDA(ctx, cudaMemcpyAsync(d.map, event_map_start, sizeof(int32_t) * n_map_total, cudaMemcpyHostToDevice, ctx->stream));
    if (n_ranks_total) {
        NPH_CUDA(ctx, cudaMemcpyAsync(d.rf, ref_ranks_fwd, sizeof(uint32_t) * n_ranks_total, cudaMemcpyHostToDevice, ctx->stream));
        NPH_CUDA(ctx, cudaMemcpyAsync(d.rr, ref_ranks_rc, sizeof(uint32_t) * n_ranks_total, cudaMemcpyHostToDevice, ctx->stream));
    }
    NPH_CUDA(ctx, cudaMemcpyAsync(d.chains, chains, sizeof(nph_ea_chain) * n_chains, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(d.order, order.data(), sizeof(uint32_t) * n_chains, cudaMemcpyHostToDevice, ctx->stream));
    NPH_CUDA(ctx, cudaMemsetAsync(ctx->d_counters.p, 0, sizeof(unsigned int) * NPH_NUM_COUNTERS, ctx->stream));
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    if (cols == 3) launch_chain<3>(p, grid, ctx->stream); else launch_chain<4>(p, grid, ctx->stream);
    NPH_CUDA(ctx, cudaGetLastError());
    NPH_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->last_launches = 1;
    ctx->timing_valid = 1;
    if (records_total) NPH_CUDA(ctx, cudaMemcpyAsync(records_out, d.rec, sizeof(nph_ea_record) * records_total, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaMemcpyAsync(results_out, d.res, sizeof(nph_ea_result) * n_chains, cudaMemcpyDeviceToHost, ctx->stream));
    NPH_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NPH_OK;
}
