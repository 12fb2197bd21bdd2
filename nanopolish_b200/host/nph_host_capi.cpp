// nph_host_capi.cpp — a thin extern "C" shim over the C++ host mirror so that the Python tests can
// drive HMMInputData / HMMInputSequence / SquiggleRead / Alphabet exactly as a C++ caller would.
#include "nph_host.hpp"
#include "nph_variants.hpp"
#include "nph_methylation.hpp"
#include "nph_raw.hpp"
#include "nph_eventalign.hpp"
#include "nph_scorereads.hpp"
#include "nph_polya.hpp"
#include <cmath>
#include <chrono>
#include <cstring>
#include <memory>

using namespace nph;

namespace {
std::vector<std::unique_ptr<PoreModel>> g_models;
std::vector<std::unique_ptr<SquiggleRead>> g_reads;
EventAligner g_aligner;
AlignBatch g_round_batch;
bool g_raw_is_rna = false;
uint32_t g_load_flags = 0;
thread_local std::string g_err;
template <typename F> int guard(F f) { try { f(); return 0; } catch (const Error& e) { g_err = e.what(); return e.status; } catch (const std::exception& e) { g_err = e.what(); return NPH_ERR_INVALID; } }
}

extern "C" {

const char* nphh_last_error() { return g_err.c_str(); }

int nphh_alphabet_op(const char* alphabet, int op, const char* in, char* out)
{
    int n = -1;
    int rc = guard([&] {
        const Alphabet* a = get_alphabet_by_name(alphabet);
        std::string s(in), r;
        switch (op) {
            case 0: r = a->reverse_complement(s); break;
            case 1: r = a->methylate(s); break;
            case 2: r = a->unmethylate(s); break;
            case 3: r = a->disambiguate(s); break;
            default: throw Error(NPH_ERR_INVALID, "bad op");
        }
        std::memcpy(out, r.c_str(), r.size() + 1);
        n = (int)r.size();
    });
    return rc ? rc : n;
}

int nphh_is_motif_match(const char* alphabet, const char* seq, size_t i)
{
    return get_alphabet_by_name(alphabet)->is_motif_match(seq, i) ? 1 : 0;
}

uint32_t nphh_kmer_rank(const char* alphabet, const char* kmer, uint32_t k) { return get_alphabet_by_name(alphabet)->kmer_rank(kmer, k); }

int nphh_lexicographic_next(const char* alphabet, const char* in, char* out)
{
    std::string s(in);
    get_alphabet_by_name(alphabet)->lexicographic_next(s);
    std::memcpy(out, s.c_str(), s.size() + 1);
    return (int)s.size();
}

// HMMInputSequence::append_kmer_ranks (the rolling pass HmmBatch::add uses) against get_kmer_rank: mismatching positions
int nphh_kmer_ranks_rolling_check(const char* alphabet, const char* seq, uint32_t k, int rc)
{
    int bad = -1;
    int st = guard([&] {
        HMMInputSequence hs(std::string(seq), get_alphabet_by_name(alphabet));
        std::vector<uint32_t> r;
        hs.append_kmer_ranks(k, rc != 0, r);
        const size_t n = hs.length() >= k ? hs.length() - k + 1 : 0;
        bad = r.size() == n ? 0 : 1;
        for (size_t i = 0; i < std::min(n, r.size()); ++i) bad += r[i] != hs.get_kmer_rank((uint32_t)i, k, rc != 0);
    });
    return st ? st : bad;
}

// HMMInputSequence::get_kmer_rank for ki = 0..n-1
int nphh_kmer_ranks(const char* alphabet, const char* seq, uint32_t k, int rc, uint32_t* out)
{
    int n = 0;
    int st = guard([&] {
        HMMInputSequence hs(std::string(seq), get_alphabet_by_name(alphabet));
        if (hs.length() < k) return;
        n = (int)(hs.length() - k + 1);
        for (int i = 0; i < n; ++i) out[i] = hs.get_kmer_rank(i, k, rc != 0);
    });
    return st ? st : n;
}

int nphh_model_create(const char* alphabet, uint32_t k, uint32_t n_states, const double* mean, const double* stdv, const double* log_stdv)
{
    int h = -1;
    int rc = guard([&] {
        std::unique_ptr<PoreModel> pm(new PoreModel(k));
        pm->pmalphabet = get_alphabet_by_name(alphabet);
        pm->states.resize(n_states);
        for (uint32_t i = 0; i < n_states; ++i) {
            pm->states[i].level_mean = mean[i];
            pm->states[i].level_stdv = stdv[i];
            pm->states[i].level_log_stdv = log_stdv ? log_stdv[i] : std::log(stdv[i]);
        }
        g_models.push_back(std::move(pm));
        h = (int)g_models.size() - 1;
    });
    return rc ? rc : h;
}

int nphh_read_create(uint32_t n_events, const float* mean, const double* start_time, double shift, double scale, double drift,
                     double var, double events_per_base, int base_model)
{
    std::unique_ptr<SquiggleRead> sr(new SquiggleRead());
    sr->pore_type = PORETYPE_R9;
    sr->base_model[0] = g_models[base_model].get();
    sr->scalings[0].set4(shift, scale, drift, var);
    sr->events_per_base[0] = events_per_base;
    sr->events[0].resize(n_events);
    for (uint32_t i = 0; i < n_events; ++i) sr->events[0][i] = SquiggleEvent{mean[i], 1.0f, start_time[i], 0.0f, 0.0f};
    sr->cache_event_means();
    g_reads.push_back(std::move(sr));
    return (int)g_reads.size() - 1;
}

void nphh_read_add_model(int read, const char* alphabet, int model) { g_reads[read]->alt_models[0][alphabet] = g_models[model].get(); }
void nphh_clear() { g_reads.clear(); }
void nphh_set_indel_bias(double v) { hmm_indel_bias_factor = v; }
void nphh_set_rna(int rna) { g_raw_is_rna = rna != 0; }        // nucleotide type of the reads nphh_load_from_raw builds
void nphh_set_load_flags(uint32_t flags) { g_load_flags = flags; }   // SquiggleReadFlags for nphh_load_from_raw
long long nphh_read_num_samples(int read) { return (long long)g_reads[read]->samples.size(); }
float nphh_read_sample(int read, size_t i) { return g_reads[read]->samples.at(i); }

// profile_hmm_score(sequence, data, flags) exactly as a nanopolish caller writes it
int nphh_profile_hmm_score(int read, int model, const char* seq, uint32_t e_start, uint32_t e_stop, int rc, uint32_t flags, float* out)
{
    return guard([&] {
        const PoreModel* pm = g_models[model].get();
        HMMInputSequence sequence(std::string(seq), pm->pmalphabet);
        HMMInputData data;
        data.read = g_reads[read].get();
        data.pore_model = pm;
        data.event_start_idx = e_start;
        data.event_stop_idx = e_stop;
        data.strand = 0;
        data.rc = rc;
        data.event_stride = rc ? -1 : 1;
        *out = profile_hmm_score(sequence, data, flags);
    });
}

// one HmmBatch over many calls (the intended integration)
int nphh_profile_hmm_score_many(size_t n, const int32_t* read, const int32_t* model, const char* seq_buf, const uint64_t* seq_off,
                                const uint32_t* e_start, const uint32_t* e_stop, const uint8_t* rc, const uint32_t* flags, float* out)
{
    return guard([&] {
        HmmBatch b;
        for (size_t j = 0; j < n; ++j) {
            const PoreModel* pm = g_models[model[j]].get();
            HMMInputSequence sequence(std::string(seq_buf + seq_off[j], seq_buf + seq_off[j + 1]), pm->pmalphabet);
            HMMInputData data;
            data.read = g_reads[read[j]].get();
            data.pore_model = pm;
            data.event_start_idx = e_start[j];
            data.event_stop_idx = e_stop[j];
            data.strand = 0;
            data.rc = rc[j];
            data.event_stride = rc[j] ? -1 : 1;
            b.add(sequence, data, flags[j]);
        }
        std::vector<float> s = b.run(Engine::thread_default());
        std::memcpy(out, s.data(), sizeof(float) * n);
    });
}

// profile_hmm_score_set over {nucleotide sequence, methylated sequence(s)}
int nphh_profile_hmm_score_set(int read, int model, int n_seqs, const char** seqs, const char** alphabets, uint32_t e_start,
                               uint32_t e_stop, int rc, uint32_t flags, float* out)
{
    return guard([&] {
        std::vector<HMMInputSequence> ss;
        for (int i = 0; i < n_seqs; ++i) ss.emplace_back(std::string(seqs[i]), get_alphabet_by_name(alphabets[i]));
        HMMInputData data;
        data.read = g_reads[read].get();
        data.pore_model = g_models[model].get();
        data.event_start_idx = e_start;
        data.event_stop_idx = e_stop;
        data.strand = 0;
        data.rc = rc;
        data.event_stride = rc ? -1 : 1;
        *out = profile_hmm_score_set(ss, data, flags);
    });
}

long long nphh_abea(int read, int model, const char* seq, int32_t* pairs_out, size_t cap)
{
    long long n = -1;
    int rc = guard([&] {
        std::vector<AlignedPair> p = adaptive_banded_simple_event_align(*g_reads[read], *g_models[model], std::string(seq));
        if (p.size() > cap) throw Error(NPH_ERR_INVALID, "cap");
        for (size_t i = 0; i < p.size(); ++i) { pairs_out[2 * i] = p[i].ref_pos; pairs_out[2 * i + 1] = p[i].read_pos; }
        n = (long long)p.size();
    });
    return rc ? rc : n;
}

int nphh_mom(int read, int model, const char* seq, double* out4)
{
    return guard([&] {
        std::vector<float> m;
        for (const SquiggleEvent& e : g_reads[read]->events[0]) m.push_back(e.mean);
        SquiggleScalings s = estimate_scalings_using_mom(std::string(seq), *g_models[model], m);
        out4[0] = s.shift; out4[1] = s.scale; out4[2] = s.drift; out4[3] = s.var;
    });
}

// ---- N2: variant scoring -------------------------------------------------------------------
// Haplotype::apply_variants on a reference string; returns the derived sequence (or -1 if a variant was refused)
int nphh_haplotype_apply(const char* ref, size_t ref_position, int n_var, const size_t* pos, const char** ref_seq, const char** alt_seq,
                         char* out)
{
    Haplotype h("ctg", ref_position, ref);
    bool good = true;
    for (int i = 0; i < n_var; ++i) { Variant v; v.ref_name = "ctg"; v.ref_position = pos[i]; v.ref_seq = ref_seq[i]; v.alt_seq = alt_seq[i]; good = h.apply_variant(v) && good; }
    std::memcpy(out, h.get_sequence().c_str(), h.get_sequence().size() + 1);
    return good ? (int)h.get_sequence().size() : -1;
}

// score_variants_thresholded over reads (handles + per-read event window) and a candidate list
int nphh_score_variants_thresholded(int n_reads, const int32_t* read, const uint32_t* e_start, const uint32_t* e_stop, const uint8_t* rc,
                                    int model, const char* base_seq, size_t ref_position, int n_var, const size_t* pos,
                                    const char** ref_seq, const char** alt_seq, uint32_t flags, uint32_t threshold,
                                    int n_meth, const char** meth_types, double indel_bias, double* quality_out)
{
    return guard([&] {
        std::vector<HMMInputData> input(n_reads);
        for (int j = 0; j < n_reads; ++j) {
            input[j].read = g_reads[read[j]].get();
            input[j].pore_model = g_models[model].get();
            input[j].event_start_idx = e_start[j];
            input[j].event_stop_idx = e_stop[j];
            input[j].strand = 0;
            input[j].rc = rc[j];
            input[j].event_stride = rc[j] ? -1 : 1;
        }
        std::vector<Variant> vars(n_var);
        for (int i = 0; i < n_var; ++i) { vars[i].ref_name = "ctg"; vars[i].ref_position = pos[i]; vars[i].ref_seq = ref_seq[i]; vars[i].alt_seq = alt_seq[i]; }
        std::vector<std::string> mt;
        for (int i = 0; i < n_meth; ++i) mt.push_back(meth_types[i]);
        Haplotype base("ctg", ref_position, base_seq);
        std::vector<Variant> out = score_variants_thresholded(vars, base, input, flags, threshold, mt, Engine::thread_default(), indel_bias);
        for (int i = 0; i < n_var; ++i) quality_out[i] = out[i].quality;
    });
}

// score_variant_group over reads and a variant group: combos_out[c] = bitmask of the variant ids of combination c,
// scores_out[c * n_reads + r]; returns the number of combinations (or a negative status)
long long nphh_score_variant_group(int n_reads, const int32_t* read, const uint32_t* e_start, const uint32_t* e_stop, const uint8_t* rc,
                                   int model, const char* base_seq, size_t ref_position, int n_var, const size_t* pos,
                                   const char** ref_seq, const char** alt_seq, int max_haplotypes, uint32_t flags,
                                   int n_meth, const char** meth_types, double indel_bias, uint32_t* combos_out, double* scores_out, size_t cap_comb)
{
    long long n = -1;
    int st = guard([&] {
        std::vector<HMMInputData> input(n_reads);
        for (int j = 0; j < n_reads; ++j) {
            input[j].read = g_reads[read[j]].get();
            input[j].pore_model = g_models[model].get();
            input[j].event_start_idx = e_start[j];
            input[j].event_stop_idx = e_stop[j];
            input[j].strand = 0;
            input[j].rc = rc[j];
            input[j].event_stride = rc[j] ? -1 : 1;
        }
        std::vector<Variant> vars(n_var);
        for (int i = 0; i < n_var; ++i) { vars[i].ref_name = "ctg"; vars[i].ref_position = pos[i]; vars[i].ref_seq = ref_seq[i]; vars[i].alt_seq = alt_seq[i]; }
        std::vector<std::string> mt;
        for (int i = 0; i < n_meth; ++i) mt.push_back(meth_types[i]);
        Haplotype base("ctg", ref_position, base_seq);
        const VariantGroupScores g = score_variant_group(vars, base, input, max_haplotypes, flags, mt, Engine::thread_default(), indel_bias);
        if (g.combinations.size() > cap_comb) throw Error(NPH_ERR_INVALID, "combination buffer too small");
        for (size_t c = 0; c < g.combinations.size(); ++c) {
            uint32_t mask = 0;
            for (size_t id : g.combinations[c]) mask |= 1u << id;
            combos_out[c] = mask;
            for (int r = 0; r < n_reads; ++r) scores_out[c * (size_t)n_reads + r] = g.scores[c][r];
        }
        n = (long long)g.combinations.size();
    });
    return st ? st : n;
}

// ---- N3: call-methylation for a batch of reads; returns the concatenated TSV ------------------------------
// aligned pairs are (ref_pos, event_idx) interleaved, pair_off[n_reads+1]
static long long call_methylation_impl(int n_reads, const int32_t* read, const char** read_names, const uint8_t* is_rev, const uint8_t* rc,
                                       const int32_t* ref_start, const char** ref_seqs, const int32_t* pairs, const uint64_t* pair_off,
                                       const char* contig, double indel_bias, char* tsv_out, size_t cap, uint64_t* n_jobs_out, double* secs4)
{
    long long n = -1;
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    int st = guard([&] {
        // one caller for the process, cleared between batches: its page-locked staging is allocated once (what a BamProcessor
        // integration does: one MethylationCaller per worker, a batch per BamProcessor round)
        static std::unique_ptr<MethylationCaller> caller;
        if (!caller) { MethylationCallingParameters params; caller.reset(new MethylationCaller(params)); }
        caller->clear();
        const double tm = now();
        // the shim's own marshalling of the test's flat arrays into the caller-side objects (not part of the product path)
        std::vector<EventAlignedRead> batch_reads((size_t)n_reads);
#pragma omp parallel for schedule(dynamic, 16) num_threads(host_threads()) if (n_reads > 64)
        for (int i = 0; i < n_reads; ++i) {
            EventAlignedRead& r = batch_reads[(size_t)i];
            r.read = g_reads[read[i]].get();
            r.read_name = read_names[i];
            r.is_reverse = is_rev[i];
            r.contig = contig;
            r.ref_start_pos = ref_start[i];
            r.ref_seq = ref_seqs[i];
            const uint64_t np = pair_off[i + 1] - pair_off[i];
            r.aligned_events[0].resize(np);
            if (np) std::memcpy(r.aligned_events[0].data(), pairs + 2 * pair_off[i], sizeof(AlignedPair) * np);
            r.rc[0] = rc[i];
        }
        const double t0 = now();
        caller->add_reads(batch_reads);
        const double t1 = now();
        caller->run(Engine::thread_default(), indel_bias);
        *n_jobs_out = caller->num_jobs();
        const double t2 = now();
        const size_t bytes = caller->tsv_all(tsv_out, cap ? cap - 1 : 0);
        if (secs4) { secs4[0] = t1 - t0; secs4[1] = t2 - t1; secs4[2] = now() - t2; secs4[3] = t0 - tm; }
        if (bytes + 1 > cap) throw Error(NPH_ERR_INVALID, "tsv buffer too small");
        tsv_out[bytes] = 0;
        n = (long long)bytes;
    });
    return st ? st : n;
}

long long nphh_call_methylation(int n_reads, const int32_t* read, const char** read_names, const uint8_t* is_rev, const uint8_t* rc,
                                const int32_t* ref_start, const char** ref_seqs, const int32_t* pairs, const uint64_t* pair_off,
                                const char* contig, double indel_bias, char* tsv_out, size_t cap, uint64_t* n_jobs_out)
{
    return call_methylation_impl(n_reads, read, read_names, is_rev, rc, ref_start, ref_seqs, pairs, pair_off, contig, indel_bias, tsv_out, cap,
                                 n_jobs_out, nullptr);
}
// the same, with the seconds spent in {staging (add_reads), flatten + device call, TSV formatting, the shim's own marshalling}: secs4[4]
long long nphh_call_methylation_timed(int n_reads, const int32_t* read, const char** read_names, const uint8_t* is_rev, const uint8_t* rc,
                                      const int32_t* ref_start, const char** ref_seqs, const int32_t* pairs, const uint64_t* pair_off,
                                      const char* contig, double indel_bias, char* tsv_out, size_t cap, uint64_t* n_jobs_out, double* secs3)
{
    return call_methylation_impl(n_reads, read, read_names, is_rev, rc, ref_start, ref_seqs, pairs, pair_off, contig, indel_bias, tsv_out, cap,
                                 n_jobs_out, secs3);
}

// call-methylation from flat host buffers (the C-ABI layout) to TSV bytes: what bench.py's end-to-end arm times.
// host_mode != 0 runs the host-side enumerator instead (reads registered with nphh_read_create; the cross-check path).
long long nphh_call_methylation_flat(const void* reads, size_t n_reads, const float* ev_mean, const double* ev_start_time, size_t n_events,
                                     const char* ref_bases, size_t n_ref, const void* aligned_events, size_t n_pairs,
                                     const int16_t* event_deltas, const int32_t* first_event, void* records, size_t n_records,
                                     int cpg_model, const char** read_names, const uint8_t* is_reverse, const char* contig, double indel_bias,
                                     char* tsv_out, size_t cap, uint64_t* n_sites_out, uint64_t* scored_events_out, double* secs2)
{
    long long n = -1;
    int st = guard([&] {
        Engine& eng = Engine::thread_default();
        const PoreModel* model = g_models[cpg_model].get();
        const uint32_t mid = eng.model_id(model);
        nph_meth_record* recs = static_cast<nph_meth_record*>(records);
        for (size_t r = 0; r < n_records; ++r) recs[r].model_id = mid;
        FlatMethylationBatch b;
        b.reads = static_cast<const nph_read*>(reads); b.n_reads = n_reads; b.ev_mean = ev_mean; b.ev_start_time = ev_start_time; b.n_events = n_events;
        b.ref_bases = ref_bases; b.n_ref = n_ref; b.aligned_events = static_cast<const nph_aligned_pair*>(aligned_events); b.n_pairs = n_pairs;
        b.event_deltas = event_deltas; b.first_event = first_event;
        b.records = recs; b.n_records = n_records; b.read_names = read_names; b.is_reverse = is_reverse; b.contig = contig;
        MethylationCallingParameters params;
        params.methylation_type = model->pmalphabet->get_name();
        params.alphabet = model->pmalphabet;
        FlatMethylationStats stats;
        const size_t bytes = call_methylation_flat(eng, b, params, model->k, indel_bias, tsv_out, cap ? cap - 1 : 0, &stats);
        if (bytes + 1 > cap) throw Error(NPH_ERR_INVALID, "tsv buffer too small");
        tsv_out[bytes] = 0;
        if (n_sites_out) *n_sites_out = stats.n_sites;
        if (scored_events_out) *scored_events_out = stats.scored_events;
        if (secs2) { secs2[0] = stats.device_seconds; secs2[1] = stats.tsv_seconds; }
        n = (long long)bytes;
    });
    return st ? st : n;
}

// modBAM tags of one record from explicit calls (start position, site sequence, strand-0 log-likelihoods); reference_mode:
// create_reference_modbam_record (seq = reference over the record, aligned pairs unused).  Returns the number of Ml entries.
long long nphh_modbam_tags(const char* seq, int ref_pos, int flag, const uint32_t* cigar, int n_cigar, int n_calls, const int32_t* start_pos,
                           const char** site_seqs, const double* ll_m0, const double* ll_u0, int reference_mode, char* mm_out, size_t mm_cap,
                           uint8_t* ml_out, size_t ml_cap)
{
    long long n = -1;
    int rc = guard([&] {
        std::map<int, ScoredSite> calls;
        for (int i = 0; i < n_calls; ++i) {
            ScoredSite ss;
            ss.start_position = start_pos[i];
            ss.sequence = site_seqs[i];
            ss.ll_methylated[0] = ll_m0[i];
            ss.ll_unmethylated[0] = ll_u0[i];
            calls[start_pos[i]] = ss;
        }
        MethylationCallingParameters params;
        ModbamTags t;
        if (reference_mode) {
            t = reference_modbam_tags(seq, ref_pos, calls, params);
        } else {
            const std::vector<AlignedSegment> segs = get_aligned_segments(ref_pos, std::vector<uint32_t>(cigar, cigar + n_cigar));
            if (segs.size() > 1) throw Error(NPH_ERR_UNSUPPORTED, "spliced alignment");       // the reference exits
            t = modbam_tags(seq, segs[0], (flag & NPH_BAM_FREVERSE) != 0, calls, params);
        }
        if (t.mm.size() + 1 > mm_cap || t.ml.size() > ml_cap) throw Error(NPH_ERR_INVALID, "tag buffers too small");
        std::memcpy(mm_out, t.mm.c_str(), t.mm.size() + 1);
        std::memcpy(ml_out, t.ml.data(), t.ml.size());
        n = (long long)t.ml.size();
    });
    return rc ? rc : n;
}

// enumeration only (no device): seconds spent in MethylationCaller::add_read over all reads, and the job count
// parallel != 0: MethylationCaller::add_reads (host_threads() workers); jobs_out / ranks_out (optional) receive the job list
double nphh_methylation_enumerate_seconds(int n_reads, const int32_t* read, const char** read_names, const uint8_t* is_rev, const uint8_t* rc,
                                          const int32_t* ref_start, const char** ref_seqs, const int32_t* pairs, const uint64_t* pair_off,
                                          const char* contig, uint64_t* n_jobs_out, int parallel, void* jobs_out, size_t cap_jobs,
                                          uint32_t* ranks_out, size_t cap_ranks, uint64_t* n_ranks_out)
{
    double secs = -1.0;
    guard([&] {
        MethylationCallingParameters params;
        MethylationCaller caller(params, MethylationCaller::Mode::HostEnumeration);
        std::vector<EventAlignedRead> rs(n_reads);
        for (int i = 0; i < n_reads; ++i) {
            EventAlignedRead& r = rs[i];
            r.read = g_reads[read[i]].get();
            r.read_name = read_names[i];
            r.is_reverse = is_rev[i];
            r.contig = contig;
            r.ref_start_pos = ref_start[i];
            r.ref_seq = ref_seqs[i];
            r.aligned_events[0].reserve(pair_off[i + 1] - pair_off[i]);
            for (uint64_t p = pair_off[i]; p < pair_off[i + 1]; ++p) r.aligned_events[0].push_back(AlignedPair{pairs[2 * p], pairs[2 * p + 1]});
            r.rc[0] = rc[i];
        }
        const auto t0 = std::chrono::steady_clock::now();
        if (parallel) caller.add_reads(rs);
        else for (int i = 0; i < n_reads; ++i) caller.add_read(rs[i]);
        secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        *n_jobs_out = caller.num_jobs();
        if (jobs_out && ranks_out) {
            const HmmBatch& b = caller.batch();
            const std::vector<uint32_t> rk = b.ranks();
            if (b.jobs().size() > cap_jobs || rk.size() > cap_ranks) throw Error(NPH_ERR_INVALID, "dump buffers too small");
            std::memcpy(jobs_out, b.jobs().data(), sizeof(nph_hmm_job) * b.jobs().size());
            std::memcpy(ranks_out, rk.data(), sizeof(uint32_t) * rk.size());
            *n_ranks_out = rk.size();
        }
    });
    return secs;
}

// ---- N4: load_from_raw over a batch -----------------------------------------------------------
// seqs: concatenated basecalled sequences (seq_off has n+1 entries); samples likewise.  Outputs per read: n_events
// (0 = failed), {shift, scale, drift, var, events_per_base} in scal5, and — into the flat arrays at ev_off[i] (room =
// n_samples/2 + 8 per read) — mean, stdv, start_time, duration.  b2e_out (optional): n_kmers IndexPairs per read at
// seq_off[i] (room = sequence length).  Returns the reads in g_reads (first handle) or a negative status.
int nphh_load_from_raw(int model, int n, const float* samples, const uint64_t* sample_off, const char* seqs, const uint64_t* seq_off,
                       double sample_rate, uint32_t* n_events, double* scal5, const uint64_t* ev_off, float* mean, float* stdv,
                       double* start_time, float* duration, int32_t* b2e_out, uint64_t* stats5)
{
    int first = -1;
    int rc = guard([&] {
        std::vector<RawRead> raw(n);
        for (int i = 0; i < n; ++i) {
            raw[i].read_name = "read" + std::to_string(i);
            raw[i].read_sequence.assign(seqs + seq_off[i], seqs + seq_off[i + 1]);
            raw[i].samples.assign(samples + sample_off[i], samples + sample_off[i + 1]);
            raw[i].sample_rate = sample_rate;
            raw[i].nucleotide_type = g_raw_is_rna ? SRNT_RNA : SRNT_DNA;
        }
        LoadFromRawStats st;
        std::vector<std::unique_ptr<SquiggleRead>> rs = load_from_raw(Engine::thread_default(), *g_models[model], raw, &st, g_load_flags);
        stats5[0] = st.total; stats5[1] = st.empty_after_trim; stats5[2] = st.failed_alignment; stats5[3] = st.failed_calibration; stats5[4] = st.qc_fail;
        first = (int)g_reads.size();
        for (int i = 0; i < n; ++i) {
            SquiggleRead& sr = *rs[i];
            n_events[i] = (uint32_t)sr.events[0].size();
            const SquiggleScalings& s = sr.scalings[0];
            scal5[5 * i] = s.shift; scal5[5 * i + 1] = s.scale; scal5[5 * i + 2] = s.drift; scal5[5 * i + 3] = s.var; scal5[5 * i + 4] = sr.events_per_base[0];
            for (size_t e = 0; e < sr.events[0].size(); ++e) {
                const SquiggleEvent& ev = sr.events[0][e];
                mean[ev_off[i] + e] = ev.mean; stdv[ev_off[i] + e] = ev.stdv; start_time[ev_off[i] + e] = ev.start_time; duration[ev_off[i] + e] = ev.duration;
            }
            if (b2e_out)
                for (size_t kk = 0; kk < sr.base_to_event_map.size(); ++kk) {
                    b2e_out[2 * (seq_off[i] + kk)] = sr.base_to_event_map[kk].indices[0].start;
                    b2e_out[2 * (seq_off[i] + kk) + 1] = sr.base_to_event_map[kk].indices[0].stop;
                }
            g_reads.push_back(std::move(rs[i]));
        }
    });
    return rc ? rc : first;
}

// ---- N1: eventalign (segment chaining around the Viterbi kernel) -------------------------------------------
// what load_from_raw leaves on a SquiggleRead beyond events and scalings
int nphh_read_set_eventalign(int read, const char* read_name, const char* read_sequence, const int32_t* map_start, const int32_t* map_stop,
                             size_t n_map, const float* stdv, const float* duration)
{
    return guard([&] {
        SquiggleRead& sr = *g_reads[read];
        sr.read_name = read_name;
        sr.read_sequence = read_sequence;
        sr.base_to_event_map.resize(n_map);
        for (size_t i = 0; i < n_map; ++i) sr.base_to_event_map[i].indices[0] = IndexPair(map_start[i], map_stop[i]);
        for (size_t i = 0; i < sr.events[0].size(); ++i) { sr.events[0][i].stdv = stdv[i]; sr.events[0][i].duration = duration[i]; }
    });
}

// the raw samples load_from_raw keeps with SRF_LOAD_RAW_SAMPLES
int nphh_read_set_samples(int read, const float* samples, size_t n, double sample_rate)
{
    return guard([&] {
        SquiggleRead& sr = *g_reads[read];
        sr.samples.assign(samples, samples + n);
        sr.sample_start_time = 0;
        sr.sample_rate = sample_rate;
    });
}

void nphh_ea_begin() { g_aligner.clear(); g_round_batch.clear(); }

int nphh_ea_add_read(int read, const char* ref_name, int ref_pos, int flag, int mapq, const uint32_t* cigar, int n_cigar, const char* ref_seq,
                     int read_idx, int region_start, int region_end)
{
    int idx = -1;
    int rc = guard([&] {
        EventAlignmentParameters p;
        p.sr = g_reads[read].get();
        p.strand_idx = 0;
        p.ref_name = ref_name; p.ref_pos = ref_pos; p.flag = (uint16_t)flag; p.mapq = (uint8_t)mapq;
        p.cigar.assign(cigar, cigar + n_cigar);
        p.ref_seq = ref_seq;
        p.read_idx = read_idx; p.region_start = region_start; p.region_end = region_end;
        idx = (int)g_aligner.add_read(p);
    });
    return rc ? rc : idx;
}

// everything on the GPU, chains walked by the chain kernel: returns the number of kernel batches (1 + fallback rounds)
long long nphh_ea_run(double indel_bias)
{
    long long rounds = -1;
    int rc = guard([&] { rounds = (long long)g_aligner.run(Engine::thread_default(), indel_bias); });
    return rc ? rc : rounds;
}

// the host-driven form (one Viterbi launch per round): returns the number of rounds
long long nphh_ea_run_rounds(double indel_bias)
{
    long long rounds = -1;
    int rc = guard([&] { rounds = (long long)g_aligner.run_rounds(Engine::thread_default(), indel_bias); });
    return rc ? rc : rounds;
}

// One round's job list without running it (host-logic tests feed the paths back through nphh_ea_consume):
// jobs_out = nph_hmm_job[cap_jobs] (job.read = index of the read in the aligner), ranks_out = uint32[cap_ranks].
// Returns the number of jobs (0 = all reads finished) or a negative status.
long long nphh_ea_next_round(void* jobs_out, size_t cap_jobs, uint32_t* ranks_out, size_t cap_ranks, uint64_t* n_ranks_out)
{
    long long n = 0;
    int rc = guard([&] {
        if (!g_aligner.next_round(g_round_batch)) { n = 0; return; }
        const std::vector<nph_hmm_job>& jobs = g_round_batch.jobs();
        if (jobs.size() > cap_jobs || g_round_batch.ranks().size() > cap_ranks) throw Error(NPH_ERR_INVALID, "round buffers too small");
        nph_hmm_job* out = static_cast<nph_hmm_job*>(jobs_out);
        for (size_t j = 0; j < jobs.size(); ++j) { out[j] = jobs[j]; out[j].read = (uint32_t)g_aligner.round_reads()[j]; }
        std::memcpy(ranks_out, g_round_batch.ranks().data(), sizeof(uint32_t) * g_round_batch.ranks().size());
        *n_ranks_out = g_round_batch.ranks().size();
        n = (long long)jobs.size();
    });
    return rc ? rc : n;
}

int nphh_ea_consume(size_t n_jobs, const uint64_t* state_off, const nph_align_state* states)
{
    return guard([&] {
        std::vector<std::vector<HMMAlignmentState>> paths(n_jobs);
        for (size_t j = 0; j < n_jobs; ++j)
            for (uint64_t i = state_off[j]; i < state_off[j + 1]; ++i)
                paths[j].push_back(HMMAlignmentState{states[i].event_idx, states[i].kmer_idx, -INFINITY, states[i].l_fm, -INFINITY, states[i].state});
        g_aligner.consume(paths);
    });
}

// what: 0 = TSV rows, 1 = TSV rows with read names, 2 = TSV rows with --scale-events, 3 = SAM line, 4 = event CIGAR, 5 = summary row,
// 6 = TSV header, 7 = header + rows with --signal-index --samples
long long nphh_ea_text(int idx, int what, char* out, size_t cap)
{
    long long n = -1;
    int rc = guard([&] {
        EventalignOptions opt;
        std::string s;
        switch (what) {
            case 0: s = g_aligner.tsv(idx, opt); break;
            case 1: opt.print_read_names = true; s = g_aligner.tsv(idx, opt); break;
            case 2: opt.scale_events = true; s = g_aligner.tsv(idx, opt); break;
            case 3: s = g_aligner.sam(idx); break;
            case 4: s = g_aligner.event_cigar(idx); break;
            case 5: s = g_aligner.summary_row(idx, "read.fast5"); break;
            case 6: s = EventAligner::tsv_header(opt); break;
            case 7: opt.write_signal_index = true; opt.write_samples = true; s = EventAligner::tsv_header(opt) + g_aligner.tsv(idx, opt); break;
            default: throw Error(NPH_ERR_INVALID, "unknown text kind");
        }
        if (s.size() + 1 > cap) throw Error(NPH_ERR_INVALID, "text buffer too small");
        std::memcpy(out, s.c_str(), s.size() + 1);
        n = (long long)s.size();
    });
    return rc ? rc : n;
}

// every read's TSV rows concatenated in read order, formatted in parallel (EventAligner::tsv_batch)
long long nphh_ea_tsv_all(char* out, size_t cap)
{
    long long n = -1;
    int rc = guard([&] {
        const std::vector<std::string> parts = g_aligner.tsv_batch();
        size_t total = 0;
        for (const std::string& s : parts) total += s.size();
        n = (long long)total;
        if (!out) return;                                   // size only (timing the formatter without the copy)
        if (total + 1 > cap) throw Error(NPH_ERR_INVALID, "text buffer too small");
        char* o = out;
        for (const std::string& s : parts) { std::memcpy(o, s.data(), s.size()); o += s.size(); }
        *o = 0;
    });
    return rc ? rc : n;
}

// format_fixed against the C library on n float bit patterns drawn from `seed` (uniform bit patterns, then values
// near printed-digit ties): returns the number of mismatches
long long nphh_format_fixed_check(uint64_t seed, size_t n)
{
    long long bad = 0;
    uint64_t x = seed * 2862933555777941757ull + 3037000493ull;
    char a[512], b[512];
    for (size_t i = 0; i < n; ++i) {
        x ^= x << 13; x ^= x >> 7; x ^= x << 17;
        float v;
        uint32_t bits = (uint32_t)(x >> 16);
        if (i % 3 == 1) {                       // magnitudes eventalign prints: 1e-4 .. 1e3, often an exact multiple of a small power of two
            const int q = (int)((x >> 8) & 0xffff) - 32768;
            v = (float)q / (float)(1 << ((x >> 48) & 15));
            if ((x >> 60) & 1) v = std::nextafterf(v, 1e9f);
        } else if (i % 3 == 2) {                // decimal ties and their float neighbours
            const int q = (int)((x >> 8) & 0xfffff);
            v = (float)((q + 0.5) / 1000.0);
            if ((x >> 62) & 1) v = -v;
        } else {
            std::memcpy(&v, &bits, 4);
        }
        for (int prec = 0; prec <= 5; ++prec) {
            format_fixed(a, v, prec);
            snprintf(b, sizeof(b), "%.*lf", prec, (double)v);
            if (std::strcmp(a, b) != 0) { if (bad < 5) g_err = std::string("format_fixed: ") + a + " vs " + b; ++bad; }
        }
        // doubles: sums/differences of floats (the log-likelihood columns), values next to decimal ties, raw bit patterns
        double d;
        if (i % 3 == 0) { std::memcpy(&d, &x, 8); }
        else if (i % 3 == 1) { float w; uint32_t wb = (uint32_t)(x >> 7); std::memcpy(&w, &wb, 4); d = (double)v + (double)w; if (!(std::fabs(d) < 1e15)) d = (double)v - 123.456; }
        else d = std::nextafter((double)((long long)(x >> 40)) / 1000.0 + 0.0005, (x & 1) ? 1e300 : -1e300);
        for (int prec = 0; prec <= 3; ++prec) {
            format_fixed(a, d, prec);
            snprintf(b, sizeof(b), "%.*lf", prec, d);
            if (std::strcmp(a, b) != 0) { if (bad < 5) g_err = std::string("format_fixed(double): ") + a + " vs " + b; ++bad; }
        }
    }
    return bad;
}

// rolling_kmer_ranks against Alphabet::kmer_rank on every k-mer of seq: number of mismatches
long long nphh_rolling_ranks_check(const char* alphabet, const char* seq, uint32_t k)
{
    long long bad = -1;
    int rc = guard([&] {
        const Alphabet* a = get_alphabet_by_name(alphabet);
        const std::string s(seq);
        std::vector<uint32_t> r(s.size() >= k ? s.size() - k + 1 : 0);
        rolling_kmer_ranks(a, s, k, r.data());
        bad = 0;
        for (size_t i = 0; i < r.size(); ++i) bad += r[i] != a->kmer_rank(s.c_str() + i, k);
    });
    return rc ? rc : bad;
}

// EventAligner::summarize: {events, steps, stays, skips, span} and {sum_duration, sum_z_score}
int nphh_ea_summary(int idx, int32_t* ints5, double* doubles2)
{
    return guard([&] {
        const EventalignSummary sm = g_aligner.summarize((size_t)idx);
        ints5[0] = sm.num_events; ints5[1] = sm.num_steps; ints5[2] = sm.num_stays; ints5[3] = sm.num_skips; ints5[4] = sm.reference_span;
        doubles2[0] = sm.sum_duration; doubles2[1] = sm.sum_z_score;
    });
}

long long nphh_ea_num_segments(int idx) { return (long long)g_aligner.num_segments(idx); }

// ---- scorereads: model_score over the reads queued in the aligner (after nphh_ea_run / the CPU round driver) ------------
// mode 0: enumerate only — jobs_out / ranks_out receive the job list (job.read = aligner read index of each job's read is NOT
// rewritten: reads are deduplicated by SquiggleRead); mode 1: also run on the device, scores3_out[3 * i] = {score, n_events,
// n_segments} per read.  ref_seqs[i] / ref_offsets[i]: the fetched reference of read i.  Returns the number of jobs.
long long nphh_scorereads(int n_reads, const int32_t* read, const char** ref_seqs, const int32_t* ref_offsets, int events_per_segment, int mode,
                          void* jobs_out, size_t cap_jobs, uint32_t* ranks_out, size_t cap_ranks, uint64_t* n_ranks_out, double* scores3_out)
{
    long long n = -1;
    int rc = guard([&] {
        ScoreReads sr((size_t)events_per_segment);
        for (int i = 0; i < n_reads; ++i) sr.add_read(*g_reads[read[i]], 0, g_aligner.alignment((size_t)i), ref_seqs[i], ref_offsets[i]);
        const HmmBatch& b = sr.batch();
        n = (long long)b.jobs().size();
        if (jobs_out && ranks_out) {
            const std::vector<uint32_t> rk = b.ranks();
            if (b.jobs().size() > cap_jobs || rk.size() > cap_ranks) throw Error(NPH_ERR_INVALID, "dump buffers too small");
            std::memcpy(jobs_out, b.jobs().data(), sizeof(nph_hmm_job) * b.jobs().size());
            std::memcpy(ranks_out, rk.data(), sizeof(uint32_t) * rk.size());
            *n_ranks_out = rk.size();
        }
        if (mode == 1) {
            sr.run(Engine::thread_default());
            for (int i = 0; i < n_reads; ++i) {
                scores3_out[3 * i] = sr.score((size_t)i).score;
                scores3_out[3 * i + 1] = (double)sr.score((size_t)i).n_events;
                scores3_out[3 * i + 2] = (double)sr.score((size_t)i).n_segments;
            }
        }
    });
    return rc ? rc : n;
}

// get_aligned_segments on a packed CIGAR: pairs_out = (ref_pos, read_pos) interleaved, seg_off[n_segments + 1]
long long nphh_aligned_segments(int ref_pos, const uint32_t* cigar, int n_cigar, int32_t* pairs_out, size_t cap_pairs, uint64_t* seg_off, size_t cap_segs)
{
    long long n = -1;
    int rc = guard([&] {
        std::vector<AlignedSegment> segs = get_aligned_segments(ref_pos, std::vector<uint32_t>(cigar, cigar + n_cigar));
        if (segs.size() + 1 > cap_segs) throw Error(NPH_ERR_INVALID, "segment buffer too small");
        size_t o = 0;
        seg_off[0] = 0;
        for (size_t i = 0; i < segs.size(); ++i) {
            if (o + segs[i].size() > cap_pairs) throw Error(NPH_ERR_INVALID, "pair buffer too small");
            for (const AlignedPair& p : segs[i]) { pairs_out[2 * o] = p.ref_pos; pairs_out[2 * o + 1] = p.read_pos; ++o; }
            seg_off[i + 1] = o;
        }
        n = (long long)segs.size();
    });
    return rc ? rc : n;
}

// ---- N5: polya ------------------------------------------------------------------------------------------------
// PolyaEstimator over the reads [first_read, first_read + n) of g_reads (names from SquiggleRead::read_name, one contig):
// add_read / run / tsv.  Returns the TSV's length (written to out if it fits cap) or a negative status.
long long nphh_polya_tsv(int first_read, int n, const char* contig, const int32_t* positions, const uint16_t* flags,
                         const uint32_t* suffix_clip, int header, char* out, size_t cap)
{
    long long len = -1;
    int rc = guard([&] {
        PolyaEstimator est;
        for (int i = 0; i < n; ++i) {
            const SquiggleRead& sr = *g_reads[first_read + i];
            est.add_read(PolyaRecord{sr.read_name, contig, positions[i], flags[i], suffix_clip[i]}, sr);
        }
        est.run(Engine::thread_default());
        const std::string t = est.tsv(header != 0);
        if (t.size() <= cap) memcpy(out, t.data(), t.size());
        len = (long long)t.size();
    });
    return rc ? rc : len;
}

// polya_from_raw over raw reads given as nphh_load_from_raw takes them (reads named "read<i>", nucleotide type from
// nphh_set_rna); returns the TSV's length (written to out if it fits cap) or a negative status
long long nphh_polya_from_raw(int model, int n, const float* samples, const uint64_t* sample_off, const char* seqs, const uint64_t* seq_off,
                              double sample_rate, const char* contig, const int32_t* positions, const uint16_t* flags,
                              const uint32_t* suffix_clip, int header, char* out, size_t cap)
{
    long long len = -1;
    int rc = guard([&] {
        std::vector<RawRead> raw(n);
        std::vector<PolyaRecord> recs(n);
        for (int i = 0; i < n; ++i) {
            raw[i].read_name = "read" + std::to_string(i);
            raw[i].read_sequence.assign(seqs + seq_off[i], seqs + seq_off[i + 1]);
            raw[i].samples.assign(samples + sample_off[i], samples + sample_off[i + 1]);
            raw[i].sample_rate = sample_rate;
            raw[i].nucleotide_type = g_raw_is_rna ? SRNT_RNA : SRNT_DNA;
            recs[i] = PolyaRecord{raw[i].read_name, contig, positions[i], flags[i], suffix_clip[i]};
        }
        const std::string t = polya_from_raw(Engine::thread_default(), *g_models[model], raw, recs, header != 0);
        if (t.size() <= cap) memcpy(out, t.data(), t.size());
        len = (long long)t.size();
    });
    return rc ? rc : len;
}

} // extern "C"

