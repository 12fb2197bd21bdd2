/* nph.h — C ABI of the B200-native nanopolish HMM engine (libnph.so).
 *
 * This is the drop-in boundary for the ONE hot path this repository accelerates
 * (SURVEY.md section 8):
 *
 *   1. the R9 profile-HMM forward score
 *        profile_hmm_score            ref: src/hmm/nanopolish_profile_hmm.cpp:23-30
 *        profile_hmm_score_r9         ref: src/hmm/nanopolish_profile_hmm_r9.cpp:35-65
 *        profile_hmm_fill_generic_r9  ref: src/hmm/nanopolish_profile_hmm_r9.inl:265-433
 *        profile_hmm_score_set        ref: src/hmm/nanopolish_profile_hmm.cpp:32-56
 *   2. the adaptive banded event-to-sequence alignment
 *        adaptive_banded_simple_event_align   ref: src/nanopolish_raw_loader.cpp:77-379
 *        estimate_scalings_using_mom          ref: src/nanopolish_raw_loader.cpp:17-60
 *   3. (section 8f "next" row N1) the Viterbi alignment with the same fill
 *        profile_hmm_align_r9         ref: src/hmm/nanopolish_profile_hmm_r9.cpp:73-204
 *   4. (row N4) the raw-signal prologue that produces the reads the calls above consume
 *        SquiggleRead::load_from_raw  ref: src/nanopolish_squiggle_read.cpp:226-336
 *        trim_and_segment_raw         ref: src/thirdparty/scrappie/scrappie_common.c:122-190
 *        detect_events                ref: src/thirdparty/scrappie/event_detection.c:268-319
 *        recalibrate_model            ref: src/nanopolish_methyltrain.cpp:204-307
 *
 * The reference has no FFI layer: its seam is those C++ free functions, called with
 * HMMInputData / HMMInputSequence / SquiggleRead.  The C++ mirror of that call surface
 * lives in nanopolish_b200/host/ and lowers onto the functions below; INTEGRATION.md shows
 * the binding a nanopolish maintainer would add.
 *
 * Conventions
 *   - plain C, plain pointers and sizes; no C++/torch/CUDA types in any signature
 *     (a CUDA stream is passed as void*).
 *   - every function returns NPH_OK (0) or a negative nph_status; nothing throws, nothing
 *     calls exit().  nph_strerror() gives a message, nph_last_error(ctx) the CUDA detail.
 *   - the caller owns every host buffer for the duration of the call; the context owns
 *     all device memory.  A context is bound to one device and one stream and must not be
 *     used from two threads at once (use one context per OpenMP thread, or a mutex).
 *   - there is NO CPU fallback: without a CUDA device nph_create() fails with
 *     NPH_ERR_NO_DEVICE and nothing else can be called.
 *   - results are bit-identical to the reference's float arithmetic (same operation order,
 *     same quantised table logsum, IEEE add/mul/div, no FMA contraction); see DESIGN.md.
 */
#ifndef NPH_H
#define NPH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NPH_VERSION_MAJOR 0
#define NPH_VERSION_MINOR 1

typedef enum {
    NPH_OK = 0,
    NPH_ERR_NO_DEVICE = -1,   /* no usable CUDA device / driver: there is no CPU path */
    NPH_ERR_CUDA = -2,        /* a CUDA runtime call failed; see nph_last_error */
    NPH_ERR_INVALID = -3,     /* bad argument (null pointer, out-of-range index, ...) */
    NPH_ERR_NOMEM = -4,       /* device or host allocation failed */
    NPH_ERR_STATE = -5,       /* call sequence error (e.g. score before load) */
    NPH_ERR_UNSUPPORTED = -6  /* a shape the kernels do not handle (documented limits) */
} nph_status;

/* flags of profile_hmm_score / profile_hmm_align.
 * ref: src/hmm/nanopolish_profile_hmm.h:34-38 (HAF_ALLOW_PRE_CLIP, HAF_ALLOW_POST_CLIP) */
#define NPH_HAF_ALLOW_PRE_CLIP  1u
#define NPH_HAF_ALLOW_POST_CLIP 2u

typedef struct nph_ctx nph_ctx;

/* One strand of one SquiggleRead: the part of it the hot path reads.
 * ref: SquiggleRead::events[strand] (src/nanopolish_squiggle_read.h:277-299),
 *      SquiggleScalings (:63-93), events_per_base[strand] (:293). 64 bytes. */
typedef struct {
    uint64_t event_off;       /* first event of this read in ev_mean[] / ev_start_time[] */
    uint32_t n_events;
    uint32_t reserved;
    double scale;             /* SquiggleScalings::scale   */
    double shift;             /*                 ::shift   */
    double drift;             /*                 ::drift   */
    double var;               /*                 ::var     */
    double log_var;           /*                 ::log_var (= log(var), cached by set4/set6) */
    double events_per_base;   /* SquiggleRead::events_per_base[strand] */
} nph_read;

/* One profile_hmm_score call == one (HMMInputSequence, HMMInputData, flags) triple.
 * ref: HMMInputData (src/common/nanopolish_common.h:53-62).  The sequence is passed as the
 * k-mer ranks HMMInputSequence::get_kmer_rank(ki, k, rc) returns for ki = 0..n_kmers-1
 * (src/hmm/nanopolish_hmm_input_sequence.h:76-91), i.e. already strand-resolved. 32 bytes. */
typedef struct {
    uint64_t rank_off;        /* first k-mer rank of this job in kmer_ranks[] */
    uint32_t read;            /* index into reads[] */
    uint32_t model_id;        /* from nph_model_upload: HMMInputData::pore_model */
    uint32_t event_start;     /* HMMInputData::event_start_idx */
    uint32_t event_stop;      /* HMMInputData::event_stop_idx (inclusive) */
    uint32_t n_kmers;         /* sequence.length() - k + 1 */
    int8_t   stride;          /* HMMInputData::event_stride: +1, or -1 when event_stop < event_start */
    uint8_t  rc;              /* HMMInputData::rc (informational: ranks are already resolved) */
    uint8_t  flags;           /* NPH_HAF_* */
    uint8_t  reserved;
} nph_hmm_job;

/* One adaptive_banded_simple_event_align call: a whole read against its basecalled sequence. */
typedef struct {
    uint64_t rank_off;        /* first k-mer rank (forward strand, alphabet->kmer_rank) in kmer_ranks[] */
    uint64_t pairs_off;       /* where this read's AlignedPairs go in pairs_out[] (in pairs) */
    uint32_t read;            /* index into reads[] (scalings as set by the MoM estimate: drift 0, var 1) */
    uint32_t n_kmers;
    uint32_t pairs_cap;       /* room at pairs_off, in pairs; n_events + n_kmers always suffices */
    uint32_t reserved;
} nph_abea_job;

/* ref: AlignedPair (src/alignment/nanopolish_anchor.h:18-22) */
typedef struct { int32_t ref_pos; int32_t read_pos; } nph_aligned_pair;

/* status of one ABEA job.  The reference returns an empty vector for every failure
 * (src/nanopolish_raw_loader.cpp:365-372); n_pairs is 0 in exactly those cases. */
#define NPH_ABEA_OK              0
#define NPH_ABEA_LOW_EMISSION    1   /* avg_log_emission < -5.0 */
#define NPH_ABEA_NOT_SPANNED     2   /* path does not run from k-mer 0 to k-mer n_kmers-1 */
#define NPH_ABEA_MAX_GAP         4   /* more than 50 consecutive skipped k-mers */
#define NPH_ABEA_NO_END_CELL     8   /* last k-mer column never inside the band (reference behaviour undefined) */
#define NPH_ABEA_PAIRS_OVERFLOW 16   /* pairs_cap too small */
typedef struct {
    uint32_t n_pairs;         /* 0 when the reference would have returned an empty vector */
    int32_t  status;          /* bit-or of NPH_ABEA_* */
    int32_t  max_gap;
    uint32_t n_aligned;       /* path length before QC (== n_pairs when status == 0) */
    double   avg_log_emission;
} nph_abea_result;

/* One Viterbi state of profile_hmm_align.  ref: HMMAlignmentState (src/common/nanopolish_common.h:65-73);
 * l_posterior and log_transition_probability are left for the host wrapper (section 8f N1). */
typedef struct {
    uint32_t event_idx;
    uint32_t kmer_idx;
    float    l_fm;
    char     state;           /* 'M', 'B' (bad event) or 'K' (k-mer skip) */
    uint8_t  reserved[3];
} nph_align_state;

/* ---- context ------------------------------------------------------------------------- */

/* Create a context on CUDA device `device` with its own non-blocking stream. */
int nph_create(nph_ctx** ctx_out, int device);
/* Same, but run everything on the caller's stream (a cudaStream_t passed as void*; NULL = legacy
 * default stream).  Lets a host framework time/sequence the kernels with its own events. */
int nph_create_on_stream(nph_ctx** ctx_out, int device, void* cuda_stream);
int nph_destroy(nph_ctx* ctx);
const char* nph_strerror(int status);
const char* nph_last_error(const nph_ctx* ctx);
int nph_version(void);                              /* major*1000 + minor */
int nph_sync(nph_ctx* ctx);                         /* wait for everything queued on the context's stream */
void* nph_stream(nph_ctx* ctx);                     /* the cudaStream_t the kernels run on */

/* PoreModel::states as three parallel arrays (level_mean, level_stdv, level_log_stdv).
 * ref: PoreModelStateParams (src/pore_model/nanopolish_poremodel.h:20-36). Uploaded once per model. */
int nph_model_upload(nph_ctx* ctx, const double* level_mean, const double* level_stdv,
                     const double* level_log_stdv, uint32_t n_states, uint32_t k,
                     uint32_t alphabet_size, uint32_t* model_id_out);

/* ---- profile_hmm_score ------------------------------------------------------------------
 * One-shot form, host buffers in, host scores out (synchronous):
 *   scores_out[j] == profile_hmm_score(sequence_j, data_j, flags_j)   for j in [0, n_jobs)
 * with hmm_indel_bias_factor (src/hmm/nanopolish_profile_hmm_r9.cpp:19) == indel_bias.
 * A job with event range or k-mer count the reference would assert on yields NPH_ERR_INVALID. */
int nph_hmm_score_batch(nph_ctx* ctx,
                        const nph_read* reads, size_t n_reads,
                        const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                        const uint32_t* kmer_ranks, size_t n_ranks_total,
                        const nph_hmm_job* jobs, size_t n_jobs,
                        double indel_bias, float* scores_out);

/* Staged form of the same computation, for callers that keep a batch resident in HBM
 * (bench.py's device-resident timing, multi-GPU shards, repeated scoring with new jobs):
 *   nph_reads_load   : H2D of events + scalings, then the per-read device prologue
 *                      (drift-scaled levels get_drift_scaled_level, squiggle_read.h:149-154;
 *                       transitions calculate_transitions, profile_hmm_r9.inl:17-76)
 *   nph_hmm_jobs_load: H2D of ranks + jobs, scheduling order
 *   nph_hmm_score    : launches the forward kernel(s) on the context's stream (asynchronous);
 *                      scores go to scores_dev if non-NULL (device pointer, n_jobs floats)
 *                      else to an internal device buffer
 *   nph_hmm_scores_fetch: D2H of the internal score buffer + stream sync                    */
int nph_reads_load(nph_ctx* ctx, const nph_read* reads, size_t n_reads,
                   const float* ev_mean, const double* ev_start_time, size_t n_events_total);
int nph_hmm_jobs_load(nph_ctx* ctx, const uint32_t* kmer_ranks, size_t n_ranks_total,
                      const nph_hmm_job* jobs, size_t n_jobs, double indel_bias);
int nph_hmm_score(nph_ctx* ctx, float* scores_dev);
int nph_hmm_scores_fetch(nph_ctx* ctx, float* scores_out, size_t n_jobs);

/* The same computation with the sequences as BASE CODES instead of k-mer ranks — one byte per base on the wire and in HBM instead
 * of four per k-mer; the forward kernel forms each k-mer's rank from the codes while it scales the k-mer's Gaussian.
 * seq_codes holds, per job, the alphabet ranks Alphabet::rank(c) of the n_kmers + k - 1 symbols of the string the job's strand
 * reads: HMMInputSequence's m_seq for rc == 0, its m_rc_seq for rc == 1 (so that k-mer i is what get_kmer_rank(i, k, rc)
 * ranks: the k symbols at i, resp. at length - i - k; src/hmm/nanopolish_hmm_input_sequence.h:76-91).  In these calls
 * nph_hmm_job::rank_off is the offset of the job's first code in seq_codes, and nph_hmm_job::rc selects the direction.
 * A code outside the job's model alphabet yields NPH_ERR_INVALID. */
int nph_hmm_score_batch_seq(nph_ctx* ctx,
                            const nph_read* reads, size_t n_reads,
                            const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                            const uint8_t* seq_codes, size_t n_codes_total,
                            const nph_hmm_job* jobs, size_t n_jobs,
                            double indel_bias, float* scores_out);
int nph_hmm_jobs_load_seq(nph_ctx* ctx, const uint8_t* seq_codes, size_t n_codes_total,
                          const nph_hmm_job* jobs, size_t n_jobs, double indel_bias);

/* profile_hmm_score_set (ref: src/hmm/nanopolish_profile_hmm.cpp:32-56): combine the per-sequence
 * scores of each group of n_alt consecutive jobs, host side, in double through the table logsum:
 *   out[g] = (+)_i ( scores[g*n_alt + i] - log(n_alt) ).  Pure host arithmetic on fetched scores. */
int nph_score_set_combine(const float* scores, size_t n_groups, uint32_t n_alt, float* out);

/* ---- adaptive_banded_simple_event_align -------------------------------------------------
 * One-shot, host buffers (synchronous). pairs_out receives, for job j, results[j].n_pairs
 * AlignedPairs at pairs_out + jobs[j].pairs_off in the reference's order (ascending). */
int nph_abea_batch(nph_ctx* ctx,
                   const nph_read* reads, size_t n_reads,
                   const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                   const uint32_t* kmer_ranks, size_t n_ranks_total,
                   const nph_abea_job* jobs, size_t n_jobs, uint32_t model_id,
                   nph_aligned_pair* pairs_out, size_t pairs_total, nph_abea_result* results);
/* Staged form (reads via nph_reads_load). */
int nph_abea_jobs_load(nph_ctx* ctx, const uint32_t* kmer_ranks, size_t n_ranks_total,
                       const nph_abea_job* jobs, size_t n_jobs, uint32_t model_id, size_t pairs_total);
int nph_abea_run(nph_ctx* ctx);
int nph_abea_fetch(nph_ctx* ctx, nph_aligned_pair* pairs_out, size_t pairs_total,
                   nph_abea_result* results, size_t n_jobs);

/* estimate_scalings_using_mom for each job's read/sequence: out[j] = {shift, scale} (drift 0, var 1). */
int nph_mom_batch(nph_ctx* ctx, const nph_read* reads, size_t n_reads,
                  const float* ev_mean, size_t n_events_total,
                  const uint32_t* kmer_ranks, size_t n_ranks_total,
                  const nph_abea_job* jobs, size_t n_jobs, uint32_t model_id, double* shift_scale_out);

/* ---- profile_hmm_align (Viterbi; section 8f N1) ------------------------------------------
 * states_out receives, for job j, n_states_out[j] HMMAlignmentStates at states_out + states_off[j] in ascending
 * event order; states_off has n_jobs + 1 entries and states_off[j+1] - states_off[j] is the room for job j
 * (n_events + n_kmers always suffices).  n_states_out[j] == 0 where the reference would trip an assert (fewer
 * than two events, or the best path runs into a -inf cell).  scores_out (optional) = l_fm of the last state.
 * Limit: the movement trace of the batch's largest window, 2 * (E + K/C + 1) * 32*C bytes per warp (C = 1..8 columns per
 * lane), is kept for every resident warp; the number of resident warps shrinks so that the arena stays within 16 GiB, and a
 * window that needs more than that for a single CTA of 16 warps (E*K beyond ~1.6e7) returns NPH_ERR_UNSUPPORTED.
 * ref: profile_hmm_align_r9, src/hmm/nanopolish_profile_hmm_r9.cpp:73-204. */
int nph_hmm_align_batch(nph_ctx* ctx,
                        const nph_read* reads, size_t n_reads,
                        const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                        const uint32_t* kmer_ranks, size_t n_ranks_total,
                        const nph_hmm_job* jobs, size_t n_jobs, double indel_bias,
                        nph_align_state* states_out, const uint64_t* states_off,
                        uint32_t* n_states_out, float* scores_out);
/* The same against the reads a preceding nph_reads_load left resident in HBM: eventalign re-aligns one ~100-base
 * segment per read per round (align_read_to_ref, src/alignment/nanopolish_eventalign.cpp:691-823), each round's
 * jobs depending on the previous round's paths, so the events go up once and only jobs/states travel per round. */
int nph_hmm_align(nph_ctx* ctx,
                  const uint32_t* kmer_ranks, size_t n_ranks_total,
                  const nph_hmm_job* jobs, size_t n_jobs, double indel_bias,
                  nph_align_state* states_out, const uint64_t* states_off,
                  uint32_t* n_states_out, float* scores_out);

/* ---- eventalign: a read's whole segment chain on the device (section 8f N1) ------------------------------
 * align_read_to_ref (src/alignment/nanopolish_eventalign.cpp:612-827) walks one BAM-aligned segment of a read in
 * ~100-base steps: pick the aligned pair ~100 reference bases ahead (get_end_pair :196-207), the event nearest to its
 * read k-mer (SquiggleRead::get_closest_event_to, src/nanopolish_squiggle_read.cpp:160-186), profile_hmm_align over
 * that window, emit up to 50 event alignments (all of them in the last section), restart from the last one emitted.
 * Each step depends on the previous path, so one warp walks one chain from start to end: cursor, Viterbi fill,
 * backtrack and emission stay on the device, and a batch of reads is ONE launch instead of one per step.
 * A chain is one BAM segment (the pieces between N operations) of one read strand, already trimmed to the region and
 * to the read's last k-mer by the caller (trim_aligned_pairs_to_ref_region / _to_kmer, :166-193).
 * Reads: the batch a preceding nph_reads_load left resident. */
typedef struct {
    uint64_t pair_off;        /* this segment's aligned pairs (ref_pos ascending, read_pos = BAM query k-mer) in pairs[] */
    uint64_t map_off;         /* the read's base_to_event_map[*].indices[strand].start in event_map_start[] (-1: none) */
    uint64_t rank_off;        /* the record's reference in ref_ranks_fwd[] / ref_ranks_rc[]: entry p = rank of the k-mer at
                                 reference offset p (fwd) / of its reverse complement as HMMInputSequence resolves it (rc) */
    uint64_t out_off;         /* where this chain's records go in records_out[] */
    uint32_t read;            /* index into the resident reads */
    uint32_t model_id;
    uint32_t n_pairs;
    uint32_t map_len;         /* base_to_event_map.size() */
    uint32_t ref_len;         /* ref_seq.length(); ref_len - k + 1 rank entries */
    uint32_t read_seq_len;    /* read_sequence.size() (SquiggleRead::flip_k_strand) */
    uint32_t out_cap;         /* room at out_off; abs(last_event - first_event) + 2 always suffices */
    int32_t  ref_offset;      /* record->core.pos */
    int32_t  first_event;     /* get_closest_event_to of the segment's first pair (after flip_k_strand if reversed) */
    int32_t  last_event;      /* ... of its last pair */
    uint8_t  do_base_rc;      /* bam_is_rev(record) */
    uint8_t  rc;              /* HMMInputData::rc == rc_flags[strand] */
    uint8_t  k;
    uint8_t  reserved;
} nph_ea_chain;
/* one EventAlignment (src/alignment/nanopolish_eventalign.h:54-71) without its strings: ref_kmer and model_kmer are
 * substrings of the reference at ref_position (model_kmer reverse-complemented for rc reads, NNNNNN for 'B') */
typedef struct { int32_t ref_position; int32_t event_idx; uint8_t hmm_state; uint8_t reserved[3]; } nph_ea_record;
#define NPH_EA_OK               0
#define NPH_EA_WINDOW_TOO_LARGE 1   /* a window has more k-mers or events than the kernel's single-strip scratch holds:
                                       re-run this read through nph_hmm_align rounds (records so far are valid) */
#define NPH_EA_RC_STRIDE        2   /* event order disagrees with rc (the reference asserts, profile_hmm_r9.inl:275) */
#define NPH_EA_OUT_OVERFLOW     4   /* out_cap too small */
#define NPH_EA_BAD_EVENT        8   /* a cursor event lies outside the read */
typedef struct { uint32_t n_records; uint32_t n_windows; int32_t status; uint32_t reserved; } nph_ea_result;
int nph_eventalign_chain(nph_ctx* ctx,
                         const nph_aligned_pair* pairs, size_t n_pairs_total,
                         const int32_t* event_map_start, size_t n_map_total,
                         const uint32_t* ref_ranks_fwd, const uint32_t* ref_ranks_rc, size_t n_ranks_total,
                         const nph_ea_chain* chains, size_t n_chains, double indel_bias,
                         nph_ea_record* records_out, size_t records_total, nph_ea_result* results_out);

/* ---- call-methylation: window enumeration + both scores per motif group on the device (section 8f N3) -----
 * calculate_methylation_for_read (src/basemods/nanopolish_basemods.cpp:238-457) from "Scan the sequence for motifs"
 * (:301) to the two profile_hmm_score calls (:383-392), for a whole BamProcessor batch in one call: the motif scan,
 * the grouping of sites closer than min_separation, the window (min_flank either side, span <= max_span, not within
 * min_separation of the alignment start), AlignmentDB::_find_by_ref_bounds on the read's event alignment
 * (src/alignment/nanopolish_alignment_db.cpp:688-731), the region filter, the unmethylated / methylated
 * HMMInputSequence pair (Alphabet::methylate, reverse_complement with its methylated-site units) as k-mer ranks, and the
 * two forward scores.  Nothing O(bases) or O(groups) is left to the host: it hands over the reference substring and
 * the event alignment of each (record, strand) and receives one nph_meth_site per scored group.
 * A record = one BAM record x one strand of its read.  ref_bases holds ref_seq of every record: the reference over
 * [record->core.pos, bam_endpos], already through gDNAAlphabet.disambiguate() (upper-case ACGT).  aligned_events holds
 * EventAlignmentRecord::aligned_events (ref_pos ascending, read_pos = event index; alignment_db.cpp:50-91). */
#define NPH_METH_MAX_SITES 4
#define NPH_METH_MAX_SITE_LEN 8
#define NPH_METH_MAX_WINDOW 1024     /* max_span + 2 * min_flank + 1 must not exceed this */
typedef struct {
    uint64_t ref_off;         /* first base of this record's ref_seq in ref_bases[] */
    uint64_t pair_off;        /* first aligned_events entry in aligned_events[] */
    uint32_t read;            /* index into reads[]: events[strand] of the record's SquiggleRead */
    uint32_t model_id;        /* sr.get_model(strand, methylation_type): the model over the methylation alphabet */
    uint32_t ref_len;         /* ref_seq.size() */
    uint32_t n_pairs;
    int32_t  ref_start_pos;   /* record->core.pos */
    uint8_t  rc;              /* EventAlignmentRecord::rc -> HMMInputData::rc */
    uint8_t  strand;          /* informational (sites of the two strands of one read are merged by the caller) */
    uint8_t  reserved[2];
} nph_meth_record;            /* 40 bytes */
typedef struct {
    int32_t  min_separation;  /* MethylationCallingParameters::min_separation (10), basemods.h:56 */
    int32_t  min_flank;       /* ::min_flank (10) */
    int32_t  max_span;        /* 200: groups spanning more are skipped, basemods.cpp:336 */
    int32_t  min_event_span;  /* 10: abs(e2 - e1) <= 10 skips the group, :363 */
    int32_t  region_start;    /* -1: no restriction (the -w window), :398-401 */
    int32_t  region_end;
    uint32_t k;               /* sr.get_model_k(strand) */
    uint32_t alphabet_size;   /* of the methylation alphabet (5 for cpg: ACGMT) */
    char     bases[8];        /* its symbols in rank order, NUL padded ("ACGMT") */
    char     complements[8];  /* complement of each symbol, same order ("TGCGA") */
    uint32_t n_sites;         /* Alphabet::num_recognition_sites() (1 for cpg, 2 for dcm) */
    uint32_t site_len;        /* Alphabet::recognition_length() */
    char     sites[NPH_METH_MAX_SITES][NPH_METH_MAX_SITE_LEN];                        /* get_recognition_site(i): "CG" */
    char     sites_methylated[NPH_METH_MAX_SITES][NPH_METH_MAX_SITE_LEN];             /* ..._methylated(i): "MG" */
    char     sites_methylated_complement[NPH_METH_MAX_SITES][NPH_METH_MAX_SITE_LEN];  /* ..._methylated_complement(i): "GM" */
} nph_meth_params;
/* One scored group of one record == the strand-specific half of a ScoredSite (basemods.h:25-43). */
typedef struct {
    int32_t  start_position;  /* first motif site of the group, reference coordinates */
    int32_t  end_position;    /* last motif site of the group */
    uint32_t n_motif;
    uint32_t record;          /* index into records[] */
    float    ll_unmethylated; /* profile_hmm_score(unmethylated, data, PRE_CLIP | POST_CLIP) */
    float    ll_methylated;
} nph_meth_site;              /* 24 bytes */
/* One-shot: host buffers in, host sites out (synchronous).  site_off_out has n_records + 1 entries: the sites of
 * record r are sites_out[site_off_out[r] .. site_off_out[r+1]) in ascending start_position.  sites_cap is the room in
 * sites_out; sum over records of (ref_len / (min_separation + 1) + 2) always suffices, NPH_ERR_INVALID if it was too
 * small (nph_last_error says how many were needed).  n_scored_events_out (optional): sum over groups of 2 * (abs(e2 - e1) + 1),
 * the unit of the events/s metric.  A group whose event indices lie outside its read (the reference would read out of
 * bounds) or whose clamped window is shorter than k yields NPH_ERR_INVALID. */
int nph_methylation_batch(nph_ctx* ctx,
                          const nph_read* reads, size_t n_reads,
                          const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                          const char* ref_bases, size_t n_ref_total,
                          const nph_aligned_pair* aligned_events, size_t n_pairs_total,
                          const nph_meth_record* records, size_t n_records,
                          const nph_meth_params* params, double indel_bias,
                          uint64_t* site_off_out, nph_meth_site* sites_out, size_t sites_cap,
                          uint64_t* n_scored_events_out);
/* The same with the event alignments in COMPACT form — 2 bytes per reference base instead of 8 per aligned pair, which matters
 * because this call is PCIe bound (the event alignment is larger than the events themselves).  event_deltas runs parallel to
 * ref_bases (entry ref_off + o belongs to reference offset o of the record): NPH_METH_NO_PAIR where aligned_events has no entry
 * with ref_pos == ref_start_pos + o (a deleted reference base, the record's boundary k-mers), else that entry's event index
 * minus the event index of the previous entry (minus first_event[record] for the record's first entry).  The device rebuilds
 * the (ref_pos, event index) list by a prefix sum; results are identical to the pair form.  records[].pair_off / n_pairs are
 * ignored.  Requires strictly increasing ref_pos inside a record (true of every EventAlignmentRecord) and event-index steps
 * that fit an int16 (a caller that meets a larger step uses the pair form). */
#define NPH_METH_NO_PAIR (-32768)
int nph_methylation_batch_compact(nph_ctx* ctx,
                                  const nph_read* reads, size_t n_reads,
                                  const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                                  const char* ref_bases, const int16_t* event_deltas, size_t n_ref_total,
                                  const int32_t* first_event,
                                  const nph_meth_record* records, size_t n_records,
                                  const nph_meth_params* params, double indel_bias,
                                  uint64_t* site_off_out, nph_meth_site* sites_out, size_t sites_cap,
                                  uint64_t* n_scored_events_out);
int nph_methylation_load_compact(nph_ctx* ctx, const char* ref_bases, const int16_t* event_deltas, size_t n_ref_total,
                                 const int32_t* first_event, const nph_meth_record* records, size_t n_records,
                                 const nph_meth_params* params, double indel_bias);
/* Staged form against the reads a preceding nph_reads_load left resident:
 *   nph_methylation_load : H2D of the reference bases, event alignments and records
 *   nph_methylation_run  : enumerate -> schedule -> score -> fill the site records, all on the device
 *                          (two small read-backs inside: the counts that size the job arrays, the schedule summary)
 *   nph_methylation_fetch: D2H of the offsets and site records */
int nph_methylation_load(nph_ctx* ctx, const char* ref_bases, size_t n_ref_total,
                         const nph_aligned_pair* aligned_events, size_t n_pairs_total,
                         const nph_meth_record* records, size_t n_records,
                         const nph_meth_params* params, double indel_bias);
int nph_methylation_run(nph_ctx* ctx);
/* counts of the most recent nph_methylation_run: scored groups, forward jobs (2 per group), scored events */
int nph_methylation_counts(nph_ctx* ctx, uint64_t* n_sites_out, uint64_t* n_jobs_out, uint64_t* n_scored_events_out);
int nph_methylation_fetch(nph_ctx* ctx, uint64_t* site_off_out, nph_meth_site* sites_out, size_t sites_cap);
/* The site records of the most recent nph_methylation_run where they lie in device memory (valid until the next call on
 * this context; ordered behind the run on the context's stream), for a caller that ships them GPU to GPU — a multi-GPU
 * driver gathering every rank's records with NCCL — without a host hop. */
int nph_methylation_sites_dev(nph_ctx* ctx, const nph_meth_site** sites_dev_out, uint64_t* n_sites_out);
/* The rows of methylation_calls.tsv for the most recent nph_methylation_run, formatted on the device — the reference's writer
 * (src/nanopolish_call_methylation.cpp:113-140: chromosome, strand, start, end, read_name, log_lik_ratio, log_lik_methylated,
 * log_lik_unmethylated, num_calling_strands, num_motifs, sequence; "%.2lf" for the three likelihoods) applied to every site
 * record in record order, for records that are their read's only scored strand (num_calling_strands 1; every 1D read).
 * contig: the chromosome name of the batch; read_names + name_off (n_records + 1 offsets into read_names, no terminators):
 * the read name of each record; is_reverse[n_records]: bam1_is_rev of each record ('-' / '+').  tsv_out receives
 * *n_bytes_out bytes (no terminator).  NPH_ERR_INVALID with *n_bytes_out set if cap was too small; NPH_ERR_UNSUPPORTED if a
 * likelihood is not finite or beyond 2^52 (the C library's arbitrary-precision path: fetch the sites and format on the host). */
int nph_methylation_tsv(nph_ctx* ctx, const char* contig, const char* read_names, const uint32_t* name_off,
                        const uint8_t* is_reverse, char* tsv_out, size_t cap, uint64_t* n_bytes_out);
/* One-shot of the whole caller: nph_methylation_batch_compact's inputs in, methylation_calls.tsv rows out (the site
 * records never cross PCIe).  On NPH_ERR_UNSUPPORTED (see nph_methylation_tsv) the batch has been scored: the caller
 * may nph_methylation_fetch the records and format them itself. */
int nph_methylation_batch_compact_tsv(nph_ctx* ctx,
                                      const nph_read* reads, size_t n_reads,
                                      const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                                      const char* ref_bases, const int16_t* event_deltas, size_t n_ref_total,
                                      const int32_t* first_event,
                                      const nph_meth_record* records, size_t n_records,
                                      const nph_meth_params* params, double indel_bias,
                                      const char* contig, const char* read_names, const uint32_t* name_off, const uint8_t* is_reverse,
                                      char* tsv_out, size_t cap, uint64_t* n_bytes_out,
                                      uint64_t* n_sites_out, uint64_t* n_scored_events_out);

/* ---- variants: candidate screening on the device (section 8f N2, BASELINE configs[4]) -----------------------------
 * generate_candidate_single_base_edits (src/nanopolish_call_variants.cpp:288-361) for a reference region: at every position i
 * the window [i - flank, i + 1 + flank] (22 bases for flank 10), up to nine candidate edits of base i — for j in ACGT order
 * the substitution to j and the insertion of j behind it (both skipped when j is the reference base), then the deletion of
 * base i (skipped when it equals base i - 1) — each scored with score_variant_thresholded
 * (src/common/nanopolish_variant.cpp:765-799): over the event sequences of the window
 * (AlignmentDB::get_event_subsequences, src/alignment/nanopolish_alignment_db.cpp:172-221: every record whose event alignment
 * bounds the window, event span below 20 events per base), in record order,
 *     if (fabs(total) < score_threshold) total += profile_hmm_score_set(variant) - profile_hmm_score_set(base)
 * — the reference's single-thread semantics (its `omp parallel for` makes the exit point racy).  The early exit is honoured
 * in the work done: reads are scored reads_per_round at a time, and only candidates whose total is still inside the
 * threshold get jobs in the next round (a candidate that leaves it mid-round ignores the rest of that round, exactly like the
 * sequential loop).  Window enumeration, the k-mer ranks of the ten sequences per position and strand, job emission, the
 * forward scores and the accumulation all run on the device; the host drives the rounds (one count read-back per round).
 * No methylation alternatives (opt::methylation_types empty, the default).
 * Records: nph_meth_record with ref_off = offset of the record's compact event alignment in event_deltas[] (ref_len entries,
 * entry o <-> reference position ref_start_pos + o; NPH_METH_NO_PAIR / steps as in nph_methylation_batch_compact),
 * pair_off / n_pairs unused, model_id = the read's base model.  Record order = AlignmentDB's m_event_records order.
 * ref_bases: the region's reference, ref_bases[p] = base at position region_start + p, n_ref_bases = region_end - region_start + 1
 * (AlignmentDB's m_region_start .. m_region_end inclusive); positions screened: region_start .. region_end - 1. */
#define NPH_SCREEN_SLOTS 9          /* per position: j = 0..3 (ACGT): slot 2j = substitution to j, 2j + 1 = insertion of j; slot 8 = deletion */
typedef struct {
    int32_t  flank;               /* opt::screen_flanking_sequence (10); the window must fit NPH_SCREEN_MAX_WINDOW */
    uint32_t score_threshold;     /* opt::screen_score_threshold (100) */
    uint32_t alignment_flags;     /* NPH_HAF_* handed to profile_hmm_score_set */
    uint32_t k;                   /* k of the reads' base model (nucleotide alphabet) */
    uint32_t reads_per_round;     /* reads of a position scored between two early-exit tests (8) */
    int32_t  region_start;        /* m_region_start */
} nph_screen_params;
#define NPH_SCREEN_MAX_WINDOW 64
/* qualities_out: NPH_SCREEN_SLOTS doubles per screened position (position region_start + p at p * NPH_SCREEN_SLOTS): the
 * Variant::quality score_variant_thresholded returns; NaN for a candidate the reference does not generate (j == reference base,
 * redundant deletion) and for positions whose window leaves the region (are_coordinates_valid fails: the reference skips them).
 * n_reads_out (optional): event sequences per position.  n_scored_events_out (optional): DP rows scored in all rounds. */
int nph_screen_edits_batch(nph_ctx* ctx,
                           const nph_read* reads, size_t n_reads,
                           const float* ev_mean, const double* ev_start_time, size_t n_events_total,
                           const char* ref_bases, size_t n_ref_bases,
                           const int16_t* event_deltas, size_t n_deltas_total, const int32_t* first_event,
                           const nph_meth_record* records, size_t n_records,
                           const nph_screen_params* params, double indel_bias,
                           double* qualities_out, uint32_t* n_reads_out, uint64_t* n_scored_events_out);
/* Staged form (reads resident): load, run (all rounds; asynchronous device work between the per-round read-backs), fetch. */
int nph_screen_load(nph_ctx* ctx, const char* ref_bases, size_t n_ref_bases, const int16_t* event_deltas, size_t n_deltas_total,
                    const int32_t* first_event, const nph_meth_record* records, size_t n_records,
                    const nph_screen_params* params, double indel_bias);
int nph_screen_run(nph_ctx* ctx);
/* counters of the most recent nph_screen_run: rounds; forward jobs and scored events (DP rows) actually run; what scoring every
 * read of every candidate (no early exit) would have cost in jobs (valid after nph_screen_fetch); and the DP rows the reference's
 * own loop scores for the same result — base and variant sequence per (candidate, read) until the candidate's total leaves the
 * threshold — the unit in which this workload's throughput is compared with the CPU arm (here the base haplotype of a read is
 * scored once per round for all its candidates, the reference scores it once per candidate) */
int nph_screen_counts(nph_ctx* ctx, uint32_t* n_rounds_out, uint64_t* n_jobs_out, uint64_t* n_scored_events_out, uint64_t* n_jobs_without_exit_out,
                      uint64_t* n_reference_events_out);
/* reference_rows_out (optional, one per position): the position's share of nph_screen_counts' n_reference_events */
int nph_screen_fetch(nph_ctx* ctx, double* qualities_out, uint32_t* n_reads_out, uint64_t* reference_rows_out);

/* ---- event detection (section 8f N4: the step before ABEA) --------------------------------------
 * scrappie's detect_events as load_from_raw calls it: t-statistics over two windows on prefix sums, a short/long
 * peak detector, events between consecutive boundaries.
 * ref: src/thirdparty/scrappie/event_detection.c:35-319, event_detection.h:15-29 (parameters),
 *      src/nanopolish_squiggle_read.cpp:229-235 (call site). */
typedef struct {
    uint32_t window_length1, window_length2;   /* 3, 6 for DNA; 7, 14 for RNA */
    float threshold1, threshold2, peak_height;  /* 1.4, 9.0, 0.2 for DNA; 2.5, 9.0, 1.0 for RNA */
    uint32_t reverse_events;  /* nph_load_from_raw_batch only: 1 for direct RNA, whose events load_from_raw turns
                                 around to 5'->3' after the MoM estimate (src/nanopolish_squiggle_read.cpp:262-265) */
} nph_event_params;
/* scrappie's event_t reduced to what it computes here (pos/state are always -1 there) */
typedef struct { uint64_t start; float length; float mean; float stdv; uint32_t reserved; } nph_event;
typedef struct {
    uint64_t sample_off;      /* first raw sample of this read in raw[] (picoamps as float, like Fast5Data::rt.raw) */
    uint64_t event_off;       /* where this read's events go in events_out[] */
    uint32_t n_samples;
    uint32_t event_cap;       /* room at event_off; n_samples always suffices, n_samples/2 does in practice */
} nph_raw_read;
/* events_out[reads[i].event_off ...] receives n_events_out[i] events in scrappie's order; n_events_out[i] == 0 with
 * NPH_ERR_UNSUPPORTED returned if some event_cap was too small (nothing else can fail: every signal has >= 1 event). */
int nph_detect_events_batch(nph_ctx* ctx, const float* raw, size_t n_samples_total, const nph_raw_read* reads, size_t n_reads,
                            const nph_event_params* params, nph_event* events_out, size_t events_total, uint32_t* n_events_out);

/* ---- raw-signal trimming (section 8f N4: the step before event detection) --------------------------
 * trim_and_segment_raw(rt, trim_start, trim_end, varseg_chunk, varseg_thresh) on a raw_table that starts at
 * {start 0, end n_samples}: median absolute deviation per chunk, chunks at or below the varseg_thresh quantile of
 * those MADs dropped from both ends, then the fixed trims.  ranges_out[i] is the surviving [start, end) relative to
 * reads[i].sample_off; {0, 0} where the reference returns an empty table (or would trip its assert: fewer samples
 * than one chunk, or no chunk above the threshold).  Only sample_off and n_samples of nph_raw_read are used.
 * ref: src/thirdparty/scrappie/scrappie_common.c:9-190; call site src/nanopolish_squiggle_read.cpp:226-233
 *      (trim_start 200, trim_end 10, varseg_chunk 100, varseg_thresh 0.0).  varseg_chunk <= 128. */
typedef struct { uint32_t start, end; } nph_raw_range;
int nph_trim_raw_batch(nph_ctx* ctx, const float* raw, size_t n_samples_total, const nph_raw_read* reads, size_t n_reads,
                       int32_t trim_start, int32_t trim_end, int32_t varseg_chunk, float varseg_thresh,
                       nph_raw_range* ranges_out);

/* ---- calibration after ABEA (section 8f N4: the step between ABEA and the HMM) ---------------------
 * For each ABEA job (same jobs[], kmer_ranks[], pairs[] and results[] as nph_abea_batch took and returned):
 *   base_to_event_out[rank_off + ki] = SquiggleRead::base_to_event_map[ki].indices[strand]   ({-1,-1}: no events)
 *   events_per_base                   = (max_event - min_event) / n_kmers
 *   shift, scale, var                 = recalibrate_model(read, model, strand,
 *                                           get_eventalignment_for_1d_basecalls(...), scale_var=true, scale_drift=false)
 * and the QC that follows.  reads[] carries the scalings the read has before the call (the MoM estimate); they come
 * back unchanged when the read is not recalibrated.  base_to_event_out may be NULL.
 * ref: src/nanopolish_squiggle_read.cpp:270-336,340-391; src/nanopolish_methyltrain.cpp:204-307. */
typedef struct { int32_t start, stop; } nph_event_range;      /* IndexPair, src/nanopolish_squiggle_read.h:32-37 */
#define NPH_CAL_OK              0
#define NPH_CAL_NOT_ALIGNED     1   /* ABEA returned no pairs: events cleared, events_per_base = 0 */
#define NPH_CAL_TOO_FEW_EVENTS  2   /* fewer than 200 'M' events: not recalibrated, events cleared */
#define NPH_CAL_HIGH_VAR        4   /* var > MIN_CALIBRATION_VAR (2.5): events cleared */
#define NPH_CAL_TOO_MANY_STAYS  8   /* events_per_base > 5.0: events cleared */
typedef struct {
    double shift, scale, drift, var;   /* arguments of SquiggleScalings::set4 */
    double events_per_base;
    uint32_t n_used;                   /* 'M' events that entered the normal equations */
    int32_t status;                    /* NPH_CAL_*; non-zero = the reference drops the read */
} nph_calibration;
int nph_recalibrate_batch(nph_ctx* ctx, const nph_read* reads, size_t n_reads, const float* ev_mean, size_t n_events_total,
                          const uint32_t* kmer_ranks, size_t n_ranks_total, const nph_abea_job* jobs, size_t n_jobs,
                          uint32_t model_id, const nph_aligned_pair* pairs, size_t pairs_total,
                          const nph_abea_result* results, nph_event_range* base_to_event_out, nph_calibration* calibrations_out);

/* ---- the whole read prologue in one call (section 8f N4) ------------------------------------------------
 * SquiggleRead::load_from_raw for a batch of reads: trim_and_segment_raw (200, 10, 100, 0.0) -> detect_events ->
 * SquiggleEvent conversion -> estimate_scalings_using_mom -> adaptive_banded_simple_event_align -> base_to_event_map,
 * events_per_base, recalibrate_model and the QC, chained on the device (the samples cross PCIe once, events never
 * come back in between).  ref: src/nanopolish_squiggle_read.cpp:226-336.
 * DNA: params = event_detection_defaults, a 6-mer nucleotide model.  Direct RNA: params = event_detection_rna with
 * reverse_events = 1, the 5-mer u_to_t_rna model, ranks of the sequence with U replaced by T (:206-213); the events
 * come back in 5'->3' order, each keeping the start time it had in acquisition order (so start times descend).
 * Outputs, per job j:  events [event_off_out[j], event_off_out[j+1]) of the four event arrays (compact, job order;
 * SquiggleEvent::log_stdv = logf(stdv) is left to the caller's libm), calibrations_out[j] (status != 0: the reference
 * clears the read's events; the arrays still hold them), base_to_event_out[rank_off + ki] (optional).
 * A read that trims to nothing (the reference aborts on it) gets no events and NPH_CAL_EMPTY_AFTER_TRIM.
 * NPH_ERR_UNSUPPORTED if events_cap is too small (n_samples_total / 3 always suffices). */
#define NPH_CAL_EMPTY_AFTER_TRIM 16
typedef struct {
    uint64_t sample_off;      /* first raw sample (picoamps, float) of this read in raw[] */
    uint64_t rank_off;        /* first k-mer rank of the basecalled sequence in kmer_ranks[] (forward strand) */
    uint32_t n_samples;
    uint32_t n_kmers;         /* read_sequence.length() - k + 1 */
    double   sample_rate;     /* Fast5Data::channel_params.sample_rate */
} nph_raw_job;
int nph_load_from_raw_batch(nph_ctx* ctx, const float* raw, size_t n_samples_total,
                            const uint32_t* kmer_ranks, size_t n_ranks_total,
                            const nph_raw_job* jobs, size_t n_jobs, uint32_t model_id, const nph_event_params* params,
                            uint64_t* event_off_out, float* ev_mean_out, float* ev_stdv_out, double* ev_start_time_out,
                            float* ev_duration_out, size_t events_cap,
                            nph_event_range* base_to_event_out, nph_calibration* calibrations_out);

/* The surviving sample range [start, end) of each job of the most recent nph_load_from_raw_batch on this context,
 * relative to the job's sample_off ({0, 0}: nothing survived).  It is what load_from_raw keeps with SRF_LOAD_RAW_SAMPLES
 * (samples[i] = rt.raw[rt.start + i], sample_start_time = 0; src/nanopolish_squiggle_read.cpp:251-258), which eventalign's
 * --samples / --signal-index read back.  NPH_ERR_STATE if n_jobs is not that call's job count. */
int nph_last_trim_ranges(nph_ctx* ctx, nph_raw_range* ranges_out, size_t n_jobs);

/* ---- poly(A) tail length of direct-RNA reads (section 8f N5: `nanopolish polya`) -------------------------------
 * Per read, what estimate_polya_for_single_read computes once load_from_raw has run (ref:
 * src/nanopolish_polya_estimator.cpp): SegmentationHMM's 6-state Viterbi over every trimmed raw sample (:204-509) with the
 * Gaussians scaled by the read's (float) scale / shift / var, segment_squiggle's region ends and cliff count,
 * estimate_unaligned_duration_profile's read rate (:564-599), estimate_polya_length (:638-662) and the two QC verdicts
 * that need no alignment record: post_segmentation_qc (NOREGION) and post_estimation_qc (ADAPTER).  SUFFCLIP comes from
 * the BAM record's last CIGAR op and is the caller's (nph::PolyaEstimator in nanopolish_b200/host/nph_polya.hpp).
 * Emissions use glibc's expf / logf restated bit for bit (csrc/polya_math.cuh), so results equal the reference's on an
 * x86-64 host with glibc >= 2.28. */
typedef struct {
    uint64_t sample_off;      /* first trimmed raw sample of the read in samples[] (acquisition order, picoamps) */
    uint64_t event_off;       /* first event duration in durations[] (the read's events in SquiggleRead order) */
    uint64_t map_off;         /* first base_to_event_map entry of the read in map[] (event indices relative to event_off) */
    uint32_t n_samples;       /* >= 2 */
    uint32_t n_events;        /* 0: the read did not load (READ_FAILED_LOAD); nothing else of the job is read */
    uint32_t n_kmers;         /* read_sequence.length() - k + 1 map entries, >= 1 */
    uint32_t reserved;
    double sample_rate;
    double shift, scale, var; /* sr.scalings[0] */
} nph_polya_job;              /* 72 bytes */
#define NPH_POLYA_NOREGION     1   /* fewer than 200 adapter or poly(A) samples */
#define NPH_POLYA_ADAPTER      2   /* more than 300 adapter nucleotides */
#define NPH_POLYA_FAILED_LOAD  4   /* no events: no other field is set */
typedef struct {
    uint64_t start, leader, adapter, polya;   /* Segmentation: last sample index of S, L, A and P/C (size_t arithmetic) */
    uint64_t cliffs;                          /* samples in state C */
    double read_rate;                         /* 1 / median per-k-mer duration */
    double polya_length;                      /* nucleotides, >= 0 */
    float end_score;                          /* viterbi_scores[n_samples-1][TRANSCRIPT] */
    uint32_t qc;                              /* NPH_POLYA_* bits */
} nph_polya_result;           /* 64 bytes */
/* One call: host buffers in, results out.  Jobs may share samples, durations and map entries.  A job with n_samples < 2, a sample / event / map range outside its buffer,
 * no map entries, or a map entry outside [0, n_events) (start -1 means "no events" and is skipped) yields NPH_ERR_INVALID. */
int nph_polya_batch(nph_ctx* ctx, const float* samples, size_t n_samples_total, const float* durations, size_t n_events_total,
                    const nph_event_range* map, size_t n_map_total, const nph_polya_job* jobs, size_t n_jobs,
                    nph_polya_result* results_out);
/* The same over the reads of the most recent nph_load_from_raw_batch on this context, from what it left in device memory:
 * the raw samples with their trim ranges, the event durations, the base_to_event_map, the calibrated scalings and the
 * sample rates.  Nothing is uploaded.  A read whose calibration status is non-zero gets NPH_POLYA_FAILED_LOAD.  (For this,
 * nph_load_from_raw_batch keeps the batch's raw samples on the device, 4 bytes per sample, until the next such call or
 * nph_destroy.)
 * NPH_ERR_STATE if n_jobs is not that call's job count, or if another call has reused its buffers since. */
int nph_polya_after_load(nph_ctx* ctx, nph_polya_result* results_out, size_t n_jobs);

/* ---- measurement hooks (used by bench.py; not part of the reference surface) ------------- */
/* Device time in ms of the most recent nph_hmm_score / nph_abea_run kernel sequence, measured
 * with CUDA events on the context's stream (valid after a sync), and the number of kernel
 * launches it issued. */
int nph_last_kernel_ms(nph_ctx* ctx, float* ms_out, int* launches_out);
/* Pinned host memory helpers so callers can stage H2D/D2H at full PCIe speed. */
int nph_host_alloc(void** ptr_out, size_t bytes);
int nph_host_free(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* NPH_H */
