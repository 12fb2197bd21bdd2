// oracle/ref_polya_harness.cpp — TEST INFRASTRUCTURE ONLY.
//
// `nanopolish polya` (src/nanopolish_polya_estimator.cpp) keeps its segmentation HMM in a class local to that .cpp, so
// this translation unit compiles the reference's .cpp itself (#include, unmodified, from $(REF)/src) next to our
// oracle/ref_harness.cpp (whose reads — npref_read_create / npref_read_set_eventalign / npref_read_set_samples /
// npref_read_set_scalings — the functions below take by handle).  oracle/polya.mk links it with the other reference
// objects into oracle/_ref/libnpref_polya.so with --gc-sections, so the CLI code (ReadDB, BAM, faidx) is dropped.
//
// npref_polya runs the reference's own SegmentationHMM::segment_squiggle and ::viterbi (for the end score),
// estimate_unaligned_duration_profile, estimate_polya_length and the three QC functions.  Only the QC priority and the
// row of estimate_polya_for_single_read (:760-777, :803-826), which needs ReadDB and fast5, are restated.
#include "ref_harness.cpp"
#include "nanopolish_polya_estimator.cpp"

namespace {

// the row estimate_polya_for_single_read prints for one read (verbose 0); returns its length
int polya_row(SquiggleRead& sr, const char* read_name, const char* contig, int pos, uint32_t suffix_clip, int want_end_score,
              uint64_t* seg_out, double* rate_len_out, float* end_score_out, int* qc_out, char* row, size_t row_cap)
{
    if (sr.events[0].empty()) {
        *qc_out = 4;
        return snprintf(row, row_cap, "%s\t%s\t%d\t-1.0\t-1.0\t-1.0\t-1.0\t-1.00\t-1.00\tREAD_FAILED_LOAD\n", read_name, contig, pos);
    }
    std::string pre = pre_segmentation_qc(suffix_clip, 0, sr.read_sequence.length(), sr);
    SegmentationHMM hmm(static_cast<float>(sr.scalings[0].scale), static_cast<float>(sr.scalings[0].shift),
                        static_cast<float>(sr.scalings[0].var));
    Segmentation seg = hmm.segment_squiggle(sr);
    std::string post_seg = post_segmentation_qc(seg, sr);
    double read_rate = estimate_unaligned_duration_profile(sr, NULL, NULL, NULL, 0, 0);
    double polya_length = estimate_polya_length(sr, seg, read_rate);
    std::string post_est = post_estimation_qc(seg, sr, read_rate, polya_length);
    if (want_end_score) {
        ViterbiOutputs vo = hmm.viterbi(sr);
        *end_score_out = vo.scores[sr.samples.size() - 1];
    }
    std::string qc_tag;
    if (post_seg.compare("PASS") != 0) qc_tag = post_seg;
    else if (post_est.compare("PASS") != 0) qc_tag = post_est;
    else if (pre.compare("PASS") != 0) qc_tag = pre;
    else qc_tag = "PASS";
    seg_out[0] = seg.start; seg_out[1] = seg.leader; seg_out[2] = seg.adapter; seg_out[3] = seg.polya; seg_out[4] = seg.cliffs;
    rate_len_out[0] = read_rate; rate_len_out[1] = polya_length;
    *qc_out = (post_seg != "PASS" ? 1 : 0) | (post_est != "PASS" ? 2 : 0) | (pre != "PASS" ? 8 : 0);
    double leader_sample_start = seg.start + 1, adapter_sample_start = seg.leader + 1, polya_sample_start = seg.adapter + 1;
    double transcr_sample_start = seg.polya + 1;
    return snprintf(row, row_cap, "%s\t%s\t%d\t%.1lf\t%.1lf\t%.1lf\t%.1lf\t%.2lf\t%.2lf\t%s\n", read_name, contig, pos,
                    leader_sample_start, adapter_sample_start, polya_sample_start, transcr_sample_start, read_rate, polya_length,
                    qc_tag.c_str());
}

} // namespace

extern "C" {

// One read: seg_out = {start, leader, adapter, polya, cliffs}, rate_len_out = {read_rate, polya_length}, the Viterbi end
// score, qc bits (1 NOREGION, 2 ADAPTER, 4 failed load, 8 SUFFCLIP) and the TSV row.  Returns the row length.
int npref_polya(int h, const char* read_name, const char* contig, int pos, uint32_t suffix_clip, uint64_t* seg_out,
                double* rate_len_out, float* end_score_out, int* qc_out, char* row, size_t row_cap)
{
    return polya_row(*g_reads[h], read_name, contig, pos, suffix_clip, 1, seg_out, rate_len_out, end_score_out, qc_out, row, row_cap);
}

// The header line polya_main prints (:877)
const char* npref_polya_header(void)
{
    return "readname\tcontig\tposition\tleader_start\tadapter_start\tpolya_start\ttranscript_start\tread_rate\tpolya_length\tqc_tag\n";
}

// Timing of the reference's per-read work over n reads on `threads` OpenMP threads (the CLI's parallel_run over BAM
// records); the rows go to rows (row_stride bytes each).  Returns elapsed seconds.
double npref_polya_batch(const int* handles, size_t n, const char* contig, int threads, char* rows, size_t row_stride)
{
    auto t0 = std::chrono::steady_clock::now();
    #pragma omp parallel for schedule(dynamic, 1) num_threads(threads)
    for (long long i = 0; i < (long long)n; ++i) {
        SquiggleRead& sr = *g_reads[handles[i]];
        uint64_t seg[5]; double rl[2]; float es; int qc;
        polya_row(sr, sr.read_name.c_str(), contig, 0, 0, 0, seg, rl, &es, &qc, rows + i * row_stride, row_stride);
    }
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

} // extern "C"
