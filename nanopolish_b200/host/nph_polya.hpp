// nph_polya.hpp — SURVEY.md section 8(f) row N5: `nanopolish polya`, the per-read work of
//
//   estimate_polya_for_single_read      ref: src/nanopolish_polya_estimator.cpp:733-862 (header line :877)
//
// for a batch of BAM records in one device call (nph_polya_batch): the segmentation Viterbi over every trimmed raw sample,
// the read rate, the tail length and the NOREGION / ADAPTER verdicts on the device; the SUFFCLIP verdict (the record's last
// CIGAR op), the QC priority and the TSV rows here.  polya_from_raw chains it after load_from_raw without the samples
// leaving the device (nph_polya_after_load).  The reference's --verbose dumps are not reproduced.
#pragma once
#include "nph_raw.hpp"

namespace nph {

// what estimate_polya_for_single_read takes from the BAM record (:742-758)
struct PolyaRecord {
    std::string read_name;          // bam_get_qname
    std::string contig;             // hdr->target_name[core.tid]
    int32_t position = 0;           // core.pos
    uint16_t flag = 0;              // core.flag: BAM_FSECONDARY records give no row
    uint32_t suffix_clip = 0;       // bam_cigar_oplen of the LAST CIGAR op, whatever the op (:755-758)
};

// the header line polya_main prints (:877)
const std::string& polya_tsv_header();

class PolyaEstimator {
public:
    // sr: the SquiggleRead load_from_raw built with SRF_LOAD_RAW_SAMPLES (trimmed samples, events, base_to_event_map and
    // scalings; a read without events gives the READ_FAILED_LOAD row).  Returns the read's index, or -1 for a secondary record.
    long add_read(const PolyaRecord& record, const SquiggleRead& sr);
    void run(Engine& engine);                           // one device call for every read added
    // the header (optional) and one row per read in add_read order, byte for byte what the reference prints
    std::string tsv(bool header = true) const;
    const nph_polya_result& result(size_t i) const { return m_results[i]; }
    size_t num_reads() const { return m_records.size(); }
    void clear();

private:
    std::vector<PolyaRecord> m_records;
    std::vector<nph_polya_job> m_jobs;
    std::vector<float> m_samples, m_durations;
    std::vector<nph_event_range> m_map;
    std::vector<nph_polya_result> m_results;
};

// the row of one read (:765 for a failed load, :823-826 otherwise) appended to out
void append_polya_row(std::string& out, const PolyaRecord& record, const nph_polya_result& r);

// load_from_raw (direct RNA: raw[i].nucleotide_type == SRNT_RNA, the 5-mer RNA model) and polya over the same reads, with the
// samples, events, map and scalings kept on the device between the two (nph_polya_after_load).  records[i] belongs to
// raw[i].  Returns the header (optional) and the rows, as PolyaEstimator::tsv would over the reads load_from_raw builds.
std::string polya_from_raw(Engine& engine, const PoreModel& base_model, const std::vector<RawRead>& raw,
                           const std::vector<PolyaRecord>& records, bool header = true);

} // namespace nph
