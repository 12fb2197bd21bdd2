// nph_polya.cpp — see nph_polya.hpp.
#include "nph_polya.hpp"

namespace nph {

namespace {
const uint16_t kBamSecondary = 0x100;      // BAM_FSECONDARY

// estimate_polya_for_single_read's QC priority (:803-813): post-segmentation, post-estimation, then pre-segmentation (:672-683)
const char* qc_tag(const nph_polya_result& r, uint32_t suffix_clip)
{
    if (r.qc & NPH_POLYA_NOREGION) return "NOREGION";
    if (r.qc & NPH_POLYA_ADAPTER) return "ADAPTER";
    return suffix_clip > 200 ? "SUFFCLIP" : "PASS";
}
} // namespace

const std::string& polya_tsv_header()
{
    static const std::string h = "readname\tcontig\tposition\tleader_start\tadapter_start\tpolya_start\ttranscript_start\tread_rate\tpolya_length\tqc_tag\n";
    return h;
}

void append_polya_row(std::string& out, const PolyaRecord& rec, const nph_polya_result& r)
{
    out += rec.read_name; out += '\t'; out += rec.contig; out += '\t'; out += std::to_string(rec.position);
    if (r.qc & NPH_POLYA_FAILED_LOAD) {
        out += "\t-1.0\t-1.0\t-1.0\t-1.0\t-1.00\t-1.00\tREAD_FAILED_LOAD\n";
        return;
    }
    // the region ends + 1 in size_t arithmetic, printed as doubles (:816-820)
    const double cols[4] = {(double)(uint64_t)(r.start + 1), (double)(uint64_t)(r.leader + 1), (double)(uint64_t)(r.adapter + 1),
                            (double)(uint64_t)(r.polya + 1)};
    char buf[512];
    for (double c : cols) { out += '\t'; out.append(buf, format_fixed(buf, c, 1)); }
    out += '\t'; out.append(buf, format_fixed(buf, r.read_rate, 2));
    out += '\t'; out.append(buf, format_fixed(buf, r.polya_length, 2));
    out += '\t'; out += qc_tag(r, rec.suffix_clip); out += '\n';
}

long PolyaEstimator::add_read(const PolyaRecord& record, const SquiggleRead& sr)
{
    if (record.flag & kBamSecondary) return -1;
    nph_polya_job j{};
    if (!sr.events[0].empty()) {           // the reference's load check (:760-762); everything else is validated on the device
        const size_t k = sr.base_model[0] ? sr.base_model[0]->k : 0;
        if (!sr.base_model[0] || sr.read_sequence.size() < k || sr.base_to_event_map.size() != sr.read_sequence.size() - k + 1)
            throw Error(NPH_ERR_INVALID, "PolyaEstimator::add_read: the read's base_to_event_map does not cover its k-mers");
        j.sample_off = m_samples.size(); j.event_off = m_durations.size(); j.map_off = m_map.size();
        j.n_samples = (uint32_t)sr.samples.size(); j.n_events = (uint32_t)sr.events[0].size(); j.n_kmers = (uint32_t)sr.base_to_event_map.size();
        j.sample_rate = sr.sample_rate;
        j.shift = sr.scalings[0].shift; j.scale = sr.scalings[0].scale; j.var = sr.scalings[0].var;
        m_samples.insert(m_samples.end(), sr.samples.begin(), sr.samples.end());
        for (const SquiggleEvent& e : sr.events[0]) m_durations.push_back(e.duration);
        for (const auto& m : sr.base_to_event_map) m_map.push_back(nph_event_range{m.indices[0].start, m.indices[0].stop});
    }
    m_records.push_back(record);
    m_jobs.push_back(j);
    return (long)m_records.size() - 1;
}

void PolyaEstimator::run(Engine& engine)
{
    m_results.assign(m_jobs.size(), nph_polya_result{});
    if (m_jobs.empty()) return;
    engine.check(nph_polya_batch(engine.ctx(), m_samples.data(), m_samples.size(), m_durations.data(), m_durations.size(), m_map.data(), m_map.size(),
                                 m_jobs.data(), m_jobs.size(), m_results.data()),
                 "nph_polya_batch");
}

std::string PolyaEstimator::tsv(bool header) const
{
    std::string out = header ? polya_tsv_header() : std::string();
    for (size_t i = 0; i < m_records.size() && i < m_results.size(); ++i) append_polya_row(out, m_records[i], m_results[i]);
    return out;
}

void PolyaEstimator::clear()
{
    m_records.clear(); m_jobs.clear(); m_samples.clear(); m_durations.clear(); m_map.clear(); m_results.clear();
}

std::string polya_from_raw(Engine& engine, const PoreModel& base_model, const std::vector<RawRead>& raw,
                           const std::vector<PolyaRecord>& records, bool header)
{
    if (records.size() != raw.size()) throw Error(NPH_ERR_INVALID, "polya_from_raw: one record per raw read");
    std::vector<std::unique_ptr<SquiggleRead>> reads = load_from_raw(engine, base_model, raw);
    // the reads load_from_raw sent to the device, in order (the others have no events: READ_FAILED_LOAD)
    const size_t k = base_model.k;
    std::vector<long> job_of(raw.size(), -1);
    size_t n_sent = 0;
    for (size_t i = 0; i < raw.size(); ++i)
        if (!(raw[i].samples.empty() || reads[i]->read_sequence.size() < k || !(raw[i].sample_rate > 0.0))) job_of[i] = (long)n_sent++;
    std::vector<nph_polya_result> res(n_sent);
    if (n_sent) engine.check(nph_polya_after_load(engine.ctx(), res.data(), res.size()), "nph_polya_after_load");
    std::string out = header ? polya_tsv_header() : std::string();
    nph_polya_result failed{};
    failed.qc = NPH_POLYA_FAILED_LOAD;
    for (size_t i = 0; i < raw.size(); ++i) {
        if (records[i].flag & kBamSecondary) continue;
        append_polya_row(out, records[i], job_of[i] >= 0 ? res[job_of[i]] : failed);
    }
    return out;
}

} // namespace nph
