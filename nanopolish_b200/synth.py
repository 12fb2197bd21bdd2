"""Deterministic synthetic R9.4 reads and job lists in the C-ABI layout (include/nph.h).

Shapes follow SURVEY.md section 8(d): uniform ACGT sequence, 0-3 events per k-mer
(mean ~1.7 events/base), event mean ~ N(scale*mu_kmer + shift, (var*sigma_kmer)^2),
duration 0.002 s, per-read shift/scale/var jitter.  The same generator feeds the CUDA path,
the oracle and the compiled reference, so every arm of a comparison sees identical bytes.

Job builders mirror the callers of profile_hmm_score:
  * scorereads_jobs   -> 500-event segments, flags 0   (ref: src/nanopolish_scorereads.cpp:116-203)
  * methylation_jobs  -> one window per CpG group, both alleles over the cpg alphabet, flags PRE|POST
                         (ref: src/basemods/nanopolish_basemods.cpp:322-417)
  * abea_jobs         -> whole read vs its sequence (ref: src/nanopolish_squiggle_read.cpp:270)
"""
from __future__ import annotations

import os
from dataclasses import dataclass, field

import numpy as np

# ---- C-ABI PODs as numpy dtypes (must match include/nph.h) --------------------------------
READ_DT = np.dtype([
    ("event_off", "<u8"), ("n_events", "<u4"), ("reserved", "<u4"),
    ("scale", "<f8"), ("shift", "<f8"), ("drift", "<f8"), ("var", "<f8"), ("log_var", "<f8"),
    ("events_per_base", "<f8"),
], align=True)
HMM_JOB_DT = np.dtype([
    ("rank_off", "<u8"), ("read", "<u4"), ("model_id", "<u4"), ("event_start", "<u4"),
    ("event_stop", "<u4"), ("n_kmers", "<u4"), ("stride", "i1"), ("rc", "u1"), ("flags", "u1"),
    ("reserved", "u1"),
], align=True)
ABEA_JOB_DT = np.dtype([
    ("rank_off", "<u8"), ("pairs_off", "<u8"), ("read", "<u4"), ("n_kmers", "<u4"),
    ("pairs_cap", "<u4"), ("reserved", "<u4"),
], align=True)
PAIR_DT = np.dtype([("ref_pos", "<i4"), ("read_pos", "<i4")], align=True)
ABEA_RES_DT = np.dtype([
    ("n_pairs", "<u4"), ("status", "<i4"), ("max_gap", "<i4"), ("n_aligned", "<u4"),
    ("avg_log_emission", "<f8"),
], align=True)
ALIGN_STATE_DT = np.dtype([("event_idx", "<u4"), ("kmer_idx", "<u4"), ("l_fm", "<f4"), ("state", "S1"),
                           ("reserved", "u1", (3,))], align=True)
EA_CHAIN_DT = np.dtype([("pair_off", "<u8"), ("map_off", "<u8"), ("rank_off", "<u8"), ("out_off", "<u8"), ("read", "<u4"),
                        ("model_id", "<u4"), ("n_pairs", "<u4"), ("map_len", "<u4"), ("ref_len", "<u4"), ("read_seq_len", "<u4"),
                        ("out_cap", "<u4"), ("ref_offset", "<i4"), ("first_event", "<i4"), ("last_event", "<i4"),
                        ("do_base_rc", "u1"), ("rc", "u1"), ("k", "u1"), ("reserved", "u1")], align=True)
EA_RECORD_DT = np.dtype([("ref_position", "<i4"), ("event_idx", "<i4"), ("hmm_state", "S1"), ("reserved", "u1", 3)], align=True)
EA_RESULT_DT = np.dtype([("n_records", "<u4"), ("n_windows", "<u4"), ("status", "<i4"), ("reserved", "<u4")], align=True)
assert EA_CHAIN_DT.itemsize == 80 and EA_RECORD_DT.itemsize == 12 and EA_RESULT_DT.itemsize == 16
EVENT_DT = np.dtype([("start", "<u8"), ("length", "<f4"), ("mean", "<f4"), ("stdv", "<f4"), ("reserved", "<u4")], align=True)
RAW_READ_DT = np.dtype([("sample_off", "<u8"), ("event_off", "<u8"), ("n_samples", "<u4"), ("event_cap", "<u4")], align=True)
EVENT_PARAMS_DT = np.dtype([("window_length1", "<u4"), ("window_length2", "<u4"), ("threshold1", "<f4"), ("threshold2", "<f4"),
                            ("peak_height", "<f4"), ("reverse_events", "<u4")], align=True)
RAW_RANGE_DT = np.dtype([("start", "<u4"), ("end", "<u4")], align=True)
EVENT_RANGE_DT = np.dtype([("start", "<i4"), ("stop", "<i4")], align=True)
CALIBRATION_DT = np.dtype([("shift", "<f8"), ("scale", "<f8"), ("drift", "<f8"), ("var", "<f8"), ("events_per_base", "<f8"),
                           ("n_used", "<u4"), ("status", "<i4")], align=True)
assert EVENT_DT.itemsize == 24 and RAW_READ_DT.itemsize == 24 and EVENT_PARAMS_DT.itemsize == 24
RAW_JOB_DT = np.dtype([("sample_off", "<u8"), ("rank_off", "<u8"), ("n_samples", "<u4"), ("n_kmers", "<u4"), ("sample_rate", "<f8")], align=True)
assert RAW_JOB_DT.itemsize == 32
assert RAW_RANGE_DT.itemsize == 8 and EVENT_RANGE_DT.itemsize == 8 and CALIBRATION_DT.itemsize == 48
METH_RECORD_DT = np.dtype([("ref_off", "<u8"), ("pair_off", "<u8"), ("read", "<u4"), ("model_id", "<u4"), ("ref_len", "<u4"),
                           ("n_pairs", "<u4"), ("ref_start_pos", "<i4"), ("rc", "u1"), ("strand", "u1"), ("reserved", "u1", 2)], align=True)
METH_SITE_DT = np.dtype([("start_position", "<i4"), ("end_position", "<i4"), ("n_motif", "<u4"), ("record", "<u4"),
                         ("ll_unmethylated", "<f4"), ("ll_methylated", "<f4")], align=True)
METH_PARAMS_DT = np.dtype([("min_separation", "<i4"), ("min_flank", "<i4"), ("max_span", "<i4"), ("min_event_span", "<i4"),
                           ("region_start", "<i4"), ("region_end", "<i4"), ("k", "<u4"), ("alphabet_size", "<u4"),
                           ("bases", "S8"), ("complements", "S8"), ("n_sites", "<u4"), ("site_len", "<u4"),
                           ("sites", "S8", 4), ("sites_methylated", "S8", 4), ("sites_methylated_complement", "S8", 4)], align=True)
assert METH_RECORD_DT.itemsize == 40 and METH_SITE_DT.itemsize == 24 and METH_PARAMS_DT.itemsize == 152
assert ALIGN_STATE_DT.itemsize == 16
assert READ_DT.itemsize == 64 and HMM_JOB_DT.itemsize == 32 and ABEA_JOB_DT.itemsize == 32
assert PAIR_DT.itemsize == 8 and ABEA_RES_DT.itemsize == 24

HAF_ALLOW_PRE_CLIP = 1
HAF_ALLOW_POST_CLIP = 2

_GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


@dataclass
class PoreModel:
    """PoreModel::states as SoA (ref: src/pore_model/nanopolish_poremodel.h:20-36, 70-110)."""
    name: str
    k: int
    alphabet: str            # "nucleotide" (ACGT) or "cpg" (ACGMT)
    level_mean: np.ndarray   # f64[n_states]
    level_stdv: np.ndarray
    level_log_stdv: np.ndarray

    @property
    def alphabet_size(self) -> int:
        return 4 if self.alphabet == "nucleotide" else 5

    @property
    def n_states(self) -> int:
        return int(self.level_mean.shape[0])


def synthetic_model(alphabet: str = "nucleotide", k: int = 6, seed: int = 7) -> PoreModel:
    """A plausible random pore model (levels 60-125 pA, stdv 1.2-3.5) for runs without fixtures."""
    a = 4 if alphabet == "nucleotide" else 5
    rng = np.random.default_rng(seed + a)
    n = a ** k
    mean = rng.uniform(60.0, 125.0, n)
    stdv = rng.uniform(1.2, 3.5, n)
    return PoreModel(f"synthetic.{alphabet}.{k}mer", k, alphabet, mean, stdv, np.log(stdv))


def load_model(alphabet: str = "nucleotide") -> PoreModel:
    """The built-in r9.4_450bps 6-mer template table dumped from the compiled reference by
    scripts/make_golden.py (tests/golden/r9.4_450bps.<alphabet>.6mer.template.npz); falls back to
    synthetic_model() if the fixture is absent."""
    path = os.path.join(_GOLDEN, f"r9.4_450bps.{alphabet}.6mer.template.npz")
    if os.path.exists(path):
        z = np.load(path)
        return PoreModel(f"r9.4_450bps.{alphabet}.6mer.template", int(z["k"]), alphabet,
                         z["level_mean"].astype(np.float64), z["level_stdv"].astype(np.float64),
                         z["level_log_stdv"].astype(np.float64))
    return synthetic_model(alphabet)


# ---- k-mer ranks (numpy restatement for DNA / CpG strings already encoded as base codes) ----
_DNA_CODE = np.full(256, 255, np.uint8)
for _i, _c in enumerate(b"ACGT"):
    _DNA_CODE[_c] = _i
_CPG_CODE = np.full(256, 255, np.uint8)
for _i, _c in enumerate(b"ACGMT"):
    _CPG_CODE[_c] = _i


def encode(seq: bytes | str, alphabet: str) -> np.ndarray:
    b = np.frombuffer(seq.encode() if isinstance(seq, str) else seq, np.uint8)
    codes = (_DNA_CODE if alphabet == "nucleotide" else _CPG_CODE)[b]
    if (codes == 255).any():
        raise ValueError("sequence has symbols outside the alphabet")
    return codes


def kmer_ranks_from_codes(codes: np.ndarray, k: int, asize: int) -> np.ndarray:
    """rank of k-mer i = sum_j code[i+j] * asize^(k-1-j)  (ref: Alphabet::kmer_rank,
    src/common/nanopolish_alphabet.h:78-89)."""
    n = codes.shape[0] - k + 1
    if n <= 0:
        return np.zeros(0, np.uint32)
    r = np.zeros(n, np.uint32)
    for j in range(k):
        r = r * np.uint32(asize) + codes[j:j + n].astype(np.uint32)
    return r


def dna_rc_kmer_ranks(codes: np.ndarray, k: int) -> np.ndarray:
    """HMMInputSequence::_rc_kmer_rank for the plain DNA alphabet: rank of the reverse complement of
    k-mer i (ref: src/hmm/nanopolish_hmm_input_sequence.h:88-91)."""
    n = codes.shape[0] - k + 1
    r = np.zeros(n, np.uint32)
    for j in range(k):
        r = r * np.uint32(4) + (3 - codes[k - 1 - j:k - 1 - j + n]).astype(np.uint32)
    return r


@dataclass
class ReadSet:
    reads: np.ndarray                 # READ_DT[n_reads]
    ev_mean: np.ndarray               # f32[total events]
    ev_start_time: np.ndarray         # f64[total events]
    seq_codes: list                   # per read: u8 base codes (ACGT = 0..3) of the true sequence
    ev_kmer: list                     # per read: i4[n_events] index of the k-mer that emitted each event
    kmer_first_event: list = field(default_factory=list)  # per read: i4[n_kmers] first event >= that k-mer
    k: int = 6

    @property
    def n_reads(self) -> int:
        return int(self.reads.shape[0])

    @property
    def total_events(self) -> int:
        return int(self.ev_mean.shape[0])


def gen_reads(n_reads: int, n_events: int, model: PoreModel, seed: int = 42, drift: bool = False,
              rng_scalings: bool = True, cpg_keep: float = 1.0) -> ReadSet:
    """n_reads reads of ~n_events events each (exactly n_events: the sequence is extended until the
    event budget is reached).  Events are emitted from `model` (nucleotide alphabet)."""
    assert model.alphabet == "nucleotide"
    k = model.k
    reads = np.zeros(n_reads, READ_DT)
    means, times, seqs, evk, kfe = [], [], [], [], []
    off = 0
    p_nev = np.array([0.03, 0.35, 0.45, 0.17])
    for r in range(n_reads):
        rng = np.random.default_rng(seed + r)
        # enough k-mers to cover the budget with margin, then trim
        nk_guess = int(n_events / 1.76 * 1.15) + 8
        codes = rng.integers(0, 4, nk_guess + k - 1, dtype=np.uint8)
        if cpg_keep < 1.0:
            # CpG depletion: turn most CG into CA so motif groups are ~60 bp apart (SURVEY 8d, cfg 3)
            cg = np.flatnonzero((codes[:-1] == 1) & (codes[1:] == 2))
            drop = cg[rng.random(cg.shape[0]) >= cpg_keep]
            codes[drop + 1] = 0
        nev = rng.choice(4, nk_guess, p=p_nev)
        csum = np.cumsum(nev)
        nk = int(np.searchsorted(csum, n_events, side="left")) + 1
        nk = min(nk, nk_guess)
        nev = nev[:nk].copy()
        extra = int(nev.sum()) - n_events
        if extra > 0:
            nev[-1] -= extra
        elif extra < 0:
            nev[-1] += -extra
        codes = codes[:nk + k - 1]
        ranks = kmer_ranks_from_codes(codes, k, 4)
        which = np.repeat(np.arange(nk, dtype=np.int32), nev)
        E = which.shape[0]
        if rng_scalings:
            shift = rng.uniform(-5.0, 5.0)
            scale = rng.uniform(0.9, 1.1)
            var = rng.uniform(0.9, 1.3)
        else:
            shift, scale, var = 0.0, 1.0, 1.0
        dr = rng.uniform(-0.002, 0.002) if drift else 0.0
        t = (np.arange(E, dtype=np.float64) * 0.002) + rng.uniform(0.0, 100.0)
        mu = scale * model.level_mean[ranks[which]] + shift + (t - t[0]) * dr
        sd = var * model.level_stdv[ranks[which]]
        m = (mu + sd * rng.standard_normal(E)).astype(np.float32)
        reads[r]["event_off"] = off
        reads[r]["n_events"] = E
        reads[r]["scale"], reads[r]["shift"], reads[r]["drift"], reads[r]["var"] = scale, shift, dr, var
        reads[r]["log_var"] = np.log(var)
        reads[r]["events_per_base"] = E / float(nk)
        first = np.searchsorted(which, np.arange(nk), side="left").astype(np.int32)
        means.append(m); times.append(t); seqs.append(codes); evk.append(which); kfe.append(first)
        off += E
    return ReadSet(reads, np.concatenate(means), np.concatenate(times), seqs, evk, kfe, k)


def gen_reads_from_sequence(codes: np.ndarray, n_reads: int, model: PoreModel, seed: int = 42) -> ReadSet:
    """n_reads reads that all traverse the same base sequence (a pile-up over one reference window), each with its own
    event counts, noise and scalings — the input shape of variant scoring (SURVEY.md 8d, config 5)."""
    k = model.k
    nk = codes.shape[0] - k + 1
    ranks = kmer_ranks_from_codes(codes, k, 4)
    reads = np.zeros(n_reads, READ_DT)
    means, times, seqs, evk, kfe = [], [], [], [], []
    off = 0
    p_nev = np.array([0.03, 0.35, 0.45, 0.17])
    for r in range(n_reads):
        rng = np.random.default_rng(seed + r)
        nev = rng.choice(4, nk, p=p_nev)
        nev[0] = max(nev[0], 1); nev[-1] = max(nev[-1], 1)
        which = np.repeat(np.arange(nk, dtype=np.int32), nev)
        E = which.shape[0]
        shift, scale, var = rng.uniform(-5.0, 5.0), rng.uniform(0.9, 1.1), rng.uniform(0.9, 1.3)
        t = (np.arange(E, dtype=np.float64) * 0.002) + rng.uniform(0.0, 100.0)
        mu = scale * model.level_mean[ranks[which]] + shift
        sd = var * model.level_stdv[ranks[which]]
        m = (mu + sd * rng.standard_normal(E)).astype(np.float32)
        reads[r] = (off, E, 0, scale, shift, 0.0, var, np.log(var), E / float(nk))
        first = np.searchsorted(which, np.arange(nk), side="left").astype(np.int32)
        means.append(m); times.append(t); seqs.append(codes.copy()); evk.append(which); kfe.append(first)
        off += E
    return ReadSet(reads, np.concatenate(means), np.concatenate(times), seqs, evk, kfe, k)


@dataclass
class HmmJobs:
    jobs: np.ndarray          # HMM_JOB_DT[n_jobs]
    kmer_ranks: np.ndarray    # u4[total]
    scored_events: int        # sum over jobs of DP rows (the metric's unit)
    block_cells: int          # sum over jobs of E*K
    seqs: list | None = None  # optional per-job sequence strings (bytes) for the reference harness
    seq_codes: np.ndarray | None = None   # u1: per job the alphabet ranks of the string its strand reads (nph_hmm_*_seq)
    code_jobs: np.ndarray | None = None   # the same jobs with rank_off = offset of the job's first code in seq_codes


def _finish_jobs(rows, ranks_list, seqs=None, codes_list=None) -> HmmJobs:
    jobs = np.zeros(len(rows), HMM_JOB_DT)
    off = 0
    ev = 0
    cells = 0
    for j, (read, model_id, e0, e1, rc, flags) in enumerate(rows):
        nk = ranks_list[j].shape[0]
        jobs[j] = (off, read, model_id, e0, e1, nk, 1 if e1 >= e0 else -1, rc, flags, 0)
        off += nk
        E = abs(int(e1) - int(e0)) + 1
        ev += E
        cells += E * nk
    kr = np.concatenate(ranks_list).astype(np.uint32) if ranks_list else np.zeros(0, np.uint32)
    out = HmmJobs(jobs, kr, ev, cells, seqs)
    if codes_list is not None:
        cj = jobs.copy()
        lens = np.array([c.shape[0] for c in codes_list], np.uint64)
        cj["rank_off"] = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64) if len(codes_list) else np.zeros(0, np.uint64)
        out.code_jobs = cj
        out.seq_codes = np.concatenate(codes_list).astype(np.uint8) if codes_list else np.zeros(0, np.uint8)
    return out


_CODE2DNA = np.frombuffer(b"ACGT", np.uint8)


def scorereads_jobs(rs: ReadSet, events_per_segment: int = 500, model_id: int = 0, rc_every: int = 0,
                    keep_seqs: bool = False) -> HmmJobs:
    """500-event segments [i*seg, (i+1)*seg] for i >= 1 while (i+1)*seg < n_events - ... , sequence =
    bases spanned by the true alignment of the two boundary events, flags 0
    (ref: model_score, src/nanopolish_scorereads.cpp:116-203).  rc_every=n makes every n-th read a
    reverse-strand job (events walked backwards, rc k-mer ranks) to cover stride -1."""
    rows, ranks_list, seqs, codes_list = [], [], [], []
    k = rs.k
    for r in range(rs.n_reads):
        E = int(rs.reads[r]["n_events"])
        which = rs.ev_kmer[r]
        codes = rs.seq_codes[r]
        rc = 1 if (rc_every and r % rc_every == rc_every - 1) else 0
        s = events_per_segment
        while s < E - events_per_segment:
            e0, e1 = s, s + events_per_segment
            k0, k1 = int(which[e0]), int(which[e1])
            sub = codes[k0:k1 + k]           # bases of k-mers k0..k1
            if sub.shape[0] > k:
                if not rc:
                    ranks_list.append(kmer_ranks_from_codes(sub, k, 4))
                    rows.append((r, model_id, e0, e1, 0, 0))
                    codes_list.append(sub)                          # m_seq
                    if keep_seqs:
                        seqs.append(_CODE2DNA[sub].tobytes())
                else:
                    # reverse-strand read: the HMM sequence is the reverse complement of the bases the
                    # events were emitted from; events are walked from e1 down to e0.
                    rcsub = (3 - sub[::-1]).astype(np.uint8)
                    ranks_list.append(dna_rc_kmer_ranks(rcsub, k))
                    rows.append((r, model_id, e1, e0, 1, 0))
                    codes_list.append(sub)                          # m_rc_seq = reverse complement of the HMM sequence = the bases as sequenced
                    if keep_seqs:
                        seqs.append(_CODE2DNA[rcsub].tobytes())
            s += events_per_segment
    return _finish_jobs(rows, ranks_list, seqs if keep_seqs else None, codes_list)


def abea_jobs(rs: ReadSet) -> tuple[np.ndarray, np.ndarray, int]:
    """One ABEA job per read over its full true sequence. Returns (jobs, kmer_ranks, pairs_total)."""
    jobs = np.zeros(rs.n_reads, ABEA_JOB_DT)
    ranks_list = []
    roff = poff = 0
    for r in range(rs.n_reads):
        ranks = kmer_ranks_from_codes(rs.seq_codes[r], rs.k, 4)
        nk = ranks.shape[0]
        cap = int(rs.reads[r]["n_events"]) + nk
        jobs[r] = (roff, poff, r, nk, cap, 0)
        ranks_list.append(ranks)
        roff += nk
        poff += cap
    return jobs, np.concatenate(ranks_list).astype(np.uint32), poff


_CODE2CPG = np.frombuffer(b"ACGMT", np.uint8)
_DNA2CPG = np.array([0, 1, 2, 4], np.uint8)       # A C G T -> ranks in "ACGMT"


def methylation_jobs(rs: ReadSet, model_id: int = 0, min_separation: int = 10, min_flank: int = 10,
                     max_span: int = 200, keep_seqs: bool = False, max_groups_per_read: int | None = None) -> HmmJobs:
    """call-methylation windows on forward-strand reads: CG motif scan -> groups (sites <= 10 bp apart)
    -> window = [first-10, last+10] -> two jobs per group (unmethylated, methylated), both over the
    cpg alphabet (ACGMT, 5^6 states), flags PRE|POST clip.  Jobs 2g, 2g+1 are the u/m pair of group g.
    (ref: calculate_methylation_for_read, src/basemods/nanopolish_basemods.cpp:238-457)"""
    rows, ranks_list, seqs, codes_list = [], [], [], []
    k = rs.k
    flags = HAF_ALLOW_PRE_CLIP | HAF_ALLOW_POST_CLIP
    for r in range(rs.n_reads):
        codes = rs.seq_codes[r]
        nk = codes.shape[0] - k + 1
        kfe = rs.kmer_first_event[r]
        E = int(rs.reads[r]["n_events"])
        sites = np.flatnonzero((codes[:-1] == 1) & (codes[1:] == 2))
        if sites.shape[0] == 0:
            continue
        brk = np.flatnonzero(np.diff(sites) > min_separation) + 1
        starts = np.concatenate([[0], brk]); ends = np.concatenate([brk, [sites.shape[0]]])
        n_done = 0
        for gs, ge in zip(starts, ends):
            first, last = int(sites[gs]), int(sites[ge - 1])
            sub_start, sub_end = first - min_flank, last + min_flank
            span = last - first
            if sub_start <= min_separation or span > max_span or sub_end >= codes.shape[0]:
                continue
            k_lo, k_hi = sub_start, min(sub_end, nk - 1)
            e1, e2 = int(min(kfe[k_lo], E - 1)), int(min(kfe[k_hi], E - 1))
            if abs(e2 - e1) <= 10:
                continue
            sub = codes[sub_start:sub_end + 1]
            u = _DNA2CPG[sub]
            m = u.copy()
            cg = np.flatnonzero((sub[:-1] == 1) & (sub[1:] == 2))
            m[cg] = 3                                    # Alphabet::methylate: CG -> MG
            for arr in (u, m):
                ranks_list.append(kmer_ranks_from_codes(arr, k, 5))
                rows.append((r, model_id, e1, e2, 0, flags))
                codes_list.append(arr)
                if keep_seqs:
                    seqs.append(_CODE2CPG[arr].tobytes())
            n_done += 1
            if max_groups_per_read and n_done >= max_groups_per_read:
                break
    return _finish_jobs(rows, ranks_list, seqs if keep_seqs else None, codes_list)


def event_params(rna: bool = False) -> np.ndarray:
    """scrappie's event_detection_defaults / event_detection_rna (src/thirdparty/scrappie/event_detection.h:15-29)."""
    p = np.zeros(1, EVENT_PARAMS_DT)
    # reverse_events: load_from_raw turns direct-RNA events around to 5'->3' (src/nanopolish_squiggle_read.cpp:262-265)
    p[0] = (7, 14, 2.5, 9.0, 1.0, 1) if rna else (3, 6, 1.4, 9.0, 0.2, 0)
    return p


def gen_raw(n_reads: int, n_samples: int, model: PoreModel, seed: int = 42, mean_dwell: float = 9.0, return_seqs: bool = False):
    """Synthetic raw current traces (picoamps, float32): a random sequence's k-mer levels held for a geometric dwell
    (mean ~9 samples at 4 kHz / 450 bases/s) plus Gaussian noise.  Returns (raw f32[total], RAW_READ_DT[n_reads]) and,
    with return_seqs, the base codes of the stretch of sequence each trace covers (its "basecall")."""
    reads = np.zeros(n_reads, RAW_READ_DT)
    chunks = []
    seqs = []
    soff = eoff = 0
    for r in range(n_reads):
        rng = np.random.default_rng(seed + r)
        nk = int(n_samples / mean_dwell * 1.3) + 16
        codes = rng.integers(0, 4, nk + model.k - 1, dtype=np.uint8)
        ranks = kmer_ranks_from_codes(codes, model.k, 4)
        dwell = np.maximum(1, rng.geometric(1.0 / mean_dwell, nk))
        covered = min(nk, int(np.searchsorted(np.cumsum(dwell), n_samples)) + 1)
        seqs.append(codes[:covered + model.k - 1])
        lv = np.repeat(model.level_mean[ranks], dwell)[:n_samples]
        sd = np.repeat(model.level_stdv[ranks], dwell)[:n_samples]
        x = (lv + 1.2 * sd * rng.standard_normal(lv.shape[0])).astype(np.float32)
        cap = x.shape[0] // 2 + 8
        reads[r] = (soff, eoff, x.shape[0], cap)
        chunks.append(x)
        soff += x.shape[0]
        eoff += cap
    if return_seqs:
        return np.concatenate(chunks), reads, seqs
    return np.concatenate(chunks), reads


def eventalign_chains(rs: ReadSet, model_id: int = 0):
    """Inputs of nph_eventalign_chain for reads aligned to the reference they were generated from (forward strand, CIGAR all
    M, reference = the read's own sequence): one chain per read.  Returns (pairs i4[n, 2], event_map_start i4, ranks_fwd u4,
    ranks_rc u4, chains EA_CHAIN_DT).  ref: align_read_to_ref's inputs, src/alignment/nanopolish_eventalign.cpp:612-689."""
    k = rs.k
    pairs, maps, rf, rr = [], [], [], []
    chains = np.zeros(rs.n_reads, EA_CHAIN_DT)
    po = mo = ro = oo = 0
    for i in range(rs.n_reads):
        codes = rs.seq_codes[i]
        nk = codes.shape[0] - k + 1
        which = rs.ev_kmer[i]
        first = np.searchsorted(which, np.arange(nk), side="left")
        last = np.searchsorted(which, np.arange(nk), side="right") - 1
        start = np.where(last >= first, first, -1).astype(np.int32)
        has = np.flatnonzero(start >= 0)
        # get_closest_event_to of the first / last aligned k-mer: nearest k-mer with an event, looking backwards first
        first_event = int(start[has[0]])
        last_event = int(start[has[-1]])
        p = np.arange(nk, dtype=np.int32)
        pairs.append(np.stack([p, p], 1)); maps.append(start)
        rf.append(kmer_ranks_from_codes(codes, k, 4)); rr.append(dna_rc_kmer_ranks(codes, k))
        cap = abs(last_event - first_event) + 2
        chains[i] = (po, mo, ro, oo, i, model_id, nk, nk, codes.shape[0], codes.shape[0], cap, 0, first_event, last_event, 0, 0, k, 0)
        po += nk; mo += nk; ro += nk; oo += cap
    return (np.ascontiguousarray(np.concatenate(pairs)), np.concatenate(maps), np.concatenate(rf).astype(np.uint32),
            np.concatenate(rr).astype(np.uint32), chains)


_METH_ALPHABETS = {   # name: (bases, complements, sites, methylated, methylated complement); src/common/nanopolish_alphabet.cpp:15-194
    "cpg": (b"ACGMT", b"TGCGA", [b"CG"], [b"MG"], [b"GM"]),
    "gpc": (b"ACGMT", b"TGCGA", [b"GC"], [b"GM"], [b"MG"]),
    "dam": (b"ACGMT", b"TGCTA", [b"GATC"], [b"GMTC"], [b"CTMG"]),
    "dcm": (b"ACGMT", b"TGCGA", [b"CCAGG", b"CCTGG"], [b"CMAGG", b"CMTGG"], [b"GGTMC", b"GGAMC"]),
}


def meth_params(alphabet: str = "cpg", k: int = 6, min_separation: int = 10, min_flank: int = 10, max_span: int = 200,
                min_event_span: int = 10, region_start: int = -1, region_end: int = -1) -> np.ndarray:
    """nph_meth_params for one of the reference's methylation alphabets (MethylationCallingParameters defaults)."""
    bases, comps, sites, sm, smc = _METH_ALPHABETS[alphabet]
    p = np.zeros(1, METH_PARAMS_DT)
    p[0]["min_separation"], p[0]["min_flank"], p[0]["max_span"], p[0]["min_event_span"] = min_separation, min_flank, max_span, min_event_span
    p[0]["region_start"], p[0]["region_end"], p[0]["k"], p[0]["alphabet_size"] = region_start, region_end, k, len(bases)
    p[0]["bases"], p[0]["complements"], p[0]["n_sites"], p[0]["site_len"] = bases, comps, len(sites), len(sites[0])
    for i in range(len(sites)):
        p[0]["sites"][i], p[0]["sites_methylated"][i], p[0]["sites_methylated_complement"][i] = sites[i], sm[i], smc[i]
    return p


def closest_event_map(which: np.ndarray, nk: int):
    """(base_to_event_map[*].indices[0].start, .stop, closest) per k-mer of a read whose event i was emitted by k-mer which[i]:
    start/stop = first/last event of the k-mer (-1: none); closest[p] = SquiggleRead::get_closest_event_to(p) — the first event
    of the nearest k-mer at or before p that has one (within 1000 k-mers), else of the nearest one after it
    (src/nanopolish_squiggle_read.cpp:160-186)."""
    first = np.searchsorted(which, np.arange(nk), side="left")
    last = np.searchsorted(which, np.arange(nk), side="right") - 1
    has = last >= first
    start = np.where(has, first, -1).astype(np.int32)
    stop = np.where(has, last, -1).astype(np.int32)
    idx = np.arange(nk)
    prev = np.maximum.accumulate(np.where(has, idx, -1))                 # nearest k-mer <= p with an event
    nxt = np.minimum.accumulate(np.where(has, idx, nk)[::-1])[::-1]       # nearest k-mer >= p with an event
    # the backward scan covers [max(0, p - 1000) + 1, p] (its loop stops before stop_before), the forward one [p, min(p + 1000, nk - 1) - 1]
    stop_before = np.maximum(idx - 1000, 0)
    stop_after = np.minimum(idx + 1000, nk - 1)
    before = np.where((prev >= 0) & (prev > stop_before), start[np.maximum(prev, 0)], -1)
    after = np.where((nxt < nk) & (nxt < stop_after), start[np.minimum(nxt, nk - 1)], -1)
    return start, stop, np.where(before == -1, after, before).astype(np.int32)


def methylation_records(rs: ReadSet, model_id: int = 1, ref_start: int = 10_000, rc_every: int = 0):
    """call-methylation's per-record inputs for reads aligned base for base (CIGAR all M) to the sequence they were generated
    from: the reference bases (the read's own sequence; its reverse complement for every rc_every-th read, a reverse-strand
    record whose events fall as reference positions rise) and EventAlignmentRecord::aligned_events exactly as
    src/alignment/nanopolish_alignment_db.cpp:50-91 builds them (boundary k-mers dropped, get_closest_event_to of the read-strand
    k-mer).  Returns (ref_bases u8[total], pairs PAIR_DT[total], records METH_RECORD_DT[n_reads])."""
    k = rs.k
    refs, prs = [], []
    recs = np.zeros(rs.n_reads, METH_RECORD_DT)
    ro = po = 0
    for i in range(rs.n_reads):
        codes = rs.seq_codes[i]
        nk = codes.shape[0] - k + 1
        read_length = codes.shape[0]
        _, _, closest = closest_event_map(rs.ev_kmer[i], nk)
        p = np.arange(k, read_length - k)                      # read_pos >= k and read_pos + k < read_length
        p = p[p < nk]
        rc = 1 if (rc_every and i % rc_every == rc_every - 1) else 0
        if rc:
            ref = _CODE2DNA[(3 - codes[::-1]).astype(np.uint8)]
            ev = closest[read_length - p - k]                  # flip_k_strand
        else:
            ref = _CODE2DNA[codes]
            ev = closest[p]
        pr = np.zeros(p.shape[0], PAIR_DT)
        pr["ref_pos"], pr["read_pos"] = ref_start + p, ev
        if pr.shape[0] and pr["read_pos"][0] == pr["read_pos"][-1]:
            pr = pr[:0]                                        # degenerate alignment: the reference clears it
        recs[i] = (ro, po, i, model_id, ref.shape[0], pr.shape[0], ref_start, rc, 0, (0, 0))
        refs.append(ref); prs.append(pr)
        ro += ref.shape[0]; po += pr.shape[0]
    return np.concatenate(refs), np.concatenate(prs), recs


METH_NO_PAIR = -32768


def compact_event_alignment(records: np.ndarray, pairs: np.ndarray, n_ref_total: int):
    """aligned_events pair lists -> the compact form of nph_methylation_batch_compact: (event_deltas i2[n_ref_total] parallel to the
    reference bases, first_event i4[n_records]).  Raises OverflowError when an event-index step does not fit an int16."""
    deltas = np.full(n_ref_total, METH_NO_PAIR, np.int16)
    first = np.zeros(records.shape[0], np.int32)
    for i, R in enumerate(records):
        pr = pairs[int(R["pair_off"]):int(R["pair_off"]) + int(R["n_pairs"])]
        if pr.shape[0] == 0:
            continue
        off = pr["ref_pos"].astype(np.int64) - int(R["ref_start_pos"])
        assert (np.diff(off) > 0).all() and off[0] >= 0 and off[-1] < int(R["ref_len"])
        ev = pr["read_pos"].astype(np.int64)
        first[i] = ev[0]
        d = np.diff(ev, prepend=ev[0])
        if (np.abs(d) > 32767).any():
            raise OverflowError("event-index step beyond int16: use the pair form")
        deltas[int(R["ref_off"]) + off] = d.astype(np.int16)
    return deltas, first


SCREEN_PARAMS_DT = np.dtype([("flank", "<i4"), ("score_threshold", "<u4"), ("alignment_flags", "<u4"), ("k", "<u4"), ("reads_per_round", "<u4"),
                             ("region_start", "<i4")], align=True)
assert SCREEN_PARAMS_DT.itemsize == 24
SCREEN_SLOTS = 9


def screen_params(region_start: int, k: int = 6, flank: int = 10, threshold: int = 100, flags: int = 0, reads_per_round: int = 8) -> np.ndarray:
    p = np.zeros(1, SCREEN_PARAMS_DT)
    p[0] = (flank, threshold, flags, k, reads_per_round, region_start)
    return p


def gen_pileup(ref_len: int, depth: int, read_bases: int, model: PoreModel, seed: int = 42, region_start: int = 5000, n_true_variants: int = 0,
               rc_every: int = 2):
    """A draft reference of ref_len bases and ~depth-fold coverage by reads of read_bases bases sampled from the TRUTH (the draft with
    n_true_variants substitutions), aligned base for base (CIGAR all M) — the input shape of `variants --consensus` screening
    (SURVEY.md 8d, config 5).  Returns (ref_codes u1, ReadSet, records METH_RECORD_DT, pairs PAIR_DT): record r = read r, its
    EventAlignmentRecord::aligned_events built like src/alignment/nanopolish_alignment_db.cpp:50-91 (ref_off = offset of the record's
    slice in the compact event alignment, see compact_event_alignment)."""
    rng = np.random.default_rng(seed)
    k = model.k
    ref = rng.integers(0, 4, ref_len, dtype=np.uint8)
    truth = ref.copy()
    if n_true_variants:
        pos = rng.choice(np.arange(40, ref_len - 40), n_true_variants, replace=False)
        truth[pos] = (truth[pos] + rng.integers(1, 4, n_true_variants)) % 4
    n_reads = max(1, int(round(depth * ref_len / read_bases)))
    starts = np.sort(rng.integers(0, ref_len - read_bases + 1, n_reads))
    reads = np.zeros(n_reads, READ_DT)
    recs = np.zeros(n_reads, METH_RECORD_DT)
    means, times, seqs, evk, kfe, prs = [], [], [], [], [], []
    p_nev = np.array([0.03, 0.35, 0.45, 0.17])
    eoff = doff = poff = 0
    for r in range(n_reads):
        rr = np.random.default_rng(seed * 7919 + r)
        s0 = int(starts[r])
        seg = truth[s0:s0 + read_bases]
        rc = 1 if (rc_every and r % rc_every == rc_every - 1) else 0
        codes = (3 - seg[::-1]).astype(np.uint8) if rc else seg.copy()          # the bases as the pore saw them
        nk = codes.shape[0] - k + 1
        ranks = kmer_ranks_from_codes(codes, k, 4)
        nev = rr.choice(4, nk, p=p_nev)
        nev[0] = max(nev[0], 1); nev[-1] = max(nev[-1], 1)
        which = np.repeat(np.arange(nk, dtype=np.int32), nev)
        E = which.shape[0]
        shift, scale, var = rr.uniform(-5.0, 5.0), rr.uniform(0.9, 1.1), rr.uniform(0.9, 1.3)
        t = np.arange(E, dtype=np.float64) * 0.002 + rr.uniform(0.0, 100.0)
        m = (scale * model.level_mean[ranks[which]] + shift + var * model.level_stdv[ranks[which]] * rr.standard_normal(E)).astype(np.float32)
        reads[r] = (eoff, E, 0, scale, shift, 0.0, var, np.log(var), E / float(nk))
        _, _, closest = closest_event_map(which, nk)
        q = np.arange(k, read_bases - k)
        q = q[q < nk]
        ev = closest[read_bases - q - k] if rc else closest[q]
        pr = np.zeros(q.shape[0], PAIR_DT)
        pr["ref_pos"], pr["read_pos"] = region_start + s0 + q, ev
        if pr.shape[0] and pr["read_pos"][0] == pr["read_pos"][-1]:
            pr = pr[:0]
        recs[r] = (doff, poff, r, 0, read_bases, pr.shape[0], region_start + s0, rc, 0, (0, 0))
        means.append(m); times.append(t); seqs.append(codes); evk.append(which)
        kfe.append(np.searchsorted(which, np.arange(nk), side="left").astype(np.int32)); prs.append(pr)
        eoff += E; doff += read_bases; poff += pr.shape[0]
    rs = ReadSet(reads, np.concatenate(means), np.concatenate(times), seqs, evk, kfe, k)
    return ref, rs, recs, np.concatenate(prs)


# ---- poly(A) tail length (section 8f N5: `nanopolish polya`) ---------------------------------------------------------------
POLYA_JOB_DT = np.dtype([("sample_off", "<u8"), ("event_off", "<u8"), ("map_off", "<u8"), ("n_samples", "<u4"), ("n_events", "<u4"),
                         ("n_kmers", "<u4"), ("reserved", "<u4"), ("sample_rate", "<f8"), ("shift", "<f8"), ("scale", "<f8"),
                         ("var", "<f8")], align=True)
POLYA_RES_DT = np.dtype([("start", "<u8"), ("leader", "<u8"), ("adapter", "<u8"), ("polya", "<u8"), ("cliffs", "<u8"),
                         ("read_rate", "<f8"), ("polya_length", "<f8"), ("end_score", "<f4"), ("qc", "<u4")], align=True)
POLYA_NOREGION, POLYA_ADAPTER, POLYA_FAILED_LOAD = 1, 2, 4

# the reads' families: what each exercises in estimate_polya_for_single_read
POLYA_FAMILIES = ("pass", "noregion", "adapter", "suffclip", "missing", "zero_median", "failed_load", "tiny")


@dataclass
class PolyaSet:
    samples: np.ndarray          # f32, every read's trimmed raw samples in acquisition order (3'->5' for direct RNA)
    durations: np.ndarray        # f32 event durations (seconds), SquiggleRead order
    map: np.ndarray              # EVENT_RANGE_DT base_to_event_map entries
    jobs: np.ndarray             # POLYA_JOB_DT
    names: list
    suffix_clip: np.ndarray      # u4, length of each record's last CIGAR op
    family: list


def _polya_trace(rng, n_lead, n_adapt, n_polya, n_tx, shift, scale, var, cliff_rate=0.002):
    """START (Gaussian + uniform), leader, adapter mixture, poly(A) with cliff excursions, then a 5-mer-like transcript;
    levels in the HMM's unscaled picoamps, mapped through shift + scale * level with var-scaled noise."""
    n_start = int(rng.integers(150, 1500))
    s = np.where(rng.random(n_start) < 0.5, rng.normal(70.2737, 3.7743, n_start), rng.uniform(40.0, 250.0, n_start))
    lead = rng.normal(110.973, 5.237, n_lead)
    pick = rng.random(n_adapt) < 0.874
    adapt = np.where(pick, rng.normal(79.347, 8.3702, n_adapt), rng.normal(63.3126, 2.7464, n_adapt))
    pa = rng.normal(108.883, 3.257, n_polya)
    cl = rng.random(n_polya) < cliff_rate
    pa[cl] = rng.uniform(72.0, 95.0, int(cl.sum()))
    dwell = np.maximum(1, rng.geometric(1.0 / 30.0, n_tx // 20 + 2))
    lv = np.repeat(rng.uniform(70.0, 125.0, dwell.shape[0]), dwell)[:n_tx]
    tx = lv + rng.normal(0.0, 2.5, lv.shape[0])
    lv = np.concatenate([s, lead, adapt, pa, tx])
    return (shift + scale * lv + (var - 1.0) * rng.normal(0.0, 1.5, lv.shape[0])).astype(np.float32)


def gen_polya(n_reads: int, seed: int = 5, families=POLYA_FAMILIES, polya_samples=(2000, 9000), tx_samples=(4000, 20000),
              sample_rate: float = 3012.0, lengths=None) -> PolyaSet:
    """Seeded direct-RNA-shaped reads for `polya`, cycling through `families` (POLYA_FAMILIES).  lengths: the trace length of
    each read instead (cut from, or padded with, transcript)."""
    samples, durs, maps, names, clips, fam = [], [], [], [], [], []
    jobs = np.zeros(n_reads, POLYA_JOB_DT)
    so = eo = mo = 0
    for r in range(n_reads):
        rng = np.random.default_rng(seed * 100003 + r)
        f = families[r % len(families)]
        shift, scale, var = float(rng.normal(0.0, 3.0)), float(rng.uniform(0.9, 1.1)), float(rng.uniform(0.9, 1.3))
        n_lead, n_adapt = int(rng.integers(300, 1200)), int(rng.integers(1500, 5000))
        n_polya, n_tx = int(rng.integers(*polya_samples)), int(rng.integers(*tx_samples))
        if f == "noregion":
            n_polya = int(rng.integers(20, 150))
        elif f == "adapter":
            n_adapt = int(rng.integers(16000, 24000))
        elif f == "missing":
            n_lead = n_adapt = n_polya = 0
        if f == "tiny":
            n_tiny = 2 if r < len(families) else int(rng.integers(3, 40))          # n = 2: size_t wrap-around in the defaults
            x = (shift + scale * rng.uniform(40.0, 210.0, n_tiny)).astype(np.float32)
        else:
            x = _polya_trace(rng, n_lead, n_adapt, n_polya, n_tx, shift, scale, var)
            if f == "missing":
                x = x[-n_tx:]
        if lengths is not None and f != "tiny":
            want = int(lengths[r])
            x = _polya_trace(rng, n_lead, n_adapt, n_polya, max(16, want), shift, scale, var)[:want]
        n_kmers = int(rng.integers(300, 2500)) if f != "tiny" else int(rng.integers(1, 8))
        n_events = 0 if f == "failed_load" else int(n_kmers * rng.uniform(1.2, 2.0)) + 1
        d = (rng.integers(3, 60, n_events) / sample_rate).astype(np.float32)
        m = np.zeros(n_kmers, EVENT_RANGE_DT)
        if n_events:
            # monotone event ranges per k-mer; some k-mers get none (-1)
            cuts = np.sort(rng.integers(0, n_events, n_kmers))
            span = rng.integers(0, 3, n_kmers)
            m["start"] = cuts
            m["stop"] = np.minimum(cuts + span, n_events - 1)
            none = rng.random(n_kmers) < (0.7 if f == "zero_median" else 0.05)
            m["start"][none] = -1; m["stop"][none] = -1
        jobs[r] = (so, eo, mo, x.shape[0], n_events, n_kmers, 0, sample_rate, shift, scale, var)
        samples.append(x); durs.append(d); maps.append(m)
        names.append(f"{uuid_like(rng)}"); clips.append(int(rng.integers(201, 600)) if f == "suffclip" else int(rng.integers(0, 200)))
        fam.append(f)
        so += x.shape[0]; eo += n_events; mo += n_kmers
    return PolyaSet(np.concatenate(samples), np.concatenate(durs) if eo else np.zeros(0, np.float32), np.concatenate(maps), jobs,
                    names, np.asarray(clips, np.uint32), fam)


def uuid_like(rng) -> str:
    h = rng.integers(0, 16, 32)
    s = "".join("0123456789abcdef"[int(v)] for v in h)
    return f"{s[:8]}-{s[8:12]}-{s[12:16]}-{s[16:20]}-{s[20:]}"
