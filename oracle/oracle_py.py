"""ctypes bindings of the two CPU checkers — TEST INFRASTRUCTURE ONLY.

  * PortOracle : oracle/libnporacle.so, our plain-C restatement (np_oracle.c)
  * RefOracle  : oracle/_ref/libnpref.so, the unmodified reference TUs behind ref_harness.cpp

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import
this module.  Nothing under nanopolish_b200/ does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_SO = os.path.join(HERE, "libnporacle.so")
REF_SO = os.path.join(HERE, "_ref", "libnpref.so")


def build(ref: bool = True) -> None:
    """Compile the checkers (port always; the reference build only where /root/reference exists)."""
    subprocess.run(["make", "-C", HERE, "port"], check=True, stdout=subprocess.DEVNULL)
    if ref:
        subprocess.run(["make", "-C", HERE, "-j8", "ref"], check=True, stdout=subprocess.DEVNULL)


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class _NpoModel(C.Structure):
    _fields_ = [("level_mean", C.c_void_p), ("level_stdv", C.c_void_p),
                ("level_log_stdv", C.c_void_p), ("n_states", C.c_uint32)]


class PortOracle:
    def __init__(self):
        if not os.path.exists(PORT_SO):
            build(ref=False)
        self.lib = L = C.CDLL(PORT_SO)
        L.npo_logsum.restype = C.c_float
        L.npo_logsum.argtypes = [C.c_float, C.c_float]
        L.npo_log_normal_pdf.restype = C.c_float
        L.npo_log_normal_pdf.argtypes = [C.c_float] * 4
        L.npo_hmm_score_batch.restype = C.c_double
        L.npo_hmm_score_dump.restype = C.c_float
        L.npo_abea_batch.restype = C.c_double
        L.npo_score_set_combine.restype = C.c_float
        L.npo_init()
        self._keep = []

    def models(self, model_list):
        arr = (_NpoModel * len(model_list))()
        for i, m in enumerate(model_list):
            mean = np.ascontiguousarray(m.level_mean, np.float64)
            sd = np.ascontiguousarray(m.level_stdv, np.float64)
            lsd = np.ascontiguousarray(m.level_log_stdv, np.float64)
            self._keep += [mean, sd, lsd]
            arr[i] = _NpoModel(mean.ctypes.data, sd.ctypes.data, lsd.ctypes.data, mean.shape[0])
        return arr

    def logsum_table(self):
        t = np.zeros(16000, np.float32)
        self.lib.npo_logsum_table(_p(t))
        return t

    def flank_table(self, n):
        t = np.zeros(n, np.float32)
        self.lib.npo_flank_table(_p(t), C.c_size_t(n))
        return t

    def transitions(self, events_per_base, indel_bias=1.0):
        t = np.zeros(10, np.float32)
        self.lib.npo_transitions(C.c_double(events_per_base), C.c_double(indel_bias), _p(t))
        return t

    def hmm_score_batch(self, reads, ev_mean, ev_start, model_list, kmer_ranks, jobs, indel_bias=1.0,
                        threads=1):
        out = np.zeros(jobs.shape[0], np.float32)
        marr = self.models(model_list)
        secs = self.lib.npo_hmm_score_batch(_p(reads), _p(ev_mean), _p(ev_start), marr, _p(kmer_ranks),
                                            _p(jobs), C.c_size_t(jobs.shape[0]), C.c_double(indel_bias),
                                            C.c_int(threads), _p(out))
        return out, secs

    def hmm_score_dump(self, reads, ev_mean, ev_start, model_list, kmer_ranks, job, indel_bias=1.0):
        E = abs(int(job["event_stop"]) - int(job["event_start"])) + 1
        K = int(job["n_kmers"])
        fm = np.zeros((E + 1, 3 * (K + 2)), np.float32)
        marr = self.models(model_list)
        jb = np.array([job], dtype=job.dtype)
        s = self.lib.npo_hmm_score_dump(_p(reads), _p(ev_mean), _p(ev_start), marr, _p(kmer_ranks), _p(jb),
                                        C.c_double(indel_bias), _p(fm))
        return s, fm

    def hmm_align(self, reads, ev_mean, ev_start, model_list, kmer_ranks, job, indel_bias=1.0):
        from nanopolish_b200.synth import ALIGN_STATE_DT
        E = abs(int(job["event_stop"]) - int(job["event_start"])) + 1
        cap = E + int(job["n_kmers"]) + 4
        out = np.zeros(cap, ALIGN_STATE_DT)
        marr = self.models(model_list)
        jb = np.array([job], dtype=job.dtype)
        st = C.c_int()
        self.lib.npo_hmm_align.restype = C.c_uint32
        n = self.lib.npo_hmm_align(_p(reads), _p(ev_mean), _p(ev_start), marr, _p(kmer_ranks), _p(jb), C.c_double(indel_bias),
                                   _p(out), C.c_uint32(cap), C.byref(st))
        return out[:n].copy(), st.value

    def score_set_combine(self, scores):
        s = np.ascontiguousarray(scores, np.float32)
        return self.lib.npo_score_set_combine(_p(s), C.c_uint32(s.shape[0]))

    def abea_batch(self, reads, ev_mean, ev_start, model, kmer_ranks, jobs, pairs_total, threads=1):
        from nanopolish_b200.synth import PAIR_DT, ABEA_RES_DT
        pairs = np.zeros(pairs_total, PAIR_DT)
        res = np.zeros(jobs.shape[0], ABEA_RES_DT)
        marr = self.models([model])
        secs = self.lib.npo_abea_batch(_p(reads), _p(ev_mean), _p(ev_start), marr, _p(kmer_ranks), _p(jobs),
                                       C.c_size_t(jobs.shape[0]), C.c_int(threads), _p(pairs), _p(res))
        return pairs, res, secs

    def mom(self, reads, ev_mean, model, kmer_ranks, job):
        marr = self.models([model])
        sh, sc = C.c_double(), C.c_double()
        jb = np.array([job], dtype=job.dtype)
        self.lib.npo_mom(_p(reads), _p(ev_mean), marr, _p(kmer_ranks), _p(jb), C.byref(sh), C.byref(sc))
        return sh.value, sc.value

    def detect_events(self, raw, params):
        from nanopolish_b200.synth import EVENT_DT
        out = np.zeros(raw.shape[0] + 1, EVENT_DT)
        self.lib.npo_detect_events.restype = C.c_longlong
        n = self.lib.npo_detect_events(_p(raw), C.c_size_t(raw.shape[0]), _p(params), _p(out), C.c_size_t(out.shape[0]))
        return out[:n].copy()

    def trim_raw(self, raw, trim_start=200, trim_end=10, varseg_chunk=100, varseg_thresh=0.0):
        s, e = C.c_uint32(), C.c_uint32()
        ok = self.lib.npo_trim_raw(_p(raw), C.c_size_t(raw.shape[0]), C.c_int(trim_start), C.c_int(trim_end), C.c_int(varseg_chunk),
                                   C.c_float(varseg_thresh), C.byref(s), C.byref(e))
        return int(ok), s.value, e.value

    def recalibrate(self, reads, ev_mean, model, kmer_ranks, job, pairs, n_pairs):
        from nanopolish_b200.synth import EVENT_RANGE_DT, CALIBRATION_DT
        marr = self.models([model])
        jb = np.array([job], dtype=job.dtype)
        b2e = np.zeros(int(job["n_kmers"]), EVENT_RANGE_DT)
        cal = np.zeros(1, CALIBRATION_DT)
        self.lib.npo_recalibrate(_p(reads), _p(ev_mean), marr, _p(kmer_ranks), _p(jb), _p(pairs), C.c_uint32(int(n_pairs)), _p(b2e), _p(cal))
        return b2e, cal[0]

    def max_threads(self):
        return int(self.lib.npo_max_threads())


class RefOracle:
    """The compiled reference.  Reads are registered once (npref_read_create) and addressed by handle."""

    def __init__(self):
        if not os.path.exists(REF_SO):
            raise FileNotFoundError(REF_SO + " (run `make -C oracle ref` where /root/reference exists)")
        self.lib = L = C.CDLL(REF_SO)
        L.npref_score_batch.restype = C.c_double
        L.npref_abea_batch.restype = C.c_double
        L.npref_abea.restype = C.c_int64
        L.npref_add_logs.restype = C.c_float
        L.npref_add_logs.argtypes = [C.c_float, C.c_float]
        L.npref_log_probability_match_r9.restype = C.c_float
        L.npref_log_normal_pdf.restype = C.c_float
        L.npref_log_normal_pdf.argtypes = [C.c_float] * 3
        L.npref_kmer_rank.restype = C.c_uint32
        self._models = {}

    @staticmethod
    def available() -> bool:
        return os.path.exists(REF_SO)

    def builtin_model(self, alphabet="nucleotide", kit="r9.4_450bps", strand="template", k=6):
        key = (kit, alphabet, strand, k)
        if key not in self._models:
            h = self.lib.npref_model_builtin(kit.encode(), alphabet.encode(), strand.encode(), k)
            if h < 0:
                raise KeyError(key)
            self._models[key] = h
        return self._models[key]

    def custom_model(self, model):
        mean = np.ascontiguousarray(model.level_mean, np.float64)
        sd = np.ascontiguousarray(model.level_stdv, np.float64)
        return self.lib.npref_model_custom(model.alphabet.encode(), model.k, C.c_uint32(mean.shape[0]), _p(mean), _p(sd))

    def model_dump(self, h):
        k, n, a = C.c_uint32(), C.c_uint32(), C.c_uint32()
        self.lib.npref_model_info(h, C.byref(k), C.byref(n), C.byref(a))
        mean = np.zeros(n.value); sd = np.zeros(n.value); lsd = np.zeros(n.value)
        self.lib.npref_model_dump(h, _p(mean), _p(sd), _p(lsd))
        return k.value, a.value, mean, sd, lsd

    def register_reads(self, reads, ev_mean, ev_start, base_model_h):
        hs = np.zeros(reads.shape[0], np.int32)
        for i, r in enumerate(reads):
            o, n = int(r["event_off"]), int(r["n_events"])
            m = np.ascontiguousarray(ev_mean[o:o + n]); t = np.ascontiguousarray(ev_start[o:o + n])
            hs[i] = self.lib.npref_read_create(C.c_uint32(n), _p(m), _p(t), C.c_double(r["shift"]),
                                               C.c_double(r["scale"]), C.c_double(r["drift"]),
                                               C.c_double(r["var"]), C.c_double(r["events_per_base"]),
                                               base_model_h)
        return hs

    def clear_reads(self):
        self.lib.npref_reads_clear()

    def score_batch(self, read_handles, jobs, seqs, model_handles, indel_bias=1.0, threads=1):
        n = jobs.shape[0]
        rh = np.ascontiguousarray(read_handles[jobs["read"]], np.int32)
        mh = np.ascontiguousarray(np.asarray(model_handles, np.int32)[jobs["model_id"]], np.int32)
        es = np.ascontiguousarray(jobs["event_start"], np.uint32)
        ee = np.ascontiguousarray(jobs["event_stop"], np.uint32)
        rc = np.ascontiguousarray(jobs["rc"], np.uint8)
        fl = np.ascontiguousarray(jobs["flags"], np.uint32)
        buf = b"".join(seqs)
        off = np.zeros(n + 1, np.uint64)
        off[1:] = np.cumsum([len(s) for s in seqs])
        out = np.zeros(n, np.float32)
        secs = self.lib.npref_score_batch(C.c_size_t(n), _p(rh), _p(mh), _p(es), _p(ee), _p(rc), _p(fl),
                                          C.c_char_p(buf), _p(off), C.c_double(indel_bias), C.c_int(threads), _p(out))
        return out, secs

    def align(self, read_h, model_h, seq: bytes, e_start, e_stop, rc, flags, indel_bias=1.0):
        cap = abs(int(e_stop) - int(e_start)) + 1 + len(seq) + 4
        ek = np.zeros((cap, 2), np.uint32); lfm = np.zeros(cap, np.float32); st = C.create_string_buffer(cap)
        n = self.lib.npref_align(int(read_h), model_h, C.c_char_p(seq), C.c_uint32(int(e_start)), C.c_uint32(int(e_stop)), int(rc),
                                 C.c_uint32(int(flags)), C.c_double(indel_bias), _p(ek), _p(lfm), st, C.c_uint32(cap))
        return ek[:n].copy(), lfm[:n].copy(), st.raw[:n]

    def read_set_eventalign(self, read_h, name: str, read_sequence: str, b2e_start, b2e_stop, stdv, duration):
        a, b = np.ascontiguousarray(b2e_start, np.int32), np.ascontiguousarray(b2e_stop, np.int32)
        sd, du = np.ascontiguousarray(stdv, np.float32), np.ascontiguousarray(duration, np.float32)
        self.lib.npref_read_set_eventalign(int(read_h), name.encode(), read_sequence.encode(), _p(a), _p(b), C.c_size_t(a.shape[0]), _p(sd), _p(du))

    def eventalign_summary(self):
        """summarize_alignment of the most recent eventalign() call: dict of its counters"""
        ints = np.zeros(5, np.int32); dbl = np.zeros(2)
        self.lib.npref_eventalign_summary(_p(ints), _p(dbl))
        return dict(num_events=int(ints[0]), num_steps=int(ints[1]), num_stays=int(ints[2]), num_skips=int(ints[3]),
                    reference_span=int(ints[4]), sum_duration=float(dbl[0]), sum_z_score=float(dbl[1]))

    def read_set_samples(self, read_h, samples, sample_rate):
        a = np.ascontiguousarray(samples, np.float32)
        self.lib.npref_read_set_samples(int(read_h), _p(a), C.c_size_t(a.shape[0]), C.c_double(sample_rate))

    def event_samples(self, read_h, event_idx):
        """(start_idx, end_idx, scaled samples) of one event: SquiggleRead::get_event_sample_idx / get_scaled_samples_for_event"""
        idx = np.zeros(2, np.uint64); out = np.zeros(4096, np.float32)
        self.lib.npref_event_samples.restype = C.c_longlong
        n = self.lib.npref_event_samples(int(read_h), C.c_size_t(int(event_idx)), _p(idx), _p(out), C.c_size_t(out.shape[0]))
        assert n >= 0
        return int(idx[0]), int(idx[1]), out[:n].copy()

    def eventalign(self, read_h, contig_name: str, contig: str, ref_pos, flag, cigar, read_idx, region=(-1, -1), want_cigar=True):
        """align_read_to_ref + emit_event_alignment_tsv (default options) + the SAM writer's event CIGAR.
        Returns (tsv text, cigar string, int32[n, 3] of (ref_position, event_idx, ord(state)))."""
        cg = np.ascontiguousarray(cigar, np.uint32)
        cap = 1 << 22
        tsv = C.create_string_buffer(cap); cs = C.create_string_buffer(1 << 16)
        ea = np.zeros((1 << 16, 3), np.int32)
        self.lib.npref_eventalign.restype = C.c_longlong
        n = self.lib.npref_eventalign(int(read_h), contig_name.encode(), contig.encode(), int(ref_pos), int(flag), _p(cg), int(cg.shape[0]),
                                      int(read_idx), int(region[0]), int(region[1]), tsv, C.c_size_t(cap), cs, C.c_size_t((1 << 16) if want_cigar else 0),
                                      _p(ea), C.c_size_t(ea.size))
        if n < 0:
            raise RuntimeError("npref_eventalign: output buffer too small")
        return tsv.value.decode(), cs.value.decode(), ea[:n].copy()

    def call_methylation(self, read_h, read_name: str, contig_name: str, contig: str, ref_pos, flag, cigar, methylation_type="cpg",
                         region=(-1, -1), indel_bias=1.0):
        """calculate_methylation_for_read + write_methylation_results_as_tsv on a hand-built record.
        Returns (tsv text, int32[n, 4] of (start, end, n_motif, strands_scored), float64[n, 2] of strand-0 (ll_unmethylated, ll_methylated))."""
        cg = np.ascontiguousarray(cigar, np.uint32)
        cap, scap = 1 << 22, 1 << 15
        tsv = C.create_string_buffer(cap)
        sites = np.zeros((scap, 4), np.int32); ll = np.zeros((scap, 2), np.float64)
        self.lib.npref_call_methylation.restype = C.c_longlong
        n = self.lib.npref_call_methylation(int(read_h), read_name.encode(), contig_name.encode(), contig.encode(), int(ref_pos), int(flag), _p(cg),
                                            int(cg.shape[0]), methylation_type.encode(), int(region[0]), int(region[1]), C.c_double(indel_bias),
                                            tsv, C.c_size_t(cap), _p(sites), _p(ll), C.c_size_t(scap))
        if n < 0:
            raise RuntimeError("npref_call_methylation: output buffer too small")
        return tsv.value.decode(), sites[:n].copy(), ll[:n].copy()

    def calibrate(self, read_h, model_h, read_sequence: bytes, pairs):
        """The tail of load_from_raw after ABEA (base-to-event map, get_eventalignment_for_1d_basecalls, recalibrate_model):
        dict(shift, scale, drift, var, events_per_base, calibrated, n_used) or None for an empty alignment."""
        pr = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        out = np.zeros(6)
        self.lib.npref_calibrate.restype = C.c_longlong
        n = self.lib.npref_calibrate(int(read_h), int(model_h), read_sequence, _p(pr), C.c_size_t(pr.shape[0]), _p(out))
        if n < 0:
            return None
        return dict(shift=out[0], scale=out[1], drift=out[2], var=out[3], events_per_base=out[4], calibrated=bool(out[5]), n_used=int(n))

    def set_globals(self, indel_bias: float, omp_threads: int):
        """hmm_indel_bias_factor and the OpenMP thread count, process-wide (for callers that run harness calls from their own threads)"""
        self.lib.npref_set_globals(C.c_double(indel_bias), int(omp_threads))

    def score_variants_thresholded(self, read_handles, windows, rc, ref_seq: str, ref_position, variants, flags, threshold,
                                   methylation: bool, indel_bias=1.0):
        """[score_variant_thresholded(v, Haplotype(ref), reads, flags, threshold, types).quality for v in variants], single thread"""
        n, nv = len(read_handles), len(variants)
        rh = np.ascontiguousarray(read_handles, np.int32)
        es = np.array([w[0] for w in windows], np.uint32); ee = np.array([w[1] for w in windows], np.uint32)
        rcs = np.ascontiguousarray(rc, np.uint8)
        pos = (C.c_size_t * nv)(*[v[0] for v in variants])
        refs = (C.c_char_p * nv)(*[v[1].encode() for v in variants]); alts = (C.c_char_p * nv)(*[v[2].encode() for v in variants])
        q = np.zeros(nv)
        self.lib.npref_score_variants_thresholded(n, _p(rh), _p(es), _p(ee), _p(rcs), ref_seq.encode(), C.c_size_t(ref_position), nv, pos, refs,
                                                  alts, C.c_uint32(flags), C.c_uint32(threshold), int(methylation), C.c_double(indel_bias), _p(q))
        return q

    def score_variant_group(self, read_handles, windows, rc, ref_seq: str, ref_position, variants, max_haplotypes, flags, methylation=False,
                            indel_bias=1.0):
        """score_variant_group: dict {frozenset of variant ids: float64[n_reads] scores}; variants = [(pos, ref, alt)]."""
        n = len(read_handles); nv = len(variants)
        rh = np.ascontiguousarray(read_handles, np.int32)
        es = np.array([w[0] for w in windows], np.uint32); ee = np.array([w[1] for w in windows], np.uint32)
        rcs = np.ascontiguousarray(rc, np.uint8)
        cap = 1 << 12
        combos = np.zeros(cap, np.uint32); scores = np.zeros(cap * n, np.float64)
        self.lib.npref_score_variant_group.restype = C.c_longlong
        k = self.lib.npref_score_variant_group(n, _p(rh), _p(es), _p(ee), _p(rcs), ref_seq.encode(), C.c_size_t(ref_position), nv,
                                               (C.c_size_t * nv)(*[v[0] for v in variants]), (C.c_char_p * nv)(*[v[1].encode() for v in variants]),
                                               (C.c_char_p * nv)(*[v[2].encode() for v in variants]), int(max_haplotypes), int(flags),
                                               1 if methylation else 0, C.c_double(indel_bias), _p(combos), _p(scores), C.c_size_t(cap))
        if k < 0:
            raise RuntimeError("npref_score_variant_group: buffer too small")
        return {frozenset(i for i in range(nv) if combos[c] >> i & 1): scores[c * n:(c + 1) * n].copy() for c in range(k)}

    def modbam(self, seq: str, ref_pos, flag, cigar, calls):
        """create_modbam_record's Mm / Ml tags; calls = [(start_position, site sequence, ll_methylated[0], ll_unmethylated[0])]."""
        cg = np.ascontiguousarray(cigar, np.uint32)
        n = len(calls)
        sp = np.array([c[0] for c in calls], np.int32)
        seqs = (C.c_char_p * max(n, 1))(*[c[1].encode() for c in calls])
        lm = np.array([c[2] for c in calls], np.float64); lu = np.array([c[3] for c in calls], np.float64)
        mm = C.create_string_buffer(1 << 16); ml = np.zeros(1 << 14, np.uint8)
        self.lib.npref_modbam.restype = C.c_longlong
        k = self.lib.npref_modbam(seq.encode(), int(ref_pos), int(flag), _p(cg), int(cg.shape[0]), n, _p(sp), seqs, _p(lm), _p(lu),
                                  mm, C.c_size_t(1 << 16), _p(ml), C.c_size_t(ml.shape[0]))
        if k < 0:
            raise RuntimeError("npref_modbam: output buffer too small")
        return mm.value.decode(), ml[:k].copy()

    def kmer_ranks(self, model_h, seq: bytes, rc: bool):
        out = np.zeros(max(len(seq), 1), np.uint32)
        n = self.lib.npref_kmer_ranks(model_h, C.c_char_p(seq), int(rc), _p(out))
        return out[:n].copy()

    def alphabet_op(self, alphabet: str, op: int, s: bytes) -> bytes:
        out = C.create_string_buffer(len(s) + 16)
        n = self.lib.npref_alphabet_op(alphabet.encode(), op, C.c_char_p(s), out)
        return out.raw[:n]

    def abea(self, read_h, model_h, seq: bytes, cap: int):
        pairs = np.zeros((cap, 2), np.int32)
        n = self.lib.npref_abea(int(read_h), model_h, C.c_char_p(seq), _p(pairs), C.c_size_t(cap))
        return pairs[:max(n, 0)].copy(), n

    def abea_batch(self, read_handles, model_h, seqs, caps, threads=1):
        n = len(seqs)
        buf = b"".join(seqs)
        off = np.zeros(n + 1, np.uint64); off[1:] = np.cumsum([len(s) for s in seqs])
        poff = np.zeros(n + 1, np.uint64); poff[1:] = np.cumsum(caps)
        pairs = np.zeros((int(poff[-1]), 2), np.int32)
        npairs = np.zeros(n, np.int64)
        rh = np.ascontiguousarray(read_handles, np.int32)
        secs = self.lib.npref_abea_batch(C.c_size_t(n), _p(rh), model_h, C.c_char_p(buf), _p(off), C.c_int(threads),
                                         _p(pairs), _p(poff), _p(npairs))
        return pairs, poff, npairs, secs

    def detect_events(self, raw, rna=False):
        n = raw.shape[0]
        start = np.zeros(n + 1, np.uint64); length = np.zeros(n + 1, np.float32)
        mean = np.zeros(n + 1, np.float32); stdv = np.zeros(n + 1, np.float32)
        self.lib.npref_detect_events.restype = C.c_longlong
        ne = self.lib.npref_detect_events(_p(raw), C.c_size_t(n), int(rna), _p(start), _p(length), _p(mean), _p(stdv), C.c_size_t(n + 1))
        return start[:ne], length[:ne], mean[:ne], stdv[:ne]

    def trim_raw(self, raw, trim_start=200, trim_end=10, varseg_chunk=100, varseg_thresh=0.0):
        s, e = C.c_uint32(), C.c_uint32()
        ok = self.lib.npref_trim_raw(_p(raw), C.c_size_t(raw.shape[0]), C.c_int(trim_start), C.c_int(trim_end), C.c_int(varseg_chunk),
                                     C.c_float(varseg_thresh), C.byref(s), C.byref(e))
        return int(ok), s.value, e.value

    def mom(self, read_h, model_h, seq: bytes):
        out = np.zeros(4)
        self.lib.npref_mom(int(read_h), model_h, C.c_char_p(seq), _p(out))
        return out

    def logsum_table(self):
        t = np.zeros(16000, np.float32)
        self.lib.npref_logsum_table(_p(t))
        return t

    def add_logs(self, a, b):
        """add_logs(a[i], b[i]) for each i, as float32"""
        return np.array([self.lib.npref_add_logs(float(x), float(y)) for x, y in zip(a, b)], np.float32)

    def max_threads(self):
        return int(self.lib.npref_max_threads())
