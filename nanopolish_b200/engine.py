"""Python driver over the C ABI (include/nph.h) — used by tests/, bench.py and smoke().

The product is libnph.so; this wrapper only marshals numpy buffers (structured arrays with the
layouts in synth.py) into the C calls.  It never computes a score itself and has no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .synth import ABEA_RES_DT, ALIGN_STATE_DT, CALIBRATION_DT, EVENT_DT, EVENT_RANGE_DT, METH_SITE_DT, PAIR_DT, RAW_RANGE_DT


def _p(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


class Engine:
    """One nph_ctx (one device, one stream)."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self.lib = _lib.load()
        self.ctx = C.c_void_p()
        if stream is None:
            rc = self.lib.nph_create(C.byref(self.ctx), device)
        else:
            rc = self.lib.nph_create_on_stream(C.byref(self.ctx), device, C.c_void_p(stream))
        if rc != 0:
            raise _lib.NphError(rc, "nph_create", self.lib.nph_strerror(rc).decode())
        self.n_jobs = 0

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise _lib.NphError(rc, what, self.lib.nph_strerror(rc).decode() + " / " +
                                self.lib.nph_last_error(self.ctx).decode())

    def close(self):
        if self.ctx:
            self.lib.nph_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- call-methylation: enumeration + scoring on the device (include/nph.h, section N3) ----
    @staticmethod
    def meth_sites_cap(records, params) -> int:
        return int((records["ref_len"].astype(np.int64) // (int(params[0]["min_separation"]) + 1) + 2).sum())

    def methylation_batch(self, reads, ev_mean, ev_start_time, ref_bases, pairs, records, params, indel_bias: float = 1.0, out=None):
        """nph_methylation_batch: returns (site_off u8[n_records + 1], sites METH_SITE_DT[n_sites], scored_events)."""
        n = int(records.shape[0])
        cap = self.meth_sites_cap(records, params)
        site_off, sites = out if out is not None else (np.zeros(n + 1, np.uint64), np.zeros(max(cap, 1), METH_SITE_DT))
        scored = C.c_uint64()
        self._check(self.lib.nph_methylation_batch(self.ctx, _p(reads), reads.shape[0], _p(ev_mean), _p(ev_start_time), ev_mean.shape[0],
                                                   _p(ref_bases), ref_bases.shape[0], _p(pairs), pairs.shape[0], _p(records), n, _p(params),
                                                   indel_bias, _p(site_off), _p(sites), sites.shape[0], C.byref(scored)), "nph_methylation_batch")
        return site_off, sites[:int(site_off[n])], int(scored.value)

    def methylation_batch_compact(self, reads, ev_mean, ev_start_time, ref_bases, deltas, first_event, records, params, indel_bias: float = 1.0, out=None):
        """nph_methylation_batch_compact (event alignments as int16 deltas per reference base)"""
        n = int(records.shape[0])
        cap = self.meth_sites_cap(records, params)
        site_off, sites = out if out is not None else (np.zeros(n + 1, np.uint64), np.zeros(max(cap, 1), METH_SITE_DT))
        scored = C.c_uint64()
        self._check(self.lib.nph_methylation_batch_compact(self.ctx, _p(reads), reads.shape[0], _p(ev_mean), _p(ev_start_time), ev_mean.shape[0],
                                                           _p(ref_bases), _p(deltas), ref_bases.shape[0], _p(first_event), _p(records), n, _p(params),
                                                           indel_bias, _p(site_off), _p(sites), sites.shape[0], C.byref(scored)), "nph_methylation_batch_compact")
        return site_off, sites[:int(site_off[n])], int(scored.value)

    def methylation_load_compact(self, ref_bases, deltas, first_event, records, params, indel_bias: float = 1.0):
        self._check(self.lib.nph_methylation_load_compact(self.ctx, _p(ref_bases), _p(deltas), ref_bases.shape[0], _p(first_event), _p(records),
                                                          records.shape[0], _p(params), indel_bias), "nph_methylation_load_compact")
        self._meth_n = int(records.shape[0])

    def methylation_load(self, ref_bases, pairs, records, params, indel_bias: float = 1.0):
        self._check(self.lib.nph_methylation_load(self.ctx, _p(ref_bases), ref_bases.shape[0], _p(pairs), pairs.shape[0], _p(records),
                                                  records.shape[0], _p(params), indel_bias), "nph_methylation_load")
        self._meth_n = int(records.shape[0])

    def methylation_run(self):
        self._check(self.lib.nph_methylation_run(self.ctx), "nph_methylation_run")

    def methylation_counts(self):
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._check(self.lib.nph_methylation_counts(self.ctx, C.byref(a), C.byref(b), C.byref(c)), "nph_methylation_counts")
        return int(a.value), int(b.value), int(c.value)

    def methylation_sites_dev(self):
        """(device pointer, n_sites) of the last run's site records (nph_methylation_sites_dev)"""
        ptr, n = C.c_void_p(), C.c_uint64()
        self._check(self.lib.nph_methylation_sites_dev(self.ctx, C.byref(ptr), C.byref(n)), "nph_methylation_sites_dev")
        return int(ptr.value or 0), int(n.value)

    def methylation_tsv(self, contig: str, names: list, is_reverse: np.ndarray, cap: int | None = None) -> bytes:
        """nph_methylation_tsv: the methylation_calls.tsv rows of the last run, formatted on the device."""
        blob = "".join(names).encode()
        off = np.zeros(len(names) + 1, np.uint32)
        off[1:] = np.cumsum([len(n.encode()) for n in names])
        rev = np.ascontiguousarray(is_reverse, np.uint8)
        if cap is None:
            cap = 256 * max(1, self.methylation_counts()[0]) + 4096
        out = np.empty(cap, np.uint8)
        n = C.c_uint64()
        self._check(self.lib.nph_methylation_tsv(self.ctx, contig.encode(), blob, _p(off), _p(rev), _p(out), cap, C.byref(n)), "nph_methylation_tsv")
        return out[:int(n.value)].tobytes()

    def methylation_fetch(self, out=None):
        n_sites = self.methylation_counts()[0]
        site_off, sites = out if out is not None else (np.zeros(self._meth_n + 1, np.uint64), np.zeros(max(n_sites, 1), METH_SITE_DT))
        self._check(self.lib.nph_methylation_fetch(self.ctx, _p(site_off), _p(sites), sites.shape[0]), "nph_methylation_fetch")
        return site_off, sites[:n_sites]

    # ---- variants: candidate screening on the device (include/nph.h, section N2) ----
    def screen_edits_batch(self, reads, ev_mean, ev_start_time, ref_bases, deltas, first_event, records, params, indel_bias: float = 1.0):
        """nph_screen_edits_batch: returns (qualities f8[n_pos, 9], n_reads u4[n_pos], scored_events)."""
        n_pos = int(ref_bases.shape[0]) - 1
        q = np.zeros((n_pos, 9), np.float64); nr = np.zeros(n_pos, np.uint32)
        scored = C.c_uint64()
        self._check(self.lib.nph_screen_edits_batch(self.ctx, _p(reads), reads.shape[0], _p(ev_mean), _p(ev_start_time), ev_mean.shape[0],
                                                    _p(ref_bases), ref_bases.shape[0], _p(deltas), deltas.shape[0], _p(first_event), _p(records),
                                                    records.shape[0], _p(params), indel_bias, _p(q), _p(nr), C.byref(scored)), "nph_screen_edits_batch")
        return q, nr, int(scored.value)

    def screen_load(self, ref_bases, deltas, first_event, records, params, indel_bias: float = 1.0):
        self._check(self.lib.nph_screen_load(self.ctx, _p(ref_bases), ref_bases.shape[0], _p(deltas), deltas.shape[0], _p(first_event), _p(records),
                                             records.shape[0], _p(params), indel_bias), "nph_screen_load")
        self._screen_n = int(ref_bases.shape[0]) - 1

    def screen_run(self):
        self._check(self.lib.nph_screen_run(self.ctx), "nph_screen_run")

    def screen_counts(self):
        a, b, c, d, e = C.c_uint32(), C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._check(self.lib.nph_screen_counts(self.ctx, C.byref(a), C.byref(b), C.byref(c), C.byref(d), C.byref(e)), "nph_screen_counts")
        return dict(rounds=int(a.value), jobs=int(b.value), scored_events=int(c.value), jobs_without_exit=int(d.value), reference_events=int(e.value))

    def screen_fetch(self, with_reference_rows: bool = False):
        q = np.zeros((self._screen_n, 9), np.float64); nr = np.zeros(self._screen_n, np.uint32)
        rows = np.zeros(self._screen_n, np.uint64) if with_reference_rows else None
        self._check(self.lib.nph_screen_fetch(self.ctx, _p(q), _p(nr), _p(rows)), "nph_screen_fetch")
        return (q, nr, rows) if with_reference_rows else (q, nr)

    # ---- models / reads / jobs ----------------------------------------------------------
    def model_upload(self, model) -> int:
        mid = C.c_uint32()
        mean = np.ascontiguousarray(model.level_mean, np.float64)
        sd = np.ascontiguousarray(model.level_stdv, np.float64)
        lsd = np.ascontiguousarray(model.level_log_stdv, np.float64)
        self._check(self.lib.nph_model_upload(self.ctx, _p(mean), _p(sd), _p(lsd), mean.shape[0], model.k,
                                              model.alphabet_size, C.byref(mid)), "nph_model_upload")
        return mid.value

    def reads_load(self, reads, ev_mean, ev_start_time):
        self._check(self.lib.nph_reads_load(self.ctx, _p(reads), reads.shape[0], _p(ev_mean),
                                            _p(ev_start_time), ev_mean.shape[0]), "nph_reads_load")

    def hmm_jobs_load(self, kmer_ranks, jobs, indel_bias: float = 1.0):
        self._check(self.lib.nph_hmm_jobs_load(self.ctx, _p(kmer_ranks), kmer_ranks.shape[0], _p(jobs),
                                               jobs.shape[0], indel_bias), "nph_hmm_jobs_load")
        self.n_jobs = int(jobs.shape[0])

    def hmm_score(self, scores_dev_ptr: int | None = None):
        self._check(self.lib.nph_hmm_score(self.ctx, C.c_void_p(scores_dev_ptr) if scores_dev_ptr else None),
                    "nph_hmm_score")

    def hmm_scores_fetch(self, out: np.ndarray | None = None) -> np.ndarray:
        if out is None:
            out = np.empty(self.n_jobs, np.float32)
        self._check(self.lib.nph_hmm_scores_fetch(self.ctx, _p(out), out.shape[0]), "nph_hmm_scores_fetch")
        return out

    def hmm_score_batch(self, reads, ev_mean, ev_start_time, kmer_ranks, jobs, indel_bias: float = 1.0,
                        out: np.ndarray | None = None) -> np.ndarray:
        """== [profile_hmm_score(seq_j, data_j, flags_j) for j]  through the one-shot C call."""
        if out is None:
            out = np.empty(jobs.shape[0], np.float32)
        self._check(self.lib.nph_hmm_score_batch(self.ctx, _p(reads), reads.shape[0], _p(ev_mean),
                                                 _p(ev_start_time), ev_mean.shape[0], _p(kmer_ranks),
                                                 kmer_ranks.shape[0], _p(jobs), jobs.shape[0], indel_bias,
                                                 _p(out)), "nph_hmm_score_batch")
        self.n_jobs = int(jobs.shape[0])
        return out

    def hmm_score_batch_seq(self, reads, ev_mean, ev_start_time, seq_codes, jobs, indel_bias: float = 1.0,
                            out: np.ndarray | None = None) -> np.ndarray:
        """the same with base codes instead of k-mer ranks (nph_hmm_score_batch_seq; jobs' rank_off = code offsets)"""
        if out is None:
            out = np.empty(jobs.shape[0], np.float32)
        self._check(self.lib.nph_hmm_score_batch_seq(self.ctx, _p(reads), reads.shape[0], _p(ev_mean), _p(ev_start_time), ev_mean.shape[0],
                                                     _p(seq_codes), seq_codes.shape[0], _p(jobs), jobs.shape[0], indel_bias, _p(out)),
                    "nph_hmm_score_batch_seq")
        self.n_jobs = int(jobs.shape[0])
        return out

    def hmm_jobs_load_seq(self, seq_codes, jobs, indel_bias: float = 1.0):
        self._check(self.lib.nph_hmm_jobs_load_seq(self.ctx, _p(seq_codes), seq_codes.shape[0], _p(jobs), jobs.shape[0], indel_bias),
                    "nph_hmm_jobs_load_seq")
        self.n_jobs = int(jobs.shape[0])

    def score_set_combine(self, scores: np.ndarray, n_alt: int) -> np.ndarray:
        s = np.ascontiguousarray(scores, np.float32)
        g = s.shape[0] // n_alt
        out = np.empty(g, np.float32)
        self._check(self.lib.nph_score_set_combine(_p(s), g, n_alt, _p(out)), "nph_score_set_combine")
        return out

    # ---- Viterbi alignment (profile_hmm_align) -------------------------------------------
    def hmm_align_batch(self, reads, ev_mean, ev_start_time, kmer_ranks, jobs, indel_bias: float = 1.0):
        """== [profile_hmm_align(seq_j, data_j, flags_j) for j]: list of ALIGN_STATE_DT arrays (empty where the
        reference would assert), plus l_fm of each alignment's final state."""
        n = jobs.shape[0]
        E = np.abs(jobs["event_stop"].astype(np.int64) - jobs["event_start"].astype(np.int64)) + 1
        caps = E + jobs["n_kmers"].astype(np.int64) + 2
        off = np.zeros(n + 1, np.uint64)
        off[1:] = np.cumsum(caps)
        states = np.zeros(int(off[-1]), ALIGN_STATE_DT)
        counts = np.zeros(n, np.uint32)
        scores = np.zeros(n, np.float32)
        self._check(self.lib.nph_hmm_align_batch(self.ctx, _p(reads), reads.shape[0], _p(ev_mean), _p(ev_start_time),
                                                 ev_mean.shape[0], _p(kmer_ranks), kmer_ranks.shape[0], _p(jobs), n,
                                                 indel_bias, _p(states), _p(off), _p(counts), _p(scores)),
                    "nph_hmm_align_batch")
        return [states[int(off[j]):int(off[j]) + int(counts[j])] for j in range(n)], scores

    def hmm_align(self, kmer_ranks, jobs, indel_bias: float = 1.0):
        """hmm_align_batch against the reads a preceding reads_load() left resident (eventalign's chained rounds)."""
        n = jobs.shape[0]
        E = np.abs(jobs["event_stop"].astype(np.int64) - jobs["event_start"].astype(np.int64)) + 1
        off = np.zeros(n + 1, np.uint64)
        off[1:] = np.cumsum(E + jobs["n_kmers"].astype(np.int64) + 2)
        states = np.zeros(int(off[-1]), ALIGN_STATE_DT)
        counts = np.zeros(n, np.uint32)
        scores = np.zeros(n, np.float32)
        self._check(self.lib.nph_hmm_align(self.ctx, _p(kmer_ranks), kmer_ranks.shape[0], _p(jobs), n, indel_bias,
                                           _p(states), _p(off), _p(counts), _p(scores)), "nph_hmm_align")
        return [states[int(off[j]):int(off[j]) + int(counts[j])] for j in range(n)], scores

    def eventalign_chain(self, pairs, event_map_start, ref_ranks_fwd, ref_ranks_rc, chains, indel_bias: float = 1.0, out=None):
        """eventalign's segment chains (align_read_to_ref's per-segment loop) walked on the device against the resident
        reads: returns (records EA_RECORD_DT[sum out_cap], results EA_RESULT_DT[n_chains]); chain c's records are
        records[out_off : out_off + n_records]."""
        from .synth import EA_RECORD_DT, EA_RESULT_DT
        n = chains.shape[0]
        total = int((chains["out_off"] + chains["out_cap"]).max()) if n else 0
        if out is not None:                      # caller-owned (e.g. page-locked) output buffers
            records, results = out
            assert records.shape[0] >= total and results.shape[0] >= n
        else:
            records = np.zeros(total, EA_RECORD_DT)
            results = np.zeros(n, EA_RESULT_DT)
        self._check(self.lib.nph_eventalign_chain(self.ctx, _p(pairs), pairs.shape[0], _p(event_map_start), event_map_start.shape[0],
                                                  _p(ref_ranks_fwd), _p(ref_ranks_rc), ref_ranks_fwd.shape[0], _p(chains), n,
                                                  indel_bias, _p(records), total, _p(results)), "nph_eventalign_chain")
        return records, results

    # ---- ABEA ---------------------------------------------------------------------------
    def abea_batch(self, reads, ev_mean, ev_start_time, kmer_ranks, jobs, model_id: int, pairs_total: int):
        pairs = np.zeros(pairs_total, PAIR_DT)
        res = np.zeros(jobs.shape[0], ABEA_RES_DT)
        self._check(self.lib.nph_abea_batch(self.ctx, _p(reads), reads.shape[0], _p(ev_mean), _p(ev_start_time),
                                            ev_mean.shape[0], _p(kmer_ranks), kmer_ranks.shape[0], _p(jobs),
                                            jobs.shape[0], model_id, _p(pairs), pairs_total, _p(res)),
                    "nph_abea_batch")
        return pairs, res

    def abea_jobs_load(self, kmer_ranks, jobs, model_id: int, pairs_total: int):
        self._check(self.lib.nph_abea_jobs_load(self.ctx, _p(kmer_ranks), kmer_ranks.shape[0], _p(jobs),
                                                jobs.shape[0], model_id, pairs_total), "nph_abea_jobs_load")
        self._abea_n = int(jobs.shape[0])
        self._abea_pairs = int(pairs_total)

    def abea_run(self):
        self._check(self.lib.nph_abea_run(self.ctx), "nph_abea_run")

    def abea_fetch(self):
        pairs = np.zeros(self._abea_pairs, PAIR_DT)
        res = np.zeros(self._abea_n, ABEA_RES_DT)
        self._check(self.lib.nph_abea_fetch(self.ctx, _p(pairs), self._abea_pairs, _p(res), self._abea_n),
                    "nph_abea_fetch")
        return pairs, res

    def mom_batch(self, reads, ev_mean, kmer_ranks, jobs, model_id: int) -> np.ndarray:
        out = np.zeros((jobs.shape[0], 2), np.float64)
        self._check(self.lib.nph_mom_batch(self.ctx, _p(reads), reads.shape[0], _p(ev_mean), ev_mean.shape[0],
                                           _p(kmer_ranks), kmer_ranks.shape[0], _p(jobs), jobs.shape[0],
                                           model_id, _p(out)), "nph_mom_batch")
        return out

    # ---- event detection (scrappie detect_events) ---------------------------------------------
    def detect_events_batch(self, raw, reads, params, out=None):
        """== [detect_events(read_i)]: list of EVENT_DT arrays, one per raw read.  out: (events EVENT_DT[room], counts u4[n_reads]) to
        reuse (page-locked) buffers across calls."""
        total = int((reads["event_off"] + reads["event_cap"]).max()) if reads.shape[0] else 0
        events, counts = out if out is not None else (np.zeros(total, EVENT_DT), np.zeros(reads.shape[0], np.uint32))
        assert events.shape[0] >= total and counts.shape[0] >= reads.shape[0]
        self._check(self.lib.nph_detect_events_batch(self.ctx, _p(raw), raw.shape[0], _p(reads), reads.shape[0], _p(params),
                                                     _p(events), total, _p(counts)), "nph_detect_events_batch")
        return [events[int(r["event_off"]):int(r["event_off"]) + int(c)] for r, c in zip(reads, counts)]

    # ---- raw trimming and post-ABEA calibration (the rest of load_from_raw) -----------------------
    def trim_raw_batch(self, raw, reads, trim_start=200, trim_end=10, varseg_chunk=100, varseg_thresh=0.0):
        """== trim_and_segment_raw per read: RAW_RANGE_DT[n_reads], {0,0} where nothing survives."""
        out = np.zeros(reads.shape[0], RAW_RANGE_DT)
        self._check(self.lib.nph_trim_raw_batch(self.ctx, _p(raw), raw.shape[0], _p(reads), reads.shape[0], trim_start, trim_end,
                                                varseg_chunk, varseg_thresh, _p(out)), "nph_trim_raw_batch")
        return out

    def recalibrate_batch(self, reads, ev_mean, kmer_ranks, jobs, model_id, pairs, results):
        """base_to_event_map + events_per_base + recalibrate_model per ABEA job: (EVENT_RANGE_DT[n_ranks], CALIBRATION_DT[n_jobs])."""
        b2e = np.zeros(kmer_ranks.shape[0], EVENT_RANGE_DT)
        cal = np.zeros(jobs.shape[0], CALIBRATION_DT)
        self._check(self.lib.nph_recalibrate_batch(self.ctx, _p(reads), reads.shape[0], _p(ev_mean), ev_mean.shape[0], _p(kmer_ranks),
                                                   kmer_ranks.shape[0], _p(jobs), jobs.shape[0], model_id, _p(pairs), pairs.shape[0],
                                                   _p(results), _p(b2e), _p(cal)), "nph_recalibrate_batch")
        return b2e, cal

    def load_from_raw_batch(self, raw, kmer_ranks, jobs, model_id, params, events_cap=None, pinned=None):
        """SquiggleRead::load_from_raw for a batch in one call.  Returns (event_off u64[n+1], mean, stdv, start_time,
        duration, base_to_event EVENT_RANGE_DT[n_ranks], CALIBRATION_DT[n_jobs]); event arrays are compact, job order."""
        n = jobs.shape[0]
        cap = int(events_cap if events_cap is not None else raw.shape[0] // 3 + 16 * n)
        off = np.zeros(n + 1, np.uint64)
        if pinned is not None:            # caller-staged output buffers (e.g. page-locked): mean, stdv, start_time, duration, b2e, cal
            mean, stdv, start, dur, b2e, cal = pinned
        else:
            mean = np.zeros(cap, np.float32); stdv = np.zeros(cap, np.float32); start = np.zeros(cap, np.float64); dur = np.zeros(cap, np.float32)
            b2e = np.zeros(kmer_ranks.shape[0], EVENT_RANGE_DT)
            cal = np.zeros(n, CALIBRATION_DT)
        self._check(self.lib.nph_load_from_raw_batch(self.ctx, _p(raw), raw.shape[0], _p(kmer_ranks), kmer_ranks.shape[0], _p(jobs), n, model_id,
                                                     _p(params), _p(off), _p(mean), _p(stdv), _p(start), _p(dur), cap, _p(b2e), _p(cal)),
                    "nph_load_from_raw_batch")
        tot = int(off[-1])
        return off, mean[:tot], stdv[:tot], start[:tot], dur[:tot], b2e, cal

    # ---- poly(A) tail length (nanopolish polya) -------------------------------------------------
    def polya_batch(self, samples, durations, emap, jobs, out=None):
        """== the device part of estimate_polya_for_single_read per POLYA_JOB_DT job: POLYA_RES_DT[n_jobs] (segmentation, cliffs,
        read rate, tail length, Viterbi end score, NOREGION / ADAPTER / failed-load bits).  out: a (page-locked) result buffer."""
        from .synth import POLYA_RES_DT
        res = out if out is not None else np.zeros(jobs.shape[0], POLYA_RES_DT)
        self._check(self.lib.nph_polya_batch(self.ctx, _p(samples), samples.shape[0], _p(durations), durations.shape[0], _p(emap),
                                             emap.shape[0], _p(jobs), jobs.shape[0], _p(res)), "nph_polya_batch")
        return res

    def polya_after_load(self, n_jobs: int, out=None):
        """polya over the reads of the last load_from_raw_batch, from what it left on the device (nothing is uploaded)."""
        from .synth import POLYA_RES_DT
        res = out if out is not None else np.zeros(n_jobs, POLYA_RES_DT)
        self._check(self.lib.nph_polya_after_load(self.ctx, _p(res), n_jobs), "nph_polya_after_load")
        return res

    # ---- measurement ----------------------------------------------------------------------
    def last_trim_ranges(self, n_jobs: int) -> np.ndarray:
        """[start, end) of the samples each job of the last load_from_raw_batch kept (what SRF_LOAD_RAW_SAMPLES stores)."""
        from .synth import RAW_RANGE_DT
        out = np.zeros(n_jobs, RAW_RANGE_DT)
        self._check(self.lib.nph_last_trim_ranges(self.ctx, _p(out), n_jobs), "nph_last_trim_ranges")
        return out

    def sync(self):
        self._check(self.lib.nph_sync(self.ctx), "nph_sync")

    def last_kernel_ms(self):
        ms, n = C.c_float(), C.c_int()
        self._check(self.lib.nph_last_kernel_ms(self.ctx, C.byref(ms), C.byref(n)), "nph_last_kernel_ms")
        return ms.value, n.value

    def stream(self) -> int:
        return int(self.lib.nph_stream(self.ctx) or 0)
