"""`nanopolish polya` (section 8f N5) on the device: nph_polya_batch against the plain-C restatement on large batches and against
the compiled reference's recorded answers, the resident form after nph_load_from_raw_batch, malformed jobs, and the
exhaustive check of the restated expf / logf against the host's libm."""
import os
import subprocess
import types

import numpy as np
import pytest

from nanopolish_b200 import synth
from tests.test_polya import CONTIG, REF_TEST, assert_results_equal_reference, polya_reference, ref_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("start", "leader", "adapter", "polya", "cliffs", "read_rate", "polya_length", "end_score", "qc")


def assert_same(got, want):
    """every field of two POLYA_RES_DT arrays, bit for bit"""
    for k in FIELDS:
        a, b = np.ascontiguousarray(got[k]), np.ascontiguousarray(want[k])
        bad = np.nonzero((a.view(np.uint8).reshape(a.shape[0], -1) != b.view(np.uint8).reshape(b.shape[0], -1)).any(1))[0]
        assert bad.size == 0, (k, bad[:5], a[bad[:5]], b[bad[:5]])


@pytest.mark.gpu
def test_device_equals_port_on_a_large_batch(engine):
    """>= 500 reads of 2 .. 200 000 samples plus one of 1.2 x 10^6, every family, bit for bit against npo_polya"""
    from oracle.polya_py import PortPolya
    rng = np.random.default_rng(17)
    lengths = np.exp(rng.uniform(np.log(2.0), np.log(200_000.0), 560)).astype(np.int64)
    lengths[:4] = (2, 3, 200_000, 1_200_000)
    ps = synth.gen_polya(560, seed=8, lengths=lengths)
    assert ps.jobs["n_samples"].max() >= 1_000_000 and ps.jobs["n_samples"].min() == 2
    got = engine.polya_batch(ps.samples, ps.durations, ps.map, ps.jobs)
    want = PortPolya().polya(ps.samples, ps.durations, ps.map, ps.jobs)
    assert_same(got, want)
    assert set(np.unique(got["qc"])) >= {0, 1, 2, 4}


@pytest.mark.gpu
def test_device_equals_recorded_reference(engine):
    """the CPU test's reads: the device against the compiled reference's answers (replayed from that test's recording)"""
    node = types.SimpleNamespace(module=types.SimpleNamespace(__name__="tests.test_polya"), name=REF_TEST)
    ref, _ = polya_reference(node, record_dir="")
    ps, pos = ref_case()
    seg, rl, es, qc, tsv = ref.polya(ps.samples, ps.durations, ps.map, ps.jobs, ps.names, CONTIG, pos, ps.suffix_clip)
    got = engine.polya_batch(ps.samples, ps.durations, ps.map, ps.jobs)
    assert_results_equal_reference(got, seg, rl, es, qc)
    from oracle.polya_py import format_rows
    assert format_rows(got, ps.names, CONTIG, pos, ps.suffix_clip) == tsv


def _rna_reads(model, n, seed):
    """direct-RNA traces for load_from_raw: a poly(A)-shaped head (START, leader, adapter, tail) in front of a transcript
    trace, which the pore reads 3'->5' (the basecall's levels back to front)"""
    raw, rr, seqs = synth.gen_raw(n, 40000, model, seed=seed, mean_dwell=40.0, return_seqs=True)
    signals = []
    for i, r in enumerate(rr):
        rng = np.random.default_rng(seed + 1000 + i)
        tx = raw[int(r["sample_off"]):int(r["sample_off"]) + int(r["n_samples"])][::-1]
        head = synth._polya_trace(rng, 600, 2500, 4000 + 500 * i, 0, 0.0, 1.0, 1.0)
        signals.append(np.ascontiguousarray(np.concatenate([head, tx]).astype(np.float32)))
    return signals, seqs


@pytest.mark.gpu
def test_resident_form_equals_one_shot_after_load_from_raw(engine):
    """nph_polya_after_load (samples, durations, event map and scalings left on the device by nph_load_from_raw_batch) ==
    nph_polya_batch on the same values brought back to the host, on RNA traces, including a read that fails to load"""
    m6 = synth.load_model("nucleotide")
    sd5 = m6.level_stdv.reshape(1024, 4).mean(1)
    model = synth.PoreModel("derived.nucleotide.5mer", 5, "nucleotide", m6.level_mean.reshape(1024, 4).mean(1), sd5, np.log(sd5))
    mid = engine.model_upload(model)
    signals, seqs = _rna_reads(model, 4, 913)
    signals.insert(1, np.full(3000, 77.0, np.float32)); seqs.insert(1, seqs[0][:300])          # nothing survives the trim
    sizes = np.array([s.shape[0] for s in signals])
    flat = np.concatenate(signals)
    ranks = [synth.kmer_ranks_from_codes(np.ascontiguousarray(q), 5, 4) for q in seqs]
    jobs = np.zeros(len(signals), synth.RAW_JOB_DT)
    so = ro = 0
    for j, (n, rk) in enumerate(zip(sizes, ranks)):
        jobs[j] = (so, ro, n, rk.shape[0], 3012.0)
        so += n; ro += rk.shape[0]
    flat_ranks = np.concatenate(ranks).astype(np.uint32)
    off, mean, stdv, start, dur, b2e, cal = engine.load_from_raw_batch(flat, flat_ranks, jobs, mid, synth.event_params(True))
    trim = engine.last_trim_ranges(len(signals))
    resident = engine.polya_after_load(len(signals))
    pj = np.zeros(len(signals), synth.POLYA_JOB_DT)
    for j in range(len(signals)):
        ok = int(cal[j]["status"]) == 0
        pj[j] = (int(jobs[j]["sample_off"]) + int(trim[j]["start"]), int(off[j]), int(jobs[j]["rank_off"]), int(trim[j]["end"] - trim[j]["start"]),
                 int(off[j + 1] - off[j]) if ok else 0, int(jobs[j]["n_kmers"]), 0, 3012.0, cal[j]["shift"], cal[j]["scale"], cal[j]["var"])
    assert (pj["n_events"] > 0).sum() >= 3 and pj["n_events"][1] == 0
    one_shot = engine.polya_batch(flat, np.ascontiguousarray(dur), b2e, pj)
    assert_same(resident, one_shot)
    assert int(resident[1]["qc"]) == synth.POLYA_FAILED_LOAD
    from oracle.polya_py import PortPolya
    assert_same(one_shot, PortPolya().polya(flat, dur, b2e, pj))


@pytest.mark.gpu
def test_malformed_jobs_are_refused(engine):
    from nanopolish_b200 import _lib
    ps = synth.gen_polya(8, seed=4, families=("pass",))
    good = engine.polya_batch(ps.samples, ps.durations, ps.map, ps.jobs)
    assert not (good["qc"] & 4).any()

    def bad(row, field, value, in_map=False):
        j = ps.jobs.copy(); m = ps.map.copy()
        if in_map:
            m[int(j[row]["map_off"]) + 3] = value
        else:
            j[row][field] = value
        with pytest.raises(_lib.NphError) as e:
            engine.polya_batch(ps.samples, ps.durations, m, j)
        assert e.value.status == -3, (row, field)

    bad(3, "n_samples", 1)                                                       # n_samples < 2
    bad(7, "n_samples", int(ps.jobs[7]["n_samples"]) + 1)                        # samples past the buffer
    bad(5, "event_off", ps.durations.shape[0])                                   # events past the buffer
    bad(2, "n_kmers", 0)                                                         # no map entries
    bad(7, "n_kmers", int(ps.jobs[7]["n_kmers"]) + 1)                            # map past the buffer
    bad(4, None, (0, int(ps.jobs[4]["n_events"])), in_map=True)                  # event index past the read's events
    bad(1, None, (-2, 3), in_map=True)                                           # negative start other than -1
    bad(6, None, (5, 4), in_map=True)                                            # start > stop
    # a failed load reads nothing else
    j = ps.jobs.copy(); j[6]["n_events"] = 0; j[6]["n_samples"] = 0
    r = engine.polya_batch(ps.samples, ps.durations, ps.map, j)
    assert int(r[6]["qc"]) == synth.POLYA_FAILED_LOAD
    # the context is still usable
    assert_same(engine.polya_batch(ps.samples, ps.durations, ps.map, ps.jobs), good)


@pytest.mark.gpu
def test_restated_polya_math_exhaustive_on_device():
    """csrc/polya_math.cuh on the device over every float x <= 0 (expf) and x >= 0 (logf) against this host's libm"""
    exe = os.path.join(ROOT, "tests", "cuda", "check_polya_math")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "expf 0 bad" in r.stdout and "logf 0 bad" in r.stdout
