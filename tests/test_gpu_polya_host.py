"""`nanopolish polya` through the C++ host mirror (nanopolish_b200/host/nph_polya.*): PolyaEstimator's rows against the compiled
reference's, polya_from_raw against PolyaEstimator over the reads load_from_raw builds, and jobs that share samples and
event-map entries (each warp keeps its own scratch)."""
import ctypes as C
import os
import types

import numpy as np
import pytest

from nanopolish_b200 import synth
from tests.test_polya import CONTIG, REF_TEST, polya_reference, ref_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST_SO = os.path.join(ROOT, "nanopolish_b200", "libnph_host.so")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def host():
    lib = C.CDLL(HOST_SO)
    lib.nphh_last_error.restype = C.c_char_p
    lib.nphh_polya_tsv.restype = C.c_longlong
    lib.nphh_polya_from_raw.restype = C.c_longlong
    return lib


def _rna_model():
    m6 = synth.load_model("nucleotide")
    sd5 = m6.level_stdv.reshape(1024, 4).mean(1)
    return synth.PoreModel("derived.u_to_t_rna.5mer", 5, "nucleotide", m6.level_mean.reshape(1024, 4).mean(1), sd5, np.log(sd5))


def _model_handle(host, model, alphabet=b"nucleotide"):
    mean, sd, lsd = (np.ascontiguousarray(a, np.float64) for a in (model.level_mean, model.level_stdv, model.level_log_stdv))
    h = host.nphh_model_create(alphabet, model.k, mean.shape[0], _p(mean), _p(sd), _p(lsd))
    assert h >= 0, host.nphh_last_error()
    return h


def _tsv(host, fn, *args):
    cap = 1 << 20
    out = C.create_string_buffer(cap)
    n = fn(*args, out, C.c_size_t(cap))
    assert n >= 0, host.nphh_last_error()
    return out.raw[:n]


@pytest.mark.gpu
def test_estimator_tsv_equals_reference_rows(host):
    """PolyaEstimator::add_read / run / tsv on SquiggleReads assembled like load_from_raw leaves them == the reference's rows"""
    node = types.SimpleNamespace(module=types.SimpleNamespace(__name__="tests.test_polya"), name=REF_TEST)
    ref, _ = polya_reference(node, record_dir="")
    ps, pos = ref_case()
    *_, want = ref.polya(ps.samples, ps.durations, ps.map, ps.jobs, ps.names, CONTIG, pos, ps.suffix_clip)
    host.nphh_clear()
    mh = _model_handle(host, _rna_model())
    first = None
    for i, jb in enumerate(ps.jobs):
        ne, nk = int(jb["n_events"]), int(jb["n_kmers"])
        eo, mo, so, ns = int(jb["event_off"]), int(jb["map_off"]), int(jb["sample_off"]), int(jb["n_samples"])
        z = np.zeros(max(ne, 1), np.float32); t = np.zeros(max(ne, 1))
        h = host.nphh_read_create(C.c_uint32(ne), _p(z), _p(t), C.c_double(jb["shift"]), C.c_double(jb["scale"]), C.c_double(0.0),
                                  C.c_double(jb["var"]), C.c_double(0.0), mh)
        first = h if first is None else first
        m = ps.map[mo:mo + nk]
        a, b = np.ascontiguousarray(m["start"], np.int32), np.ascontiguousarray(m["stop"], np.int32)
        du = np.ascontiguousarray(ps.durations[eo:eo + ne], np.float32); sd = np.ones(max(ne, 1), np.float32)
        assert host.nphh_read_set_eventalign(h, ps.names[i].encode(), b"A" * (nk + 4), _p(a), _p(b), C.c_size_t(nk), _p(sd), _p(du)) == 0
        x = np.ascontiguousarray(ps.samples[so:so + ns], np.float32)
        assert host.nphh_read_set_samples(h, _p(x), C.c_size_t(ns), C.c_double(jb["sample_rate"])) == 0
    n = ps.jobs.shape[0]
    positions = np.ascontiguousarray(pos, np.int32)
    flags = np.zeros(n, np.uint16)
    clips = np.ascontiguousarray(ps.suffix_clip, np.uint32)
    got = _tsv(host, host.nphh_polya_tsv, first, n, CONTIG.encode(), _p(positions), _p(flags), _p(clips), 1)
    assert got == want
    # a secondary record gives no row
    flags[3] = 0x100
    got = _tsv(host, host.nphh_polya_tsv, first, n, CONTIG.encode(), _p(positions), _p(flags), _p(clips), 0)
    rows = want.splitlines(keepends=True)[1:]
    assert got == b"".join(rows[:3] + rows[4:])
    host.nphh_clear()


@pytest.mark.gpu
def test_polya_from_raw_equals_estimator_after_load_from_raw(host):
    """polya_from_raw (nph_polya_after_load: nothing uploaded after load_from_raw) == PolyaEstimator over the SquiggleReads
    load_from_raw builds with SRF_LOAD_RAW_SAMPLES, on direct-RNA traces with a poly(A)-shaped head, one that trims to nothing
    and one too short to align"""
    model = _rna_model()
    raw, rr, seqs = synth.gen_raw(4, 40000, model, seed=517, mean_dwell=40.0, return_seqs=True)
    signals = []
    for i, r in enumerate(rr):
        rng = np.random.default_rng(517 + i)
        tx = raw[int(r["sample_off"]):int(r["sample_off"]) + int(r["n_samples"])][::-1]
        signals.append(np.concatenate([synth._polya_trace(rng, 700, 3000, 4500 + 700 * i, 0, 0.0, 1.0, 1.0), tx]).astype(np.float32))
    signals.insert(1, np.full(3000, 77.0, np.float32)); seqs.insert(1, seqs[0][:300])
    short, _, sq = synth.gen_raw(1, 2400, model, seed=78, mean_dwell=40.0, return_seqs=True)
    signals.append(np.ascontiguousarray(short[::-1])); seqs.append(sq[0])
    n = len(signals)
    host.nphh_clear()
    mh = _model_handle(host, model, b"u_to_t_rna")
    soff = np.zeros(n + 1, np.uint64); soff[1:] = np.cumsum([s.shape[0] for s in signals])
    qoff = np.zeros(n + 1, np.uint64); qoff[1:] = np.cumsum([c.shape[0] for c in seqs])
    seqbuf = b"".join(synth._CODE2DNA[c].tobytes() for c in seqs).replace(b"T", b"U")
    eoff = np.zeros(n, np.uint64); eoff[1:] = np.cumsum([s.shape[0] // 2 + 8 for s in signals])[:-1]
    room = int(eoff[-1]) + signals[-1].shape[0] // 2 + 8
    n_events = np.zeros(n, np.uint32); scal = np.zeros((n, 5)); stats = np.zeros(5, np.uint64)
    mean = np.zeros(room, np.float32); stdv = np.zeros(room, np.float32); start = np.zeros(room, np.float64); dur = np.zeros(room, np.float32)
    flat = np.concatenate(signals)
    positions = np.arange(n, dtype=np.int32) * 11; flags = np.zeros(n, np.uint16); clips = np.array([0, 0, 250, 0, 0, 0], np.uint32)[:n]
    host.nphh_set_rna(1)
    host.nphh_set_load_flags(2)                                 # SRF_LOAD_RAW_SAMPLES
    try:
        first = host.nphh_load_from_raw(mh, n, _p(flat), _p(soff), seqbuf, _p(qoff), C.c_double(3012.0), _p(n_events), _p(scal), _p(eoff),
                                        _p(mean), _p(stdv), _p(start), _p(dur), None, _p(stats))
        assert first >= 0, host.nphh_last_error()
        want = _tsv(host, host.nphh_polya_tsv, first, n, CONTIG.encode(), _p(positions), _p(flags), _p(clips), 1)
        got = _tsv(host, host.nphh_polya_from_raw, mh, n, _p(flat), _p(soff), seqbuf, _p(qoff), C.c_double(3012.0), CONTIG.encode(),
                   _p(positions), _p(flags), _p(clips), 1)
    finally:
        host.nphh_set_load_flags(0)
        host.nphh_set_rna(0)
        host.nphh_clear()
    assert got == want
    tags = [ln.split(b"\t")[-1] for ln in got.splitlines()[1:]]
    assert tags[1] == b"READ_FAILED_LOAD" and sum(t != b"READ_FAILED_LOAD" for t in tags) >= 3, tags


@pytest.mark.gpu
def test_jobs_sharing_samples_and_map(engine):
    """jobs over the same samples, durations and map entries with different scalings (and trims) are independent reads"""
    from oracle.polya_py import PortPolya
    ps = synth.gen_polya(6, seed=31, families=("pass",))
    base = ps.jobs.copy()
    jobs = []
    for k in range(48):
        j = base[k % 6].copy()
        j["shift"] = float(j["shift"]) + 0.7 * (k // 6)
        j["scale"] = float(j["scale"]) * (1.0 + 0.02 * (k // 6))
        if k % 5 == 4:                                            # another trim of the same signal
            j["sample_off"] = int(j["sample_off"]) + 97; j["n_samples"] = int(j["n_samples"]) - 200
        jobs.append(j)
    jobs = np.array(jobs, synth.POLYA_JOB_DT)
    got = engine.polya_batch(ps.samples, ps.durations, ps.map, jobs)
    want = PortPolya().polya(ps.samples, ps.durations, ps.map, jobs)
    for k in ("start", "leader", "adapter", "polya", "cliffs", "read_rate", "polya_length", "end_score", "qc"):
        a, b = np.ascontiguousarray(got[k]), np.ascontiguousarray(want[k])
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), k
    assert len(set(got["end_score"].tolist())) > 6                  # the scalings do change the reads
