"""`nanopolish polya` (section 8f N5) on the CPU: the plain-C restatement (oracle/np_polya.c) against the compiled reference
(live where oracle/_ref/libnpref_polya.so is built, replayed from tests/golden/ref_calls/ elsewhere), the rows, the restated
expf / logf of csrc/polya_math.cuh against the C library, and the ABI layouts."""
import os
import re
import subprocess

import numpy as np
import pytest

from nanopolish_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONTIG = "chrIV"

# the CPU reads the device is also checked on (tests/test_gpu_polya.py replays this test's recording)
REF_READS = dict(n_reads=48, seed=21)
REF_TEST = "test_port_equals_compiled_reference"


def ref_case():
    ps = synth.gen_polya(REF_READS["n_reads"], seed=REF_READS["seed"])
    positions = (np.arange(ps.jobs.shape[0]) * 37 + 1000).astype(np.int64)
    return ps, positions


def polya_reference(node, record_dir=None):
    """the compiled reference's polya, live or replayed for the test `node` (the ref_oracle fixture's scheme, tests/ref_replay.py)"""
    from oracle.polya_py import RefPolya
    from tests.ref_replay import ReplayedRef
    live = RefPolya() if RefPolya.available() else None
    record_dir = record_dir if record_dir is not None else os.environ.get("NPH_RECORD_REF")
    if record_dir and live is None:
        pytest.fail("NPH_RECORD_REF is set but oracle/_ref/libnpref_polya.so is not built")
    if live is not None and not record_dir:
        return live, None
    rep = ReplayedRef(node, live, record_dir or None)
    return rep, rep


@pytest.fixture
def polya_ref(request):
    ref, rep = polya_reference(request.node)
    yield ref
    if rep is not None:
        rep.finish()


def assert_results_equal_reference(res, seg, rl, es, qc):
    for i, r in enumerate(res):
        assert int(r["qc"]) & 4 == int(qc[i]) & 4, i
        if int(r["qc"]) & 4:
            continue
        got = [int(r[k]) for k in ("start", "leader", "adapter", "polya", "cliffs")]
        assert got == [int(v) for v in seg[i]], (i, got, seg[i])
        assert np.float32(r["end_score"]).view(np.uint32) == np.float32(es[i]).view(np.uint32), (i, r["end_score"], es[i])
        assert np.float64(r["read_rate"]).view(np.uint64) == np.float64(rl[i][0]).view(np.uint64), i
        assert np.float64(r["polya_length"]).view(np.uint64) == np.float64(rl[i][1]).view(np.uint64), i
        assert int(r["qc"]) & 3 == int(qc[i]) & 3, i


def test_port_equals_compiled_reference(polya_ref):
    """npo_polya == the reference's segment_squiggle / viterbi / estimate_* / QC on every synthetic family, bit for bit"""
    from oracle.polya_py import PortPolya, format_rows
    ps, pos = ref_case()
    seg, rl, es, qc, tsv = polya_ref.polya(ps.samples, ps.durations, ps.map, ps.jobs, ps.names, CONTIG, pos, ps.suffix_clip)
    port = PortPolya().polya(ps.samples, ps.durations, ps.map, ps.jobs)
    assert_results_equal_reference(port, seg, rl, es, qc)
    # every family reaches the branch it is there for
    tags = [ln.split(b"\t")[-1] for ln in tsv.splitlines()[1:]]
    for fam, want in (("noregion", b"NOREGION"), ("adapter", b"ADAPTER"), ("suffclip", b"SUFFCLIP"), ("failed_load", b"READ_FAILED_LOAD"),
                      ("pass", b"PASS")):
        assert any(f == fam and t == want for f, t in zip(ps.family, tags)), fam
    assert any(np.isinf(rl[i][0]) for i, f in enumerate(ps.family) if f == "zero_median")
    n = ps.jobs["n_samples"]
    assert any(int(seg[i][2]) == int(n[i]) - 2 and int(seg[i][3]) == int(n[i]) - 1 for i in range(len(n)) if not qc[i] & 4)   # defaults
    assert any(int(seg[i][1]) == 2 ** 64 - 1 for i in range(len(n)))                                                        # n = 2 wraps
    # the rows restated from our values are the reference's bytes
    assert format_rows(port, ps.names, CONTIG, pos, ps.suffix_clip) == tsv


def test_restated_polya_math_on_host():
    """the host copy of csrc/polya_math.cuh (expf on x <= 0, logf on x >= 0) against this machine's libm on 2 x 10^7 inputs"""
    exe = os.path.join(ROOT, "tests", "cuda", "check_polya_math")
    r = subprocess.run([exe, "--host-only", "10000000"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "expf 0 bad" in r.stdout and "logf 0 bad" in r.stdout


def test_polya_abi_layouts_match_header():
    hdr = open(os.path.join(ROOT, "include", "nph.h")).read()
    assert re.search(r"\} nph_polya_job;\s+/\* 72 bytes \*/", hdr) and re.search(r"\} nph_polya_result;\s+/\* 64 bytes \*/", hdr)
    assert synth.POLYA_JOB_DT.itemsize == 72 and synth.POLYA_RES_DT.itemsize == 64
    f = synth.POLYA_JOB_DT.fields
    assert [f[k][1] for k in ("sample_off", "event_off", "map_off", "n_samples", "n_events", "n_kmers", "sample_rate", "shift", "scale", "var")] == \
        [0, 8, 16, 24, 28, 32, 40, 48, 56, 64]
    g = synth.POLYA_RES_DT.fields
    assert [g[k][1] for k in ("start", "leader", "adapter", "polya", "cliffs", "read_rate", "polya_length", "end_score", "qc")] == \
        [0, 8, 16, 24, 32, 40, 48, 56, 60]
    for name, v in (("NPH_POLYA_NOREGION", synth.POLYA_NOREGION), ("NPH_POLYA_ADAPTER", synth.POLYA_ADAPTER),
                    ("NPH_POLYA_FAILED_LOAD", synth.POLYA_FAILED_LOAD)):
        assert re.search(rf"#define {name}\s+{v}\b", hdr), name
