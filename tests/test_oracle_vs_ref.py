"""Pin the plain-C oracle (oracle/np_oracle.c) to the COMPILED REFERENCE (oracle/_ref/libnpref.so),
bit for bit.  Where the reference is not compiled, its answers are replayed from tests/golden/ref_calls/
(tests/ref_replay.py)."""
import numpy as np
import pytest

from nanopolish_b200 import synth
from tests.golden_cases import make_abea_cases, make_hmm_cases


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_logsum_table_and_samples(port_oracle, ref_oracle):
    assert np.array_equal(_bits(port_oracle.logsum_table()), _bits(ref_oracle.logsum_table()))
    rng = np.random.default_rng(0)
    a = rng.uniform(-50, 0, 20000).astype(np.float32)
    b = (a + rng.uniform(-20, 20, 20000)).astype(np.float32)
    a[:50] = -np.inf
    b[25:75] = -np.inf
    r = ref_oracle.add_logs(a, b)
    for x, y, rx in zip(a, b, r):
        p = port_oracle.lib.npo_logsum(float(x), float(y))
        assert rx.view(np.uint32) == np.float32(p).view(np.uint32)


@pytest.mark.parametrize("name", ["segments", "short_bias08", "methylation"])
def test_hmm_score_bit_identical(port_oracle, ref_oracle, name):
    case = make_hmm_cases()[name]
    rs, jobs = case["rs"], case["jobs"]
    ref_oracle.clear_reads()
    handles = [ref_oracle.builtin_model(a) for a in case["alphabets"]]
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, handles[0])
    s_ref, _ = ref_oracle.score_batch(rh, jobs.jobs, jobs.seqs, handles, indel_bias=case["indel_bias"])
    models = [synth.load_model(a) for a in case["alphabets"]]
    s_port, _ = port_oracle.hmm_score_batch(rs.reads, rs.ev_mean, rs.ev_start_time, models, jobs.kmer_ranks,
                                            jobs.jobs, indel_bias=case["indel_bias"])
    assert np.isfinite(s_ref).all()
    assert np.array_equal(_bits(s_ref), _bits(s_port))


def test_kmer_ranks_match_reference(ref_oracle):
    """synth's numpy rank arithmetic == HMMInputSequence::get_kmer_rank (both strands, both alphabets)."""
    case = make_hmm_cases()["segments"]
    h = ref_oracle.builtin_model("nucleotide")
    jobs = case["jobs"]
    for j in range(jobs.jobs.shape[0]):
        jb = jobs.jobs[j]
        want = ref_oracle.kmer_ranks(h, jobs.seqs[j], bool(jb["rc"]))
        got = jobs.kmer_ranks[int(jb["rank_off"]):int(jb["rank_off"]) + int(jb["n_kmers"])]
        assert np.array_equal(want, got)
    case = make_hmm_cases()["methylation"]
    hc = ref_oracle.builtin_model("cpg")
    jobs = case["jobs"]
    for j in range(0, jobs.jobs.shape[0], 7):
        jb = jobs.jobs[j]
        want = ref_oracle.kmer_ranks(hc, jobs.seqs[j], False)
        got = jobs.kmer_ranks[int(jb["rank_off"]):int(jb["rank_off"]) + int(jb["n_kmers"])]
        assert np.array_equal(want, got)


@pytest.mark.parametrize("name", ["reads_2k", "reads_short"])
def test_abea_identical(port_oracle, ref_oracle, name):
    rs = make_abea_cases()[name]["rs"]
    model = synth.load_model("nucleotide")
    ref_oracle.clear_reads()
    h = ref_oracle.builtin_model("nucleotide")
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, h)
    seqs = [synth._CODE2DNA[c].tobytes() for c in rs.seq_codes]
    jobs, ranks, total = synth.abea_jobs(rs)
    caps = [int(j["pairs_cap"]) for j in jobs]
    pr, poff, npairs, _ = ref_oracle.abea_batch(rh, h, seqs, caps)
    pp, res, _ = port_oracle.abea_batch(rs.reads, rs.ev_mean, rs.ev_start_time, model, ranks, jobs, total)
    for i in range(len(seqs)):
        n = int(npairs[i])
        assert n == int(res[i]["n_pairs"]) and n > 0
        a = pr[int(poff[i]):int(poff[i]) + n]
        b = pp[int(jobs[i]["pairs_off"]):int(jobs[i]["pairs_off"]) + n]
        assert np.array_equal(a[:, 0], b["ref_pos"]) and np.array_equal(a[:, 1], b["read_pos"])


def test_abea_qc_failure_matches(port_oracle, ref_oracle):
    """Events unrelated to the sequence: the reference returns an empty vector; so must the oracle."""
    model = synth.load_model("nucleotide")
    rs = synth.gen_reads(2, 400, model, seed=9, rng_scalings=False)
    rng = np.random.default_rng(5)
    rs.ev_mean[:] = rng.uniform(60, 120, rs.ev_mean.shape[0]).astype(np.float32)
    ref_oracle.clear_reads()
    h = ref_oracle.builtin_model("nucleotide")
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, h)
    seqs = [synth._CODE2DNA[c].tobytes() for c in rs.seq_codes]
    jobs, ranks, total = synth.abea_jobs(rs)
    _, _, npairs, _ = ref_oracle.abea_batch(rh, h, seqs, [int(j["pairs_cap"]) for j in jobs])
    _, res, _ = port_oracle.abea_batch(rs.reads, rs.ev_mean, rs.ev_start_time, model, ranks, jobs, total)
    assert list(npairs) == [int(x) for x in res["n_pairs"]]


def test_mom_matches(port_oracle, ref_oracle):
    model = synth.load_model("nucleotide")
    rs = synth.gen_reads(3, 800, model, seed=77)
    ref_oracle.clear_reads()
    h = ref_oracle.builtin_model("nucleotide")
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, h)
    jobs, ranks, _ = synth.abea_jobs(rs)
    for i in range(rs.n_reads):
        want = ref_oracle.mom(rh[i], h, synth._CODE2DNA[rs.seq_codes[i]].tobytes())
        sh, sc = port_oracle.mom(rs.reads, rs.ev_mean, model, ranks, jobs[i])
        assert want[0] == sh and want[1] == sc and want[2] == 0.0 and want[3] == 1.0


def test_viterbi_align_identical(port_oracle, ref_oracle):
    """profile_hmm_align: identical paths, states and bit-identical l_fm (both strands, flags 0 and PRE|POST)."""
    nuc = synth.load_model("nucleotide")
    rs = synth.gen_reads(3, 900, nuc, seed=21, drift=True)
    jobs = synth.scorereads_jobs(rs, 170, rc_every=2, keep_seqs=True)
    ref_oracle.clear_reads()
    h = ref_oracle.builtin_model("nucleotide")
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, h)
    for j in range(jobs.jobs.shape[0]):
        for flags in (0, 3):
            jb = jobs.jobs[j].copy(); jb["flags"] = flags
            ek, lfm, st = ref_oracle.align(rh[int(jb["read"])], h, jobs.seqs[j], jb["event_start"], jb["event_stop"], jb["rc"], flags)
            out, status = port_oracle.hmm_align(rs.reads, rs.ev_mean, rs.ev_start_time, [nuc], jobs.kmer_ranks, jb)
            assert status == 0 and out.shape[0] == ek.shape[0] > 0
            assert np.array_equal(out["event_idx"], ek[:, 0]) and np.array_equal(out["kmer_idx"], ek[:, 1])
            assert np.array_equal(out["l_fm"].view(np.uint32), lfm.view(np.uint32)) and out["state"].tobytes() == st


@pytest.mark.parametrize("rna", [False, True])
def test_event_detection_identical(port_oracle, ref_oracle, rna):
    """scrappie detect_events (compiled C) vs the restatement: identical boundaries, bit-identical mean/stdv."""
    nuc = synth.load_model("nucleotide")
    raw, reads = synth.gen_raw(4, 30000, nuc, seed=77, mean_dwell=30.0 if rna else 9.0)
    prm = synth.event_params(rna)
    for r in reads:
        x = np.ascontiguousarray(raw[int(r["sample_off"]):int(r["sample_off"]) + int(r["n_samples"])])
        st, ln, mn, sd = ref_oracle.detect_events(x, rna)
        ev = port_oracle.detect_events(x, prm)
        assert ev.shape[0] == st.shape[0] > 500
        assert np.array_equal(ev["start"], st) and np.array_equal(ev["length"].view(np.uint32), ln.view(np.uint32))
        assert np.array_equal(ev["mean"].view(np.uint32), mn.view(np.uint32)) and np.array_equal(ev["stdv"].view(np.uint32), sd.view(np.uint32))
    # (a signal without any peak makes the reference read peaks[-1]: undefined there, one whole-signal event here)
    ev = port_oracle.detect_events(raw[:5].copy(), prm)
    assert ev.shape[0] == 1 and ev["start"][0] == 0 and ev["length"][0] == 5.0


def _raw_with_stalls(seed, n, leader=0, tail=0):
    """A synthetic trace with an optional constant (ADC-flat, MAD exactly 0) leader and tail, as a stalled pore gives."""
    nuc = synth.load_model("nucleotide")
    raw, reads = synth.gen_raw(1, n, nuc, seed=seed)
    x = raw[:int(reads[0]["n_samples"])]
    return np.concatenate([np.full(leader, 210.0, np.float32), x, np.full(tail, 95.5, np.float32)]).astype(np.float32)


@pytest.mark.parametrize("perc,chunk", [(0.0, 100), (0.0, 64), (0.3, 100), (0.77, 37), (1.0, 100)])
def test_trim_and_segment_raw_identical(port_oracle, ref_oracle, perc, chunk):
    """scrappie trim_and_segment_raw (compiled C) vs the restatement: same surviving range, including the quantile
    interpolation of the MAD threshold and the flat-leader case the default perc 0.0 actually trims."""
    cases = [_raw_with_stalls(5, 12000), _raw_with_stalls(6, 9000, leader=730), _raw_with_stalls(7, 9037, leader=300, tail=1250),
             _raw_with_stalls(8, 150, leader=100), _raw_with_stalls(9, 260)]
    seen_trim = False
    for x in cases:
        if perc == 1.0:
            # no chunk exceeds the maximum MAD: the reference asserts; the port reports "nothing survives"
            assert port_oracle.trim_raw(x, 200, 10, chunk, perc)[0] == 0
            continue
        want = ref_oracle.trim_raw(x, 200, 10, chunk, perc)
        got = port_oracle.trim_raw(x, 200, 10, chunk, perc)
        assert want == got
        seen_trim |= want[0] == 1 and want[1] > 200
    if perc != 1.0:
        assert seen_trim


def test_recalibrate_port_solves_the_weighted_least_squares(port_oracle):
    """recalibrate_model cannot be compiled here (Eigen, HDF5), so the restatement is checked against what the function
    is defined to compute: the weighted least-squares fit of event level on model level over the 'M' events."""
    model = synth.load_model("nucleotide")
    rs = synth.gen_reads(3, 1500, model, seed=31, rng_scalings=True)
    jobs, ranks, total = synth.abea_jobs(rs)
    pairs, res, _ = port_oracle.abea_batch(rs.reads, rs.ev_mean, rs.ev_start_time, model, ranks, jobs, total)
    for j in range(jobs.shape[0]):
        n = int(res[j]["n_pairs"])
        assert n > 0
        b2e, cal = port_oracle.recalibrate(rs.reads, rs.ev_mean, model, ranks, jobs[j], pairs, n)
        pr = pairs[int(jobs[j]["pairs_off"]):int(jobs[j]["pairs_off"]) + n]
        rk = ranks[int(jobs[j]["rank_off"]):int(jobs[j]["rank_off"]) + int(jobs[j]["n_kmers"])]
        ev = rs.ev_mean[int(rs.reads[j]["event_off"]):][:int(rs.reads[j]["n_events"])]
        # independent restatement of the bookkeeping
        first = {}
        prev = -1
        for k, e in zip(pr["ref_pos"], pr["read_pos"]):
            if e != prev:
                first.setdefault(int(k), [int(e), int(e)])[1] = int(e)
            prev = e
        for k in range(rk.shape[0]):
            assert (int(b2e[k]["start"]), int(b2e[k]["stop"])) == tuple(first.get(k, (-1, -1)))
        sel, prev_rank = [], -1
        for k in sorted(first):
            if rk[k] != prev_rank:
                sel.append((k, first[k][0]))
            prev_rank = rk[k]
        assert int(cal["n_used"]) == len(sel) >= 200
        mu = model.level_mean[rk[[k for k, _ in sel]]]; sd = model.level_stdv[rk[[k for k, _ in sel]]]
        e = ev[[i for _, i in sel]].astype(np.float64)
        w = 1.0 / sd ** 2
        A = np.array([[w.sum(), (mu * w).sum()], [(mu * w).sum(), (mu * mu * w).sum()]])
        shift, scale = np.linalg.solve(A, np.array([(e * w).sum(), (mu * e * w).sum()]))
        var = np.sqrt((((e - shift - scale * mu) / sd) ** 2).mean())
        assert abs(cal["shift"] - shift) < 1e-8 and abs(cal["scale"] - scale) < 1e-10 and abs(cal["var"] - var) < 1e-10
        assert cal["drift"] == 0.0 and int(cal["status"]) == 0
        assert cal["events_per_base"] == (int(pr["read_pos"].max()) - int(pr["read_pos"].min())) / rk.shape[0]
        # recovered scalings are close to the ones the read was simulated with
        assert abs(cal["shift"] - rs.reads[j]["shift"]) < 1.5 and abs(cal["scale"] - rs.reads[j]["scale"]) < 0.02


def _meth_expected(port_oracle, rs, models, i, case):
    """the restatement's TSV + (sites, scores) for one case: EventAlignmentRecord -> enumeration -> oracle scores -> rows"""
    from tests import meth_cases as mc, meth_restatement as mr
    pairs, rc = mc.event_alignment_record(case)
    ref = mc.fetched_reference(case)
    groups = mr.enumerate_record(ref, case["ref_pos"], [p[0] for p in pairs], [p[1] for p in pairs], rc, "cpg", mc.K)
    rows, lls = [], []
    for (sp, ep, nm, e1, e2, ru, rm, seq) in groups:
        jobs = np.zeros(2, synth.HMM_JOB_DT)
        st = 1 if e1 <= e2 else -1
        jobs[0] = (0, i, 1, e1, e2, ru.shape[0], st, rc, 3, 0)
        jobs[1] = (ru.shape[0], i, 1, e1, e2, rm.shape[0], st, rc, 3, 0)
        sc, _ = port_oracle.hmm_score_batch(rs.reads, rs.ev_mean, rs.ev_start_time, models, np.concatenate([ru, rm]).astype(np.uint32), jobs)
        rows.append((sp, ep, nm, sc[0], sc[1], seq)); lls.append((float(sc[0]), float(sc[1])))
    tsv = mc.tsv_rows("chr1", "-" if case["flag"] & 16 else "+", case["name"], rows)
    return tsv, rows, np.array(lls, np.float64).reshape(-1, 2)


def test_call_methylation_restatement_pinned(port_oracle, ref_oracle):
    """tests/meth_restatement.py + tests/meth_cases.py (EventAlignmentRecord, reference fetch, TSV row) reproduce the compiled
    reference's calculate_methylation_for_read + write_methylation_results_as_tsv byte for byte: forward and reverse records,
    CIGARs with insertions / deletions / soft clips, IUPAC and lower-case reference bases."""
    from tests import meth_cases as mc
    nuc, cpg = synth.load_model("nucleotide"), synth.load_model("cpg")
    rs = synth.gen_reads(6, 2200, nuc, seed=515, cpg_keep=0.35)
    ref_oracle.clear_reads()
    mh = ref_oracle.builtin_model("nucleotide")
    ref_oracle.builtin_model("cpg")
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, mh)
    rng = np.random.default_rng(7)
    total = 0
    for i in range(rs.n_reads):
        case = mc.make_case(i, rs, rng)
        one = np.ones(int(rs.reads[i]["n_events"]), np.float32)
        ref_oracle.read_set_eventalign(rh[i], case["name"], case["read_sequence"], case["b2e_start"], case["b2e_stop"], one, one)
        tsv_ref, sites_ref, ll_ref = ref_oracle.call_methylation(rh[i], case["name"], "chr1", case["contig"], case["ref_pos"], case["flag"], case["cigar"])
        tsv, rows, ll = _meth_expected(port_oracle, rs, [nuc, cpg], i, case)
        assert tsv == tsv_ref
        assert np.array_equal(sites_ref[:, :3], np.array([r[:3] for r in rows], np.int32).reshape(-1, 3))
        assert np.array_equal(ll_ref, ll)                      # float scores widened to double: exact
        total += len(rows)
    assert total > 120
    # the output window (-w): the same filter on both sides
    case = mc.make_case(0, rs, np.random.default_rng(7))
    lo, hi = case["ref_pos"] + 400, case["ref_pos"] + 1100
    tsv_ref, sites_ref, _ = ref_oracle.call_methylation(rh[0], case["name"], "chr1", case["contig"], case["ref_pos"], case["flag"], case["cigar"], region=(lo, hi))
    assert 0 < sites_ref.shape[0] < 40 and (sites_ref[:, 0] >= lo).all() and (sites_ref[:, 1] < hi).all()


def test_recalibrate_pinned_to_compiled_reference(port_oracle, ref_oracle):
    """npo_recalibrate against the reference's own get_eventalignment_for_1d_basecalls + recalibrate_model
    (src/nanopolish_squiggle_read.cpp:340-391, src/nanopolish_methyltrain.cpp:204-307, compiled unmodified into oracle/_ref):
    identical doubles for shift, scale, var, events_per_base and the same 'M'-event count.  The one thing that is NOT the
    reference's object code is Eigen's FullPivLU (un-vendored, absent here): recalibrate_model is compiled against
    oracle/shim/Eigen/Dense, which restates the published algorithm; the sums that feed it and the residual variance that
    follows are the reference's own loops."""
    model = synth.load_model("nucleotide")
    rs = synth.gen_reads(5, 1500, model, seed=31, rng_scalings=True)
    jobs, ranks, total = synth.abea_jobs(rs)
    pairs, res, _ = port_oracle.abea_batch(rs.reads, rs.ev_mean, rs.ev_start_time, model, ranks, jobs, total)
    ref_oracle.clear_reads()
    mh = ref_oracle.builtin_model("nucleotide")
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, mh)
    for j in range(jobs.shape[0]):
        n = int(res[j]["n_pairs"])
        assert n > 0
        _, cal = port_oracle.recalibrate(rs.reads, rs.ev_mean, model, ranks, jobs[j], pairs, n)
        pr = pairs[int(jobs[j]["pairs_off"]):int(jobs[j]["pairs_off"]) + n]
        seq = synth._CODE2DNA[rs.seq_codes[j]].tobytes()
        want = ref_oracle.calibrate(rh[j], mh, seq, np.stack([pr["ref_pos"], pr["read_pos"]], 1))
        assert want is not None and want["calibrated"] and want["n_used"] == int(cal["n_used"]) >= 200
        for key in ("shift", "scale", "drift", "var", "events_per_base"):
            assert np.float64(want[key]).view(np.uint64) == np.float64(cal[key]).view(np.uint64), key
    # fewer than 200 'M' events: not recalibrated, scalings untouched
    short = synth.gen_reads(1, 260, model, seed=5, rng_scalings=True)
    jobs, ranks, total = synth.abea_jobs(short)
    pairs, res, _ = port_oracle.abea_batch(short.reads, short.ev_mean, short.ev_start_time, model, ranks, jobs, total)
    n = int(res[0]["n_pairs"])
    if n:
        ref_oracle.clear_reads()
        rh = ref_oracle.register_reads(short.reads, short.ev_mean, short.ev_start_time, mh)
        pr = pairs[:n]
        want = ref_oracle.calibrate(rh[0], mh, synth._CODE2DNA[short.seq_codes[0]].tobytes(), np.stack([pr["ref_pos"], pr["read_pos"]], 1))
        _, cal = port_oracle.recalibrate(short.reads, short.ev_mean, model, ranks, jobs[0], pairs, n)
        assert not want["calibrated"] and int(cal["status"]) == 2 and want["n_used"] == int(cal["n_used"]) < 200


from tests.random_cases import HMM_SHAPES, random_hmm_jobs


@pytest.mark.parametrize("shape", HMM_SHAPES)
def test_random_hmm_shapes_pinned(port_oracle, ref_oracle, shape):
    """The shape families the GPU parity test draws (K = 1 and E = 1 jobs, methylation-window sizes, scorereads segments,
    multi-strip widths with few rows, wide-and-tall, every flag combination, both strands, drift, indel bias 0.9): the port
    oracle the CUDA path is compared with equals the compiled reference bit for bit on exactly those jobs."""
    nuc = synth.load_model("nucleotide")
    rs = synth.gen_reads(8, 2600, nuc, seed=900 + shape["kmin"], drift=True)
    rng = np.random.default_rng(shape["kmin"] * 7 + 1)
    jobs = random_hmm_jobs(rs, rng, shape["n"], shape["kmin"], shape["kmax"], shape["emin"], shape["emax"], [0, 1, 2, 3])
    ref_oracle.clear_reads()
    h = ref_oracle.builtin_model("nucleotide")
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, h)
    s_ref, _ = ref_oracle.score_batch(rh, jobs.jobs, jobs.seqs, [h], indel_bias=0.9, threads=8)
    s_port, _ = port_oracle.hmm_score_batch(rs.reads, rs.ev_mean, rs.ev_start_time, [nuc], jobs.kmer_ranks, jobs.jobs, indel_bias=0.9, threads=8)
    assert np.array_equal(_bits(s_ref), _bits(s_port))


def _abea_ref_vs_port(port_oracle, ref_oracle, rs, jobs, ranks, total, seqs):
    model = synth.load_model("nucleotide")
    ref_oracle.clear_reads()
    h = ref_oracle.builtin_model("nucleotide")
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, h)
    pr, poff, npairs, _ = ref_oracle.abea_batch(rh, h, seqs, [int(j["pairs_cap"]) for j in jobs], threads=8)
    pp, res, _ = port_oracle.abea_batch(rs.reads, rs.ev_mean, rs.ev_start_time, model, ranks, jobs, total, threads=8)
    assert [int(x) for x in npairs] == [int(x) for x in res["n_pairs"]]
    for i in range(len(seqs)):
        n = int(npairs[i])
        a = pr[int(poff[i]):int(poff[i]) + n]
        b = pp[int(jobs[i]["pairs_off"]):int(jobs[i]["pairs_off"]) + n]
        assert np.array_equal(a[:, 0], b["ref_pos"]) and np.array_equal(a[:, 1], b["read_pos"]), f"read {i}"
    return res


@pytest.mark.parametrize("n_events,n_reads,scaled", [(60, 12, False), (900, 10, True), (4000, 6, False), (8000, 3, True)])
def test_abea_random_reads_pinned(port_oracle, ref_oracle, n_events, n_reads, scaled):
    """the read families of tests/test_gpu_abea.py::test_random_reads_identical_paths through the compiled reference"""
    model = synth.load_model("nucleotide")
    rs = synth.gen_reads(n_reads, n_events, model, seed=7000 + n_events, rng_scalings=scaled)
    jobs, ranks, total = synth.abea_jobs(rs)
    res = _abea_ref_vs_port(port_oracle, ref_oracle, rs, jobs, ranks, total, [synth._CODE2DNA[c].tobytes() for c in rs.seq_codes])
    assert (res["n_pairs"] > 0).all()


def test_abea_qc_mixed_and_truncated_pinned(port_oracle, ref_oracle):
    """test_gpu_abea.py's QC / mixed-batch and truncated-sequence cases through the compiled reference: a read of noise and
    one with a long stall (empty results where the reference's QC rejects), half a sequence, a 3-k-mer sequence."""
    model = synth.load_model("nucleotide")
    rs = synth.gen_reads(6, 500, model, seed=99, rng_scalings=False)
    rng = np.random.default_rng(1)
    o, n = int(rs.reads[1]["event_off"]), int(rs.reads[1]["n_events"])
    rs.ev_mean[o:o + n] = rng.uniform(60, 120, n).astype(np.float32)
    o, n = int(rs.reads[4]["event_off"]), int(rs.reads[4]["n_events"])
    rs.ev_mean[o + 100:o + 300] = rs.ev_mean[o + 100]
    jobs, ranks, total = synth.abea_jobs(rs)
    res = _abea_ref_vs_port(port_oracle, ref_oracle, rs, jobs, ranks, total, [synth._CODE2DNA[c].tobytes() for c in rs.seq_codes])
    assert int(res[1]["n_pairs"]) == 0
    rs = synth.gen_reads(4, 700, model, seed=123, rng_scalings=False)
    jobs, ranks, total = synth.abea_jobs(rs)
    jobs = jobs.copy()
    jobs[0]["n_kmers"] = jobs[0]["n_kmers"] // 2
    jobs[1]["n_kmers"] = 3
    seqs = [synth._CODE2DNA[c[:int(j["n_kmers"]) + 5]].tobytes() for c, j in zip(rs.seq_codes, jobs)]
    _abea_ref_vs_port(port_oracle, ref_oracle, rs, jobs, ranks, total, seqs)


def test_variant_screening_restatement_pinned(port_oracle, ref_oracle):
    """tests/var_restatement.py (candidate list, the windows' event sequences, the read-order early exit) gives, for every candidate of
    sampled positions, the double the compiled reference's score_variant_thresholded returns (src/common/nanopolish_variant.cpp:765-799,
    one OpenMP thread): substitutions, insertions and the deletion, forward and reverse-strand reads, PRE|POST clip, indel bias 0.9."""
    from tests import var_restatement as vr
    nuc = synth.load_model("nucleotide")
    REGION = 5000
    ref, rs, recs, pairs = synth.gen_pileup(150, 14, 110, nuc, seed=11, region_start=REGION, n_true_variants=3)
    ref_s = synth._CODE2DNA[ref].tobytes().decode()
    ref_oracle.clear_reads()
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, ref_oracle.builtin_model("nucleotide"))
    checked = exited = 0
    for pi in range(20, 128, 6):
        i = REGION + pi
        cs, ce = i - 10, i + 11
        want, n_seq, seqs = vr.screen_position(port_oracle, rs, nuc, ref_s, REGION, i, recs, pairs, 10, 40, 3, 0.9, 6)
        if n_seq == 0:
            continue
        cands = vr.candidates(ref_s, pi)
        got = ref_oracle.score_variants_thresholded([rh[r] for r, _, _ in seqs], [(e1, e2) for _, e1, e2 in seqs],
                                                    np.array([recs[r]["rc"] for r, _, _ in seqs], np.uint8), ref_s[cs - REGION:ce - REGION + 1], cs,
                                                    [(REGION + off, rseq, aseq) for _, off, rseq, aseq in cands], 3, 40, False, indel_bias=0.9)
        for (slot, _, _, _), v in zip(cands, got):
            assert want[slot] == float(v), (pi, slot, want[slot], float(v))
            checked += 1; exited += abs(float(v)) >= 40
    ref_oracle.clear_reads()
    assert checked > 80 and exited > 40
