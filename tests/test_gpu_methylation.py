"""SURVEY.md 8(f) row N3 on the device — nph_methylation_batch (csrc/methylation.cu) through the C ABI.

The checker is tests/meth_restatement.py: a plain-Python restatement of calculate_methylation_for_read
(src/basemods/nanopolish_basemods.cpp:301-417; pinned to the compiled reference in tests/test_oracle_vs_ref.py)
whose windows are scored by the oracle.  The device must return the same groups (positions, motif counts, order),
bit-identical scores, and the same scored-event count; edge cases: reverse-strand records, windows cut by the end of
the reference, records without sites / without an event alignment, region filters, non-default window parameters,
and a multi-symbol alphabet (dam: GATC -> GMTC) with a random 5^6 model."""
import numpy as np
import pytest

from nanopolish_b200 import synth
from tests import meth_restatement as mr

pytestmark = pytest.mark.gpu
K = 6


def _expected(port_oracle, rs, models, ref_bases, pairs, records, alphabet, **kw):
    site_rows, jobs, ranks = mr.enumerate_batch(ref_bases, pairs, records, alphabet, K, **kw)
    if jobs.shape[0]:
        scores, _ = port_oracle.hmm_score_batch(rs.reads, rs.ev_mean, rs.ev_start_time, models, ranks, jobs)
    else:
        scores = np.zeros(0, np.float32)
    return site_rows, jobs, scores


def _check(engine, port_oracle, rs, models, ref_bases, pairs, records, alphabet, **kw):
    params = synth.meth_params(alphabet, K, **kw)
    site_off, sites, scored = engine.methylation_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ref_bases, pairs, records, params)
    rows, jobs, scores = _expected(port_oracle, rs, models, ref_bases, pairs, records, alphabet, **kw)
    assert sites.shape[0] == len(rows)
    want_off = np.zeros(records.shape[0] + 1, np.uint64)
    for r in rows:
        want_off[r[0] + 1] += 1
    want_off = np.cumsum(want_off).astype(np.uint64)
    assert np.array_equal(site_off, want_off)
    if rows:
        w = np.array([(r[1], r[2], r[3], r[0]) for r in rows], np.int64)
        assert np.array_equal(sites["start_position"], w[:, 0]) and np.array_equal(sites["end_position"], w[:, 1])
        assert np.array_equal(sites["n_motif"], w[:, 2]) and np.array_equal(sites["record"], w[:, 3])
        assert np.array_equal(sites["ll_unmethylated"].view(np.uint32), scores[0::2].view(np.uint32))
        assert np.array_equal(sites["ll_methylated"].view(np.uint32), scores[1::2].view(np.uint32))
        E = np.abs(jobs["event_stop"].astype(np.int64) - jobs["event_start"].astype(np.int64)) + 1
        assert scored == int(E.sum())
    return sites


def _batch(n_reads, n_events, seed, rc_every=3):
    nuc, cpg = synth.load_model("nucleotide"), synth.load_model("cpg")
    rs = synth.gen_reads(n_reads, n_events, nuc, seed=seed, cpg_keep=0.3)
    ref, pairs, recs = synth.methylation_records(rs, model_id=1, rc_every=rc_every)
    return rs, [nuc, cpg], ref, pairs, recs


@pytest.fixture(scope="module")
def eng2(engine):
    # engine fixture is shared: models 0 = nucleotide, 1 = cpg must exist in this order for these tests
    from nanopolish_b200.engine import Engine
    e = Engine(0)
    e.model_upload(synth.load_model("nucleotide"))
    e.model_upload(synth.load_model("cpg"))
    yield e
    e.close()


def test_cpg_groups_and_scores_identical(eng2, port_oracle):
    rs, models, ref, pairs, recs = _batch(12, 2500, 77)
    sites = _check(eng2, port_oracle, rs, models, ref, pairs, recs, "cpg")
    assert sites.shape[0] > 150 and (sites["n_motif"] > 1).any()


def test_edge_records(eng2, port_oracle):
    rs, models, ref, pairs, recs = _batch(8, 1200, 5)
    recs = recs.copy()
    ref = ref.copy()
    # record 0: no CG at all; record 1: no event alignment; record 2: alignment that stops halfway (unbounded windows);
    # record 3: reference cut right after a site so that the last window is clipped by substr
    r0 = recs[0]; seg = ref[int(r0["ref_off"]):int(r0["ref_off"]) + int(r0["ref_len"])]
    seg[seg == ord("G")] = ord("A")
    recs[1]["n_pairs"] = 0
    recs[2]["n_pairs"] = recs[2]["n_pairs"] // 2
    r3 = recs[3]; seg3 = ref[int(r3["ref_off"]):int(r3["ref_off"]) + int(r3["ref_len"])]
    cg = np.flatnonzero((seg3[:-1] == ord("C")) & (seg3[1:] == ord("G")))
    cut = int(cg[len(cg) // 2]) + 2 + 3            # 3 bases after a site: its window (+10) runs past the end
    recs[3]["ref_len"] = cut
    _check(eng2, port_oracle, rs, models, ref, pairs, recs, "cpg")


def test_region_and_window_parameters(eng2, port_oracle):
    rs, models, ref, pairs, recs = _batch(6, 2000, 19)
    _check(eng2, port_oracle, rs, models, ref, pairs, recs, "cpg", region_start=10_300, region_end=10_900)
    _check(eng2, port_oracle, rs, models, ref, pairs, recs, "cpg", min_separation=5, min_flank=12, max_span=40, min_event_span=20)


def test_dam_alphabet(port_oracle):
    """GATC -> GMTC / CTMG: a four-symbol site whose methylated symbol is not the first one; random 5^6 model."""
    from nanopolish_b200.engine import Engine
    nuc = synth.load_model("nucleotide")
    dam = synth.synthetic_model("cpg", 6, seed=99)          # any ACGMT table serves: the alphabet only fixes the symbols' ranks
    rng = np.random.default_rng(4)
    rs = synth.gen_reads(6, 2500, nuc, seed=31)
    # plant GATC every ~40-70 bases (and some pairs 6 apart) in the read sequences' reference copies
    ref, pairs, recs = synth.methylation_records(rs, model_id=1, rc_every=2)
    ref = ref.copy()
    for r in recs:
        o, n = int(r["ref_off"]), int(r["ref_len"])
        pos = 30
        while pos + 12 < n:
            ref[o + pos:o + pos + 4] = np.frombuffer(b"GATC", np.uint8)
            if rng.random() < 0.3:
                ref[o + pos + 6:o + pos + 10] = np.frombuffer(b"GATC", np.uint8)
            pos += int(rng.integers(40, 70))
    e = Engine(0)
    try:
        e.model_upload(nuc); e.model_upload(dam)
        sites = _check(e, port_oracle, rs, [nuc, dam], ref, pairs, recs, "dam")
        assert sites.shape[0] > 100
    finally:
        e.close()


def test_staged_form_matches_one_shot(eng2):
    rs, models, ref, pairs, recs = _batch(10, 1500, 123)
    params = synth.meth_params("cpg", K)
    off1, s1, ev1 = eng2.methylation_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ref, pairs, recs, params)
    eng2.reads_load(rs.reads, rs.ev_mean, rs.ev_start_time)
    eng2.methylation_load(ref, pairs, recs, params)
    for _ in range(2):                                   # repeatable on the resident batch
        eng2.methylation_run()
        off2, s2 = eng2.methylation_fetch()
        n_sites, n_jobs, ev2 = eng2.methylation_counts()
        assert n_sites == s1.shape[0] and n_jobs == 2 * n_sites and ev2 == ev1
        assert np.array_equal(off1, off2) and s1.tobytes() == s2.tobytes()


def test_large_batch_pipelined_upload(eng2, port_oracle):
    """> 2^20 events: the one-shot call streams the event levels behind the enumeration (progress words)."""
    rs, models, ref, pairs, recs = _batch(300, 4000, 999, rc_every=4)
    params = synth.meth_params("cpg", K)
    off1, s1, ev1 = eng2.methylation_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ref, pairs, recs, params)
    eng2.reads_load(rs.reads, rs.ev_mean, rs.ev_start_time)
    eng2.methylation_load(ref, pairs, recs, params)
    eng2.methylation_run()
    off2, s2 = eng2.methylation_fetch()
    assert np.array_equal(off1, off2) and s1.tobytes() == s2.tobytes()
    # and a sample of it against the oracle
    sub = recs[:5].copy()
    _check(eng2, port_oracle, rs, models, ref, pairs, sub, "cpg")


def test_invalid_inputs(eng2):
    rs, models, ref, pairs, recs = _batch(3, 800, 8)
    params = synth.meth_params("cpg", K)
    from nanopolish_b200._lib import NphError
    bad = recs.copy(); bad[1]["read"] = 99
    with pytest.raises(NphError):
        eng2.methylation_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ref, pairs, bad, params)
    bad = recs.copy(); bad[0]["ref_off"] = 2 ** 63
    with pytest.raises(NphError):
        eng2.methylation_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ref, pairs, bad, params)
    badp = pairs.copy(); badp["read_pos"][5:400:3] = 10 ** 6        # event indices outside the read (one end of some window): the reference would read out of bounds
    with pytest.raises(NphError):
        eng2.methylation_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ref, badp, recs, params)
    p5 = synth.meth_params("cpg", 5)                                 # k disagrees with the model
    with pytest.raises(NphError):
        eng2.methylation_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ref, pairs, recs, p5)


def test_device_equals_compiled_reference(eng2, ref_oracle):
    """nph_methylation_batch against the compiled reference's own calculate_methylation_for_read + TSV writer (oracle/_ref,
    or its answers recorded under tests/golden/ref_calls/): records built the way BAM / FASTA / SquiggleRead present them
    (tests/meth_cases.py)."""
    from tests import meth_cases as mc
    nuc = synth.load_model("nucleotide")
    rs = synth.gen_reads(9, 2200, nuc, seed=4242, cpg_keep=0.35)
    ref_oracle.clear_reads()
    mh = ref_oracle.builtin_model("nucleotide")
    ref_oracle.builtin_model("cpg")
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, mh)
    rng = np.random.default_rng(11)
    refs, prs, want_tsv, want_ll, cases = [], [], [], [], []
    recs = np.zeros(rs.n_reads, synth.METH_RECORD_DT)
    ro = po = 0
    for i in range(rs.n_reads):
        case = mc.make_case(i, rs, rng)
        one = np.ones(int(rs.reads[i]["n_events"]), np.float32)
        ref_oracle.read_set_eventalign(rh[i], case["name"], case["read_sequence"], case["b2e_start"], case["b2e_stop"], one, one)
        tsv_ref, sites_ref, ll_ref = ref_oracle.call_methylation(rh[i], case["name"], "chr1", case["contig"], case["ref_pos"], case["flag"], case["cigar"])
        pairs, rc = mc.event_alignment_record(case)
        ref = np.frombuffer(mc.fetched_reference(case).encode(), np.uint8)
        pr = np.zeros(len(pairs), synth.PAIR_DT)
        if pairs:
            pr["ref_pos"], pr["read_pos"] = [p[0] for p in pairs], [p[1] for p in pairs]
        recs[i] = (ro, po, i, 1, ref.shape[0], pr.shape[0], case["ref_pos"], rc, 0, (0, 0))
        refs.append(ref); prs.append(pr); want_tsv.append(tsv_ref); want_ll.append(ll_ref); cases.append(case)
        ro += ref.shape[0]; po += pr.shape[0]
    ref_bases, pairs = np.concatenate(refs), np.concatenate(prs)
    site_off, sites, _ = eng2.methylation_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ref_bases, pairs, recs, synth.meth_params("cpg", K))
    total = 0
    for i, case in enumerate(cases):
        s = sites[int(site_off[i]):int(site_off[i + 1])]
        ll = want_ll[i]
        assert s.shape[0] == ll.shape[0]
        assert np.array_equal(s["ll_unmethylated"].astype(np.float64), ll[:, 0]) and np.array_equal(s["ll_methylated"].astype(np.float64), ll[:, 1])
        fetched = mc.fetched_reference(case)
        rows = [(int(x["start_position"]), int(x["end_position"]), int(x["n_motif"]), x["ll_unmethylated"], x["ll_methylated"],
                 fetched[int(x["start_position"]) - case["ref_pos"] - K + 1:int(x["end_position"]) - case["ref_pos"] + K]) for x in s]
        assert mc.tsv_rows("chr1", "-" if case["flag"] & 16 else "+", case["name"], rows) == want_tsv[i]
        total += s.shape[0]
    assert total > 150
    # the rows the DEVICE formats (nph_methylation_tsv) are the compiled reference's TSV, byte for byte: records with insertions /
    # deletions / soft clips, reverse strand, IUPAC and lower-case reference bases
    got = eng2.methylation_tsv("chr1", [c["name"] for c in cases], np.array([1 if c["flag"] & 16 else 0 for c in cases], np.uint8))
    assert got.decode() == "".join(want_tsv)


def test_compact_event_alignment_form(eng2, ref_oracle):
    """nph_methylation_batch_compact (int16 event-index deltas per reference base, 2 B/base on the wire instead of 8 B/pair) returns
    exactly what the pair form returns: synthetic all-M records, and the CIGAR cases with deletions / insertions / clipped ends
    (reference bases without an entry, boundary k-mers dropped, reverse strand = falling event indices)."""
    rs, models, ref, pairs, recs = _batch(40, 2500, 31, rc_every=2)
    recs = recs.copy(); recs[3]["n_pairs"] = 0; recs[5]["n_pairs"] //= 2
    params = synth.meth_params("cpg", K)
    deltas, first = synth.compact_event_alignment(recs, pairs, ref.shape[0])
    a = eng2.methylation_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ref, pairs, recs, params)
    b = eng2.methylation_batch_compact(rs.reads, rs.ev_mean, rs.ev_start_time, ref, deltas, first, recs, params)
    assert np.array_equal(a[0], b[0]) and a[1].tobytes() == b[1].tobytes() and a[2] == b[2] and a[1].shape[0] > 500
    # staged
    eng2.reads_load(rs.reads, rs.ev_mean, rs.ev_start_time)
    eng2.methylation_load_compact(ref, deltas, first, recs, params)
    eng2.methylation_run()
    off2, s2 = eng2.methylation_fetch()
    assert np.array_equal(a[0], off2) and a[1].tobytes() == s2.tobytes()
    # records with indels
    from tests import meth_cases as mc
    nuc = synth.load_model("nucleotide")
    rs = synth.gen_reads(6, 2200, nuc, seed=77, cpg_keep=0.35)
    rng = np.random.default_rng(3)
    refs, prs = [], []
    recs = np.zeros(rs.n_reads, synth.METH_RECORD_DT)
    ro = po = 0
    for i in range(rs.n_reads):
        case = mc.make_case(i, rs, rng)
        pl, rc = mc.event_alignment_record(case)
        r = np.frombuffer(mc.fetched_reference(case).encode(), np.uint8)
        pr = np.zeros(len(pl), synth.PAIR_DT)
        pr["ref_pos"], pr["read_pos"] = [p[0] for p in pl], [p[1] for p in pl]
        recs[i] = (ro, po, i, 1, r.shape[0], pr.shape[0], case["ref_pos"], rc, 0, (0, 0))
        refs.append(r); prs.append(pr); ro += r.shape[0]; po += pr.shape[0]
    ref, pairs = np.concatenate(refs), np.concatenate(prs)
    deltas, first = synth.compact_event_alignment(recs, pairs, ref.shape[0])
    assert (deltas == synth.METH_NO_PAIR).sum() > 20
    a = eng2.methylation_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ref, pairs, recs, params)
    b = eng2.methylation_batch_compact(rs.reads, rs.ev_mean, rs.ev_start_time, ref, deltas, first, recs, params)
    assert np.array_equal(a[0], b[0]) and a[1].tobytes() == b[1].tobytes() and a[1].shape[0] > 100


def _expected_rows(sites, site_off, recs, ref, names, is_rev, contig, k):
    """the reference's writer (src/nanopolish_call_methylation.cpp:113-140) over site records, formatted by Python's correctly
    rounded %.2f — the C library's %.2lf"""
    out = []
    for r in range(recs.shape[0]):
        R = recs[r]
        seg = ref[int(R["ref_off"]):int(R["ref_off"]) + int(R["ref_len"])].tobytes().decode()
        for s in sites[int(site_off[r]):int(site_off[r + 1])]:
            ll_m, ll_u = float(s["ll_methylated"]) + 0.0, float(s["ll_unmethylated"]) + 0.0
            b = int(s["start_position"]) - int(R["ref_start_pos"]) - k + 1
            e = min(int(s["end_position"]) - int(R["ref_start_pos"]) + k, int(R["ref_len"]))
            out.append("%s\t%s\t%d\t%d\t%s\t%.2f\t%.2f\t%.2f\t%d\t%d\t%s\n" % (
                contig, "-" if is_rev[r] else "+", int(s["start_position"]), int(s["end_position"]), names[r], ll_m - ll_u, ll_m, ll_u, 1,
                int(s["n_motif"]), seg[b:e]))
    return "".join(out)


def test_tsv_rows_formatted_on_the_device(eng2):
    """nph_methylation_tsv: every field of every row, against Python's formatting of the same site records (forward and reverse records,
    a record without sites, a window clipped by the end of the record's reference, read names of different lengths)."""
    rs, models, ref, pairs, recs = _batch(14, 2500, 4242, rc_every=3)
    recs = recs.copy(); ref = ref.copy()
    r0 = recs[0]; seg = ref[int(r0["ref_off"]):int(r0["ref_off"]) + int(r0["ref_len"])]
    seg[seg == ord("G")] = ord("A")                                      # record 0: no site at all
    r3 = recs[3]; seg3 = ref[int(r3["ref_off"]):int(r3["ref_off"]) + int(r3["ref_len"])]
    cg = np.flatnonzero((seg3[:-1] == ord("C")) & (seg3[1:] == ord("G")))
    recs[3]["ref_len"] = int(cg[len(cg) // 2]) + 2 + 3                   # the sequence column of the last row is cut by the end
    params = synth.meth_params("cpg", K)
    site_off, sites, _ = eng2.methylation_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ref, pairs, recs, params)
    names = ["r%d_%s" % (i, "x" * (i % 7)) for i in range(recs.shape[0])]
    is_rev = (np.arange(recs.shape[0]) % 2).astype(np.uint8)
    got = eng2.methylation_tsv("chr20", names, is_rev).decode()
    want = _expected_rows(sites, site_off, recs, ref, names, is_rev, "chr20", K)
    assert want.count("\n") == sites.shape[0] > 150
    assert got == want
    # a destination that is too small reports the size needed
    from nanopolish_b200._lib import NphError
    with pytest.raises(NphError):
        eng2.methylation_tsv("chr20", names, is_rev, cap=100)


def test_tsv_number_formatting_on_device():
    """csrc/tsv_format.cuh == printf("%.2lf") / printf("%d") on 6.6e6 doubles (scores, differences, exact halves at the second decimal,
    every binade, random bit patterns, refusals beyond 2^52) — host and device copies of the same functions."""
    import os, subprocess
    exe = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cuda", "check_tsv_format")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "device: 0 bad" in r.stdout
