"""SURVEY.md 8(f) row N1, host half — eventalign's segment chaining around the Viterbi kernel
(nanopolish_b200/host/nph_eventalign.*: align_read_to_ref, src/alignment/nanopolish_eventalign.cpp:612-827, and its
TSV / SAM / summary writers).

  * the Python restatement (oracle/eventalign_py.py) against the COMPILED reference's align_read_to_ref +
    emit_event_alignment_tsv (oracle/_ref, or its answers recorded under tests/golden/ref_calls/) and against the outputs recorded from it
    (tests/golden/eventalign_golden.npz) anywhere;
  * the C++ cursor logic on the CPU: rounds are pulled out of EventAligner, the paths come from the plain-C Viterbi
    oracle and are fed back — the text it then writes must equal the reference's, byte for byte;
  * on the GPU the same through EventAligner::run (one Viterbi launch per round, events resident after round one).

Pin status of what is compared here: the default TSV, the event CIGAR and the summary NUMBERS are pinned to the compiled reference;
`-n` (read names), `--scale-events`, the SAM text around the CIGAR and the formatting of the summary row / `--samples` columns are
checked against the restatement only (oracle/eventalign_py.py follows eventalign.cpp:398-484 for them; the harness does not drive
those writer options).
"""
import ctypes as C
import os

import numpy as np
import pytest

from nanopolish_b200 import synth
from oracle import eventalign_py as EP
from tests import eventalign_cases as EC
from tests.test_host_mirror import HOST_SO, _register, _register_reads

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "eventalign_golden.npz")


@pytest.fixture(scope="module")
def cases():
    return EC.build_cases()


@pytest.fixture(scope="module")
def golden():
    z = np.load(GOLD)
    return {k: z[k].tobytes().decode() for k in z.files}


@pytest.fixture(scope="module")
def restated(cases, port_oracle):
    model, rs, cs = cases
    out = []
    for c in cs:
        st = {}
        al = EP.align_read_to_ref(c["read"], c["contig_name"], c["fetched"], c["ref_pos"], c["flag"], c["cigar"], c["read_idx"],
                                  EC.port_align_fn(port_oracle, rs, model, EC.read_slot(c, rs.n_reads)), *c["region"], stats=st)
        out.append((al, st.get("segments", 0)))
    return out


def _single_segment(c):
    return not any((int(x) & 15) == 3 for x in c["cigar"])


def test_restatement_matches_compiled_reference(cases, restated, ref_oracle):
    model, rs, cs = cases
    ref_oracle.clear_reads()
    mh = ref_oracle.builtin_model("nucleotide")
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, mh)
    for c, (al, _) in zip(cs, restated):
        slot, r = EC.read_slot(c, rs.n_reads), c["read"]
        ref_oracle.read_set_eventalign(rh[slot], r.name, r.read_sequence, r.b2e_start, c["b2e_stop"], r.stdv, r.duration)
        tsv, cigar, ea = ref_oracle.eventalign(rh[slot], c["contig_name"], c["contig"], c["ref_pos"], c["flag"], c["cigar"],
                                               c["read_idx"], c["region"], want_cigar=_single_segment(c))
        assert EP.tsv(r, al) == tsv
        assert [(a.ref_position, a.event_idx, ord(a.hmm_state)) for a in al] == [tuple(int(v) for v in row) for row in ea]
        assert ref_oracle.eventalign_summary() == EP.summarize(r, al)                  # summarize_alignment's counters and sums
        if _single_segment(c):
            assert EP.event_cigar(al) == cigar
    ref_oracle.clear_reads()


def test_sample_columns_match_compiled_reference(cases, ref_oracle):
    """What --signal-index / --samples print per event — SquiggleRead::get_event_sample_idx and
    get_scaled_samples_for_event — from the reference's own nanopolish_squiggle_read.cpp (compiled into oracle/_ref)
    against the restatement the writer tests use (drift, shift and scale all non-trivial in these reads)."""
    model, rs, cs = cases
    ref_oracle.clear_reads()
    rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, ref_oracle.builtin_model("nucleotide"))
    for c in cs[:2]:
        slot, r = EC.read_slot(c, rs.n_reads), c["read"]
        ref_oracle.read_set_eventalign(rh[slot], r.name, r.read_sequence, r.b2e_start, c["b2e_stop"], r.stdv, r.duration)
        smp = _raw_samples(slot)
        ref_oracle.read_set_samples(rh[slot], smp, 4000.0)
        for e in (0, 1, 17, 400, int(rs.reads[slot]["n_events"]) - 1):
            a, b, v = ref_oracle.event_samples(rh[slot], e)
            assert (a, b) == EP.event_sample_idx(r, e, 4000.0)
            want = np.array(EP.scaled_samples(r, e, smp, 4000.0), np.float32)
            assert v.shape == want.shape and np.array_equal(v.view(np.uint32), want.view(np.uint32))
    ref_oracle.clear_reads()


def test_restatement_matches_golden(cases, restated, golden):
    model, rs, cs = cases
    rows = 0
    for c, (al, segs) in zip(cs, restated):
        assert EP.tsv(c["read"], al) == golden[f"tsv_{c['read_idx']}"]
        if _single_segment(c):
            assert EP.event_cigar(al) == golden[f"cigar_{c['read_idx']}"]
        rows += len(al)
    assert rows > 6000                                   # forward, reverse, two-segment, windowed and unmapped records
    assert golden["tsv_4"] == ""                         # the unmapped record aligns nothing


# ---- the C++ host side --------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host():
    lib = C.CDLL(HOST_SO)
    lib.nphh_last_error.restype = C.c_char_p
    for f in ("nphh_ea_run", "nphh_ea_next_round", "nphh_ea_text", "nphh_ea_num_segments", "nphh_aligned_segments"):
        getattr(lib, f).restype = C.c_longlong
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _setup(host, cases):
    model, rs, cs = cases
    host.nphh_clear()
    mh = _register(host, model)
    rh = _register_reads(host, rs, mh)
    host.nphh_ea_begin()
    for c in cs:
        slot, r = EC.read_slot(c, rs.n_reads), c["read"]
        a, b = np.ascontiguousarray(r.b2e_start, np.int32), np.ascontiguousarray(c["b2e_stop"], np.int32)
        assert host.nphh_read_set_eventalign(rh[slot], r.name.encode(), r.read_sequence.encode(), _p(a), _p(b), C.c_size_t(a.shape[0]),
                                             _p(np.ascontiguousarray(r.stdv)), _p(np.ascontiguousarray(r.duration))) == 0
        smp = _raw_samples(slot)
        assert host.nphh_read_set_samples(rh[slot], _p(smp), C.c_size_t(smp.shape[0]), C.c_double(4000.0)) == 0
        idx = host.nphh_ea_add_read(rh[slot], c["contig_name"].encode(), c["ref_pos"], c["flag"], c["mapq"], _p(c["cigar"]),
                                    int(c["cigar"].shape[0]), c["fetched"].encode(), c["read_idx"], c["region"][0], c["region"][1])
        assert idx == c["read_idx"], host.nphh_last_error()


def _raw_samples(slot):
    """stand-in for the trimmed raw samples SRF_LOAD_RAW_SAMPLES keeps: enough of them to cover every event's time span"""
    return np.random.default_rng(900 + slot).normal(90.0, 12.0, 420_000).astype(np.float32)


def _text(host, idx, what):
    buf = C.create_string_buffer(1 << 23)
    n = host.nphh_ea_text(idx, what, buf, C.c_size_t(1 << 23))
    assert n >= 0, host.nphh_last_error()
    return buf.value.decode()


def _check_outputs(host, cases, restated, golden):
    model, rs, cs = cases
    for c, (al, segs) in zip(cs, restated):
        i, r = c["read_idx"], c["read"]
        assert _text(host, i, 0) == golden[f"tsv_{i}"]                                     # the compiled reference's bytes
        assert _text(host, i, 1) == EP.tsv(r, al, print_read_names=True)                   # -n
        assert _text(host, i, 2) == EP.tsv(r, al, scale_events=True)                       # --scale-events
        hdr = _text(host, 0, 6)[:-1] + "\tstart_idx\tend_idx\tsamples\n"
        assert _text(host, i, 7) == hdr + EP.tsv(r, al, samples=_raw_samples(EC.read_slot(c, rs.n_reads)), sample_rate=4000.0)   # --signal-index --samples
        ints, dbl = np.zeros(5, np.int32), np.zeros(2)
        assert host.nphh_ea_summary(i, _p(ints), _p(dbl)) == 0
        sm = EP.summarize(r, al)
        assert [int(v) for v in ints] == [sm["num_events"], sm["num_steps"], sm["num_stays"], sm["num_skips"], sm["reference_span"]]
        assert (float(dbl[0]), float(dbl[1])) == (sm["sum_duration"], sm["sum_z_score"])
        assert host.nphh_ea_num_segments(i) == segs
        assert _text(host, i, 5) == EP.summary_row(r, al, i, "read.fast5").replace(r.model_name, "")   # host test models carry no name
        if _single_segment(c):
            assert _text(host, i, 4) == golden[f"cigar_{i}"]
            assert _text(host, i, 3) == EP.sam(r, al, c["mapq"])
    host.nphh_ea_tsv_all.restype = C.c_longlong
    buf = C.create_string_buffer(1 << 22)
    assert host.nphh_ea_tsv_all(buf, C.c_size_t(1 << 22)) >= 0, host.nphh_last_error()
    assert buf.value.decode() == "".join(golden[f"tsv_{c['read_idx']}"] for c in cs)           # tsv_batch: all reads, in parallel
    assert _text(host, 0, 6) == ("contig\tposition\treference_kmer\tread_index\tstrand\tevent_index\tevent_level_mean\tevent_stdv\t"
                                 "event_length\tmodel_kmer\tmodel_mean\tmodel_stdv\tstandardized_level\n")


def test_host_chaining_logic_on_cpu(host, cases, restated, golden, port_oracle):
    """EventAligner's cursors, fed with the plain-C Viterbi's paths (no device involved)."""
    model, rs, cs = cases
    _setup(host, cases)
    jobs = np.zeros(len(cs), synth.HMM_JOB_DT)
    ranks = np.zeros(len(cs) * 400, np.uint32)
    n_ranks = C.c_uint64()
    rounds = 0
    while True:
        n = host.nphh_ea_next_round(_p(jobs), C.c_size_t(jobs.shape[0]), _p(ranks), C.c_size_t(ranks.shape[0]), C.byref(n_ranks))
        assert n >= 0, host.nphh_last_error()
        if n == 0:
            break
        paths, off = [], [0]
        for j in range(n):
            jb = jobs[j].copy()
            jb["read"] = EC.read_slot(cs[int(jb["read"])], rs.n_reads)      # aligner index -> synthetic read
            st, status = port_oracle.hmm_align(rs.reads, rs.ev_mean, rs.ev_start_time, [model], ranks, jb)
            paths.append(st); off.append(off[-1] + st.shape[0])
        flat = np.concatenate(paths) if off[-1] else np.zeros(0, synth.ALIGN_STATE_DT)
        assert host.nphh_ea_consume(C.c_size_t(n), _p(np.array(off, np.uint64)), _p(flat)) == 0, host.nphh_last_error()
        rounds += 1
    assert rounds == max(s for _, s in restated)          # launches = the longest read's segment count
    _check_outputs(host, cases, restated, golden)
    host.nphh_ea_begin()


def _drive_rounds(host, cs, rs, model, port_oracle):
    """pull every round's jobs out of the C++ cursors and feed back the plain-C Viterbi's paths"""
    jobs = np.zeros(max(len(cs), 1), synth.HMM_JOB_DT)
    ranks = np.zeros(len(cs) * 400 + 400, np.uint32)
    n_ranks = C.c_uint64()
    rounds = 0
    while True:
        n = host.nphh_ea_next_round(_p(jobs), C.c_size_t(jobs.shape[0]), _p(ranks), C.c_size_t(ranks.shape[0]), C.byref(n_ranks))
        assert n >= 0, host.nphh_last_error()
        if n == 0:
            return rounds
        paths, off = [], [0]
        for j in range(n):
            jb = jobs[j].copy()
            jb["read"] = EC.read_slot(cs[int(jb["read"])], rs.n_reads)
            st, _ = port_oracle.hmm_align(rs.reads, rs.ev_mean, rs.ev_start_time, [model], ranks, jb)
            paths.append(st); off.append(off[-1] + st.shape[0])
        flat = np.concatenate(paths) if off[-1] else np.zeros(0, synth.ALIGN_STATE_DT)
        assert host.nphh_ea_consume(C.c_size_t(n), _p(np.array(off, np.uint64)), _p(flat)) == 0, host.nphh_last_error()
        rounds += 1


def test_eventalign_edge_cases_against_compiled_reference(host, cases, ref_oracle, port_oracle):
    """Records the seeded cases do not reach: a window outside the alignment, a window that empties a later BAM segment
    (the reference then returns from align_read_to_ref: later segments are not aligned either), hard clips and =/X
    operations, a read whose k-mers near the segment ends have no events.  C++ cursors == restatement == compiled reference."""
    model, rs, base = cases
    variants = _edge_variants(base)
    # the map with holes needs its own read slot on the C++ side: run that one in a second batch
    for batch in (variants[:4], variants[4:]):
        for i, v in enumerate(batch):
            v["read_idx"] = i
        _setup(host, (model, rs, batch))
        _drive_rounds(host, batch, rs, model, port_oracle)
        ref_oracle.clear_reads()
        mh = ref_oracle.builtin_model("nucleotide")
        rh = ref_oracle.register_reads(rs.reads, rs.ev_mean, rs.ev_start_time, mh)
        for v in batch:
            slot, r = EC.read_slot(v, rs.n_reads), v["read"]
            ref_oracle.read_set_eventalign(rh[slot], r.name, r.read_sequence, r.b2e_start, v["b2e_stop"], r.stdv, r.duration)
            want, _, _ = ref_oracle.eventalign(rh[slot], v["contig_name"], v["contig"], v["ref_pos"], v["flag"], v["cigar"], v["read_idx"],
                                               v["region"], want_cigar=False)
            al = EP.align_read_to_ref(r, v["contig_name"], v["fetched"], v["ref_pos"], v["flag"], v["cigar"], v["read_idx"],
                                      EC.port_align_fn(port_oracle, rs, model, slot), *v["region"])
            assert EP.tsv(r, al) == want
            assert _text(host, v["read_idx"], 0) == want
        host.nphh_ea_begin()
    ref_oracle.clear_reads()


@pytest.mark.gpu
def test_eventalign_edge_cases_on_device(host, cases, port_oracle):
    """the same records through the chain kernel (EventAligner::run)"""
    model, rs, base = cases
    variants = _edge_variants(base)
    for batch in (variants[:4], variants[4:]):
        for i, v in enumerate(batch):
            v["read_idx"] = i
        _setup(host, (model, rs, batch))
        assert host.nphh_ea_run(C.c_double(1.0)) >= 0, host.nphh_last_error()
        for v in batch:
            slot, r = EC.read_slot(v, rs.n_reads), v["read"]
            al = EP.align_read_to_ref(r, v["contig_name"], v["fetched"], v["ref_pos"], v["flag"], v["cigar"], v["read_idx"],
                                      EC.port_align_fn(port_oracle, rs, model, slot), *v["region"])
            assert _text(host, v["read_idx"], 0) == EP.tsv(r, al)
        host.nphh_ea_begin()


def _edge_variants(base):
    c0, c2 = base[0], base[2]                               # forward single-segment record; forward record with an N
    assert not _single_segment(c2)
    variants = []
    v = dict(c0); v["region"] = (5, 20); variants.append(v)                                    # nothing of the alignment inside
    seg_pairs = EP.get_aligned_segments(c2["ref_pos"], c2["cigar"])
    first_end = seg_pairs[0][-1][0]
    v = dict(c2); v["region"] = (c2["ref_pos"] + 50, first_end - 10); variants.append(v)       # second segment trims to nothing
    v = dict(c2); v["region"] = (seg_pairs[1][0][0] + 30, seg_pairs[1][-1][0]); variants.append(v)   # FIRST segment empty: nothing at all
    ops = [(int(x) >> 4, EP.CIGAR_OPS[int(x) & 15]) for x in c0["cigar"]]
    ops2 = [(7, "H")] + [(n, "=" if (i % 2 and o == "M") else ("X" if (i % 3 == 0 and o == "M") else o)) for i, (n, o) in enumerate(ops)] + [(3, "H")]
    v = dict(c0); v["cigar"] = EP.pack_cigar(ops2); variants.append(v)
    holes = c0["read"].b2e_start.copy()                                                       # no events for the first / last k-mers of the read
    holes[:12] = -1; holes[-9:] = -1
    stop = c0["b2e_stop"].copy(); stop[:12] = -1; stop[-9:] = -1
    import dataclasses
    v = dict(c0); v["read"] = dataclasses.replace(c0["read"], b2e_start=holes); v["b2e_stop"] = stop; variants.append(v)
    return variants


def test_format_fixed_matches_printf(host):
    """The TSV writer's %.2lf / %.3lf / %.5lf replacement (exact integer arithmetic on the float) against snprintf on
    6 x 600k values: uniform bit patterns, dyadic fractions, decimal ties and their neighbours, inf/nan, +-0."""
    host.nphh_format_fixed_check.restype = C.c_longlong
    assert host.nphh_format_fixed_check(C.c_uint64(20240923), C.c_size_t(600_000)) == 0, host.nphh_last_error()


def test_rolling_kmer_ranks(host):
    """the rank tables EventAligner::run hands the chain kernel (one rolling pass per reference) == Alphabet::kmer_rank"""
    host.nphh_rolling_ranks_check.restype = C.c_longlong
    rng = np.random.default_rng(4)
    dna = "".join("ACGT"[c] for c in rng.integers(0, 4, 3000))
    cpg = "".join("ACGMT"[c] for c in rng.integers(0, 5, 3000))
    assert host.nphh_rolling_ranks_check(b"nucleotide", dna.encode(), 6) == 0
    assert host.nphh_rolling_ranks_check(b"nucleotide", dna.encode(), 5) == 0
    assert host.nphh_rolling_ranks_check(b"cpg", cpg.encode(), 6) == 0
    assert host.nphh_rolling_ranks_check(b"nucleotide", b"ACGTA", 6) == 0          # shorter than k: no k-mers


def test_get_aligned_segments(host):
    ops = [(5, "S"), (10, "M"), (2, "I"), (3, "D"), (4, "="), (7, "N"), (6, "X"), (3, "H")]
    cigar = EP.pack_cigar(ops)
    want = EP.get_aligned_segments(1000, cigar)
    pairs = np.zeros((64, 2), np.int32)
    seg_off = np.zeros(8, np.uint64)
    n = host.nphh_aligned_segments(1000, _p(cigar), int(cigar.shape[0]), _p(pairs), C.c_size_t(64), _p(seg_off), C.c_size_t(8))
    assert n == len(want) == 2
    for s in range(n):
        got = [tuple(int(v) for v in p) for p in pairs[int(seg_off[s]):int(seg_off[s + 1])]]
        assert got == want[s]
    assert want[0][0] == (1000, 5) and want[1][0] == (1000 + 10 + 3 + 4 + 7, 5 + 10 + 2 + 4)
    bad = EP.pack_cigar([(3, "P")])
    assert host.nphh_aligned_segments(0, _p(bad), 1, _p(pairs), C.c_size_t(64), _p(seg_off), C.c_size_t(8)) < 0     # the reference asserts


@pytest.mark.gpu
def test_eventalign_on_device(host, cases, restated, golden):
    """The whole thing on the device: every (read, BAM segment) chain walked start to end by one warp of
    eventalign_chain_kernel in ONE launch; text identical to the reference's."""
    _setup(host, cases)
    batches = host.nphh_ea_run(C.c_double(1.0))
    assert batches == 1, host.nphh_last_error()            # no window needed the host-driven fallback
    _check_outputs(host, cases, restated, golden)
    host.nphh_ea_begin()


@pytest.mark.gpu
def test_eventalign_host_rounds_on_device(host, cases, restated, golden):
    """The host-driven form: one hmm_viterbi_kernel launch per round over the next window of every unfinished read."""
    _setup(host, cases)
    rounds = host.nphh_ea_run_rounds(C.c_double(1.0))
    assert rounds >= 0, host.nphh_last_error()
    assert rounds == max(s for _, s in restated)
    _check_outputs(host, cases, restated, golden)
    host.nphh_ea_begin()


@pytest.mark.gpu
def test_eventalign_chain_falls_back_for_large_windows(host, cases, restated, golden):
    """A window with more events than the chain kernel's scratch holds flags its read; EventAligner re-runs those reads
    through the round driver and the output does not change."""
    _setup(host, cases)
    os.environ["NPH_EA_EVENT_CAP"] = "150"                  # most windows span ~170 events
    try:
        batches = host.nphh_ea_run(C.c_double(1.0))
    finally:
        del os.environ["NPH_EA_EVENT_CAP"]
    assert batches > 1, host.nphh_last_error()
    _check_outputs(host, cases, restated, golden)
    host.nphh_ea_begin()


@pytest.mark.gpu
def test_eventalign_chain_abi(engine, cases, restated):
    """nph_eventalign_chain called directly (what EventAligner::run does underneath): records per chain."""
    _chain_abi(engine, cases, restated)


@pytest.mark.gpu
def test_eventalign_chain_abi_5mer(engine, port_oracle):
    """5-mers (the RNA model's k): a 101-base window holds 97 k-mers, so the chain kernel runs four columns per lane."""
    model = EC.five_mer_model()
    cases5 = EC.build_cases(3, 1200, seed=505, model=model)
    _, rs, cs = cases5
    restated5 = []
    for c in cs:
        st = {}
        al = EP.align_read_to_ref(c["read"], c["contig_name"], c["fetched"], c["ref_pos"], c["flag"], c["cigar"], c["read_idx"],
                                  EC.port_align_fn(port_oracle, rs, model, EC.read_slot(c, rs.n_reads)), *c["region"], stats=st)
        restated5.append((al, st.get("segments", 0)))
    assert sum(len(al) for al, _ in restated5) > 2000
    _chain_abi(engine, cases5, restated5)


def _chain_abi(engine, cases, restated):
    model, rs, cs = cases
    K = model.k
    mid = engine.model_upload(model)
    engine.reads_load(rs.reads, rs.ev_mean, rs.ev_start_time)
    chains = np.zeros(0, synth.EA_CHAIN_DT)
    pairs, maps, rf, rr, want = [], [], [], [], []
    map_off = {}
    out_off = 0
    rows = []
    for c, (al, segs) in zip(cs, restated):
        if c["flag"] & EP.BAM_FUNMAP or c["region"] != (-1, -1) or not _single_segment(c):
            continue
        r, slot = c["read"], EC.read_slot(c, rs.n_reads)
        if slot not in map_off:
            map_off[slot] = sum(m.shape[0] for m in maps)
            maps.append(np.ascontiguousarray(r.b2e_start, np.int32))
        ref = EP.disambiguate(c["fetched"])
        codes = synth.encode(ref, "nucleotide")
        seg = EP.get_aligned_segments(c["ref_pos"], c["cigar"])[0]
        seg = [p for p in seg if p[1] <= len(r.read_sequence) - K]
        rev = bool(c["flag"] & EP.BAM_FREVERSE)
        k0, k1 = seg[0][1], seg[-1][1]
        if rev:
            k0, k1 = r.flip_k_strand(k0), r.flip_k_strand(k1)
        first, last = r.get_closest_event_to(k0), r.get_closest_event_to(k1)
        rows.append((sum(len(p) for p in pairs), map_off[slot], sum(x.shape[0] for x in rf), out_off, slot, mid, len(seg), r.b2e_start.shape[0],
                     len(ref), len(r.read_sequence), abs(last - first) + 2, c["ref_pos"], first, last, int(rev), int(rev), K, 0))
        out_off += abs(last - first) + 2
        pairs.append(seg)
        rf.append(synth.kmer_ranks_from_codes(codes, K, 4).astype(np.uint32))
        rr.append(synth.dna_rc_kmer_ranks(codes, K).astype(np.uint32))
        want.append((al, segs))
    chains = np.array(rows, synth.EA_CHAIN_DT)
    flat_pairs = np.array([p for seg in pairs for p in seg], np.int32).reshape(-1, 2)
    records, results = engine.eventalign_chain(flat_pairs, np.concatenate(maps), np.concatenate(rf), np.concatenate(rr), chains)
    assert len(want) >= 3 and (results["status"] == 0).all()
    for i, (al, segs) in enumerate(want):
        o, n = int(chains[i]["out_off"]), int(results[i]["n_records"])
        got = [(int(x["ref_position"]), int(x["event_idx"]), x["hmm_state"].decode()) for x in records[o:o + n]]
        assert got == [(a.ref_position, a.event_idx, a.hmm_state) for a in al]
        assert int(results[i]["n_windows"]) == segs
    ms, launches = engine.last_kernel_ms()
    assert ms > 0 and launches == 1
