#!/usr/bin/env python
"""bench_polya.py — `nanopolish polya` (section 8f N5) on the device: reads/s and samples/s of nph_polya_batch.

    python scripts/bench_polya.py [--reads 4096] [--samples 60000] [--steps 5] [--warmup 2] [--ref-reads 64] [--out FILE]

Workload: --reads seeded direct-RNA-shaped traces of --samples trimmed raw samples each (4096 x 60000 = 983 MB of float32
samples, more than the 126 MB of L2), a PASS / NOREGION / ADAPTER / SUFFCLIP mix.  One JSON line in bench.py's shape:
  value      reads/s with the inputs resident on the device (CUDA events around the Viterbi kernel, median of --steps)
  e2e        the one-shot nph_polya_batch from page-locked host buffers, wall clock (upload, validation, kernel, results)
  resident   nph_polya_after_load after nph_load_from_raw_batch on --lfr-reads direct-RNA traces (nothing uploaded)
  cpu_baseline  the compiled reference (oracle/_ref/libnpref_polya.so) on every host thread over --ref-reads of the reads,
             whose rows must equal ours
  small      device time of batches of 1, 32 and 148 reads (per-read Viterbi latency: ~one dependent step per sample)
The GPU's name and power limit are read in the same run.  Writes nothing to the tree (--out goes where it is told).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from nanopolish_b200 import _lib, synth                      # noqa: E402
from nanopolish_b200.engine import Engine                    # noqa: E402

FAMILIES = ("pass", "pass", "pass", "noregion", "adapter", "suffclip")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "power_limit": None, "error": str(e)}


def pinned_like(lib, a):
    """a copy of a in page-locked memory (nph_host_alloc), and the pointer to free"""
    p = C.c_void_p()
    if lib.nph_host_alloc(C.byref(p), max(a.nbytes, 1)) != 0:
        raise RuntimeError("nph_host_alloc failed")
    buf = (C.c_uint8 * max(a.nbytes, 1)).from_address(p.value)
    out = np.frombuffer(buf, dtype=a.dtype, count=a.shape[0])
    out[...] = a
    return out, p


def rna_traces(n, n_samples, seed):
    """direct-RNA traces for load_from_raw: poly(A)-shaped head, then a transcript read 3'->5' (the 5-mer model of the
    RNA prologue test, tests/test_gpu_prep.py)"""
    m6 = synth.load_model("nucleotide")
    sd5 = m6.level_stdv.reshape(1024, 4).mean(1)
    model = synth.PoreModel("derived.nucleotide.5mer", 5, "nucleotide", m6.level_mean.reshape(1024, 4).mean(1), sd5, np.log(sd5))
    raw, rr, seqs = synth.gen_raw(n, n_samples, model, seed=seed, mean_dwell=40.0, return_seqs=True)
    sig, ranks = [], []
    for i, r in enumerate(rr):
        rng = np.random.default_rng(seed + 7 * i)
        tx = raw[int(r["sample_off"]):int(r["sample_off"]) + int(r["n_samples"])][::-1]
        sig.append(np.concatenate([synth._polya_trace(rng, 600, 2500, 5000, 0, 0.0, 1.0, 1.0), tx]).astype(np.float32))
        ranks.append(synth.kmer_ranks_from_codes(np.ascontiguousarray(seqs[i]), 5, 4))
    jobs = np.zeros(n, synth.RAW_JOB_DT)
    so = ro = 0
    for j in range(n):
        jobs[j] = (so, ro, sig[j].shape[0], ranks[j].shape[0], 3012.0)
        so += sig[j].shape[0]; ro += ranks[j].shape[0]
    return model, np.concatenate(sig), np.concatenate(ranks).astype(np.uint32), jobs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=4096)
    ap.add_argument("--samples", type=int, default=60000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--ref-reads", type=int, default=64)
    ap.add_argument("--lfr-reads", type=int, default=512)
    ap.add_argument("--out", default=None, help="also append the line to this file")
    args = ap.parse_args()
    info = gpu_info()

    t0 = time.time()
    ps = synth.gen_polya(args.reads, seed=2024, families=FAMILIES, lengths=np.full(args.reads, args.samples))
    gen_s = time.time() - t0
    n_samples = int(ps.jobs["n_samples"].sum())
    eng = Engine(0)
    lib = eng.lib

    # ---- inputs resident: kernel time by CUDA events (nph_last_kernel_ms) ----
    res = None
    for _ in range(args.warmup):
        res = eng.polya_batch(ps.samples, ps.durations, ps.map, ps.jobs)
    ks = []
    for _ in range(args.steps):
        res = eng.polya_batch(ps.samples, ps.durations, ps.map, ps.jobs)
        ks.append(eng.last_kernel_ms()[0])
    k_ms = statistics.median(ks)

    # ---- one-shot end to end from page-locked buffers ----
    pins = [pinned_like(lib, a) for a in (ps.samples, ps.durations, ps.map, ps.jobs, np.zeros(args.reads, synth.POLYA_RES_DT))]
    (s_p, _), (d_p, _), (m_p, _), (j_p, _), (r_p, _) = pins
    e2e = []
    for i in range(args.warmup + args.steps):
        t = time.perf_counter()
        eng.polya_batch(s_p, d_p, m_p, j_p, out=r_p)
        if i >= args.warmup:
            e2e.append(time.perf_counter() - t)
    e2e_s = statistics.median(e2e)
    same_e2e = bool(np.array_equal(r_p.view(np.uint8), res.view(np.uint8)))
    for _, p in pins:
        lib.nph_host_free(p)

    # ---- small batches: per-read latency ----
    small = {}
    for nb in (1, 32, 148):
        sub = ps.jobs[:nb]
        eng.polya_batch(ps.samples, ps.durations, ps.map, sub)
        eng.polya_batch(ps.samples, ps.durations, ps.map, sub)
        small[str(nb)] = round(eng.last_kernel_ms()[0], 3)

    # ---- resident form after load_from_raw ----
    model, raw, ranks, rj = rna_traces(args.lfr_reads, 45000, seed=77)
    mid = eng.model_upload(model)
    lfr = []
    n_live = 0
    for i in range(args.warmup + args.steps):
        off, mean, stdv, start, dur, b2e, cal = eng.load_from_raw_batch(raw, ranks, rj, mid, synth.event_params(True))
        t = time.perf_counter()
        ra = eng.polya_after_load(rj.shape[0])
        if i >= args.warmup:
            lfr.append((time.perf_counter() - t, eng.last_kernel_ms()[0]))
        n_live = int((cal["status"] == 0).sum())
    trim = eng.last_trim_ranges(rj.shape[0])
    lfr_samples = int((trim["end"].astype(np.int64) - trim["start"]).sum())
    lfr_wall = statistics.median(x[0] for x in lfr)
    lfr_k = statistics.median(x[1] for x in lfr)

    # ---- compiled reference on all host threads over a sample of the reads; rows must equal ours ----
    cpu = None
    from oracle.polya_py import RefPolya, format_rows
    if RefPolya.available() and args.ref_reads > 0:
        nr = min(args.ref_reads, args.reads)
        threads = os.cpu_count() or 1
        ref = RefPolya()
        sub = ps.jobs[:nr]
        secs, rows = ref.polya_timed(ps.samples, ps.durations, ps.map, sub, ps.names[:nr], "chr1", threads)
        ours = format_rows(res[:nr], ps.names[:nr], "chr1", np.zeros(nr, np.int64), np.zeros(nr, np.uint32))
        ours = ours[ours.index(b"\n") + 1:]
        sub_samples = int(sub["n_samples"].sum())
        cpu = {"value": nr / secs, "unit": "reads/s", "samples_per_sec": sub_samples / secs, "threads": threads, "reads": nr,
               "rows_equal": rows == ours, "kind": "compiled reference (src/nanopolish_polya_estimator.cpp), one read per OpenMP thread",
               "cpu_ms_per_read_per_thread": secs * threads / nr * 1e3}

    qc = np.bincount(res["qc"].astype(np.int64), minlength=8)
    line = {
        "metric": "polya_reads_per_sec", "value": args.reads / (k_ms * 1e-3), "unit": "reads/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": k_ms, "higher_is_better": True, "scaling": "none", "vs_baseline": None,
        "dtype": "f32+f64", "data": "synthetic",
        "config": {"workload": f"polya: {args.reads} direct-RNA-shaped reads x {args.samples} trimmed raw samples ({n_samples * 4 / 1e6:.0f} MB), "
                               f"families {FAMILIES}", "samples_per_sec_device": n_samples / (k_ms * 1e-3),
                   "kernel_ms_steps": [round(x, 3) for x in ks], "qc_counts": {"pass": int(qc[0]), "noregion": int(qc[1]), "adapter": int(qc[2]),
                                                                                "both": int(qc[3])}, "gen_seconds": round(gen_s, 1)},
        "e2e": {"value": args.reads / e2e_s, "unit": "reads/s", "samples_per_sec": n_samples / e2e_s, "ms": e2e_s * 1e3,
                "h2d_bytes": int(ps.samples.nbytes + ps.durations.nbytes + ps.map.nbytes + ps.jobs.nbytes), "api": "nph_polya_batch",
                "host_buffers": "page-locked (nph_host_alloc)", "results_equal_resident": same_e2e},
        "resident_after_load": {"value": args.lfr_reads / lfr_wall, "unit": "reads/s", "ms": lfr_wall * 1e3, "kernel_ms": lfr_k,
                                "reads": args.lfr_reads, "reads_loaded": n_live, "samples": lfr_samples, "api": "nph_polya_after_load"},
        "small_batches_kernel_ms": small,
        "cpu_baseline": cpu,
        "gpu_launches": 2,
        **info,
    }
    s = json.dumps(line)
    print(s, flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")
    eng.close()


if __name__ == "__main__":
    main()
