#!/usr/bin/env python
"""bench.py — HMM-scored events/sec through profile_hmm_score on synthetic R9.4 reads.

    python bench.py --gpus N --steps K --warmup W                 # our arm (CUDA, through the C ABI)
    python bench.py --impl reference --gpus N --steps K --warmup W  # the reference's CPU path on host cores

Workload (BASELINE.json configs[1]): scorereads-shaped jobs — synthetic reads x 4000 events, k=6
r9.4_450bps nucleotide model, 500-event segments (E=501, K~290), flags 0; --reads per GPU (default
10000 => ~60k jobs, 3.0e7 scored events per step).  One "step" = one pass of the forward kernel over
the whole resident batch.  Weak scaling: every rank owns its own --reads reads (seeded by rank) and
the per-job scores are gathered to rank 0 with one NCCL gather per step.

JSON line keys follow the driver's contract; see DESIGN.md "Measurement" for what each means here.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "hmm_scored_events_per_sec"
UNIT = "events/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="scorereads",
                    choices=["scorereads", "methylation", "call_methylation", "variants", "abea", "events", "prologue", "eventalign"])
    ap.add_argument("--region", type=int, default=200000, help="--workload variants: reference positions per GPU (50x coverage by 2300-base reads)")
    ap.add_argument("--meth-reads", type=int, default=0,
                    help="reads per GPU of the call-methylation block (default 10000 at N=1; 12500 at N>1 = BASELINE configs[2]'s 100k reads at N=8)")
    ap.add_argument("--no-call-methylation", action="store_true", help="skip the configs.call_methylation block of the default line")
    ap.add_argument("--reads", type=int, default=10000, help="reads per GPU")
    ap.add_argument("--events", type=int, default=4000, help="events per read")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the per-job scores of the last step to DIR/scores.npy (float32, job order; "
                         "every rank's jobs in rank order at --gpus N), so that two builds can be compared on identical inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "scorereads" or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of the default workload (--workload scorereads, --impl ours)")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_quota():
    """CPUs' worth of time the container may use (cgroup v2 cpu.max / v1 cfs quota), or None when unlimited/unknown.
    The GPU boxes expose 128 logical CPUs under a 16-CPU quota: the CPU arm runs that many threads on that much time."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / per
    except Exception:
        return None


def cpu_threads():
    """Threads for the CPU arm: every logical CPU, unless a cgroup quota makes that oversubscription — measured on the
    B200 boxes (profiles/r01_cpu_threads.json): 128 threads under a 16-CPU quota run the reference 28 % slower than 32.
    Twice the quota is the fastest setting there, so that is what the reference gets."""
    n = os.cpu_count() or 1
    q = cpu_quota()
    return n if not q else max(1, min(n, int(round(2 * q))))


class ClockSampler:
    """nvidia-smi sampled every 200 ms DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.proc = None
        self.lines = []
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()          # the exact PID we started
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        sm, smmax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smmax = float(f[2])
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smmax,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_workload(args, rank):
    from nanopolish_b200 import synth
    nuc = synth.load_model("nucleotide")
    models = [nuc]
    seed = 42 + 1_000_003 * rank
    if args.workload == "scorereads":
        rs = synth.gen_reads(args.reads, args.events, nuc, seed=seed)
        jobs = synth.scorereads_jobs(rs, 500, model_id=0)
    else:
        cpg = synth.load_model("cpg")
        models.append(cpg)
        rs = synth.gen_reads(args.reads, args.events, nuc, seed=seed, cpg_keep=0.3)
        jobs = synth.methylation_jobs(rs, model_id=1)
    return rs, jobs, models


def k1_rooflines(args, jobs, kernel_ms, clocks):
    """The two rooflines that do bound K1 (DESIGN.md section 3.4), from MEASURED counters: profiles/r02_k1_counters.json holds ncu's executed
    warp instructions and shared-memory wavefronts of one pass of the forward kernels over this workload (same reads, same job list);
    per block-cell they do not depend on the clock, so the live kernel time turns them into rates.
      issue : warp instructions per second against 148 SMs x 4 schedulers x SM clock
      shared: shared-memory wavefronts per second against 148 SMs x 1 wavefront per clock (the table look-ups replay on bank conflicts)"""
    out = {}
    try:
        c = json.load(open(os.path.join(ROOT, "profiles", "r02_k1_counters.json"))).get(args.workload)
    except Exception:
        c = None
    clk = ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
    if c and c.get("reads") == args.reads and args.events == 4000:
        inst_per_cell = c["inst_executed"] * 32.0 / float(jobs.block_cells)       # lane-instructions per block-cell, as ncu counted them
        issue = c["inst_executed"] / (kernel_ms * 1e-3)
        shared = c["lds_wavefronts"] / (kernel_ms * 1e-3)
        out["issue"] = {"achieved": issue, "unit": "warp-instructions/s", "peak": 148 * 4 * clk, "frac": issue / (148 * 4 * clk),
                        "instructions_per_block_cell": inst_per_cell, "source": "measured: smsp__inst_executed (profiles/r02_k1_counters.json) / live kernel time"}
        out["shared_memory"] = {"achieved": shared, "unit": "wavefronts/s", "peak": 148 * clk, "frac": shared / (148 * clk),
                                "bank_conflict_share": c["lds_conflict_wavefronts"] / c["lds_wavefronts"],
                                "source": "measured: l1tex__data_pipe_lsu_wavefronts_mem_shared / live kernel time"}
        if c.get("dram_bytes"):
            out["traffic"] = c["dram_bytes"]
    return out


def algorithmic_bytes(jobs, k=6):
    """SURVEY.md 8(d): B_alg = 4*E + L + 36 bytes per job (event levels as f32, base codes, job record, score)."""
    j = jobs.jobs
    E = np.abs(j["event_stop"].astype(np.int64) - j["event_start"].astype(np.int64)) + 1
    L = j["n_kmers"].astype(np.int64) + (k - 1)
    return int((4 * E + L + 36).sum())


class CpuArm:
    """The reference's CPU path (oracle/_ref when it was compiled, else the plain-C port) over a bounded
    sample of the same job list, OpenMP over jobs with all host threads — the way the reference
    parallelises over reads (src/common/nanopolish_bam_processor.cpp:99)."""

    def __init__(self, rs, jobs, models, want_ref=True):
        from oracle.oracle_py import PortOracle, RefOracle
        self.rs, self.jobs, self.models = rs, jobs, models
        self.cores = cpu_threads()
        j = jobs.jobs
        self.E = np.abs(j["event_stop"].astype(np.int64) - j["event_start"].astype(np.int64)) + 1
        self.cells = self.E * j["n_kmers"].astype(np.int64)
        self.use_ref = want_ref and RefOracle.available()
        if self.use_ref:
            self.ref = RefOracle()
            self.mh = [self.ref.builtin_model(m.alphabet) for m in models]
            max_read = int(min(rs.n_reads, 2048))      # only reads the bounded sample can touch
            self.rh = self.ref.register_reads(rs.reads[:max_read], rs.ev_mean, rs.ev_start_time, self.mh[0])
            self.eligible = np.flatnonzero(j["read"] < max_read)
        else:
            self.port = PortOracle()
            self.eligible = np.arange(j.shape[0])
        self._seq_cache = {}

    def _seq(self, jb):
        """the harness takes sequences as strings: rebuild one from the job's forward k-mer ranks"""
        key = int(jb["rank_off"])
        if key not in self._seq_cache:
            r = self.jobs.kmer_ranks[key:key + int(jb["n_kmers"])]
            asz = self.models[int(jb["model_id"])].alphabet_size
            first = [(int(r[0]) // asz ** (5 - i)) % asz for i in range(6)]
            alpha = b"ACGT" if asz == 4 else b"ACGMT"
            self._seq_cache[key] = bytes(alpha[c] for c in first + (r[1:] % asz).tolist())
        return self._seq_cache[key]

    def time(self, idx):
        sub = np.ascontiguousarray(self.jobs.jobs[idx])
        if self.use_ref:
            seqs = [self._seq(jb) for jb in sub]
            _, secs = self.ref.score_batch(self.rh, sub, seqs, self.mh, threads=self.cores)
        else:
            _, secs = self.port.hmm_score_batch(self.rs.reads, self.rs.ev_mean, self.rs.ev_start_time, self.models,
                                                self.jobs.kmer_ranks, sub, threads=self.cores)
        return secs

    def sample_for(self, seconds_target):
        cal = self.eligible[:max(2 * self.cores, 16)]
        t_cal = self.time(cal)
        rate = self.cells[cal].sum() / max(t_cal, 1e-6)
        csum = np.cumsum(self.cells[self.eligible])
        m = int(np.searchsorted(csum, rate * seconds_target)) + 1
        return self.eligible[:min(m, self.eligible.shape[0])]

    def report(self, idx, secs):
        ev = int(self.E[idx].sum())
        return {"value": ev / secs, "unit": UNIT, "cores": self.cores, "cpu_quota": cpu_quota(),
                "kind": "reference" if self.use_ref else "port",
                "sample": f"{idx.shape[0]} jobs ({ev} scored events, {int(self.cells[idx].sum())} block-cells) of the "
                          f"same job list, {secs:.2f} s per pass, OpenMP over jobs with {self.cores} threads",
                "block_cells_per_sec": float(self.cells[idx].sum() / secs)}


def run_reference(args, rank, world, saved_stdout):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores.
    Rank 0 alone runs it; each step is one pass over a bounded sample of the workload's job list."""
    if rank != 0:
        return
    # rank 0's full job list of the own arm (same generator, same seed): the sample is drawn from it, and `config` is the own arm's
    rs, jobs, models = build_workload(args, 0)
    arm = CpuArm(rs, jobs, models)
    steps, warm = args.steps, args.warmup
    per_step = max(0.5, min(6.0, 120.0 / max(1, steps + warm)))   # whole run within a few minutes
    idx = arm.sample_for(per_step)
    for _ in range(warm):
        arm.time(idx)
    secs = [arm.time(idx) for _ in range(steps)]
    mean_s = float(np.mean(secs))
    base = arm.report(idx, mean_s)
    full = argparse.Namespace(**vars(args))
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": mean_s * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {**workload_config(full, jobs), "jobs_per_gpu": int(jobs.jobs.shape[0]),
                       "scored_events_per_step": float(jobs.scored_events) * args.gpus},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line, saved_stdout)


def workload_config(args, jobs, reads_override=None):
    j = jobs.jobs
    E = np.abs(j["event_stop"].astype(np.int64) - j["event_start"].astype(np.int64)) + 1
    return {"workload": f"{args.workload}: synthetic R9.4 reads x {args.events} events, k=6 r9.4_450bps "
                        + ("nucleotide model, 500-event segments, flags 0" if args.workload == "scorereads"
                           else "cpg model, CpG-group windows u/m pairs, flags PRE|POST"),
            "reads_per_gpu": reads_override or args.reads, "events_per_read": args.events,
            "mean_E": float(E.mean()), "mean_K": float(j["n_kmers"].mean()),
            "parallelism": f"read-shard x{args.gpus}", "l2": "inputs larger than L2 (levels+ranks+scratch > 126 MB)"}


# ------------------------------------------------------------------------------------------------------------------
# call-methylation end to end (BASELINE.json's metric names this caller; configs[2]): reference bases + event
# alignments in, per-site log-likelihood pairs / TSV rows out — enumeration, scheduling and scoring all on the device.
# ------------------------------------------------------------------------------------------------------------------
class _DevBytes:
    """zero-copy view of device memory for torch (CUDA array interface)"""
    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def call_methylation_block(args, rank, world, local, steps, warmup):
    """One step = nph_methylation_run over the resident batch (motif scan, grouping, event bounds, k-mer ranks, schedule,
    both forward scores per group, site records) and, at N > 1, ONE variable-length NCCL gather of the site records to
    rank 0 straight from device memory.  e2e = the C++ host's flat entry (libnph_host.so nphh_call_methylation_flat): page-locked
    host buffers in, methylation_calls.tsv bytes out, plus at N > 1 the gather of the TSV bytes to rank 0."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from nanopolish_b200 import synth
    from nanopolish_b200.dist import gather_records_to_rank0, gather_to_rank0
    from nanopolish_b200.engine import Engine

    dev = torch.device("cuda", local)
    n_reads = args.meth_reads or (10000 if world == 1 else 12500)
    nuc, cpg = synth.load_model("nucleotide"), synth.load_model("cpg")
    rs = synth.gen_reads(n_reads, args.events, nuc, seed=7_000_003 + 1_000_003 * rank, cpg_keep=0.3)
    ref, pairs, recs = synth.methylation_records(rs, model_id=1, rc_every=2)
    params = synth.meth_params("cpg", 6)
    stream = torch.cuda.current_stream().cuda_stream
    eng = Engine(local, stream=stream)
    eng.model_upload(nuc); eng.model_upload(cpg)

    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).pin_memory()
        return t, t.numpy().view(a.dtype).reshape(a.shape)
    keep = []
    def P(a):
        t, v = pin(a); keep.append(t); return v
    deltas, first_event = synth.compact_event_alignment(recs, pairs, ref.shape[0])       # 2 B per reference base instead of 8 B per pair
    h_reads, h_mean, h_ref, h_recs = P(rs.reads), P(rs.ev_mean), P(ref), P(recs)
    h_deltas, h_first = P(deltas), P(first_event)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm ----
    eng.reads_load(h_reads, h_mean, rs.ev_start_time)
    eng.methylation_load_compact(h_ref, h_deltas, h_first, h_recs, params)

    def step():
        eng.methylation_run()
        if world > 1:
            ptr, n = eng.methylation_sites_dev()
            raw = torch.as_tensor(_DevBytes(ptr, max(n, 1) * 24), device=dev)[:n * 24]
            return gather_to_rank0(raw, None)           # tiny all_gather of the byte counts + ONE padded NCCL gather
        return None

    for _ in range(max(3, warmup)):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        gathered = step()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    n_sites, n_jobs, scored = eng.methylation_counts()
    kern = []
    for _ in range(5):
        eng.methylation_run(); eng.sync(); kern.append(eng.last_kernel_ms())
    kernel_ms, launches = float(np.mean([k[0] for k in kern])), int(kern[-1][1])
    site_off, sites = eng.methylation_fetch()
    tot = torch.tensor([float(scored), float(n_sites), float(n_reads)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot)
        if rank == 0:
            assert sum(int(g.shape[0]) for g in gathered) == int(tot[1].item()) * 24, "gathered site records"
    scored_all, sites_all, reads_all = (float(x) for x in tot.tolist())
    value = scored_all * steps / (total_ms * 1e-3)

    # ---- e2e arm: host buffers -> TSV bytes through the C++ host ----
    os.environ["NPH_DEVICE"] = str(local)
    # the C++ host formats rows with an OpenMP team; torchrun exports OMP_NUM_THREADS=1 to every rank, which would serialise it
    # (measured at N=2: 44 ms of TSV instead of 7) — each rank takes its share of the box's CPUs, as a multi-GPU caller would set it
    host_threads = max(1, min(32, cpu_threads() // max(1, world)))
    os.environ.setdefault("NPH_HOST_THREADS", str(host_threads))
    host = C.CDLL(os.path.join(ROOT, "nanopolish_b200", "libnph_host.so"))
    host.nphh_last_error.restype = C.c_char_p
    host.nphh_call_methylation_flat.restype = C.c_longlong
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    cm = np.ascontiguousarray(cpg.level_mean); cs = np.ascontiguousarray(cpg.level_stdv); cl = np.ascontiguousarray(cpg.level_log_stdv)
    mh = host.nphh_model_create(b"cpg", 6, cm.shape[0], vp(cm), vp(cs), vp(cl))
    names = (C.c_char_p * n_reads)(*[f"read_{rank}_{i}".encode() for i in range(n_reads)])
    is_rev = np.ascontiguousarray(recs["rc"])
    cap = 128 * int(n_sites) + 4096
    t_tsv = torch.empty(cap, dtype=torch.uint8).pin_memory(); keep.append(t_tsv)
    tsv = t_tsv.numpy()
    secs2 = np.zeros(2)
    ns, se = C.c_uint64(), C.c_uint64()

    from nanopolish_b200.dist import ByteGather
    tsv_gather = None
    if world > 1:
        cap_t = torch.tensor([cap], dtype=torch.int64, device=dev)
        dist.all_reduce(cap_t, op=dist.ReduceOp.MAX)
        tsv_gather = ByteGather(int(cap_t.item()), device=dev)            # page-locked staging, allocated once

    def e2e_step():
        n = host.nphh_call_methylation_flat(vp(h_reads), C.c_size_t(n_reads), vp(h_mean), None, C.c_size_t(h_mean.shape[0]),
                                            vp(h_ref), C.c_size_t(h_ref.shape[0]), None, C.c_size_t(0), vp(h_deltas), vp(h_first),
                                            vp(h_recs), C.c_size_t(n_reads), mh, names, vp(is_rev), b"chr1", C.c_double(1.0),
                                            vp(tsv), C.c_size_t(cap), C.byref(ns), C.byref(se), vp(secs2))
        if n < 0:
            raise RuntimeError("nphh_call_methylation_flat: " + host.nphh_last_error().decode())
        if world > 1:
            tsv_gather.gather(t_tsv, int(n))
        return int(n)

    for _ in range(2):
        tsv_bytes = e2e_step()
    barrier()
    e2e_steps = steps
    stage = np.zeros(2)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        tsv_bytes = e2e_step(); stage += secs2
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    assert int(ns.value) == n_sites and int(se.value) == scored
    h2d = h_reads.nbytes + h_mean.nbytes + h_ref.nbytes + h_deltas.nbytes + h_first.nbytes + h_recs.nbytes + 8 * (n_reads + 1) + 8 * n_reads
    device_tsv = not os.environ.get("NPH_METH_HOST_TSV")
    # rows formatted on the device (nph_methylation_batch_compact_tsv): the TSV bytes are what comes back; with the host formatter the
    # 24-byte site records and their offsets do
    d2h = (tsv_bytes + 16) if device_tsv else (24 * n_sites + 8 * (n_reads + 1) + 64)

    out = None
    if rank == 0:
        peak, peak_src = peaks()
        # algorithmic bytes of the forward kernels (SURVEY.md 8d: 4E + L + 36 per job); L from the site records
        span = (sites["end_position"].astype(np.int64) - sites["start_position"].astype(np.int64)) + 21
        b_alg = 4 * scored + 2 * int(span.sum()) + 36 * n_jobs
        achieved = b_alg / (kernel_ms * 1e-3) / 1e9
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": max(3, warmup),
               "ms_per_step": total_ms / steps, "scaling": "weak", "dtype": "f32", "data": "synthetic",
               "config": {"workload": f"call-methylation: synthetic R9.4 reads x {args.events} events aligned to their own sequence (CIGAR all M, half "
                                      "the records reverse strand; event alignments in the 2 B/base compact form), CpG groups ~60 bp apart, cpg model (5^6 states), PRE|POST clip; motif scan, "
                                      "grouping, event bounds, k-mer ranks, scheduling and both scores per group on the device",
                          "reads_per_gpu": n_reads, "reads_total": reads_all, "events_per_read": args.events, "sites_per_step": sites_all,
                          "jobs_per_gpu": n_jobs, "scored_events_per_step": scored_all, "parallelism": f"read-shard x{world}",
                          "multi_gpu": "one variable-length NCCL gather of the 24-byte site records to rank 0 per step" if world > 1 else None,
                          "l2": "inputs larger than L2 (levels + event alignments + reference > 126 MB)"},
               "e2e": {"value": scored_all * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                       "steps": e2e_steps, "tsv_bytes_per_step": tsv_bytes, "ms_per_step": e2e_s / e2e_steps * 1e3,
                       "stage_ms": {"device_call": float(stage[0] / e2e_steps * 1e3), "host_side": float(stage[1] / e2e_steps * 1e3)},
                       "rows_formatted_on": "device (nph_methylation_tsv)" if device_tsv else "host (OpenMP formatter)",
                       "host_threads_per_rank": int(os.environ["NPH_HOST_THREADS"]),
                       "api": "libnph_host.so nphh_call_methylation_flat (nph::call_methylation_flat: page-locked host buffers in, TSV bytes out"
                              + ("; TSV bytes gathered to rank 0 over NCCL)" if world > 1 else ")")},
               "gpu_launches": launches * steps,
               "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                            "peak_source": peak_src, "kernel": "hmm_forward_kernel<C,4..32> over the enumerated windows", "kernel_ms": kernel_ms,
                            "algorithmic_bytes_per_step": int(b_alg),
                            "note": "kernel_ms = the forward kernels alone (CUDA events around them); the step also holds the enumeration, the "
                                    "schedule and two small read-backs, see ms_per_step"}}
        if world == 1 and not args.no_cpu_baseline:
            try:
                out["cpu_baseline"] = call_methylation_cpu(rs, recs, ref, pairs, site_off, sites, tsv[:tsv_bytes].tobytes().decode())
            except Exception as ex:
                out["cpu_baseline"] = {"value": None, "unit": UNIT, "kind": "unavailable", "sample": f"failed: {ex}"}
    eng.close()
    return out


def call_methylation_cpu(rs, recs, ref, pairs, site_off, sites, tsv_ours):
    """The compiled reference's own calculate_methylation_for_read + write_methylation_results_as_tsv over a bounded sample of the
    same reads, one read per thread like the reference's OpenMP loop; its rows must equal ours for those reads."""
    from concurrent.futures import ThreadPoolExecutor
    from nanopolish_b200 import synth
    from oracle.oracle_py import RefOracle
    if not RefOracle.available():
        raise RuntimeError("oracle/_ref/libnpref.so not present")
    ro = RefOracle()
    cores = cpu_threads()
    ns = int(min(rs.n_reads, max(4 * cores, 128)))
    mh = ro.builtin_model("nucleotide"); ro.builtin_model("cpg")
    rh = ro.register_reads(rs.reads[:ns], rs.ev_mean, rs.ev_start_time, mh)
    k = rs.k
    inputs = []
    for i in range(ns):
        codes = rs.seq_codes[i]
        nk = codes.shape[0] - k + 1
        st, sp, _ = synth.closest_event_map(rs.ev_kmer[i], nk)
        seq = synth._CODE2DNA[codes].tobytes().decode()
        one = np.ones(int(rs.reads[i]["n_events"]), np.float32)
        ro.read_set_eventalign(rh[i], f"read_0_{i}", seq, st, sp, one, one)
        R = recs[i]
        contig = "A" * int(R["ref_start_pos"]) + ref[int(R["ref_off"]):int(R["ref_off"]) + int(R["ref_len"])].tobytes().decode()
        inputs.append((contig, int(R["ref_start_pos"]), 16 if R["rc"] else 0, np.array([(len(seq) << 4) | 0], np.uint32)))
    def one_read(i):
        c = inputs[i]
        return ro.call_methylation(rh[i], f"read_0_{i}", "chr1", c[0], c[1], c[2], c[3])[0]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(cores) as ex:                  # the compiled reference releases the GIL inside each call
        rows = list(ex.map(one_read, range(ns)))
    secs = time.perf_counter() - t0
    # same rows as ours for these reads
    ours = tsv_ours.split("\n")
    cut = int(site_off[ns])
    assert "".join(rows) == "".join(x + "\n" for x in ours[:cut]), "reference TSV differs from ours on the sampled reads"
    # scored events of the sample: both jobs of a site walk the events between the two lower_bounds of its window
    ev = 0
    for i in range(ns):
        R = recs[i]
        pr = pairs[int(R["pair_off"]):int(R["pair_off"]) + int(R["n_pairs"])]
        s_ = sites[int(site_off[i]):int(site_off[i + 1])]
        a = np.searchsorted(pr["ref_pos"], s_["start_position"] - 10)
        b = np.searchsorted(pr["ref_pos"], s_["end_position"] + 10)
        ev += int((2 * (np.abs(pr["read_pos"][b].astype(np.int64) - pr["read_pos"][a].astype(np.int64)) + 1)).sum())
    return {"value": ev / secs, "unit": UNIT, "cores": cores, "cpu_quota": cpu_quota(), "kind": "reference", "seconds": secs, "sample_sites": cut,
            "sample": f"{ns} of the reads through the compiled reference's calculate_methylation_for_read + TSV writer, one read per thread "
                      f"({cores} threads), {cut} sites, rows identical to ours"}


# ------------------------------------------------------------------------------------------------------------------
# variants --consensus candidate screening (BASELINE configs[4]): every single-base edit of every position of a region scored
# against the pile-up with the reference's early-exit rule; enumeration, rounds and accumulation on the device.
# ------------------------------------------------------------------------------------------------------------------
def variants_block(args, rank, world, local, steps, warmup):
    """One step = nph_screen_run over the resident pile-up (windows' event sequences, edited-window ranks, rounds of
    reads_per_round reads with the early exit applied between rounds, qualities) + fetch of the 9 qualities per position; at N > 1
    the region is cut into one slice per rank (positions are independent: no data-path collective) and the slices' qualities are
    gathered to rank 0 with one NCCL gather.  Unit: the DP rows the reference's own loop scores for the same result (base and
    variant sequence per candidate and read until its total leaves the threshold), so that our rate and the CPU arm's are
    comparable; `our_dp_rows` is what the device actually ran (the base haplotype once per read and round, not once per candidate)."""
    import torch
    import torch.distributed as dist
    from nanopolish_b200 import synth
    from nanopolish_b200.dist import gather_to_rank0
    from nanopolish_b200.engine import Engine

    dev = torch.device("cuda", local)
    nuc = synth.load_model("nucleotide")
    region_start = 1_000_000 + rank * args.region
    ref, rs, recs, pairs = synth.gen_pileup(args.region, 50, 2300, nuc, seed=424_243 + rank, region_start=region_start,
                                            n_true_variants=max(1, args.region // 2000))
    deltas, first = synth.compact_event_alignment(recs, pairs, int(recs["ref_len"].sum()))
    ref_chars = synth._CODE2DNA[ref]
    params = synth.screen_params(region_start, 6, 10, 100, 3, 8)
    indel_bias = 0.9                                   # nanopolish variants' hmm_indel_bias_factor for the screening pass
    eng = Engine(local, stream=torch.cuda.current_stream().cuda_stream)
    eng.model_upload(nuc)
    keep = []
    def P(a):
        t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).pin_memory(); keep.append(t)
        return t.numpy().view(a.dtype).reshape(a.shape)
    h_reads, h_mean, h_ref, h_deltas, h_first, h_recs = P(rs.reads), P(rs.ev_mean), P(ref_chars), P(deltas), P(first), P(recs)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng.reads_load(h_reads, h_mean, rs.ev_start_time)
    eng.screen_load(h_ref, h_deltas, h_first, h_recs, params, indel_bias)

    def step():
        eng.screen_run()
        q, nr = eng.screen_fetch()
        if world > 1:
            gather_to_rank0(torch.from_numpy(q.reshape(-1)).to(dev), None)
        return q, nr

    for _ in range(max(3, warmup)):
        q, nr = step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    kms = []
    for _ in range(steps):
        q, nr = step(); kms.append(eng.last_kernel_ms())
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    cnt = eng.screen_counts()
    kernel_ms, launches = float(np.mean([k[0] for k in kms])), int(kms[-1][1])
    tot = torch.tensor([float(cnt["reference_events"]), float(cnt["scored_events"]), float(cnt["jobs"]), float(cnt["jobs_without_exit"])],
                       dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot)
    ref_events_all, our_rows_all, jobs_all, jobs_noexit_all = (float(x) for x in tot.tolist())
    value = ref_events_all * steps / (total_ms * 1e-3)

    # ---- e2e: the one-shot call with host buffers (events, reference, compact event alignments up; qualities back) ----
    def e2e_step():
        return eng.screen_edits_batch(h_reads, h_mean, rs.ev_start_time, h_ref, h_deltas, h_first, h_recs, params, indel_bias)
    for _ in range(2):
        e2e_step()
    barrier()
    e2e_steps = steps
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        q2, nr2, _ = e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    assert np.array_equal(np.nan_to_num(q, nan=-1e300), np.nan_to_num(q2, nan=-1e300))
    h2d = h_reads.nbytes + h_mean.nbytes + h_ref.nbytes + h_deltas.nbytes + h_first.nbytes + h_recs.nbytes
    d2h = q.nbytes + nr.nbytes

    out = None
    if rank == 0:
        peak, peak_src = peaks()
        b_alg = 4 * cnt["scored_events"] + (22 + 36) * cnt["jobs"]          # SURVEY.md 8d per job: 4E + L + 36
        achieved = b_alg / (kernel_ms * 1e-3) / 1e9
        n_pos_q = int((~np.isnan(q)).any(axis=1).sum())
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": max(3, warmup),
               "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": {"workload": f"variants --consensus candidate screening: {args.region} reference positions per GPU, 50x coverage by 2300-base "
                                      "reads (~4000 events) aligned base for base, up to 9 single-base edits per position, 22-base windows, "
                                      "threshold 100, PRE|POST clip, indel bias 0.9; reads scored 8 at a time with the early exit applied between rounds",
                          "positions_per_gpu": args.region, "positions_screened": n_pos_q, "reads_per_gpu": int(rs.n_reads),
                          "mean_event_sequences_per_position": float(nr.mean()), "rounds": cnt["rounds"],
                          "unit_definition": "DP rows the reference's loop scores for the same qualities (2 sequences per candidate and read until exit)",
                          "reference_dp_rows_per_step": ref_events_all, "our_dp_rows_per_step": our_rows_all, "jobs_per_step": jobs_all,
                          "jobs_without_early_exit": jobs_noexit_all, "parallelism": f"region-slice x{world}",
                          "multi_gpu": "positions are independent: one region slice per rank, one NCCL gather of the qualities" if world > 1 else None,
                          "l2": "inputs larger than L2 (events + rank pool > 126 MB)"},
               "e2e": {"value": ref_events_all * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                       "steps": e2e_steps, "ms_per_step": e2e_s / e2e_steps * 1e3, "api": "nph_screen_edits_batch (host buffers in, qualities out)"},
               "gpu_launches": launches * steps,
               "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                            "peak_source": peak_src, "kernel": "hmm_forward_kernel<C,4> over the rounds' jobs", "kernel_ms": kernel_ms,
                            "algorithmic_bytes_per_step": int(b_alg),
                            "note": "kernel_ms = the forward kernels of all rounds (CUDA events around each); the step also holds the window / rank / "
                                    "job kernels and two read-backs per round"}}
        if world == 1 and not args.no_cpu_baseline:
            try:
                eng.screen_run()
                _, _, ref_rows = eng.screen_fetch(with_reference_rows=True)
                out["cpu_baseline"] = variants_cpu(rs, recs, pairs, ref_chars, region_start, q, ref_rows, indel_bias)
            except Exception as ex:
                out["cpu_baseline"] = {"value": None, "unit": UNIT, "kind": "unavailable", "sample": f"failed: {type(ex).__name__}: {ex}"}
    eng.close()
    return out


def variants_cpu(rs, recs, pairs, ref_chars, region_start, q_ours, ref_rows, indel_bias):
    """The compiled reference's score_variant_thresholded for every candidate of a bounded sample of positions (one position per
    thread, each call single-threaded so that its early exit follows read order); the qualities must equal ours exactly."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle.oracle_py import RefOracle
    from tests import var_restatement as vr
    if not RefOracle.available():
        raise RuntimeError("oracle/_ref/libnpref.so not present")
    ro = RefOracle()
    cores = cpu_threads()
    ref_s = ref_chars.tobytes().decode()
    n_pos = len(ref_s) - 1
    # positions inside the first 40 kb (only the reads that can reach them are registered with the harness)
    span = min(n_pos, 40_000)
    sel = np.flatnonzero(recs["ref_start_pos"] - region_start < span + 64)
    ro.clear_reads()
    rh = ro.register_reads(rs.reads[:int(sel.max()) + 1], rs.ev_mean, rs.ev_start_time, ro.builtin_model("nucleotide"))
    sub_recs = recs[:int(sel.max()) + 1]
    sample = list(range(2000, span - 200, max(1, (span - 2200) // max(64, 24 * cores))))
    work = []
    for pi in sample:
        i = region_start + pi
        cs, ce = i - 10, i + 11
        seqs = vr.event_sequences(sub_recs, pairs, cs, ce)
        cands = vr.candidates(ref_s, pi)
        work.append((pi, cs, seqs, cands, ref_s[cs - region_start:ce - region_start + 1]))
    def one(w):
        pi, cs, seqs, cands, window = w
        return ro.score_variants_thresholded([rh[r] for r, _, _ in seqs], [(e1, e2) for _, e1, e2 in seqs],
                                             np.array([sub_recs[r]["rc"] for r, _, _ in seqs], np.uint8), window, cs,
                                             [(region_start + off, a, b) for _, off, a, b in cands], 3, 100, False, indel_bias=indel_bias)
    ro.set_globals(indel_bias, 1)          # the calls below run concurrently: each must find the globals it sets already in place
    one(work[0])
    t0 = time.perf_counter()
    with ThreadPoolExecutor(cores) as ex:
        got = list(ex.map(one, work))
    secs = time.perf_counter() - t0
    ro.set_globals(1.0, cores)
    same = True
    for (pi, cs, seqs, cands, window), g in zip(work, got):
        for (slot, _, _, _), v in zip(cands, g):
            same &= float(q_ours[pi, slot]) == float(v)
    # identical qualities mean identical exit points, so the DP rows the reference scored at these positions are the device's
    # per-position account of the reference's loop (nph_screen_fetch: reference_rows)
    rows = int(ref_rows[[w[0] for w in work]].sum())
    ro.clear_reads()
    return {"value": rows / secs, "unit": UNIT, "cores": cores, "cpu_quota": cpu_quota(), "kind": "reference", "seconds": secs, "positions": len(work),
            "candidates": int(sum(len(w[3]) for w in work)), "qualities_identical": bool(same), "dp_rows": rows,
            "sample": f"{len(work)} positions ({sum(len(w[3]) for w in work)} candidates) through the compiled reference's score_variant_thresholded, "
                      f"one position per thread ({cores} threads), each call single-threaded"}


def run_aux(args, rank, world, local, saved_stdout):
    """Auxiliary single-GPU measurements of the other kernels of the path (not the headline metric):
    --workload abea   : adaptive banded event alignment, reads x 8000 events (BASELINE configs[3] shape), events/s
    --workload events : scrappie event detection, reads x 36000 raw samples, samples/s
    --workload prologue : SquiggleRead::load_from_raw in one call (trim, events, MoM, ABEA, calibration), samples/s
    --workload eventalign : eventalign's segment chains (align_read_to_ref) walked on the device, reads x 4000 events, events/s"""
    if rank != 0:
        return
    import torch
    from nanopolish_b200 import synth
    from nanopolish_b200.engine import Engine
    nuc = synth.load_model("nucleotide")
    eng = Engine(local)
    mid = eng.model_upload(nuc)
    peak, peak_src = peaks()
    if args.workload == "abea":
        n_reads = min(args.reads, 4736)
        rs = synth.gen_reads(n_reads, 8000, nuc, seed=42, rng_scalings=False)
        jobs, ranks, total = synth.abea_jobs(rs)
        eng.reads_load(rs.reads, rs.ev_mean, rs.ev_start_time)
        eng.abea_jobs_load(ranks, jobs, mid, total)
        for _ in range(max(3, args.warmup)):
            eng.abea_run()
        eng.sync()
        ms = []
        for _ in range(args.steps):
            eng.abea_run(); eng.sync(); ms.append(eng.last_kernel_ms()[0])
        t = float(np.mean(ms))
        ev = int(rs.reads["n_events"].sum())
        b_alg = int((12 * rs.reads["n_events"].astype(np.int64) + 50 * (rs.reads["n_events"].astype(np.int64) + jobs["n_kmers"])).sum())
        t0 = time.perf_counter(); eng.abea_batch(rs.reads, rs.ev_mean, rs.ev_start_time, ranks, jobs, mid, total); e2e_s = time.perf_counter() - t0
        line = {"metric": "abea_events_per_sec", "value": ev / (t * 1e-3), "unit": "events/s", "n_gpus": 1, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": t, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32+f64", "data": "synthetic",
                "config": {"workload": f"abea: {n_reads} synthetic R9.4 reads x 8000 events, k=6 nucleotide model, band 100"},
                "e2e": {"value": ev / e2e_s, "unit": "events/s", "h2d_bytes_per_step": int(rs.ev_mean.nbytes + ranks.nbytes + jobs.nbytes),
                        "d2h_bytes_per_step": int(total * 8), "steps": 1, "api": "nph_abea_batch"},
                "gpu_launches": args.steps,
                "roofline": {"bound": "hbm", "achieved": b_alg / (t * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": b_alg / (t * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src, "kernel": "abea_kernel",
                             "note": "sequentially dependent bands: issue/latency bound (DESIGN.md section 5)"}}
        if not args.no_cpu_baseline:
            # the compiled reference's adaptive_banded_simple_event_align over a bounded sample of the same reads, OpenMP over reads
            from oracle.oracle_py import RefOracle
            if RefOracle.available():
                ro = RefOracle()
                cores = cpu_threads()
                ns = int(min(n_reads, max(2 * cores, 64)))
                h = ro.builtin_model("nucleotide")
                rh = ro.register_reads(rs.reads[:ns], rs.ev_mean, rs.ev_start_time, h)
                seqs = [synth._CODE2DNA[c].tobytes() for c in rs.seq_codes[:ns]]
                caps = [int(j["pairs_cap"]) for j in jobs[:ns]]
                ro.abea_batch(rh[:8], h, seqs[:8], caps[:8], threads=cores)
                pr, poff, npairs, secs = ro.abea_batch(rh, h, seqs, caps, threads=cores)
                pg, rg = eng.abea_fetch()
                same = all(int(npairs[i]) == int(rg[i]["n_pairs"]) for i in range(ns))
                line["cpu_baseline"] = {"value": int(rs.reads["n_events"][:ns].sum()) / secs, "unit": "events/s", "cores": cores, "cpu_quota": cpu_quota(),
                                        "kind": "reference", "seconds": secs, "same_pair_counts": bool(same),
                                        "sample": f"{ns} of the {n_reads} reads through the compiled reference's adaptive_banded_simple_event_align, "
                                                  f"OpenMP over reads with {cores} threads"}
    elif args.workload == "eventalign":
        n_reads = min(args.reads, 4736)
        rs = synth.gen_reads(n_reads, args.events, nuc, seed=42)
        pairs, maps, rf, rr, chains = synth.eventalign_chains(rs, mid)
        ev = int(rs.reads["n_events"].sum())
        # page-locked host buffers, like a caller staging a batch
        def pin(a):
            t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).pin_memory()
            return t.numpy().view(a.dtype).reshape(a.shape)
        ev_mean, pairs, maps, rf, rr, chains_p = pin(rs.ev_mean), pin(pairs), pin(maps), pin(rf), pin(rr), pin(chains)
        total_rec = int((chains["out_off"] + chains["out_cap"]).max())
        out = (pin(np.zeros(total_rec, synth.EA_RECORD_DT)), pin(np.zeros(n_reads, synth.EA_RESULT_DT)))
        chains = chains_p
        ms, e2e = [], []
        for it in range(max(3, args.warmup) + args.steps):
            t0 = time.perf_counter()
            eng.reads_load(rs.reads, ev_mean, rs.ev_start_time)
            records, results = eng.eventalign_chain(pairs, maps, rf, rr, chains, out=out)
            dt = time.perf_counter() - t0
            if it >= max(3, args.warmup):
                ms.append(eng.last_kernel_ms()[0]); e2e.append(dt)
        t = float(np.mean(ms))
        assert (results["status"] == 0).all()
        n_rec, n_win = int(results["n_records"].sum()), int(results["n_windows"].sum())
        # algorithmic bytes: event levels once (4 B), pairs (8 B) + map (4 B) + two rank tables (8 B) per k-mer, 12 B per record out
        nk_total = int(chains["n_pairs"].sum())
        b_alg = 4 * ev + 20 * nk_total + 12 * n_rec
        cpu = None
        if not args.no_cpu_baseline:
            from concurrent.futures import ThreadPoolExecutor
            from oracle.oracle_py import RefOracle
            if RefOracle.available():
                ro = RefOracle()
                cores = cpu_threads()
                ns = min(n_reads, max(cores, 32) * 2)
                rh = ro.register_reads(rs.reads[:ns], rs.ev_mean, rs.ev_start_time, ro.builtin_model("nucleotide"))
                seqs = [synth._CODE2DNA[c].tobytes().decode() for c in rs.seq_codes[:ns]]
                one = np.ones(args.events + 8, np.float32)
                for i in range(ns):
                    o, nk = int(chains[i]["map_off"]), int(chains[i]["map_len"])
                    ro.read_set_eventalign(rh[i], f"read_{i}", seqs[i], maps[o:o + nk], maps[o:o + nk], one, one)
                cig = lambda i: np.array([(len(seqs[i]) << 4) | 0], np.uint32)
                t0 = time.perf_counter()
                with ThreadPoolExecutor(cores) as ex:       # the compiled reference releases the GIL inside each call
                    rows = list(ex.map(lambda i: ro.eventalign(rh[i], "contig", seqs[i], 0, 0, cig(i), i, want_cigar=False)[2].shape[0], range(ns)))
                cs = time.perf_counter() - t0
                assert rows == [int(v) for v in results["n_records"][:ns]]
                cpu = {"value": int(rs.reads["n_events"][:ns].sum()) / cs, "unit": "events/s", "cores": cores, "cpu_quota": cpu_quota(), "kind": "reference",
                       "sample": f"{ns} of the {n_reads} reads through the compiled reference's align_read_to_ref + TSV writer, one read per thread"}
        line = {"metric": "eventalign_events_per_sec", "value": ev / (t * 1e-3), "unit": "events/s", "n_gpus": 1, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": t, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"eventalign: {n_reads} synthetic R9.4 reads x {args.events} events aligned to their own reference "
                                       f"(CIGAR all M), k=6 nucleotide model, 100-base windows, {n_win} Viterbi windows, {n_rec} event alignments",
                           "reads_per_sec_device": n_reads / (t * 1e-3), "reads_per_sec_e2e": n_reads / float(np.mean(e2e))},
                "e2e": {"value": ev / float(np.mean(e2e)), "unit": "events/s",
                        "h2d_bytes_per_step": int(rs.ev_mean.nbytes + pairs.nbytes + maps.nbytes + rf.nbytes + rr.nbytes + chains.nbytes),
                        "d2h_bytes_per_step": int(records.nbytes + results.nbytes), "steps": args.steps,
                        "api": "nph_reads_load + nph_eventalign_chain (page-locked host buffers in, records out)"},
                "gpu_launches": args.steps,
                "roofline": {"bound": "hbm", "achieved": b_alg / (t * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": b_alg / (t * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src, "kernel": "eventalign_chain_kernel<3>",
                             "note": "one warp walks one read's sequentially dependent windows: issue/latency bound like K3; "
                                     "algorithmic bytes = 4 B/event + 20 B/k-mer in, 12 B/record out"}}
        if cpu:
            line["cpu_baseline"] = cpu
    elif args.workload == "prologue":
        n_reads = min(args.reads, 2048)
        base = min(n_reads, 256)
        raw, rr, seqs = synth.gen_raw(base, 36000, nuc, seed=5, return_seqs=True)
        signals = [raw[int(r["sample_off"]):int(r["sample_off"]) + int(r["n_samples"])] for r in rr]
        reps = max(1, n_reads // base)
        jobs = np.zeros(base * reps, synth.RAW_JOB_DT)
        rk = [synth.kmer_ranks_from_codes(c, nuc.k, 4) for c in seqs]
        soff = roff = 0
        for i in range(base * reps):
            b = i % base
            jobs[i] = (soff, roff, signals[b].shape[0], rk[b].shape[0], 4000.0)
            soff += signals[b].shape[0]; roff += rk[b].shape[0]
        flat = torch.from_numpy(np.tile(raw, reps)).pin_memory().numpy()          # pinned host buffers, like a caller staging a batch
        ranks = torch.from_numpy(np.tile(np.concatenate(rk).astype(np.uint32), reps).view(np.int32)).pin_memory().numpy().view(np.uint32)
        cap = flat.shape[0] // 3 + 16 * jobs.shape[0]
        pin = lambda n, dt: torch.empty(n, dtype=dt).pin_memory().numpy()
        pinned = (pin(cap, torch.float32), pin(cap, torch.float32), pin(cap, torch.float64), pin(cap, torch.float32),
                  pin(2 * ranks.shape[0], torch.int32).view(synth.EVENT_RANGE_DT), pin(48 * jobs.shape[0], torch.uint8).view(synth.CALIBRATION_DT))
        prm = synth.event_params(False)
        ms, e2e = [], []
        for it in range(max(3, args.warmup) + args.steps):
            t0 = time.perf_counter()
            off, mean, stdv, start, dur, b2e, cal = eng.load_from_raw_batch(flat, ranks, jobs, mid, prm, events_cap=cap, pinned=pinned)
            dt = time.perf_counter() - t0
            if it >= max(3, args.warmup):
                m, nl = eng.last_kernel_ms(); ms.append(m); e2e.append(dt)
        t = float(np.mean(ms))
        n_ev = int(off[-1])
        ok = int((cal["status"] == 0).sum())
        b_alg = flat.nbytes + 20 * n_ev + 8 * ranks.shape[0] + 48 * jobs.shape[0]
        cpu = None
        if not args.no_cpu_baseline:
            from concurrent.futures import ThreadPoolExecutor
            from oracle.oracle_py import PortOracle
            from oracle.prep_chain import oracle_chain
            port = PortOracle()
            cores = cpu_threads()
            ns = min(base, max(cores, 32))
            t0 = time.perf_counter()
            with ThreadPoolExecutor(cores) as ex:       # the C restatement releases the GIL inside each call
                list(ex.map(lambda i: oracle_chain(port, nuc, [signals[i]], [seqs[i]]), range(ns)))
            cs = time.perf_counter() - t0
            cpu = {"value": sum(signals[i].shape[0] for i in range(ns)) / cs, "unit": "samples/s", "cores": cores, "cpu_quota": cpu_quota(), "kind": "port",
                   "sample": f"{ns} of the {jobs.shape[0]} reads through oracle/ (trim, events, MoM, ABEA, calibration), one read per thread"}
        line = {"metric": "load_from_raw_samples_per_sec", "value": flat.shape[0] / (t * 1e-3), "unit": "samples/s", "n_gpus": 1,
                "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": t, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
                "config": {"workload": f"prologue: {jobs.shape[0]} synthetic raw reads x 36000 samples -> calibrated SquiggleReads "
                                       f"({n_ev} events, {ok} reads pass QC), scrappie DNA parameters, k=6 nucleotide model",
                           "reads_per_sec_device": jobs.shape[0] / (t * 1e-3), "reads_per_sec_e2e": jobs.shape[0] / float(np.mean(e2e))},
                "e2e": {"value": flat.shape[0] / float(np.mean(e2e)), "unit": "samples/s", "h2d_bytes_per_step": int(flat.nbytes + ranks.nbytes + jobs.nbytes),
                        "d2h_bytes_per_step": int(20 * n_ev + 8 * ranks.shape[0] + 48 * jobs.shape[0]), "steps": args.steps,
                        "api": "nph_load_from_raw_batch"},
                "gpu_launches": int(nl) * args.steps,
                "roofline": {"bound": "hbm", "achieved": b_alg / (t * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": b_alg / (t * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                             "kernel": "trim + ed_* + convert + mom + abea + recalibrate (summed device time of the stages)",
                             "note": "algorithmic bytes = 4 B/sample in + 20 B/event + 8 B/k-mer + 48 B/read out; dominated by the "
                                     "latency-bound ABEA walk at this batch size"}}
        if cpu:
            line["cpu_baseline"] = cpu
    else:
        n_reads = min(args.reads, 8192)
        raw, reads = synth.gen_raw(min(n_reads, 512), 36000, nuc, seed=5)
        if n_reads > 512:
            reps = n_reads // 512; per = raw.shape[0]; estride = int(reads["event_off"][-1] + reads["event_cap"][-1])
            raw = np.tile(raw, reps); reads = np.tile(reads, reps)
            for r in range(reps):
                reads["sample_off"][r * 512:(r + 1) * 512] += r * per
                reads["event_off"][r * 512:(r + 1) * 512] += r * estride
        prm = synth.event_params(False)
        # page-locked host buffers for the samples and the events, allocated once (the e2e figure is host buffers -> host events)
        room = int((reads["event_off"] + reads["event_cap"]).max())
        t_raw = torch.from_numpy(raw).pin_memory(); raw = t_raw.numpy()
        t_ev = torch.empty(room * synth.EVENT_DT.itemsize, dtype=torch.uint8).pin_memory()
        ev_buf = (t_ev.numpy().view(synth.EVENT_DT), np.zeros(reads.shape[0], np.uint32))
        ms, e2e = [], []
        for it in range(max(3, args.warmup) + args.steps):
            t0 = time.perf_counter(); ev = eng.detect_events_batch(raw, reads, prm, out=ev_buf); dt = time.perf_counter() - t0
            if it >= max(3, args.warmup):
                ms.append(eng.last_kernel_ms()[0]); e2e.append(dt)
        t = float(np.mean(ms))
        n_ev = sum(e.shape[0] for e in ev)
        b_alg = raw.nbytes + 24 * n_ev
        line = {"metric": "event_detection_samples_per_sec", "value": raw.shape[0] / (t * 1e-3), "unit": "samples/s", "n_gpus": 1,
                "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": t, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
                "config": {"workload": f"events: {reads.shape[0]} synthetic raw reads x 36000 samples, scrappie DNA parameters"},
                "e2e": {"value": raw.shape[0] / float(np.mean(e2e)), "unit": "samples/s", "h2d_bytes_per_step": int(raw.nbytes),
                        "d2h_bytes_per_step": int(24 * n_ev), "steps": args.steps,
                        "api": "nph_detect_events_batch"},
                "gpu_launches": 2 * args.steps,
                "roofline": {"bound": "hbm", "achieved": b_alg / (t * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": b_alg / (t * 1e-3) / 1e9 / peak,
                             # DRAM bytes of the two kernels for the 4 096-read shape (profiles/r02_events_summary.md: 1.07 GB + 1.35 GB)
                             "traffic": 2.42e9 if reads.shape[0] == 4096 else None, "peak_source": peak_src,
                             "kernel": "ed_fused_kernel + ed_events_kernel",
                             "note": "algorithmic bytes = 4 B/sample in + 24 B/event out; the fused kernel is bound by the float<->double "
                                     "conversion unit and FP64 latency, not by HBM (DESIGN.md section 11)",
                             # compute_tstat needs >= 24 conversions per sample position (after staging each sample once), 8.5 clk per
                             # warp instruction and sub-partition (profiles/r02_ubench_cvt.txt), x 1.11 for the 128-sample warm-ups
                             "conversion_unit": {"floor_ms": raw.shape[0] / 32 * 24 * 1.11 * 8.5 / (148 * 4 * 1.965e6),
                                                 "frac": raw.shape[0] / 32 * 24 * 1.11 * 8.5 / (148 * 4 * 1.965e6) / t,
                                                 "unit": "share of the step the conversion unit alone would need"}}}
    emit(line, saved_stdout)
    eng.close()


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """DIR/<name>.npy of each device tensor, as the caller of the timed path receives it"""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def emit(line: dict, saved_stdout: int) -> None:
    """Exactly one JSON line on the real stdout (libraries such as NCCL print banners to fd 1)."""
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)            # anything a library prints goes to stderr; the JSON line is emitted via emit()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload in ("abea", "events", "prologue", "eventalign"):
        run_aux(args, rank, world, local, saved_stdout)
        return
    if args.workload == "variants" and args.impl != "reference":
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        if world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        blk = variants_block(args, rank, world, local, args.steps, args.warmup)
        if rank == 0:
            blk["clocks"] = sampler.stop()
            emit(blk, saved_stdout)
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return
    if args.workload == "call_methylation" and args.impl != "reference":
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        if world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        blk = call_methylation_block(args, rank, world, local, args.steps, args.warmup)
        if rank == 0:
            blk.update({"higher_is_better": True, "vs_baseline": None, "clocks": sampler.stop()})
            emit(blk, saved_stdout)
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return
    if args.impl == "reference":
        run_reference(args, rank, world, saved_stdout)
        return

    import torch
    import torch.distributed as dist
    from nanopolish_b200.engine import Engine

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    rs, jobs, models = build_workload(args, rank)
    n_jobs = int(jobs.jobs.shape[0])
    stream = torch.cuda.current_stream().cuda_stream
    eng = Engine(local, stream=stream)
    for m in models:
        eng.model_upload(m)

    # pinned host copies (the caller-owned host buffers of the e2e path)
    def pin(a):
        t = torch.from_numpy(a).pin_memory()
        return t, t.numpy()
    keep = []
    t_reads, h_reads = pin(rs.reads.view(np.uint8)); keep.append(t_reads); h_reads = h_reads.view(rs.reads.dtype)
    t_mean, h_mean = pin(rs.ev_mean); keep.append(t_mean)
    t_time, h_time = pin(rs.ev_start_time); keep.append(t_time)
    # sequences cross the boundary as base codes (1 B/base; nph_hmm_*_seq), the jobs' rank_off indexing them
    use_ranks = bool(os.environ.get("NPH_BENCH_RANKS"))          # development A/B: the uint32-rank form of the same calls
    t_ranks, h_ranks = pin(jobs.kmer_ranks if use_ranks else jobs.seq_codes); keep.append(t_ranks)
    t_jobs, h_jobs = pin((jobs.jobs if use_ranks else jobs.code_jobs).view(np.uint8)); keep.append(t_jobs); h_jobs = h_jobs.view(jobs.jobs.dtype)
    t_out = torch.empty(n_jobs, dtype=torch.float32).pin_memory(); h_out = t_out.numpy()

    # ---- device-resident arm: inputs already in HBM when the timed region starts ----------
    eng.reads_load(h_reads, h_mean, h_time)
    (eng.hmm_jobs_load if use_ranks else eng.hmm_jobs_load_seq)(h_ranks, h_jobs)
    scores = torch.empty(n_jobs, dtype=torch.float32, device=dev)
    counts = None
    gathered = None
    if world > 1:
        cnt = torch.tensor([n_jobs], dtype=torch.int64, device=dev)
        allc = [torch.zeros_like(cnt) for _ in range(world)]
        dist.all_gather(allc, cnt)
        counts = [int(c.item()) for c in allc]
        maxc = max(counts)
        scores = torch.zeros(maxc, dtype=torch.float32, device=dev)   # padded so one ncclGather suffices
    from nanopolish_b200.dist import gather_to_rank0

    def step():
        nonlocal gathered
        eng.hmm_score(scores.data_ptr())
        if world > 1:
            gathered = gather_to_rank0(scores, counts)           # one NCCL gather of per-job log-likelihoods over NVLink

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern_ms = []
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    total_ms = e0.elapsed_time(e1)
    km, launches_per_step = eng.last_kernel_ms()
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"scores": torch.cat(gathered) if world > 1 else scores[:n_jobs]})

    # kernel-only duration for the roofline: CUDA events around each kernel sequence, on its stream
    for _ in range(5):
        eng.hmm_score(scores.data_ptr()); eng.sync()
        kern_ms.append(eng.last_kernel_ms()[0])
    kernel_ms = float(np.mean(kern_ms))

    ev_local = int(jobs.scored_events)
    ev_t = torch.tensor([ev_local], dtype=torch.float64, device=dev)
    cells_t = torch.tensor([float(jobs.block_cells)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ev_t); dist.all_reduce(cells_t)
    ev_all, cells_all = float(ev_t.item()), float(cells_t.item())
    value = ev_all * args.steps / (total_ms * 1e-3)

    # ---- e2e arm: the one-shot C-ABI call with HOST buffers, H2D + D2H inside the timed region ----
    def e2e_step():
        (eng.hmm_score_batch if use_ranks else eng.hmm_score_batch_seq)(h_reads, h_mean, h_time, h_ranks, h_jobs, out=h_out)

    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    e2e_value = ev_all * e2e_steps / e2e_s
    any_drift = bool((rs.reads["drift"] != 0).any())
    h2d = rs.reads.nbytes + rs.ev_mean.nbytes + (rs.ev_start_time.nbytes if any_drift else 0) + jobs.seq_codes.nbytes \
        + jobs.jobs.nbytes + 4 * n_jobs + 8 * rs.n_reads
    d2h = 4 * n_jobs

    if rank == 0:
        peak, peak_src = peaks()
        b_alg = algorithmic_bytes(jobs)
        achieved = b_alg / (kernel_ms * 1e-3) / 1e9
        traffic = None          # filled from profiles/r02_k1_counters.json by k1_rooflines when the workload matches the capture
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {**workload_config(args, jobs), "jobs_per_gpu": n_jobs,
                       "scored_events_per_step": ev_all},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": e2e_steps, "api": "nph_hmm_score_batch_seq (host buffers in: events + 1 B/base sequence codes + jobs; host scores out)"},
            "gpu_launches": int(launches_per_step) * args.steps,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": "hmm_forward_kernel<C>",
                         "kernel_ms": kernel_ms, "algorithmic_bytes_per_step": b_alg,
                         "note": "scalar log-semiring DP: issue/shared-memory bound, not HBM bound (DESIGN.md); "
                                 "block-cells/s below is the figure that moves",
                         "block_cells_per_sec_per_gpu": float(jobs.block_cells) / (kernel_ms * 1e-3)},
        }
        line["roofline"].update(k1_rooflines(args, jobs, kernel_ms, clocks))
        if world == 1 and not args.no_cpu_baseline:
            try:
                arm = CpuArm(rs, jobs, models)
                idx = arm.sample_for(12.0)
                line["cpu_baseline"] = arm.report(idx, arm.time(idx))
            except Exception as ex:   # the baseline is a reported extra; never lose the GPU line over it
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "unavailable",
                                        "sample": f"failed: {ex}"}
    eng.close()
    # ---- the caller BASELINE.json's metric is named after, end to end, in the same line ----
    cm = None
    if not args.no_call_methylation:
        try:
            cm = call_methylation_block(args, rank, world, local, args.steps, args.warmup)
        except Exception as ex:          # never lose the headline line over the extra block
            cm = {"error": f"{type(ex).__name__}: {ex}"} if rank == 0 else None
    if rank == 0:
        if cm is not None:
            line["configs"] = {"call_methylation": cm}
        emit(line, saved_stdout)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
