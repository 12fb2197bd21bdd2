"""ctypes front ends of the `nanopolish polya` checkers (TEST INFRASTRUCTURE ONLY; built by oracle/polya.mk):
PortPolya, the plain-C restatement (oracle/np_polya.c), and RefPolya, the reference's src/nanopolish_polya_estimator.cpp
compiled in place (oracle/_ref/libnpref_polya.so, where the reference sources exist)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_SO = os.path.join(HERE, "libnpo_polya.so")
REF_SO = os.path.join(HERE, "_ref", "libnpref_polya.so")

HEADER = ("readname\tcontig\tposition\tleader_start\tadapter_start\tpolya_start\ttranscript_start\tread_rate\tpolya_length\t"
          "qc_tag\n")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class PortPolya:
    def __init__(self):
        if not os.path.exists(PORT_SO):
            raise FileNotFoundError(PORT_SO + " (run `make -C oracle -f polya.mk polya-port`)")
        self.lib = C.CDLL(PORT_SO)

    def polya(self, samples, durations, emap, jobs, threads=None):
        """npo_polya over POLYA_JOB_DT jobs: POLYA_RES_DT results"""
        from nanopolish_b200.synth import POLYA_RES_DT
        out = np.zeros(jobs.shape[0], POLYA_RES_DT)
        s = np.ascontiguousarray(samples, np.float32); d = np.ascontiguousarray(durations, np.float32)
        m = np.ascontiguousarray(emap); j = np.ascontiguousarray(jobs)
        self.lib.npo_polya(_p(s), _p(d), _p(m), _p(j), C.c_size_t(j.shape[0]), _p(out), C.c_int(threads or os.cpu_count() or 1))
        return out


class RefPolya:
    """The compiled reference, on reads assembled with its harness's npref_read_create / npref_read_set_eventalign /
    npref_read_set_samples / npref_read_set_scalings."""

    def __init__(self):
        if not os.path.exists(REF_SO):
            raise FileNotFoundError(REF_SO + " (run `make -C oracle -f polya.mk polya-ref` where the reference sources exist)")
        self.lib = L = C.CDLL(REF_SO)
        L.npref_polya_batch.restype = C.c_double
        mean = np.full(1024, 90.0); sd = np.full(1024, 2.0)
        self._model = L.npref_model_custom(b"nucleotide", 5, C.c_uint32(1024), _p(mean), _p(sd))   # only k = 5 is read

    @staticmethod
    def available() -> bool:
        return os.path.exists(REF_SO)

    def _register(self, samples, durations, emap, jobs, names):
        L = self.lib
        L.npref_reads_clear()
        hs = []
        for i, jb in enumerate(jobs):
            ne, nk = int(jb["n_events"]), int(jb["n_kmers"])
            eo, mo, so, ns = int(jb["event_off"]), int(jb["map_off"]), int(jb["sample_off"]), int(jb["n_samples"])
            mean = np.zeros(max(ne, 1), np.float32); t = np.zeros(max(ne, 1))
            h = L.npref_read_create(C.c_uint32(ne), _p(mean), _p(t), C.c_double(jb["shift"]), C.c_double(jb["scale"]), C.c_double(0.0),
                                    C.c_double(jb["var"]), C.c_double(0.0), self._model)
            m = emap[mo:mo + nk]
            a = np.ascontiguousarray(m["start"], np.int32); b = np.ascontiguousarray(m["stop"], np.int32)
            du = np.ascontiguousarray(durations[eo:eo + ne], np.float32); sd = np.ones(max(ne, 1), np.float32)
            seq = ("A" * (nk + 4)).encode()                  # only its length (n_kmers + k - 1) is read
            L.npref_read_set_eventalign(h, names[i].encode(), seq, _p(a), _p(b), C.c_size_t(nk), _p(sd), _p(du))
            x = np.ascontiguousarray(samples[so:so + ns], np.float32)
            L.npref_read_set_samples(h, _p(x), C.c_size_t(ns), C.c_double(jb["sample_rate"]))
            L.npref_read_set_scalings(h, C.c_double(jb["shift"]), C.c_double(jb["scale"]), C.c_double(0.0), C.c_double(jb["var"]), C.c_double(0.0))
            hs.append(h)
        return np.asarray(hs, np.int32)

    def polya(self, samples, durations, emap, jobs, names, contig, positions, suffix_clip):
        """Per read: (seg u8[n,5] = start, leader, adapter, polya, cliffs; rate_len f8[n,2]; end_score f4[n]; qc i4[n]) and the
        TSV (header + rows) the reference writes for them."""
        hs = self._register(samples, durations, emap, jobs, names)
        n = jobs.shape[0]
        seg = np.zeros((n, 5), np.uint64); rl = np.zeros((n, 2)); es = np.zeros(n, np.float32); qc = np.zeros(n, np.int32)
        rows = [HEADER.encode()]
        buf = C.create_string_buffer(4096)
        for i in range(n):
            s5 = np.zeros(5, np.uint64); r2 = np.zeros(2); e1 = np.zeros(1, np.float32); q1 = np.zeros(1, np.int32)
            k = self.lib.npref_polya(int(hs[i]), names[i].encode(), contig.encode(), int(positions[i]), C.c_uint32(int(suffix_clip[i])),
                                     _p(s5), _p(r2), _p(e1), _p(q1), buf, C.c_size_t(4096))
            rows.append(buf.raw[:k])
            seg[i] = s5; rl[i] = r2; es[i] = e1[0]; qc[i] = q1[0]
        self.lib.npref_reads_clear()
        return seg, rl, es, qc, b"".join(rows)

    def polya_timed(self, samples, durations, emap, jobs, names, contig, threads):
        """The reference's per-read work on `threads` OpenMP threads: (seconds, TSV rows without header, positions 0)"""
        hs = self._register(samples, durations, emap, jobs, names)
        stride = 512
        rows = C.create_string_buffer(stride * len(hs))
        secs = self.lib.npref_polya_batch(_p(hs), C.c_size_t(len(hs)), contig.encode(), int(threads), rows, C.c_size_t(stride))
        raw = rows.raw
        out = b"".join(raw[i * stride:(i + 1) * stride].split(b"\0", 1)[0] for i in range(len(hs)))
        self.lib.npref_reads_clear()
        return secs, out


def qc_tag(qc: int, suffix_clip: int) -> str:
    """estimate_polya_for_single_read's QC priority (:803-813): post-segmentation, post-estimation, pre-segmentation"""
    if qc & 4:
        return "READ_FAILED_LOAD"
    if qc & 1:
        return "NOREGION"
    if qc & 2:
        return "ADAPTER"
    return "SUFFCLIP" if suffix_clip > 200 else "PASS"


def format_rows(results, names, contig, positions, suffix_clip) -> bytes:
    """The header and rows polya writes (:765, :823-826, :877) from POLYA_RES_DT results; Python's %-formatting of a double
    is the correctly rounded decimal glibc's printf prints, and spells inf / nan the same way."""
    out = [HEADER]
    for i, r in enumerate(results):
        q = int(r["qc"])
        if q & 4:
            out.append(f"{names[i]}\t{contig}\t{int(positions[i])}\t-1.0\t-1.0\t-1.0\t-1.0\t-1.00\t-1.00\tREAD_FAILED_LOAD\n")
            continue
        m = 1 << 64
        cols = [float((int(r["start"]) + 1) % m), float((int(r["leader"]) + 1) % m), float((int(r["adapter"]) + 1) % m),
                float((int(r["polya"]) + 1) % m)]
        out.append("%s\t%s\t%d\t%.1f\t%.1f\t%.1f\t%.1f\t%.2f\t%.2f\t%s\n" % (names[i], contig, int(positions[i]), *cols, float(r["read_rate"]),
                                                                          float(r["polya_length"]), qc_tag(q, int(suffix_clip[i]))))
    return "".join(out).encode()
