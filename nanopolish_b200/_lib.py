"""ctypes loader of libnph.so (the C ABI of include/nph.h).

There is no fallback: if the shared library is missing (run `python -c "import __graft_entry__ as g;
g.build()"` or `make -C nanopolish_b200/csrc`) importing this module raises, and if no CUDA device is
usable nph_create() returns NPH_ERR_NO_DEVICE and Engine() raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NPH_LIB_PATH") or os.path.join(HERE, "libnph.so")     # NPH_LIB_PATH: development aid (A/B builds of the kernels)

NPH_OK = 0
NPH_ERR_NO_DEVICE = -1


class NphError(RuntimeError):
    def __init__(self, status: int, what: str, detail: str = ""):
        self.status = status
        super().__init__(f"{what}: status {status} ({detail})")


def load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(
            f"{LIB_PATH} is not built; the engine has no CPU path. Build it with "
            f"`make -C {os.path.join(HERE, 'csrc')}` (nvcc, sm_100a).")
    lib = C.CDLL(LIB_PATH)
    vp, sz, u32, dbl = C.c_void_p, C.c_size_t, C.c_uint32, C.c_double
    lib.nph_strerror.restype = C.c_char_p
    lib.nph_strerror.argtypes = [C.c_int]
    lib.nph_last_error.restype = C.c_char_p
    lib.nph_last_error.argtypes = [vp]
    lib.nph_stream.restype = vp
    lib.nph_stream.argtypes = [vp]
    lib.nph_create.argtypes = [C.POINTER(vp), C.c_int]
    lib.nph_create_on_stream.argtypes = [C.POINTER(vp), C.c_int, vp]
    lib.nph_destroy.argtypes = [vp]
    lib.nph_sync.argtypes = [vp]
    lib.nph_model_upload.argtypes = [vp, vp, vp, vp, u32, u32, u32, C.POINTER(u32)]
    lib.nph_reads_load.argtypes = [vp, vp, sz, vp, vp, sz]
    lib.nph_hmm_jobs_load.argtypes = [vp, vp, sz, vp, sz, dbl]
    lib.nph_hmm_score.argtypes = [vp, vp]
    lib.nph_hmm_scores_fetch.argtypes = [vp, vp, sz]
    lib.nph_hmm_score_batch.argtypes = [vp, vp, sz, vp, vp, sz, vp, sz, vp, sz, dbl, vp]
    lib.nph_hmm_score_batch_seq.argtypes = [vp, vp, sz, vp, vp, sz, vp, sz, vp, sz, dbl, vp]
    lib.nph_hmm_jobs_load_seq.argtypes = [vp, vp, sz, vp, sz, dbl]
    lib.nph_score_set_combine.argtypes = [vp, sz, u32, vp]
    lib.nph_abea_batch.argtypes = [vp, vp, sz, vp, vp, sz, vp, sz, vp, sz, u32, vp, sz, vp]
    lib.nph_abea_jobs_load.argtypes = [vp, vp, sz, vp, sz, u32, sz]
    lib.nph_abea_run.argtypes = [vp]
    lib.nph_abea_fetch.argtypes = [vp, vp, sz, vp, sz]
    lib.nph_mom_batch.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, sz, u32, vp]
    lib.nph_hmm_align_batch.argtypes = [vp, vp, sz, vp, vp, sz, vp, sz, vp, sz, dbl, vp, vp, vp, vp]
    lib.nph_hmm_align.argtypes = [vp, vp, sz, vp, sz, dbl, vp, vp, vp, vp]
    lib.nph_eventalign_chain.argtypes = [vp, vp, sz, vp, sz, vp, vp, sz, vp, sz, dbl, vp, sz, vp]
    lib.nph_detect_events_batch.argtypes = [vp, vp, sz, vp, sz, vp, vp, sz, vp]
    lib.nph_trim_raw_batch.argtypes = [vp, vp, sz, vp, sz, C.c_int32, C.c_int32, C.c_int32, C.c_float, vp]
    lib.nph_recalibrate_batch.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, sz, u32, vp, sz, vp, vp, vp]
    lib.nph_load_from_raw_batch.argtypes = [vp, vp, sz, vp, sz, vp, sz, u32, vp, vp, vp, vp, vp, vp, sz, vp, vp]
    lib.nph_last_trim_ranges.argtypes = [vp, vp, sz]
    lib.nph_methylation_batch.argtypes = [vp, vp, sz, vp, vp, sz, vp, sz, vp, sz, vp, sz, vp, dbl, vp, vp, sz, vp]
    lib.nph_methylation_load.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, dbl]
    lib.nph_methylation_batch_compact.argtypes = [vp, vp, sz, vp, vp, sz, vp, vp, sz, vp, vp, sz, vp, dbl, vp, vp, sz, vp]
    lib.nph_methylation_load_compact.argtypes = [vp, vp, vp, sz, vp, vp, sz, vp, dbl]
    lib.nph_methylation_run.argtypes = [vp]
    lib.nph_methylation_counts.argtypes = [vp, vp, vp, vp]
    lib.nph_methylation_fetch.argtypes = [vp, vp, vp, sz]
    lib.nph_methylation_sites_dev.argtypes = [vp, vp, vp]
    lib.nph_methylation_tsv.argtypes = [vp, C.c_char_p, vp, vp, vp, vp, C.c_size_t, vp]
    lib.nph_screen_edits_batch.argtypes = [vp, vp, sz, vp, vp, sz, vp, sz, vp, sz, vp, vp, sz, vp, dbl, vp, vp, vp]
    lib.nph_screen_load.argtypes = [vp, vp, sz, vp, sz, vp, vp, sz, vp, dbl]
    lib.nph_screen_run.argtypes = [vp]
    lib.nph_screen_counts.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.nph_screen_fetch.argtypes = [vp, vp, vp, vp]
    lib.nph_polya_batch.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, sz, vp]
    lib.nph_polya_after_load.argtypes = [vp, vp, sz]
    lib.nph_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_int)]
    lib.nph_host_alloc.argtypes = [C.POINTER(vp), sz]
    lib.nph_host_free.argtypes = [vp]
    return lib


# every symbol include/nph.h declares (tests check the library exports all of them)
EXPORTS = [
    "nph_create", "nph_create_on_stream", "nph_destroy", "nph_strerror", "nph_last_error", "nph_version",
    "nph_sync", "nph_stream", "nph_model_upload", "nph_hmm_score_batch", "nph_hmm_score_batch_seq", "nph_hmm_jobs_load_seq", "nph_reads_load",
    "nph_hmm_jobs_load", "nph_hmm_score", "nph_hmm_scores_fetch", "nph_score_set_combine",
    "nph_abea_batch", "nph_abea_jobs_load", "nph_abea_run", "nph_abea_fetch", "nph_mom_batch",
    "nph_hmm_align_batch", "nph_hmm_align", "nph_eventalign_chain", "nph_detect_events_batch", "nph_trim_raw_batch", "nph_recalibrate_batch", "nph_load_from_raw_batch", "nph_last_trim_ranges", "nph_methylation_batch", "nph_methylation_batch_compact", "nph_methylation_load", "nph_methylation_load_compact", "nph_methylation_run", "nph_methylation_counts", "nph_methylation_fetch", "nph_methylation_sites_dev", "nph_methylation_tsv", "nph_methylation_batch_compact_tsv", "nph_screen_edits_batch", "nph_screen_load", "nph_screen_run", "nph_screen_counts", "nph_screen_fetch", "nph_polya_batch", "nph_polya_after_load", "nph_last_kernel_ms", "nph_host_alloc", "nph_host_free",
]
