"""ctypes binding of libhammock_b200.so (C ABI: include/hammock_b200.h).

No CPU fallback: if the CUDA library is missing or no GPU is usable, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HMK_LIB") or os.path.join(HERE, "libhammock_b200.so")

FLAG_P2_REUSED, FLAG_XHIT_OVERFLOW, FLAG_ASYMMETRIC = 1, 2, 4
STATUS_OK, STATUS_SHIFT_TOO_BIG, STATUS_NULL_CLUSTER, STATUS_BAD_RESIDUE, STATUS_CUDA, STATUS_BAD_ARG, STATUS_UNSUPPORTED = range(7)


class GreedyIn(C.Structure):
    _fields_ = [("n", C.c_int32), ("residues", C.POINTER(C.c_uint8)), ("offsets", C.POINTER(C.c_int32)),
                ("abundance", C.POINTER(C.c_int32)), ("matrix", C.POINTER(C.c_int32)),
                ("threshold", C.c_int32), ("max_shift", C.c_int32), ("shift_penalty", C.c_int32),
                ("max_clusters", C.c_int32)]


class GreedyOut(C.Structure):
    _fields_ = [("cluster_id", C.POINTER(C.c_int32)), ("member_rank", C.POINTER(C.c_int32)),
                ("result_order", C.POINTER(C.c_int32)), ("n_result", C.c_int32), ("n_multi", C.c_int32),
                ("error_step", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("bulk_pairs", C.c_int64), ("scalar_pairs", C.c_int64), ("bulk_cells", C.c_int64),
                ("bulk_ops", C.c_int64), ("bulk_kernel_ms", C.c_double), ("total_ms", C.c_double),
                ("phase1_ms", C.c_double), ("phase2_ms", C.c_double), ("bulk_launches", C.c_int32),
                ("total_launches", C.c_int32), ("p1_steps", C.c_int32), ("p1_joins", C.c_int32),
                ("p1_new_clusters", C.c_int32), ("p1_orphans", C.c_int32), ("p1_batches", C.c_int32),
                ("p1_restarts", C.c_int32), ("p2_queries", C.c_int32), ("p2_assigned", C.c_int32),
                ("p2_rounds", C.c_int32), ("p2_hits", C.c_int64), ("p2_candidates", C.c_int64),
                ("fast_path", C.c_int32), ("lane_bits", C.c_int32), ("error_step", C.c_int32),
                ("flags", C.c_int32), ("xhits_kept", C.c_int64), ("xhits_capacity", C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class BatchProbeOut(C.Structure):
    _fields_ = [("nq_out", C.c_int32), ("qid", C.POINTER(C.c_int32)), ("bk_key", C.POINTER(C.c_uint64)),
                ("bk_cnt", C.POINTER(C.c_int32)), ("bk_ovf", C.POINTER(C.c_int32)), ("ib", C.POINTER(C.c_int32)),
                ("ibm", C.POINTER(C.c_uint32)), ("ibm2", C.POINTER(C.c_uint32)), ("pcand", C.POINTER(C.c_int32)),
                ("pd", C.POINTER(C.c_int32)), ("fhits", C.POINTER(C.c_int32)), ("fhit_cap", C.c_int64),
                ("fhit_count", C.c_int64), ("ac_cnt", C.POINTER(C.c_int32)), ("ac_slot", C.POINTER(C.c_int32)),
                ("ac_score", C.POINTER(C.c_int32)), ("ac_best", C.POINTER(C.c_int32)), ("kernel", C.c_int32 * 11)]


EXPORTS = ["hmk_abi_version", "hmk_greedy_cluster", "hmk_greedy_cluster_multi", "hmk_clinkage_cluster", "hmk_clinkage_run", "hmk_create", "hmk_destroy", "hmk_upload", "hmk_run",
           "hmk_download", "hmk_get_stats", "hmk_get_section_ms", "hmk_set_option", "hmk_score_block", "hmk_bulk_probe",
           "hmk_batch_probe", "hmk_score_graph", "hmk_score_pairs", "hmk_nearest",
           "hmk_timer_begin", "hmk_timer_end", "hmk_measure_peaks", "hmk_nccl_unique_id", "hmk_init_distributed", "hmk_release_cached"]
SECTIONS = ["p1_select", "p1_partner", "p1_cluster", "p1_intra", "p1_resolve", "p2_setup", "p2_filter", "p2_check",
            "p2_sort", "p2_base", "p2_iterate", "p2_commit", "final"]

_lib = None


def load():
    """Load the CUDA library; raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m hammock_b200.build` "
            "(hammock_b200 has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, cp, sz = C.c_void_p, C.c_char_p, C.c_size_t
    i32p = C.POINTER(C.c_int32)
    L.hmk_abi_version.restype = C.c_int
    L.hmk_greedy_cluster.restype = C.c_int
    L.hmk_greedy_cluster.argtypes = [C.POINTER(GreedyIn), C.POINTER(GreedyOut), C.c_int, cp, sz]
    L.hmk_greedy_cluster_multi.restype = C.c_int
    L.hmk_greedy_cluster_multi.argtypes = [C.POINTER(GreedyIn), C.POINTER(GreedyOut), i32p, C.c_int32, cp, sz]
    L.hmk_clinkage_cluster.restype = C.c_int
    L.hmk_clinkage_cluster.argtypes = [C.POINTER(GreedyIn), C.POINTER(GreedyOut), C.c_int, cp, sz]
    L.hmk_clinkage_run.restype = C.c_int
    L.hmk_clinkage_run.argtypes = [vp, C.POINTER(GreedyIn), C.POINTER(GreedyOut), cp, sz]
    L.hmk_create.restype = C.c_int
    L.hmk_create.argtypes = [C.POINTER(vp), C.c_int, cp, sz]
    L.hmk_destroy.restype = None
    L.hmk_destroy.argtypes = [vp]
    L.hmk_upload.restype = C.c_int
    L.hmk_upload.argtypes = [vp, C.POINTER(GreedyIn), cp, sz]
    L.hmk_run.restype = C.c_int
    L.hmk_run.argtypes = [vp, cp, sz]
    L.hmk_download.restype = C.c_int
    L.hmk_download.argtypes = [vp, C.POINTER(GreedyOut), cp, sz]
    L.hmk_get_stats.restype = C.c_int
    L.hmk_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.hmk_get_section_ms.restype = C.c_int
    L.hmk_get_section_ms.argtypes = [vp, C.POINTER(C.c_double), C.c_int]
    L.hmk_timer_begin.restype = C.c_int
    L.hmk_timer_begin.argtypes = [vp]
    L.hmk_timer_end.restype = C.c_int
    L.hmk_timer_end.argtypes = [vp, C.POINTER(C.c_double)]
    L.hmk_measure_peaks.restype = C.c_int
    L.hmk_measure_peaks.argtypes = [vp, C.POINTER(C.c_double), cp, sz]
    L.hmk_nccl_unique_id.restype = C.c_int
    L.hmk_nccl_unique_id.argtypes = [C.c_void_p, cp, sz]
    L.hmk_init_distributed.restype = C.c_int
    L.hmk_init_distributed.argtypes = [vp, C.c_int, C.c_int, C.c_void_p, cp, sz]
    L.hmk_release_cached.restype = None
    L.hmk_release_cached.argtypes = []
    L.hmk_set_option.restype = C.c_int
    L.hmk_set_option.argtypes = [vp, cp, C.c_int64]
    L.hmk_score_block.restype = C.c_int
    L.hmk_score_block.argtypes = [vp, i32p, C.c_int32, i32p, C.c_int32, i32p, cp, sz]
    L.hmk_bulk_probe.restype = C.c_int
    L.hmk_bulk_probe.argtypes = [vp, C.c_int32, i32p, C.c_int32, i32p, C.c_int32, C.c_int32, C.POINTER(C.c_uint8),
                                 C.POINTER(C.c_uint64), i32p, i32p, i32p, C.c_int64, C.POINTER(C.c_int64), i32p, cp, sz]
    L.hmk_batch_probe.restype = C.c_int
    L.hmk_batch_probe.argtypes = [vp, i32p, i32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                  C.POINTER(BatchProbeOut), cp, sz]
    L.hmk_score_graph.restype = C.c_int
    L.hmk_score_graph.argtypes = [vp, C.POINTER(C.c_int64), vp, C.c_int64, C.POINTER(C.c_int64), cp, sz]
    L.hmk_score_pairs.restype = C.c_int
    L.hmk_score_pairs.argtypes = [vp, i32p, i32p, C.c_int32, i32p, i32p, cp, sz]
    L.hmk_nearest.restype = C.c_int
    L.hmk_nearest.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, i32p, i32p, i32p, i32p, i32p, cp, sz]
    _lib = L
    return L
