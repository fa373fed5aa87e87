"""ctypes binding of libamira_gmg.so (include/amira_gmg.h).  There is no CPU fallback: if the
library is missing or no CUDA device is present, every entry point fails loudly."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AMIRA_LIB_PATH", os.path.join(HERE, "libamira_gmg.so"))   # override: developer experiments

OK = 0
E_BLANK_GENE, E_BAD_STRAND, E_EMPTY_NAME, E_UNKNOWN_GENE, E_PALINDROME, E_EMPTY_GENEMER, E_MULTI_EDGE = 1, 2, 3, 4, 5, 6, 7
E_ARG, E_STATE, E_CUDA, E_NOMEM, E_NCCL = 8, 9, 10, 11, 12
PHASES = ("h2d", "windows", "insert", "order", "remap", "incidence", "adjacency", "components", "filter",
          "exchange", "emit", "insert_kernel", "emit_nodes", "exchange_edges")

EXPORTED = (
    "amira_last_error", "amira_version", "amira_vocab_encode", "amira_host_tuple_sha", "amira_host_edge_keys", "amira_gmg_create", "amira_gmg_destroy",
    "amira_gmg_reserve", "amira_gmg_set_profiling", "amira_gmg_phase_ms", "amira_gmg_kernel_launches",
    "amira_gmg_build", "amira_gmg_sync", "amira_gmg_sizes", "amira_gmg_export_nodes", "amira_gmg_export_edges",
    "amira_gmg_export_reads", "amira_gmg_remove_low_coverage_components", "amira_gmg_filter",
    "amira_gmg_filter_mask_sizes", "amira_gmg_export_filter_masks", "amira_gmg_nccl_unique_id", "amira_gmg_comm_init", "amira_gmg_atomic_peak", "amira_gmg_debug_layout", "amira_gmg_debug_segsort",
    "amira_gmg_read_length_coverages", "amira_gmg_node_coverage_stats", "amira_gmg_junk_read_mask", "amira_gmg_nodes_containing",
    "amira_gmg_remove_nodes", "amira_gmg_remove_nodes_without_reads_of", "amira_gmg_linear_steps", "amira_gmg_linear_walks",
    "amira_gmg_unitigs", "amira_gmg_unitig_links", "amira_gmg_read_unitig_paths", "amira_gmg_bubbles",
    "amira_gmg_correct_bubble_reads", "amira_gmg_bubble_policy", "amira_gmg_input_calls",
)

_lib = None


class AmiraLibraryError(RuntimeError):
    pass


def load():
    """dlopen the in-tree library; raises if it has not been built (python -m amira_b200.build)"""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AmiraLibraryError(
            "libamira_gmg.so is not built (%s). Run `python -m amira_b200.build`; there is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.amira_last_error.restype = C.c_char_p
    lib.amira_version.restype = C.c_char_p
    vp, i64, i32, u32 = C.c_void_p, C.c_int64, C.c_int32, C.c_uint32
    lib.amira_vocab_encode.argtypes = [vp, vp, i64, vp, vp, i32, vp, vp]
    lib.amira_host_tuple_sha.argtypes = [vp, vp, i64, i32, vp]
    lib.amira_host_edge_keys.argtypes = [vp, vp, vp, vp, vp, i64, vp]
    lib.amira_gmg_create.argtypes = [C.POINTER(vp), C.c_int, vp]
    lib.amira_gmg_destroy.argtypes = [vp]
    lib.amira_gmg_destroy.restype = None
    lib.amira_gmg_reserve.argtypes = [vp, i64, i64]
    lib.amira_gmg_set_profiling.argtypes = [vp, C.c_int]
    lib.amira_gmg_phase_ms.argtypes = [vp, C.c_int, C.POINTER(C.c_float)]
    lib.amira_gmg_kernel_launches.argtypes = [vp, C.POINTER(i64)]
    lib.amira_gmg_build.argtypes = [vp, vp, vp, i64, i32, vp, vp, C.c_int]
    lib.amira_gmg_sync.argtypes = [vp]
    lib.amira_gmg_sizes.argtypes = [vp] + [C.POINTER(i64)] * 7
    lib.amira_gmg_export_nodes.argtypes = [vp] * 11
    lib.amira_gmg_export_edges.argtypes = [vp] * 6
    lib.amira_gmg_export_reads.argtypes = [vp] * 8
    lib.amira_gmg_remove_low_coverage_components.argtypes = [vp, u32]
    lib.amira_gmg_filter.argtypes = [vp, u32, u32]
    lib.amira_gmg_filter_mask_sizes.argtypes = [vp, C.POINTER(i64), C.POINTER(i64)]
    lib.amira_gmg_export_filter_masks.argtypes = [vp, vp, vp]
    lib.amira_gmg_nccl_unique_id.argtypes = [vp]
    lib.amira_gmg_comm_init.argtypes = [vp, vp, C.c_int, C.c_int]
    lib.amira_gmg_read_length_coverages.argtypes = [vp, vp, i32, vp]
    lib.amira_gmg_node_coverage_stats.argtypes = [vp, C.POINTER(i64), C.POINTER(u32)]
    lib.amira_gmg_junk_read_mask.argtypes = [vp, C.c_double, vp]
    lib.amira_gmg_nodes_containing.argtypes = [vp, vp, i32, vp]
    lib.amira_gmg_remove_nodes.argtypes = [vp, vp]
    lib.amira_gmg_remove_nodes_without_reads_of.argtypes = [vp, vp, i32]
    lib.amira_gmg_linear_steps.argtypes = [vp] * 8
    lib.amira_gmg_linear_walks.argtypes = [vp, vp, i64, C.c_int, vp, vp]
    lib.amira_gmg_unitigs.argtypes = [vp] * 12
    lib.amira_gmg_unitig_links.argtypes = [vp] * 8
    lib.amira_gmg_read_unitig_paths.argtypes = [vp] * 7
    lib.amira_gmg_bubbles.argtypes = [vp] * 9
    lib.amira_gmg_correct_bubble_reads.argtypes = [vp] * 9 + [C.c_int]
    lib.amira_gmg_bubble_policy.argtypes = [vp, vp, i32, vp, vp]
    lib.amira_gmg_input_calls.argtypes = [vp, vp, i64, i64]
    lib.amira_gmg_debug_layout.argtypes = [vp, C.c_int]
    lib.amira_gmg_debug_segsort.argtypes = [vp, vp, vp, i64, vp, C.POINTER(i64), C.c_int, i64]
    lib.amira_gmg_atomic_peak.argtypes = [vp, i64, i64] + [C.POINTER(C.c_double)] * 3
    _lib = lib
    return lib


def last_error() -> str:
    return load().amira_last_error().decode("utf-8", "replace")


def check(status: int):
    """map a C-ABI status to the exception upstream raises at the same point"""
    if status == OK:
        return
    msg = last_error()
    if status in (E_BLANK_GENE, E_BAD_STRAND, E_EMPTY_NAME, E_PALINDROME, E_EMPTY_GENEMER):
        raise AssertionError(msg)
    if status == E_UNKNOWN_GENE:
        raise KeyError(msg)
    if status == E_MULTI_EDGE:
        raise TypeError(msg)
    if status == E_ARG:
        raise ValueError(msg)
    if status == E_NOMEM:
        raise MemoryError(msg)
    raise AmiraLibraryError("amira_gmg status %d: %s" % (status, msg))
