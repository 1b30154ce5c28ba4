"""ctypes binding of libbadger_b200.so (include/badger_b200.h).

The shared library is built in-tree by ``__graft_entry__.build()`` / ``make -C badger_b200/csrc``.
There is no CPU fallback: if the library is missing, or no B200 is visible, every operator raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libbadger_b200.so")

BDG_OK, BDG_ERR_CUDA, BDG_ERR_OOM, BDG_ERR_ARG, BDG_ERR_NODEVICE, BDG_ERR_CAPACITY, BDG_ERR_UNSUPPORTED, BDG_ERR_IO = 0, -1, -2, -3, -4, -5, -6, -7
ROW_TILE = 2048  # BDG_ROW_TILE


class BadgerB200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("libbadger_b200: %s (code %d)" % (msg, code))
        self.code = code


_lib = None
_vp, _sz, _i = C.c_void_p, C.c_size_t, C.c_int


def lib():
    """Load the library once; raise loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BadgerB200Error(BDG_ERR_NODEVICE, "%s not found - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "or `make -C badger_b200/csrc`; there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.bdg_last_error.restype = C.c_char_p
    L.bdg_version.restype = C.c_char_p
    L.bdg_init.argtypes = [_vp, _i]
    L.bdg_device_count.restype = _i
    L.bdg_launch_count.restype = C.c_ulonglong
    L.bdg_host_alloc.argtypes = [_sz, C.POINTER(_vp)]
    L.bdg_host_free.argtypes = [_vp]
    L.bdg_host_free.restype = None
    L.bdg_pack16.argtypes = [_vp, _sz, _vp, _vp]
    L.bdg_pack16_sorted.argtypes = [_vp, _sz, _vp, C.POINTER(_sz)]
    L.bdg_assign_reads32.argtypes = [C.c_ulonglong, _vp, _sz, _vp, _vp, _sz, C.POINTER(_sz)]
    L.bdg_dedup_fetch.argtypes = [C.c_ulonglong, _vp, _vp, _vp, _vp]
    L.bdg_centres_above.argtypes = [C.c_ulonglong, _sz, _vp, _sz, _vp, _vp, _vp, _sz, C.POINTER(_sz), C.POINTER(C.c_double)]
    L.bdg_centres_rest.argtypes = [C.c_ulonglong, C.c_double, _sz, _vp, C.POINTER(_sz)]
    L.bdg_cluster_resident.argtypes = [_vp, _sz, _vp, _sz, _i, C.POINTER(_sz)]
    L.bdg_tsv_write_assignments32.argtypes = [_vp, C.c_char_p, _vp, _vp, _i]
    L.bdg_dedup_first_seen.argtypes = [_vp, _sz, _vp, _vp, _vp, _vp, C.POINTER(_sz)]
    L.bdg_dedup_reads.argtypes = [_vp, _vp, _sz, _vp, _vp, _vp, _vp, C.POINTER(_sz), C.POINTER(_sz), C.POINTER(C.c_ulonglong)]
    L.bdg_edges_build.argtypes = [_vp, _sz, _i, C.POINTER(_vp)]
    L.bdg_edges_build_part.argtypes = [_vp, _sz, _i, _i, _i, C.POINTER(_vp)]
    L.bdg_edges_build_resident.argtypes = [C.c_ulonglong, _i, C.POINTER(_vp)]
    L.bdg_edges_build_into.argtypes = [_vp, _sz, _i, _i, _i, _vp, _vp, _vp, _sz, C.POINTER(_sz)]
    L.bdg_edges_count.argtypes = [_vp]
    L.bdg_edges_count.restype = _sz
    L.bdg_edges_copy.argtypes = [_vp, _vp, _vp, _vp]
    L.bdg_edges_free.argtypes = [_vp]
    L.bdg_edges_free.restype = None
    L.bdg_cluster_levels.argtypes = [_vp, _sz, _vp, _vp, _sz, _vp, _sz, _i, _vp, _vp]
    L.bdg_cluster_levels_from_edges.argtypes = [_vp, _sz, _vp, _sz, _i, _vp, _vp]
    L.bdg_member_sorted.argtypes = [_vp, _sz, _vp, _sz, _vp]
    L.bdg_nearest_bounded.argtypes = [_vp, _sz, _vp, _sz, _i, _vp, _vp]
    L.bdg_kmer_score.argtypes = [_vp, _sz, _vp, _sz, _i, _sz, _vp, _vp, _vp, _vp, C.POINTER(_sz)]
    L.bdg_kmer_index_create.argtypes = [_vp, _sz, C.POINTER(_vp)]
    L.bdg_kmer_index_query.argtypes = [_vp, _vp, _sz, _i, _sz, _vp, _vp, _vp, _vp, C.POINTER(_sz)]
    L.bdg_kmer_index_free.argtypes = [_vp]
    L.bdg_kmer_index_free.restype = None
    L.bdg_kmer_index_info.argtypes = [_vp, C.POINTER(C.c_int), C.POINTER(C.c_double)]
    L.bdg_dev_edges_build.argtypes = [_vp, _sz, _i, _i, _i, _vp, _vp, _vp, _sz, _vp, _vp]
    L.bdg_set_edge_mode.argtypes = [_i]
    L.bdg_dev_edges_stats.argtypes = [C.POINTER(C.c_ulonglong), _vp]
    L.bdg_dev_edges_stats_raw.argtypes = [C.POINTER(C.c_ulonglong), _vp]
    L.bdg_join_lane_stats.argtypes = [C.POINTER(C.c_ulonglong), _i]
    L.bdg_dev_edges_balance.argtypes = [C.POINTER(C.c_ulonglong), _vp]
    L.bdg_dev_pack16.argtypes = [_vp, _sz, _vp, _vp, _vp]
    L.bdg_dev_member_sorted.argtypes = [_vp, _sz, _vp, _sz, _vp, _vp]
    L.bdg_dev_nearest_bounded.argtypes = [_vp, _sz, _vp, _sz, _i, _vp, _vp, _vp, _vp]
    L.bdg_dev_dedup_reads.argtypes = [_vp, _vp, _sz, C.POINTER(_sz), C.POINTER(_sz), C.POINTER(C.c_ulonglong), _vp]
    L.bdg_dev_dedup_fetch.argtypes = [C.c_ulonglong, _vp, _vp, _vp, _vp, _vp]
    L.bdg_dev_pack16_sorted.argtypes = [_vp, _sz, _vp, C.POINTER(_sz), _vp]
    L.bdg_dev_centres_above.argtypes = [C.c_ulonglong, _sz, _vp, _sz, _vp, _vp, _vp, _sz, C.POINTER(_sz), C.POINTER(C.c_double), _vp]
    L.bdg_dev_edges_copy.argtypes = [_vp, _vp, _vp, _vp, _vp]
    L.bdg_dev_assign_reads32.argtypes = [C.c_ulonglong, _vp, _sz, _vp, _vp, _sz, C.POINTER(_sz), _vp]
    L.bdg_dev_dedup_merge.argtypes = [C.c_ulonglong, _vp, _vp, _vp, _vp, _vp, _i, _i, C.POINTER(_sz), C.POINTER(C.c_ulonglong), _vp]
    L.bdg_dev_index_edges.argtypes = [_vp, _sz, _vp, _vp, _sz, _vp, _vp, _vp]
    L.bdg_dev_cluster_init.argtypes = [_vp, _sz, _vp, _sz, _vp, _vp, _vp, _vp, _vp]
    L.bdg_dev_cluster_mark.argtypes = [_vp, _vp, _sz, _vp, _vp, _vp]
    L.bdg_dev_cluster_claim.argtypes = [_vp, _vp, _sz, _i, _vp, _vp, _vp, _vp, _vp]
    L.bdg_dev_cluster_resolve.argtypes = [_vp, _vp, _vp, _vp, _sz, _i, _vp]
    L.bdg_dev_whitelist_check.argtypes = [_vp, _sz, _vp]
    L.bdg_dev_kmer_index_create.argtypes = [_vp, _sz, _vp, C.POINTER(_vp)]
    L.bdg_dev_kmer_index_query.argtypes = [_vp, _vp, _sz, _i, _sz, _vp, _vp, _vp, _vp, C.POINTER(_sz), _vp]
    L.bdg_dev_kmer_score.argtypes = [_vp, _sz, _vp, _sz, _i, _sz, _vp, _vp, _vp, _vp, C.POINTER(_sz), _vp]
    L.bdg_tally_create.argtypes = [C.POINTER(_vp)]
    L.bdg_tally_free.argtypes = [_vp]
    L.bdg_tally_free.restype = None
    L.bdg_tally_add.argtypes = [_vp, _vp, _vp, _sz, C.POINTER(_sz)]
    L.bdg_dev_tally_add.argtypes = [_vp, _vp, _vp, _sz, C.POINTER(_sz), _vp]
    L.bdg_tally_finish.argtypes = [_vp, C.POINTER(_sz), C.POINTER(_sz), C.POINTER(C.c_ulonglong)]
    L.bdg_dev_tally_finish.argtypes = [_vp, C.POINTER(_sz), C.POINTER(_sz), C.POINTER(C.c_ulonglong), _vp]
    L.bdg_tally_info.argtypes = [_vp, C.POINTER(_sz), C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]
    L.bdg_dev_tally_copy.argtypes = [_vp, _vp, _vp, _vp, _vp]
    L.bdg_dev_tally_merge_parts.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, C.c_ulonglong, C.c_ulonglong, _vp]
    L.bdg_assign_lookup32.argtypes = [C.c_ulonglong, _vp, _sz, _vp, _vp, _sz, _vp, _vp, C.POINTER(_sz), C.POINTER(_sz)]
    L.bdg_dev_assign_lookup32.argtypes = [C.c_ulonglong, _vp, _sz, _vp, _vp, _sz, _vp, _vp, C.POINTER(_sz), C.POINTER(_sz), _vp]
    L.bdg_part_pairs.argtypes = [_sz, _i, _i]
    L.bdg_part_pairs.restype = C.c_ulonglong
    L.bdg_dev_pipe_probe.argtypes = [_i, _i, _i, _vp, C.POINTER(C.c_ulonglong), _vp]
    L.bdg_tsv_open.argtypes = [C.c_char_p, _i, _i, C.POINTER(_vp)]
    L.bdg_tsv_rows.argtypes = [_vp]
    L.bdg_tsv_rows.restype = _sz
    L.bdg_tsv_barcodes.argtypes = [_vp, _vp, _vp]
    L.bdg_tsv_write_assignments.argtypes = [_vp, C.c_char_p, _vp, _i]
    L.bdg_tsv_close.argtypes = [_vp]
    L.bdg_tsv_close.restype = None
    L.bdg_lines16_open.argtypes = [C.c_char_p, C.POINTER(_vp)]
    L.bdg_lines16_count.argtypes = [_vp]
    L.bdg_lines16_count.restype = _sz
    L.bdg_lines16_data.argtypes = [_vp]
    L.bdg_lines16_data.restype = _vp
    L.bdg_lines16_close.argtypes = [_vp]
    L.bdg_lines16_close.restype = None
    for name in ("bdg_init", "bdg_host_alloc", "bdg_pack16", "bdg_dedup_first_seen", "bdg_edges_build", "bdg_edges_build_part", "bdg_edges_build_resident", "bdg_edges_build_into", "bdg_edges_copy", "bdg_cluster_levels", "bdg_cluster_levels_from_edges", "bdg_member_sorted",
                 "bdg_nearest_bounded", "bdg_kmer_score", "bdg_kmer_index_create", "bdg_kmer_index_query", "bdg_dev_edges_build", "bdg_set_edge_mode", "bdg_dev_edges_stats", "bdg_dev_edges_stats_raw", "bdg_dev_edges_balance", "bdg_join_lane_stats", "bdg_dev_pack16", "bdg_dev_member_sorted",
                 "bdg_dev_nearest_bounded", "bdg_dev_pipe_probe", "bdg_tsv_open", "bdg_tsv_barcodes", "bdg_tsv_write_assignments", "bdg_lines16_open", "bdg_dedup_reads", "bdg_pack16_sorted", "bdg_assign_reads32", "bdg_dedup_fetch", "bdg_centres_above", "bdg_centres_rest", "bdg_cluster_resident",
                 "bdg_tsv_write_assignments32", "bdg_dev_dedup_reads", "bdg_dev_dedup_fetch", "bdg_dev_pack16_sorted", "bdg_dev_centres_above",
                 "bdg_dev_edges_copy", "bdg_dev_assign_reads32", "bdg_dev_dedup_merge", "bdg_dev_index_edges", "bdg_dev_cluster_init",
                 "bdg_dev_cluster_mark", "bdg_dev_cluster_claim", "bdg_dev_cluster_resolve", "bdg_dev_whitelist_check",
                 "bdg_dev_kmer_index_create", "bdg_dev_kmer_index_query", "bdg_dev_kmer_score", "bdg_tally_create", "bdg_tally_add",
                 "bdg_dev_tally_add", "bdg_tally_finish", "bdg_dev_tally_finish", "bdg_tally_info", "bdg_dev_tally_copy",
                 "bdg_dev_tally_merge_parts", "bdg_assign_lookup32", "bdg_dev_assign_lookup32"):
        getattr(L, name).restype = _i
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != BDG_OK:
        raise BadgerB200Error(rc, (lib().bdg_last_error() or b"").decode(errors="replace"))


_first_device = 0        # the first device of the last successful init (a call that initialises the library itself claims all, from 0)


def init(device_ids=None) -> int:
    """bdg_init: claim the listed CUDA devices (default: all visible). Returns the device count."""
    global _first_device
    L = lib()
    if not device_ids:
        check(L.bdg_init(None, 0))
        _first_device = 0
    else:
        arr = (C.c_int * len(device_ids))(*device_ids)
        check(L.bdg_init(arr, len(device_ids)))
        _first_device = int(device_ids[0])
    return L.bdg_device_count()


def first_device() -> int:
    """The CUDA device the read map and the bdg_dev_* correction-step calls live on: the first device given to init()."""
    return _first_device


def ptr(a: np.ndarray):
    return a.ctypes.data if a.size else None
