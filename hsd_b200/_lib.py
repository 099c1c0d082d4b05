"""ctypes binding of libhsd_b200.so (the C-ABI in include/hsd_b200.h).

There is deliberately NO fallback: if the library has not been built, importing
this module raises, and every wrapper raises RuntimeError on a non-zero return
code with the library's own message.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_int32, c_int64, c_void_p, POINTER

from .build import LIB

HEADER_SYMBOLS = [
    "hsd_version", "hsd_last_error_string", "hsd_ring_signature_degree", "hsd_ring_signature_degree_allgather", "hsd_bfs_rings",
    "hsd_bfs_workspace_words", "hsd_bfs_set_workspace",
    "hsd_signature_transpose", "hsd_scatter_symmetric", "hsd_pairwise_l1", "hsd_pairwise_l1_sharded", "hsd_pairwise_l1_tile_list", "hsd_ring_signature_values",
    "hsd_pairwise_w1_merge", "hsd_pairwise_aligned", "hsd_pairwise_worker", "hsd_cheb_spmm", "hsd_laplacian_spmv", "hsd_ring_reduce", "hsd_characteristic_function", "hsd_topk_rows",
    "hsd_fp32_peak_probe", "hsd_copy2d_to_host", "hsd_mirror_upper_to_lower_host", "hsd_exact_wavelets", "hsd_ring_dense_workspace_words", "hsd_ring_signature_degree_dense",
    "hsd_ring_cols_workspace_words", "hsd_ring_counts_dense_cols", "hsd_ring_signature_from_counts",
    "hsd_topk_merge", "hsd_topk_merge_cols",
    "hsd_radius_count", "hsd_radius_emit_rows", "hsd_radius_emit_cols", "hsd_radius_scatter",
    "hsd_radius_merge_parts",
    "hsd_mst_panel_min", "hsd_mst_list_candidates", "hsd_single_linkage_host",
    "hsd_mst_panel_min_mreach", "hsd_mst_list_candidates_mreach", "hsd_hdbscan_host",
]


class HSDLibraryMissing(ImportError):
    pass


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB):
        raise HSDLibraryMissing(
            f"{LIB} is missing: build it with `python -m hsd_b200.build` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "hsd_b200 has no CPU fallback.")
    return ctypes.CDLL(LIB)


lib = _load()
_missing = [s for s in HEADER_SYMBOLS if not hasattr(lib, s)]
if _missing:
    raise HSDLibraryMissing(f"{LIB} is stale (missing {_missing}); rebuild it with `python hsd_b200/build.py --force`")

_P = c_void_p
lib.hsd_version.restype = c_int32
lib.hsd_last_error_string.restype = c_char_p
lib.hsd_ring_signature_degree.argtypes = [_P, _P, c_int32, _P, _P, c_int32, c_int32,
                                          _P, _P, c_int32, _P, c_int64, _P, _P, c_int32, _P, c_int32, _P]
lib.hsd_ring_signature_degree_allgather.argtypes = [_P, _P, c_int32, _P, _P, c_int32, c_int32, _P, _P, c_int32,
                                                    _P, c_int64, _P, c_int32, _P, c_int32, _P, c_int32, _P]
lib.hsd_bfs_workspace_words.argtypes = [c_int32]
lib.hsd_ring_dense_workspace_words.argtypes = [c_int32]
lib.hsd_ring_cols_workspace_words.argtypes = [c_int32, c_int32, c_int32]
lib.hsd_ring_counts_dense_cols.argtypes = [_P, _P, c_int32, c_int64, c_int32, _P, c_int32, c_int32, c_int32, _P, c_int64,
                                           _P, c_int64, _P]
lib.hsd_ring_signature_from_counts.argtypes = [_P, _P, c_int64, _P, _P, c_int32, c_int32, _P, c_int32, _P, c_int64,
                                               _P, c_int32, _P, _P]
lib.hsd_ring_signature_degree_dense.argtypes = [_P, _P, c_int32, _P, _P, c_int32, c_int32, _P, _P, c_int32,
                                                _P, c_int64, _P, c_int32, _P, _P, c_int32, _P, _P, c_int64, c_int64, _P]
lib.hsd_bfs_set_workspace.argtypes = [_P, c_int64]
lib.hsd_bfs_rings.argtypes = [_P, _P, c_int32, _P, _P, c_int32, c_int32, _P, _P, _P]
lib.hsd_signature_transpose.argtypes = [_P, c_int64, c_int32, c_int32, _P, c_int64, c_int32, _P, _P]
lib.hsd_scatter_symmetric.argtypes = [_P, c_int64, c_int32, c_int32, _P, _P, c_int64, c_int32, _P]
lib.hsd_pairwise_l1.argtypes = [_P, c_int32, c_int64, c_int32, c_int32, c_int32, c_int32, c_int32,
                                _P, c_int64, _P]
lib.hsd_pairwise_l1_sharded.argtypes = [_P, c_int32, c_int64, c_int32, c_int32, c_int32, c_int32, _P, c_int64, _P]
lib.hsd_pairwise_l1_tile_list.argtypes = [_P, c_int32, c_int64, c_int32, _P, c_int32, c_int32, c_int32, _P, c_int64, _P]
lib.hsd_ring_signature_values.argtypes = [_P, c_int64, _P, _P, _P, _P, c_int32, c_int32, c_int32,
                                          c_int32, _P, _P]
lib.hsd_pairwise_w1_merge.argtypes = [_P, _P, _P, c_int32, c_int32, c_int32, c_int32, c_int32,
                                      c_int32, _P, c_int64, _P, _P]
lib.hsd_pairwise_aligned.argtypes = [_P, _P, _P, c_int32, c_int32, c_int32, c_int32, c_int32,
                                     c_int32, c_int32, _P, c_int64, _P]
lib.hsd_pairwise_worker.argtypes = [_P, _P, _P, _P, _P, c_int32, c_int32, c_int32, c_int32, c_int32,
                                    c_int32, _P, c_int64, _P]
lib.hsd_cheb_spmm.argtypes = [_P, _P, c_int32, c_double, _P, c_int32, c_int32, c_int32, c_int32,
                              c_double, _P, _P, _P]
lib.hsd_laplacian_spmv.argtypes = [_P, _P, c_int32, _P, _P, _P]
lib.hsd_ring_reduce.argtypes = [_P, c_int32, c_int32, c_int32, _P, _P, _P, c_int32, c_int32, _P, _P, c_int64, _P]
lib.hsd_characteristic_function.argtypes = [_P, c_int64, c_int32, c_int32, _P, c_int32, _P, _P]
lib.hsd_topk_rows.argtypes = [_P, c_int64, c_int32, c_int32, c_int32, c_int32, _P, _P, _P, _P]
lib.hsd_topk_merge.argtypes = [_P, _P, c_int32, c_int64, c_int32, c_int32, c_int32, _P, _P, _P]
lib.hsd_topk_merge_cols.argtypes = [_P, c_int64, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P, _P]
lib.hsd_radius_count.argtypes = [_P, c_int32, c_int64, c_int32, c_int32, c_double, _P, c_int64, _P, _P, _P]
lib.hsd_radius_emit_rows.argtypes = [_P, c_int32, c_int64, c_int32, c_int32, _P, c_int64, _P, c_int32, _P, _P, _P]
lib.hsd_radius_emit_cols.argtypes = [_P, c_int32, c_int64, c_int32, c_int32, _P, c_int64, _P, c_int32, _P, _P, _P]
lib.hsd_radius_scatter.argtypes = [_P, _P, c_int32, _P, c_int32, c_int32, _P, _P, _P, _P, _P]
lib.hsd_radius_merge_parts.argtypes = [c_int32, c_int32, _P, _P, _P, _P, c_int32, _P, _P, _P, _P]
lib.hsd_mst_panel_min.argtypes = [_P, c_int64, c_int32, c_int32, c_int32, _P, _P, _P]
lib.hsd_mst_list_candidates.argtypes = [_P, _P, c_int32, c_int32, _P, _P, _P, _P]
lib.hsd_single_linkage_host.argtypes = [_P, _P, _P, c_int32, _P]
lib.hsd_mst_panel_min_mreach.argtypes = [_P, c_int64, c_int32, c_int32, c_int32, _P, _P, _P, _P]
lib.hsd_mst_list_candidates_mreach.argtypes = [_P, _P, c_int32, c_int32, _P, _P, _P, _P, _P]
lib.hsd_hdbscan_host.argtypes = [_P, c_int32, c_int32, c_int32, c_int32, _P, _P]
lib.hsd_fp32_peak_probe.argtypes = [_P, c_int32, POINTER(c_int64), _P]
lib.hsd_exact_wavelets.argtypes = [_P, c_int64, _P, c_int32, c_double, c_double, c_int32, _P, c_int64, _P]
lib.hsd_copy2d_to_host.argtypes = [_P, c_int64, _P, c_int64, c_int64, c_int64, _P]
lib.hsd_mirror_upper_to_lower_host.argtypes = [_P, c_int64, c_int32, c_int32, c_int32, c_int32]
for _name in HEADER_SYMBOLS:
    if _name not in ("hsd_last_error_string", "hsd_bfs_workspace_words", "hsd_ring_dense_workspace_words",
                     "hsd_ring_cols_workspace_words"):
        getattr(lib, _name).restype = c_int32
lib.hsd_bfs_workspace_words.restype = c_int64
lib.hsd_ring_dense_workspace_words.restype = c_int64
lib.hsd_ring_cols_workspace_words.restype = c_int64


class HSDError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libhsd_b200 error {code}: {msg}")
        self.code = code


def check(rc: int) -> None:
    if rc != 0:
        raise HSDError(rc, (lib.hsd_last_error_string() or b"").decode())
