"""Host-side parts of the minimum spanning tree / single linkage (engine.degree_mst, HSD.single_linkage) that need
no GPU: the MST -> linkage labeller against scipy, and argument validation of the hsd_mst_* entry points."""
import ctypes

import numpy as np
import pytest


def kruskal(D):
    """(u, v, dist) of Kruskal in the order E = (D[u, v], u, v), u < v, over the upper triangle of D.  The
    edges' ranks in that order are distinct weights, so scipy's MST of the rank matrix is that Kruskal's tree."""
    from scipy.sparse.csgraph import minimum_spanning_tree
    n = D.shape[0]
    iu, ju = np.triu_indices(n, 1)
    d = D[iu, ju]
    o = np.lexsort((ju, iu, d))
    W = np.zeros((n, n))
    W[iu[o], ju[o]] = np.arange(1, o.size + 1)
    r = np.sort(minimum_spanning_tree(W).tocoo().data.astype(np.int64) - 1)
    return iu[o][r].astype(np.int32), ju[o][r].astype(np.int32), d[o][r]


def _symmetric(rng, n, levels=None):
    """Symmetric float32 matrix, zero diagonal: distinct pair values (levels None) or a few value levels."""
    D = np.zeros((n, n), np.float32)
    iu = np.triu_indices(n, 1)
    if levels is None:
        D[iu] = (rng.permutation(iu[0].size) + 1).astype(np.float32) / np.float32(1024)
    else:
        D[iu] = rng.integers(0, levels, iu[0].size).astype(np.float32) * np.float32(0.25)
    return D + D.T


def _same_partition(a, b):
    """Two flat-cluster labelings describe the same partition (labels may differ)."""
    _, ia = np.unique(a, return_inverse=True)
    _, ib = np.unique(b, return_inverse=True)
    pairs = np.unique(np.stack([ia, ib], 1), axis=0)
    return pairs.shape[0] == ia.max() + 1 == ib.max() + 1


@pytest.mark.parametrize("n", [3, 7, 40, 200])
def test_linkage_equals_scipy_without_ties(n):
    from scipy.cluster.hierarchy import linkage
    from scipy.spatial.distance import squareform
    from hsd_b200.engine import single_linkage_host
    rng = np.random.default_rng(n)
    for _ in range(5):
        D = _symmetric(rng, n)
        iu = np.triu_indices(n, 1)
        assert np.unique(D[iu]).size == iu[0].size                     # tie-free
        Z = single_linkage_host(*kruskal(D), n)
        want = linkage(squareform(D, checks=False), "single")
        assert Z.dtype == np.float64 and Z.shape == (n - 1, 4)
        assert np.array_equal(Z, want)


@pytest.mark.parametrize("n,levels", [(30, 1), (30, 2), (60, 3), (150, 5), (300, 4)])
def test_linkage_heights_and_partitions_with_ties(n, levels):
    """Many equal distances: the dendrogram is no longer unique, but its heights are, and so is the partition
    fcluster cuts at every height."""
    from scipy.cluster.hierarchy import fcluster, linkage
    from scipy.spatial.distance import squareform
    from hsd_b200.engine import single_linkage_host
    D = _symmetric(np.random.default_rng(n + levels), n, levels)
    Z = single_linkage_host(*kruskal(D), n)
    want = linkage(squareform(D, checks=False), "single")
    assert np.array_equal(Z[:, 2], want[:, 2])
    assert Z[-1, 3] == n and np.all(Z[:, 0] < Z[:, 1])
    for h in np.unique(Z[:, 2]):
        assert _same_partition(fcluster(Z, h, "distance"), fcluster(want, h, "distance")), h


def test_linkage_small_n():
    from hsd_b200.engine import single_linkage_host
    e = np.zeros(0, np.int32)
    assert single_linkage_host(e, e, np.zeros(0, np.float32), 1).shape == (0, 4)
    assert single_linkage_host(e, e, np.zeros(0, np.float32), 0).shape == (0, 4)
    Z = single_linkage_host(np.array([0], np.int32), np.array([1], np.int32), np.array([0.5], np.float32), 2)
    assert np.array_equal(Z, [[0.0, 1.0, 0.5, 2.0]])
    with pytest.raises(ValueError, match="n - 1"):
        single_linkage_host(e, e, np.zeros(0, np.float32), 2)


@pytest.fixture
def buf():
    b = (ctypes.c_int64 * 256)()
    return b, ctypes.addressof(b)


def test_single_linkage_host_argument_validation():
    from hsd_b200._lib import lib
    err = lib.hsd_last_error_string

    def arr(ct, vals):
        a = (ct * max(len(vals), 1))(*vals)
        return ctypes.addressof(a), a

    Z = (ctypes.c_double * 64)()
    z = ctypes.addressof(Z)
    (u, _a), (v, _b), (d, _c) = arr(ctypes.c_int32, [0, 1]), arr(ctypes.c_int32, [1, 2]), arr(ctypes.c_float, [1, 2])
    assert lib.hsd_single_linkage_host(u, v, d, 3, z) == 0 and list(Z[:8]) == [0, 1, 1, 2, 2, 3, 2, 3]
    assert lib.hsd_single_linkage_host(None, v, d, 3, z) == -1 and b"null" in err()
    assert lib.hsd_single_linkage_host(u, v, d, 3, None) == -1 and b"null" in err()
    assert lib.hsd_single_linkage_host(u, v, d, -1, z) == -1 and b"n must be" in err()
    assert lib.hsd_single_linkage_host(None, None, None, 1, None) == 0                  # no edges
    bad_v, _d = arr(ctypes.c_int32, [1, 3])
    assert lib.hsd_single_linkage_host(u, bad_v, d, 3, z) == -1 and b"distinct nodes" in err()
    self_v, _e = arr(ctypes.c_int32, [0, 2])
    assert lib.hsd_single_linkage_host(u, self_v, d, 3, z) == -1 and b"distinct nodes" in err()
    cyc_u, _f = arr(ctypes.c_int32, [0, 1])
    cyc_v, _g = arr(ctypes.c_int32, [1, 0])
    assert lib.hsd_single_linkage_host(cyc_u, cyc_v, d, 3, z) == -1 and b"cycle" in err()
    down, _h = arr(ctypes.c_float, [2, 1])
    assert lib.hsd_single_linkage_host(u, v, down, 3, z) == -1 and b"non-decreasing" in err()
    nan, _i = arr(ctypes.c_float, [1, float("nan")])
    assert lib.hsd_single_linkage_host(u, v, nan, 3, z) == -1 and b"finite" in err()
    neg, _j = arr(ctypes.c_float, [-1, 2])
    assert lib.hsd_single_linkage_host(u, v, neg, 3, z) == -1 and b">= 0" in err()


def test_mst_panel_min_argument_validation_without_gpu(buf):
    """Bad arguments are rejected before any CUDA call, with an error string."""
    from hsd_b200._lib import lib
    _, p = buf
    err = lib.hsd_last_error_string
    # hsd_mst_panel_min(blk, ld, n_rows, n_cols, node0, comp, key_io, stream)
    assert lib.hsd_mst_panel_min(None, 8, 2, 8, 0, p, p, None) == -1 and b"null" in err()
    assert lib.hsd_mst_panel_min(p, 8, 2, 8, 0, None, p, None) == -1 and b"null" in err()
    assert lib.hsd_mst_panel_min(p, 8, 2, 8, 0, p, None, None) == -1 and b"null" in err()
    assert lib.hsd_mst_panel_min(p, 7, 2, 8, 0, p, p, None) == -1 and b"ld" in err()
    assert lib.hsd_mst_panel_min(p, 8, -1, 8, 0, p, p, None) == -1 and b"bad sizes" in err()
    assert lib.hsd_mst_panel_min(p, 8, 9, 8, 0, p, p, None) == -1 and b"n_rows must be <= n_cols" in err()
    assert lib.hsd_mst_panel_min(p, 8, 2, 8, -1, p, p, None) == -1 and b"node ids" in err()
    assert lib.hsd_mst_panel_min(p, 8, 2, 8, 2**31 - 4, p, p, None) == -1 and b"node ids" in err()
    assert lib.hsd_mst_panel_min(p, 8, 0, 8, 0, p, p, None) == 0                          # no rows


def test_mst_list_candidates_argument_validation_without_gpu(buf):
    from hsd_b200._lib import lib
    _, p = buf
    err = lib.hsd_last_error_string
    # hsd_mst_list_candidates(idx, val, n, k, comp, key_out, bound_out, stream)
    for i in range(5):
        args = [p, p, 4, 8, p, p, p, None]
        args[(0, 1, 4, 5, 6)[i]] = None
        assert lib.hsd_mst_list_candidates(*args) == -1 and b"null" in err()
    assert lib.hsd_mst_list_candidates(p, p, 4, 0, p, p, p, None) == -1 and b"k must be" in err()
    assert lib.hsd_mst_list_candidates(p, p, 4, 65, p, p, p, None) == -1 and b"k must be" in err()
    assert lib.hsd_mst_list_candidates(p, p, -1, 8, p, p, p, None) == -1 and b"n must be" in err()
    assert lib.hsd_mst_list_candidates(p, p, 0, 8, p, p, p, None) == 0                    # no nodes


def test_degree_mst_rejects_bad_arguments():
    from hsd_b200 import engine
    with pytest.raises(ValueError, match="cand_k"):
        engine.degree_mst(None, 2, cand_k=65)
    with pytest.raises(ValueError, match="empty"):
        engine.degree_mst(None, 2, empty="skip")
