"""Host-side parts of HDBSCAN (engine.hdbscan_host, HSD.hdbscan) that need no GPU: the labeller against
scikit-learn's tree_to_labels bit for bit, the conventions (core distances, mutual reachability) against
sklearn.cluster.HDBSCAN(metric="precomputed").fit, and argument validation of the new C-ABI entry points."""
import ctypes

import numpy as np
import pytest

from test_host_mst import _symmetric, kruskal


def hierarchy(Z):
    """Z float64[N-1, 4] as scikit-learn's HIERARCHY_dtype."""
    from sklearn.cluster._hdbscan._tree import HIERARCHY_dtype
    H = np.empty(Z.shape[0], dtype=HIERARCHY_dtype)
    H["left_node"], H["right_node"] = Z[:, 0].astype(np.intp), Z[:, 1].astype(np.intp)
    H["value"], H["cluster_size"] = Z[:, 2], Z[:, 3].astype(np.intp)
    return H


def core_distances(D, min_samples):
    """scikit-learn's core distance: the min_samples-th smallest of a row, its zero diagonal counted."""
    return np.partition(D, min_samples - 1, axis=1)[:, min_samples - 1]


def mreach(D, min_samples):
    core = core_distances(D, min_samples)
    return np.maximum(D, np.maximum(core[:, None], core[None, :]))


def _assert_tree_to_labels(Z, n, mcs, method, single):
    from sklearn.cluster._hdbscan._tree import tree_to_labels
    from hsd_b200.engine import hdbscan_host
    want_l, want_p = tree_to_labels(hierarchy(Z), mcs, method, single, 0.0, None)
    got_l, got_p = hdbscan_host(Z, n, mcs, method, single)
    assert got_l.dtype == np.int64 and got_p.dtype == np.float64
    assert np.array_equal(got_l, want_l), (mcs, method, single)
    assert np.array_equal(got_p.view(np.int64), want_p.view(np.int64)), (mcs, method, single)


def _cases(D, n):
    for mcs in sorted({2, 3, 5, n} - {0, 1}):
        for method in ("eom", "leaf"):
            for single in (False, True):
                yield mcs, method, single


@pytest.mark.parametrize("n", [2, 3, 9, 60, 400, 2000])
@pytest.mark.parametrize("kind", ["tie_free", "quantized", "zeros", "mreach5"])
def test_hdbscan_host_equals_tree_to_labels(n, kind):
    """Z of Kruskal in the order E over: a tie-free matrix, a few value levels (many ties, many zero heights:
    lambda = +inf), the all-zero matrix, and the mutual reachability of a quantized matrix at min_samples = 5."""
    from hsd_b200.engine import single_linkage_host
    rng = np.random.default_rng(n * 31 + len(kind))
    D = {"tie_free": lambda: _symmetric(rng, n),
         "quantized": lambda: _symmetric(rng, n, 3),
         "zeros": lambda: np.zeros((n, n), np.float32),
         "mreach5": lambda: mreach(_symmetric(rng, n, 6), min(5, n))}[kind]()
    Z = single_linkage_host(*kruskal(D), n)
    if kind == "zeros" or (kind == "quantized" and n >= 9):
        assert (Z[:, 2] == 0).any()
    for mcs, method, single in _cases(D, n):
        _assert_tree_to_labels(Z, n, mcs, method, single)


def _same_partition(a, b):
    _, ia = np.unique(a, return_inverse=True)
    _, ib = np.unique(b, return_inverse=True)
    return np.unique(np.stack([ia, ib], 1), axis=0).shape[0] == ia.max() + 1 == ib.max() + 1


@pytest.mark.parametrize("n,mcs,min_samples,seed,distinct", [
    (50, 2, 1, 1, True), (50, 2, 2, 2, True), (50, 2, 5, 22, True), (200, 5, 1, 1, True), (200, 5, 2, 2, True),
    (500, 10, 1, 1, True), (500, 10, 2, 2, True), (200, 5, 5, 5, False), (500, 10, 5, 5, False)])
def test_conventions_equal_sklearn_fit(n, mcs, min_samples, seed, distinct):
    """numpy core distances, d_mr and Kruskal's tree from D of a few blobs of points in the plane, labelled, against
    scikit-learn's fit.  The sorted heights are the same for every minimal tree: they must match sklearn's, which
    pins "min_samples includes the point itself".  Where they are pairwise distinct (asserted per case: rare at
    min_samples = 5, where many edges equal some point's core distance) the minimal tree is unique, and the
    partition, the noise set and the probabilities must match too."""
    from sklearn.cluster import HDBSCAN
    from hsd_b200.engine import hdbscan_host, single_linkage_host
    rng = np.random.default_rng(seed)
    pts = rng.normal(size=(n, 2)) + rng.integers(0, 4, n)[:, None] * 6.0
    D = np.sqrt(((pts[:, None] - pts[None, :]) ** 2).sum(-1)).astype(np.float32)
    np.fill_diagonal(D, 0)
    u, v, d = kruskal(mreach(D, min_samples))
    assert (np.unique(d).size == d.size) == distinct
    Z = single_linkage_host(u, v, d, n)
    for method in ("eom", "leaf"):
        for single in (False, True):
            fit = HDBSCAN(metric="precomputed", min_cluster_size=mcs, min_samples=min_samples, copy=True,
                          cluster_selection_method=method, allow_single_cluster=single).fit(D.astype(np.float64))
            assert np.array_equal(np.sort(fit._single_linkage_tree_["value"]), d.astype(np.float64))
            if distinct:
                labels, prob = hdbscan_host(Z, n, mcs, method, single)
                assert np.array_equal(labels == -1, fit.labels_ == -1)
                assert _same_partition(labels, fit.labels_)
                assert np.array_equal(prob, fit.probabilities_)


# ---------------------------------------------------------------- argument validation
def test_hdbscan_host_argument_validation():
    from hsd_b200._lib import lib
    from hsd_b200.engine import hdbscan_host
    err = lib.hsd_last_error_string
    Z = np.array([[0, 1, 0.5, 2], [2, 3, 1.0, 3]], np.float64)
    labels = np.empty(3, np.int64)
    prob = np.empty(3, np.float64)
    z, lp, pp = Z.ctypes.data, labels.ctypes.data, prob.ctypes.data
    assert lib.hsd_hdbscan_host(z, 3, 2, 0, 0, lp, pp) == 0
    assert lib.hsd_hdbscan_host(None, 3, 2, 0, 0, lp, pp) == -1 and b"null" in err()
    assert lib.hsd_hdbscan_host(z, 3, 2, 0, 0, None, pp) == -1 and b"null" in err()
    assert lib.hsd_hdbscan_host(z, 3, 2, 0, 0, lp, None) == -1 and b"null" in err()
    for n in (1, 0, -1):
        assert lib.hsd_hdbscan_host(z, n, 2, 0, 0, lp, pp) == -1 and b"n must be" in err()
    assert lib.hsd_hdbscan_host(z, 3, 1, 0, 0, lp, pp) == -1 and b"min_cluster_size" in err()
    for m in (-1, 2):
        assert lib.hsd_hdbscan_host(z, 3, 2, m, 0, lp, pp) == -1 and b"method" in err()
    for bad in ([[0, 1, 0.5, 2], [0, 3, 1.0, 3]],          # node 0 merged twice
                [[0, 1, 0.5, 2], [2, 4, 1.0, 3]],          # cluster 4 is not formed before row 1
                [[0, 0, 0.5, 2], [1, 2, 1.0, 3]],          # a node merged with itself
                [[0, 1.5, 0.5, 2], [2, 3, 1.0, 3]]):       # not an id
        B = np.array(bad, np.float64)
        assert lib.hsd_hdbscan_host(B.ctypes.data, 3, 2, 0, 0, lp, pp) == -1 and b"row" in err()
    B = np.array([[0, 1, 0.5, 2], [2, 3, 1.0, 4]], np.float64)
    assert lib.hsd_hdbscan_host(B.ctypes.data, 3, 2, 0, 0, lp, pp) == -1 and b"cluster size" in err()
    with pytest.raises(ValueError, match="eom"):
        hdbscan_host(Z, 3, 2, "dbscan")
    with pytest.raises(ValueError, match="n - 1"):
        hdbscan_host(Z, 4, 2)


@pytest.fixture
def buf():
    b = (ctypes.c_int64 * 256)()
    return b, ctypes.addressof(b)


def test_mst_panel_min_mreach_argument_validation_without_gpu(buf):
    from hsd_b200._lib import lib
    _, p = buf
    err = lib.hsd_last_error_string
    # hsd_mst_panel_min_mreach(blk, ld, n_rows, n_cols, node0, comp, core, key_io, stream)
    for i in (0, 5, 6, 7):
        args = [p, 8, 2, 8, 0, p, p, p, None]
        args[i] = None
        assert lib.hsd_mst_panel_min_mreach(*args) == -1 and b"null" in err()
    assert lib.hsd_mst_panel_min_mreach(p, 7, 2, 8, 0, p, p, p, None) == -1 and b"ld" in err()
    assert lib.hsd_mst_panel_min_mreach(p, 8, -1, 8, 0, p, p, p, None) == -1 and b"bad sizes" in err()
    assert lib.hsd_mst_panel_min_mreach(p, 8, 9, 8, 0, p, p, p, None) == -1 and b"n_rows must be <= n_cols" in err()
    assert lib.hsd_mst_panel_min_mreach(p, 8, 2, 8, -1, p, p, p, None) == -1 and b"node ids" in err()
    assert lib.hsd_mst_panel_min_mreach(p, 8, 2, 8, 2**31 - 4, p, p, p, None) == -1 and b"node ids" in err()
    assert lib.hsd_mst_panel_min_mreach(p, 8, 0, 8, 0, p, p, p, None) == 0                # no rows


def test_mst_list_candidates_mreach_argument_validation_without_gpu(buf):
    from hsd_b200._lib import lib
    _, p = buf
    err = lib.hsd_last_error_string
    # hsd_mst_list_candidates_mreach(idx, val, n, k, comp, core, key_out, bound_out, stream)
    for i in (0, 1, 4, 5, 6, 7):
        args = [p, p, 4, 8, p, p, p, p, None]
        args[i] = None
        assert lib.hsd_mst_list_candidates_mreach(*args) == -1 and b"null" in err()
    assert lib.hsd_mst_list_candidates_mreach(p, p, 4, 0, p, p, p, p, None) == -1 and b"k must be" in err()
    assert lib.hsd_mst_list_candidates_mreach(p, p, 4, 65, p, p, p, p, None) == -1 and b"k must be" in err()
    assert lib.hsd_mst_list_candidates_mreach(p, p, -1, 8, p, p, p, p, None) == -1 and b"n must be" in err()
    assert lib.hsd_mst_list_candidates_mreach(p, p, 0, 8, p, p, p, p, None) == 0          # no nodes


def test_degree_mreach_mst_rejects_bad_arguments():
    from types import SimpleNamespace
    from hsd_b200 import engine
    dg = SimpleNamespace(n=10)
    for ms in (0, 66, 11):
        with pytest.raises(ValueError, match="min_samples"):
            engine.degree_mreach_mst(dg, 2, ms)
    with pytest.raises(ValueError, match="cand_k"):
        engine.degree_mreach_mst(dg, 2, 5, cand_k=65)
    with pytest.raises(ValueError, match="empty"):
        engine.degree_mreach_mst(dg, 2, 5, empty="skip")
