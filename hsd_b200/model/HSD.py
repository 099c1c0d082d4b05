"""Drop-in for the reference's ``model/HSD.py`` (class HSD, model/HSD.py:17-161).

Same constructor, attributes and method names; the bodies run on the B200
through libhsd_b200.  Differences a caller can see, all additive:

* ``signal`` (ctor keyword, default "wavelet"): "degree" switches the ring
  signal from Psi[i, j] to deg(j) — the formulation the large synthetic
  configs use (BASELINE.json); then ``scale`` / ``approx`` are ignored.
* ``A`` / ``L`` are built lazily (dense N x N is 80 GB at N = 100k).
* ``init()`` builds the rings with the BFS kernel when no ``.layers`` file is
  configured (the reference reads a hard-coded absolute path, tools/const.py:12).
* drift aliases the reference's own callers use but its class lacks
  (SURVEY.md F8): ``construct_hierarchy()``, ``laplacian``, ``wavelets``.
* ``n_workers`` arguments are accepted and ignored (one process per GPU).
"""
from __future__ import annotations

import os

import networkx as nx
import numpy as np
import torch

from .. import engine, rings as _rings, wavelets as _wav
from ..graph import CSRGraph, has_nonunit_weights
from ..tools import hierarchy as _hierarchy
from ..tools import util
from ._device import on_model_device


class HSD(object):

    CHEB_ORDER = 50          # model/HSD.py:53
    THRESHOLD_COEFF = 1e-4   # model/HSD.py:65

    def __init__(self, graph, graphName, scale, hop, metric, signal="wavelet", device=None):
        """
        Hierarchical Structural Distance model (model/HSD.py:19-40).
        :param graph: nx.Graph
        :param graphName: the name of graph
        :param scale: the heat coefficient
        :param hop: k-hop local neighborhoods
        :param metric: 'Wasserstein' or 'Hellinger'
        :param signal: 'wavelet' (reference) or 'degree'
        """
        if signal not in ("wavelet", "degree"):
            raise ValueError("signal must be 'wavelet' or 'degree'")
        self.graph = graph
        self.graphName = graphName
        self.scale = scale
        self.hop = hop
        self.metric = metric
        self.signal = signal
        self.device = device

        self.nodes = list(nx.nodes(graph))
        self.n_node = len(self.nodes)
        self.idx2node, self.node2idx = util.build_node_idx_map(graph)
        self._hierarchy = None
        self._hierarchy_lazy = False
        self.wavelets = None
        self.distMat = None
        self.eigenvalues = None
        self.eigenvectors = None
        self.lmax = None
        self.empty = "raise"   # empty-ring policy in degree mode: 'raise' (scipy) | 'zero'

        self.csr = CSRGraph.from_networkx(graph)
        # every edge list the reference ships is unweighted; the CSR kernels assume unit weights
        self._weighted = has_nonunit_weights(graph)
        self._A = None
        self._L = None
        self._dg = None
        self._dcsr = None
        self._ringset = None
        self._ringset_src = None
        self._host_pipe = None

    # ---- lazy dense matrices (model/HSD.py:33-34) ----
    @property
    def A(self):
        if self._A is None:
            self._A = nx.adjacency_matrix(self.graph).todense()
        return self._A

    @property
    def L(self):
        if self._L is None:
            self._L = nx.laplacian_matrix(self.graph).todense()
        return self._L

    @property
    def laplacian(self):  # alias read by main.py:21, tests/robust_test/main.py:174
        return self.L

    # ---- rings in the reference's dict form; built from the device bitmaps on first read ----
    @property
    def hierarchy(self):
        if self._hierarchy is None and self._hierarchy_lazy:
            with torch.cuda.device(self._device()):
                self._hierarchy = self._rings().to_hierarchy(self.nodes)
            self._ringset_src = self._hierarchy   # same rings: keep the device copy
            self._hierarchy_lazy = False
        return self._hierarchy

    @hierarchy.setter
    def hierarchy(self, value):
        self._hierarchy = value
        self._hierarchy_lazy = False

    # ---- device state ----
    def _device(self):
        """The CUDA device of this model (the ctor's `device`, else the current device).  The C
        library launches on the CURRENT device, so every public entry point that reaches a
        kernel runs under `torch.cuda.device(self._device())` (see _on_model_device)."""
        if self.device is None:
            return engine.require_cuda()
        return torch.device(self.device)

    def _device_graph(self, include_zero=False) -> engine.DeviceGraph:
        if self._dg is None or self._dg.include_zero != include_zero:
            self._dg = engine.DeviceGraph.upload(self.csr, include_zero=include_zero, device=self._device())
        return self._dg

    def _device_csr(self) -> _wav.DeviceCSR:
        if self._dcsr is None:
            self._dcsr = _wav.DeviceCSR(self.csr, self._device())
        return self._dcsr

    def _rings(self) -> _rings.RingSet:
        """Rings as device bitmaps: from a caller-assigned dict (tests/robust_test/main.py:179)
        when there is one, else from the BFS kernel."""
        if self._hierarchy is not None:
            if self._ringset is None or self._ringset_src is not self._hierarchy:
                self._ringset = _rings.RingSet.from_hierarchy(self._hierarchy, self.nodes, self.node2idx,
                                                              self.hop, self._device())
                self._ringset_src = self._hierarchy
            return self._ringset
        if self._ringset is None or self._ringset.hops != self.hop or self._ringset_src is not None:
            self._ringset = _rings.RingSet.bfs(self._device_graph(), self.hop)
            self._ringset_src = None
        return self._ringset

    # init HSD model (model/HSD.py:43-44)
    def init(self):
        path = os.environ.get("HSD_HIERARCHY_DIR")
        if path and os.path.exists(os.path.join(path, f"{self.graphName}.layers")):
            self.hierarchy = _hierarchy.read_hierarchy(os.path.join(path, f"{self.graphName}.layers"), self.hop)
        else:
            self.construct_hierarchy()

    def construct_hierarchy(self):
        """Alias used by main.py:15: (re)build the k-hop rings with the BFS kernel.  Lazy: the
        kernel runs when the rings are first needed, and the dict form (``model.hierarchy``) is
        materialised from the device bitmaps on first read — the degree-signal path never needs
        the ring bitmaps at all (they are 6 GB at N = 100k, hop 4)."""
        self._hierarchy = None
        self._ringset = None
        self._ringset_src = None
        self._hierarchy_lazy = True   # the BFS runs on first use (distances / embeddings / model.hierarchy)

    # ---- wavelets (model/HSD.py:48-67) ----
    def _wavelets_device(self, scale, approx=True) -> torch.Tensor:
        if approx:
            if self._weighted:
                raise NotImplementedError("the Chebyshev kernel takes unit edge weights; use approx=False "
                                          "(dense eigh honours weights like the reference)")
            if self.lmax is None:
                self.lmax = _wav.estimate_lmax(self.csr, device=self._device())
            return _wav.cheb_wavelets_dense(self._device_csr(), float(scale), self.lmax,
                                            self.CHEB_ORDER, self.THRESHOLD_COEFF)
        if self.eigenvalues is not None and self.eigenvectors is not None:
            eig = (torch.as_tensor(np.asarray(self.eigenvalues), dtype=torch.float64, device=self._device()),
                   torch.as_tensor(np.asarray(self.eigenvectors), dtype=torch.float64, device=self._device()))
        else:
            eig = None
        L = torch.as_tensor(np.asarray(self.L, dtype=np.float64), device=self._device())
        return _wav.exact_wavelets_dense(L, float(scale), self.THRESHOLD_COEFF, eig)

    @on_model_device
    def calculate_wavelets(self, scale, approx=True) -> np.ndarray:
        psi = self._wavelets_device(scale, approx)
        self.wavelets = psi.cpu().numpy()
        return self.wavelets

    # model/HSD.py:71-83
    @on_model_device
    def get_hierarchical_coeffcients(self, wavelets) -> dict:
        mem = self._rings().members_host()
        w = np.asarray(wavelets)
        return {node: [list(w[i, layer]) for layer in mem[i]] for i, node in enumerate(self.nodes)}

    # model/HSD.py:87-94
    @on_model_device
    def get_nodes_hierarchical_degree(self) -> dict:
        sizes = self._rings().sizes.cpu().numpy()
        out = {}
        for i, node in enumerate(self.nodes):
            hop_degree = [int(x) for x in sizes[i]]
            if len(hop_degree) < self.hop:
                hop_degree = hop_degree + [0] * (self.hop - len(hop_degree))
            out[node] = hop_degree
        return out

    # ---- distances ----
    @on_model_device
    def structural_distance_device(self, scale=None, approx=False) -> torch.Tensor:
        """Device-resident result (float32 in degree mode, float64 in wavelet mode)."""
        if self.signal == "degree":
            dg = self._device_graph(include_zero=(self.empty == "zero"))
            D, _ = engine.degree_distance_device(dg, self.hop, empty=self.empty)
            return D
        psi = self._wavelets_device(self.scale if scale is None else scale, approx)
        return _rings.value_distance(psi, self._rings(), 0, self.hop + 1, mode="w1")

    @on_model_device
    def calculate_structural_distance(self, scale, approx=False, out=None):
        """model/HSD.py:98-114: D[i, j] = sum_{h=0..hop} W1(ring signal_i[h], ring signal_j[h]).
        Returns a float64 ndarray like the reference; ``out`` (a pinned float32/float64
        host tensor or ndarray of shape (N, N)) receives the result instead when given."""
        if out is not None and self.signal == "degree":
            # host-buffer pipeline: H2D of the CSR, kernels, and the D2H of finished row panels
            # overlapped with the panels still computing (engine.HostDegreePipeline)
            dst = out if isinstance(out, torch.Tensor) else torch.from_numpy(out)
            pipe = self._host_pipe
            if pipe is None or pipe.g is not self.csr or pipe.hops != self.hop or pipe.empty != self.empty:
                pipe = self._host_pipe = engine.HostDegreePipeline(self.csr, self.hop, empty=self.empty,
                                                                   device=self._device())
            if dst.dtype == torch.float32:
                pipe.run(dst)
            elif dst.dtype == torch.float64:
                # the kernels produce float32: stage through a pinned float32 buffer, widen on the host
                if getattr(self, "_host_stage", None) is None or self._host_stage.shape != dst.shape:
                    self._host_stage = torch.empty(dst.shape, dtype=torch.float32).pin_memory()
                pipe.run(self._host_stage)
                dst.copy_(self._host_stage)
            else:
                raise ValueError("out must be float32 or float64")
            return out
        D = self.structural_distance_device(scale, approx)
        if out is not None:
            dst = out if isinstance(out, torch.Tensor) else torch.from_numpy(out)
            dst.copy_(D, non_blocking=False)
            return out
        return D.cpu().numpy().astype(np.float64, copy=False)

    @on_model_device
    def nearest_neighbors(self, k, scale=None, approx=False, block_bytes=None):
        """(idx, dist): the k structurally closest nodes of every node, selected on the device
        — what a precomputed-metric KNN (tools/evaluate.py:61-69) needs, without moving the N x N
        matrix to the host.  idx are node indices (model.nodes), ordered by (distance, index).
        Degree mode sweeps the matrix in row panels of at most ``block_bytes`` (default: half the
        free device memory) and never holds it whole (engine.degree_knn), so graphs whose matrix
        exceeds the device memory work too; wavelet mode selects from the resident matrix."""
        if self.signal == "degree":
            dg = self._device_graph(include_zero=(self.empty == "zero"))
            idx, val = engine.degree_knn(dg, self.hop, k, empty=self.empty, block_bytes=block_bytes)
            return idx.cpu().numpy(), val.cpu().numpy()
        D = self.structural_distance_device(scale, approx)
        if D.dtype != torch.float32:
            D = D.to(torch.float32)
        idx, val = engine.topk_rows(D.contiguous(), k)
        return idx.cpu().numpy(), val.cpu().numpy()

    @on_model_device
    def radius_neighbors(self, radius, scale=None, approx=False, block_bytes=None, max_pairs=None):
        """(indptr, indices, dist): the radius graph — every pair of nodes whose structural distance is
        at most ``radius`` — as a canonical CSR over node indices (model.nodes): row i lists every j != i
        with float(D[i, j]) <= radius in ascending j, D being the matrix structural_distance_device holds.
        The graph is exactly symmetric and keeps distance-0 pairs (radius 0 lists the pairs the distance
        cannot tell apart), so ``scipy.sparse.csr_matrix((dist, indices, indptr), shape=(N, N))`` is
        what DBSCAN(metric="precomputed") and graph clustering take.  indptr int64[N+1], indices
        int32[nnz], dist float32 (degree mode) / float64 (wavelet mode).
        radius: >= 0 (+inf: every pair); NaN or negative raise ValueError.
        block_bytes: as for nearest_neighbors — degree mode sweeps the matrix in row panels of at most
        this size (engine.degree_radius) and never holds it whole; wavelet mode thresholds the resident
        matrix (engine.radius_resident).
        max_pairs: cap on nnz (stored entries, twice the pairs); the default is engine.radius_max_pairs
        of the free device memory.  Past it ValueError, and the call's device buffers are released."""
        radius = engine.check_radius(radius)
        if self.signal == "degree":
            dg = self._device_graph(include_zero=(self.empty == "zero"))
            out = engine.degree_radius(dg, self.hop, radius, empty=self.empty, block_bytes=block_bytes,
                                       max_pairs=max_pairs)
        else:
            D = self.structural_distance_device(scale, approx)
            try:
                out = engine.radius_resident(D, radius, max_pairs=max_pairs)
            finally:
                del D                    # also on the max_pairs error: its traceback keeps this frame
        return tuple(t.cpu().numpy() for t in out)

    @on_model_device
    def nearest_neighbors_sharded(self, k, rank, world, group=None, block_bytes=None):
        """nearest_neighbors over `world` GPUs (degree mode; one process per GPU, torch.distributed
        initialised): every rank builds its dealt share of the signatures and sweeps its share of the
        row panels; every rank returns the whole (idx, dist), equal to the one-GPU result bit for bit."""
        if self.signal != "degree":
            raise NotImplementedError("nearest_neighbors_sharded is degree mode only (signal='degree')")
        if not 0 <= rank < world:
            raise ValueError("rank must be in 0..world-1")
        import torch.distributed as dist
        if world > 1 and not (dist.is_available() and dist.is_initialized()):
            # without a process group the ranks' lists could not be combined: this rank's would be partial
            raise RuntimeError("nearest_neighbors_sharded with world > 1 needs an initialised torch.distributed "
                               "process group (one process per GPU)")
        dg = self._device_graph(include_zero=(self.empty == "zero"))
        idx, val = engine.degree_knn(dg, self.hop, k, empty=self.empty, block_bytes=block_bytes,
                                     rank=rank, world=world, group=group)
        return idx.cpu().numpy(), val.cpu().numpy()

    @on_model_device
    def radius_neighbors_sharded(self, radius, rank, world, group=None, block_bytes=None, max_pairs=None):
        """radius_neighbors over `world` GPUs (degree mode; one process per GPU, torch.distributed
        initialised): every rank builds its dealt share of the signatures and sweeps its share of the row
        panels, then the ranks' partial graphs are gathered and merged on every rank.  Every rank returns
        the whole (indptr, indices, dist), equal to the one-GPU result bit for bit.  max_pairs caps the
        global nnz (default engine.radius_sharded_max_pairs, the MIN over the ranks); past it every rank
        raises the same ValueError."""
        if self.signal != "degree":
            raise NotImplementedError("radius_neighbors_sharded is degree mode only (signal='degree')")
        if not 0 <= rank < world:
            raise ValueError("rank must be in 0..world-1")
        radius = engine.check_radius(radius)
        import torch.distributed as dist
        if world > 1 and not (dist.is_available() and dist.is_initialized()):
            # without a process group the ranks' graphs could not be combined: this rank's would be partial
            raise RuntimeError("radius_neighbors_sharded with world > 1 needs an initialised torch.distributed "
                               "process group (one process per GPU)")
        dg = self._device_graph(include_zero=(self.empty == "zero"))
        out = engine.degree_radius(dg, self.hop, radius, empty=self.empty, block_bytes=block_bytes,
                                   max_pairs=max_pairs, rank=rank, world=world, group=group)
        return tuple(t.cpu().numpy() for t in out)

    @on_model_device
    def minimum_spanning_tree(self, block_bytes=None):
        """(u, v, dist): the minimum spanning tree of the complete graph over the nodes under the structural
        distance (degree mode).  u < v are int32[N-1] node indices (model.nodes), dist float32[N-1], sorted by
        (dist, u, v).  It is the unique MST under the order E(u, v) = (float(D[u, v]), u, v), D being the matrix
        structural_distance_device holds: Kruskal in that order on D, bit for bit.  Built by Borůvka rounds over
        row panels of at most ``block_bytes`` (as for nearest_neighbors; engine.degree_mst), so graphs whose
        matrix exceeds the device memory work too."""
        if self.signal != "degree":
            raise NotImplementedError("minimum_spanning_tree is degree mode only (signal='degree')")
        if self.n_node == 0:
            return np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32)
        dg = self._device_graph(include_zero=(self.empty == "zero"))
        out = engine.degree_mst(dg, self.hop, empty=self.empty, block_bytes=block_bytes)
        return tuple(t.cpu().numpy() for t in out)

    def single_linkage(self, block_bytes=None):
        """Z float64[N-1, 4]: the single-linkage dendrogram in scipy's linkage format, which
        scipy.cluster.hierarchy.fcluster and dendrogram take as is.  Row t merges clusters Z[t, 0] < Z[t, 1] at
        height Z[t, 2], the t-th edge of minimum_spanning_tree, into a cluster of Z[t, 3] nodes; ids below N are
        nodes (model.nodes), N + t is the cluster row t formed.  Where all pair distances differ, Z equals
        scipy.cluster.hierarchy.linkage(squareform(D), "single").  Cutting it at height r
        (fcluster(Z, r, "distance")) gives the connected components of radius_neighbors(r)."""
        u, v, dist = self.minimum_spanning_tree(block_bytes=block_bytes)
        return engine.single_linkage_host(u, v, dist, self.n_node)

    @on_model_device
    def mutual_reachability_mst(self, min_samples=5, block_bytes=None):
        """(u, v, dist): the minimum spanning tree of HDBSCAN's mutual-reachability distance (degree mode), the tree
        hdbscan labels.  core(i) is the (min_samples - 1)-th smallest D[i, j] over j != i, 0 when min_samples = 1
        (scikit-learn's convention: min_samples includes the point itself), and d_mr(i, j) = max(core(i), core(j),
        D[i, j]), D being the matrix structural_distance_device holds.  u < v are int32[N-1] node indices
        (model.nodes), dist = d_mr float32[N-1], sorted by (dist, u, v): the unique MST under the order
        E(u, v) = (d_mr(u, v), u, v), Kruskal in that order on the dense d_mr, bit for bit.  Built without the
        N x N matrix (engine.degree_mreach_mst), in row panels of at most ``block_bytes`` as for
        nearest_neighbors.  min_samples: 1..65 and at most N, else ValueError."""
        if self.signal != "degree":
            raise NotImplementedError("mutual_reachability_mst is degree mode only (signal='degree')")
        dg = self._device_graph(include_zero=(self.empty == "zero"))
        out = engine.degree_mreach_mst(dg, self.hop, min_samples, empty=self.empty, block_bytes=block_bytes)
        return tuple(t.cpu().numpy() for t in out[:3])

    def hdbscan(self, min_cluster_size=5, min_samples=None, cluster_selection_method="eom",
                allow_single_cluster=False, block_bytes=None):
        """(labels int64[N], probabilities float64[N]): HDBSCAN of the structural distance (degree mode), what
        sklearn.cluster.HDBSCAN(metric="precomputed", ...).fit(D) computes, without the N x N matrix.  labels are
        cluster ids 0, 1, ... over node indices (model.nodes), -1 for noise; probabilities are the membership
        strengths (0 for noise).  min_samples=None means min_cluster_size, as in scikit-learn.

        The labels are scikit-learn's tree_to_labels(Z, min_cluster_size, cluster_selection_method,
        allow_single_cluster, 0.0, None) bit for bit, Z being single_linkage_host's linkage of
        mutual_reachability_mst(min_samples) (engine.hdbscan_host).  Ties: when several spanning trees are minimal
        (many pairs at distance 0, many edges at some node's core distance), HDBSCAN's output depends on the one
        chosen.  This one takes the unique tree under E = (d_mr, u, v), so the output is well defined;
        scikit-learn's fit chooses among tied trees by Prim's order and an unstable sort, and matches it where the
        tree's heights are pairwise distinct.  The sorted heights are the same for every minimal tree.
        ValueError, as scikit-learn's: N < 2, min_samples > N, min_cluster_size < 2, an unknown
        cluster_selection_method; also min_samples > 65.  NotImplementedError in wavelet mode.  Empty rings follow
        model.empty, as in the other degree-mode methods."""
        if int(min_cluster_size) != min_cluster_size or min_cluster_size < 2:
            raise ValueError(f"min_cluster_size must be an integer >= 2 (got {min_cluster_size!r})")
        if min_samples is None:
            min_samples = min_cluster_size
        if int(min_samples) != min_samples or min_samples < 1:
            raise ValueError(f"min_samples must be None or an integer >= 1 (got {min_samples!r})")
        if cluster_selection_method not in engine.HDBSCAN_METHODS:
            raise ValueError(f"cluster_selection_method must be 'eom' or 'leaf' (got {cluster_selection_method!r})")
        if self.signal != "degree":
            raise NotImplementedError("hdbscan is degree mode only (signal='degree')")
        n = self.n_node
        if n < 2:
            raise ValueError(f"n_samples={n} while HDBSCAN requires more than one sample")
        if min_samples > n:
            raise ValueError(f"min_samples ({min_samples}) must be at most the number of samples ({n})")
        u, v, dist = self.mutual_reachability_mst(int(min_samples), block_bytes=block_bytes)
        Z = engine.single_linkage_host(u, v, dist, n)
        return engine.hdbscan_host(Z, n, int(min_cluster_size), cluster_selection_method, allow_single_cluster)

    @on_model_device
    def parallel_calculate_HSD(self, n_workers=3, row_signal="reference"):
        """model/HSD.py:118-137 with the worker of :140-161: hops 0..hop-1 of the zero-padded
        'aligned' distance (tools/metrics.py:151-192).  row_signal="reference" reproduces the
        worker as written — both ring signals are read from wavelet row ``startIndex``
        (:152,:155); row_signal="own" reads node j's signal from its own row j."""
        if self.wavelets is None:
            raise AttributeError("'HSD' object has no attribute 'wavelets' "
                                 "(assign model.wavelets = model.calculate_wavelets(...) first)")
        psi = torch.as_tensor(np.asarray(self.wavelets, dtype=np.float64), device=self._device())
        if row_signal == "reference":
            D = _rings.worker_distance(psi, self._rings(), self.hop, self.metric)
        elif row_signal == "own":
            D = _rings.value_distance(psi, self._rings(), 0, self.hop, mode="aligned", metric=self.metric)
        else:
            raise ValueError("row_signal must be 'reference' or 'own'")
        self.distMat = D.cpu().numpy()
        return self.distMat

    def _calculate_worker(self, startIndex: int) -> np.ndarray:
        """One row of the above (columns > startIndex, zeros elsewhere; model/HSD.py:140-161)."""
        if self.distMat is None:
            self.parallel_calculate_HSD()
        row = np.array(self.distMat[startIndex], dtype=float)
        row[:startIndex + 1] = 0.0
        return row
