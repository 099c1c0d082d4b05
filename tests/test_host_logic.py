"""Host-side logic that needs no GPU: CSR ingest, degree ordering, support tables,
sharding / panel plans, the C-ABI surface and its argument validation."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "hsd_b200.h")).read()
    declared = set(re.findall(r"\b(hsd_[a-z0-9_]+)\s*\(", hdr))
    from hsd_b200._lib import HEADER_SYMBOLS, lib
    assert declared == set(HEADER_SYMBOLS), declared ^ set(HEADER_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.hsd_version() >= 100


def test_c_abi_argument_validation_without_gpu():
    """Bad arguments are rejected before any CUDA call, with an error string."""
    from hsd_b200._lib import HSDError, check, lib
    rc = lib.hsd_pairwise_l1(None, 16, 128, 0, 1, 0, 1, 0, None, 128, None)
    assert rc == -1 and b"null" in lib.hsd_last_error_string()
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    assert lib.hsd_pairwise_l1(p, 0, 128, 0, 1, 0, 1, 0, p, 128, None) == -1      # k_used > 0
    assert lib.hsd_pairwise_l1(p, 16, 130, 0, 1, 0, 1, 0, p, 130, None) == -1     # n_pad % 4
    assert lib.hsd_pairwise_l1(p, 16, 128, 0, 64, 0, 32, 1, p, 128, None) == -1   # symmetric trapezoid
    assert lib.hsd_pairwise_l1(p, 16, 128, 2, 64, 0, 32, 0, p, 128, None) == -1   # TMA origin alignment
    assert lib.hsd_ring_signature_degree(None, None, 4, None, None, 1, 2, None, None, 1, None, 0,
                                         None, None, 0, None, 0, None) == -1
    assert lib.hsd_pairwise_aligned(p, p, p, 4, 2, 0, 3, 7, 0, 1, p, 4, None) == -1  # metric id
    assert lib.hsd_ring_reduce(p, 1, 4, 4, p, p, None, 9, 0, p, p, 64, None) == -1   # hops > 7
    with pytest.raises(HSDError):
        check(lib.hsd_cheb_spmm(p, p, 4, -1.0, p, 1, 3, 0, 4, 0.0, p, p, None))
    assert lib.hsd_topk_rows(p, 8, 4, 8, 65, 0, None, p, p, None) == -1              # k <= 64
    assert lib.hsd_topk_rows(p, 4, 4, 8, 2, 0, None, p, p, None) == -1               # ld >= n_cols
    assert lib.hsd_scatter_symmetric(None, 8, 2, 8, p, p, 8, 1, None) == -1 and b"null" in lib.hsd_last_error_string()
    assert lib.hsd_scatter_symmetric(p, 4, 2, 8, p, p, 8, 1, None) == -1             # blk_ld >= n
    # round-2 entry points
    assert lib.hsd_exact_wavelets(None, 4, p, 4, 1.0, 0.0, 1, p, 4, None) == -1 and b"null" in lib.hsd_last_error_string()
    assert lib.hsd_exact_wavelets(p, 2, p, 4, 1.0, 0.0, 1, p, 4, None) == -1          # ldu >= n
    assert lib.hsd_copy2d_to_host(None, 16, p, 16, 16, 1, None) == -1
    assert lib.hsd_copy2d_to_host(p, 8, p, 16, 16, 1, None) == -1                    # pitch >= width
    assert lib.hsd_copy2d_to_host(p, 16, p, 16, 0, 0, None) == 0                     # empty window: nothing to do
    words = lib.hsd_ring_dense_workspace_words(1000)
    assert words == 2 * 1000 * 32 + 1000                                            # two 1000 x 1024-bit tables + the row map
    assert lib.hsd_ring_signature_degree_dense(p, p, 1000, p, p, 10, 2, p, p, 3, p, 8, None, 0, p, None, 0, p,
                                               p, words - 1, 5000, None) == -1       # workspace too small
    assert lib.hsd_ring_signature_degree_dense(p, p, 1000, p, p, 10, 0, p, p, 3, p, 8, None, 0, p, None, 0, p,
                                               p, words, 5000, None) == -1 and b"hops >= 1" in lib.hsd_last_error_string()
    # graphs whose four N-bit bitmaps fit shared memory need no BFS workspace; larger ones say how much
    assert lib.hsd_bfs_workspace_words(100000) == 0
    words = lib.hsd_bfs_workspace_words(450000)
    assert words > 0 and words % (4 * ((450000 + 31) // 32)) == 0


def test_no_cpu_fallback():
    """Without a CUDA device the entry points raise instead of computing on the host.  The checks run in
    a child process that sees no device, so that they hold on a machine with a GPU as well."""
    import subprocess
    import sys
    code = "\n".join([
        "import pytest, torch",
        "from hsd_b200 import engine",
        "from hsd_b200.graph import powerlaw_graph",
        "assert not torch.cuda.is_available()",
        "with pytest.raises(RuntimeError):",
        "    engine.require_cuda()",
        "with pytest.raises(RuntimeError):",
        "    engine._ptr(torch.zeros(4))",
        "with pytest.raises(RuntimeError):",
        "    engine.DeviceGraph.upload(powerlaw_graph(50))",
        "print('raised')",
    ])
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=300,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stderr[-1500:]
    assert out.stdout.strip().splitlines()[-1] == "raised"


def test_csr_from_networkx_keeps_first_appearance_order():
    import networkx as nx
    from hsd_b200.graph import CSRGraph
    g = nx.Graph()
    g.add_edges_from([("b", "a"), ("a", "c"), ("d", "b"), ("a", "b")])
    csr = CSRGraph.from_networkx(g)
    assert csr.nodes == ["b", "a", "c", "d"]                     # tools/util.py:11-24 ordering
    assert csr.degree.tolist() == [2, 2, 1, 1]
    assert csr.neighbors(0).tolist() == [1, 3] and csr.neighbors(1).tolist() == [0, 2]
    A = nx.adjacency_matrix(g).todense()
    dense = np.zeros((4, 4), dtype=int)
    for i in range(4):
        dense[i, csr.neighbors(i)] = 1
    assert np.array_equal(dense, np.asarray(A).astype(int))


def test_degree_order_and_support_tables():
    from hsd_b200.graph import powerlaw_graph
    g = powerlaw_graph(3000, 5, seed=0)
    o = g.degree_order()
    deg = g.degree
    assert np.all(np.diff(o.sorted_degree) >= 0)
    assert np.array_equal(np.sort(o.orig_of), np.arange(g.n))
    assert np.array_equal(o.new_of[o.orig_of], np.arange(g.n))
    assert np.array_equal(deg[o.orig_of], o.sorted_degree)
    # relabelled adjacency is the same graph
    for new in [0, 17, g.n - 1]:
        nb = o.col[o.rowptr[new]:o.rowptr[new + 1]]
        assert sorted(o.orig_of[nb].tolist()) == g.neighbors(o.orig_of[new]).tolist()
        assert np.all(np.diff(nb) > 0)
    assert len(o.col) % 4 == 0 and len(o.col) >= g.nnz + 4      # LDG.128 padding
    sup, bin_end, delta = o.support()
    assert np.array_equal(sup, np.unique(deg)) and bin_end[-1] == g.n
    for b in range(len(sup)):
        assert bin_end[b] == np.sum(deg <= sup[b])
    assert np.array_equal(delta, np.diff(sup).astype(np.float32))
    sup0, be0, _ = o.support(include_zero=True)
    assert sup0[0] == 0 and be0[0] == 0 and len(sup0) == len(sup) + 1


def test_edge_insertion_and_dedup():
    from hsd_b200.graph import CSRGraph
    g = CSRGraph.from_edges(5, np.array([[0, 1], [1, 0], [1, 2], [3, 3]]))
    assert g.degree.tolist() == [1, 2, 1, 1, 0]                  # duplicate collapsed, self-loop once
    g2 = g.with_edges_added(np.array([[4, 0], [2, 1]]))
    assert g2.degree.tolist() == [2, 2, 1, 1, 1]
    with pytest.raises(ValueError):
        CSRGraph.from_edges(3, np.array([[0, 3]]))
    with pytest.raises(ValueError):
        g.with_edges_added(np.array([[0, 5]]))


def test_sorted_merge_insertion_equals_a_rebuild():
    """with_edges_added merges the new entries into the sorted CSR (binary search + insert); it
    must equal a rebuild from the full edge list: duplicates of existing edges, both orientations,
    repeated new edges, a self-loop, first / last rows, and insertion into an empty graph."""
    import networkx as nx
    from hsd_b200.graph import CSRGraph
    rng = np.random.default_rng(5)
    G = nx.barabasi_albert_graph(400, 3, seed=2)
    g = CSRGraph.from_networkx(G)
    existing = np.array(list(G.edges()))[:5]
    new = np.concatenate([rng.integers(0, 400, size=(60, 2)), existing, existing[:, ::-1],
                          [[0, 399], [399, 0], [0, 399], [7, 7], [398, 399]]])
    got = g.with_edges_added(new)
    G2 = G.copy()
    G2.add_edges_from(new.tolist())
    want = CSRGraph.from_networkx(G2)
    assert np.array_equal(got.rowptr, want.rowptr) and np.array_equal(got.col, want.col)
    assert got.col.dtype == np.int32 and got.rowptr.dtype == np.int32
    same = g.with_edges_added(np.zeros((0, 2), dtype=np.int64))
    assert np.array_equal(same.col, g.col) and np.array_equal(same.rowptr, g.rowptr)
    empty = CSRGraph.from_edges(6, np.zeros((0, 2)))
    e2 = empty.with_edges_added(np.array([[0, 5], [2, 3], [5, 0]]))
    assert e2.rowptr.tolist() == [0, 1, 1, 2, 3, 3, 4] and e2.col.tolist() == [5, 3, 2, 0]


@pytest.mark.parametrize("n,world", [(20000, 1), (20000, 8), (10, 4), (3, 8), (1190, 2)])
def test_shard_rows_cover_every_row_once(n, world):
    from hsd_b200.sharded import shard_rows
    seen = []
    for r in range(world):
        row0, nr, per = shard_rows(n, world, r)
        assert per * world >= n and nr <= per and (nr == 0 or row0 % 4 == 0)
        seen += list(range(row0, row0 + nr))
    assert seen == list(range(n))


def test_host_pipeline_panels_tile_the_rows():
    from hsd_b200.engine import HostDegreePipeline
    for n_rows, n, full in [(20000, 20000, True), (2500, 20000, False), (100, 100, True), (129, 129, True)]:
        p = HostDegreePipeline.__new__(HostDegreePipeline)     # the panel plan alone: no device buffers
        p.n_rows, p.n, p.full = n_rows, n, full
        panels = p._plan_panels(8)
        assert panels[0][0] == 0 and sum(r for _, r in panels) == n_rows
        for (a, ra), (b, _) in zip(panels[:-1], panels[1:]):
            assert a + ra == b and a % 128 == 0
        if full and n_rows > 2000:
            assert panels[0][1] < panels[-1][1]          # equal-work trapezoids start narrow


def test_reference_arm_of_bench_runs_on_cpu():
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--workload", "1500x2"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["unit"] == "node-pairs/s"


def test_bench_rejects_a_run_without_timed_steps():
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 2 and "--steps" in out.stderr


def test_product_package_never_touches_the_oracle_or_reference():
    """oracle/ is test infrastructure: nothing under hsd_b200/, model/ or tools/ may import it,
    and nothing shipped may read /root/reference."""
    import glob
    bad = []
    for path in glob.glob(os.path.join(ROOT, "hsd_b200", "**", "*.py"), recursive=True) + \
            glob.glob(os.path.join(ROOT, "model", "*.py")) + glob.glob(os.path.join(ROOT, "tools", "*.py")):
        src = open(path).read()
        if re.search(r"^\s*(from|import)\s+oracle\b", src, re.M) or "/root/reference" in src:
            bad.append(path)
    assert not bad, bad
    for path in [os.path.join(ROOT, "bench.py"), os.path.join(ROOT, "__graft_entry__.py")]:
        assert "/root/reference" not in open(path).read()


def test_rw_formats_round_trip(tmp_path, robust_csv):
    """tools/rw.py formats: the CSV layout of the reference's golden robust.csv and the
    distance edge list."""
    from tools import rw, save_vectors_dict
    vecs = {int(n): list(v[:12]) for n, v in zip(robust_csv["node"], robust_csv["values"])}
    p = tmp_path / "v.csv"
    save_vectors_dict(vecs, str(p))
    first = open(p).readline().strip().split(",")
    assert first[0] == str(int(robust_csv["node"][0])) and first[1] == "%.8f" % robust_csv["values"][0][0]
    back = rw.read_vectors(str(p))
    assert np.allclose(back[str(int(robust_csv["node"][3]))], robust_csv["values"][3][:12], atol=1e-8)
    D = np.array([[0, 1.5, 2.0], [1.5, 0, 0.25], [2.0, 0.25, 0]])
    q = tmp_path / "d.edgelist"
    rw.save_distance_edgelist(str(q), [0, 1, 2], D)
    assert np.array_equal(rw.read_distance(str(q), 3), D)
    with pytest.raises(FileNotFoundError):
        rw.read_vectors(str(tmp_path / "missing.csv"))


def test_reference_side_modules_stay_importable_through_the_shim(tmp_path):
    """With $HSD_REFERENCE_ROOT set, `from tools import evaluate, dataloader` (main.py:7 of the
    reference) resolves to the reference's own files while tools.hierarchy / tools.rw stay ours.
    The reference checkout is stood in for by a tools/ directory with the same module names: the
    modules the shim does not provide, and decoys of the ones it must keep providing itself."""
    import subprocess
    import sys
    ref = str(tmp_path / "reference")
    os.makedirs(os.path.join(ref, "tools"))
    for name in ("__init__", "evaluate", "dataloader", "hierarchy", "rw", "util"):
        with open(os.path.join(ref, "tools", name + ".py"), "w") as f:
            f.write("" if name in ("__init__", "evaluate", "dataloader") else "raise ImportError('reference copy')\n")
    code = ("import tools; from tools import evaluate, dataloader, rw, util, hierarchy; "
            "import model; "
            "print(evaluate.__file__); print(hierarchy.__name__); print(rw.__name__); print(model.HSD.__module__)")
    env = dict(os.environ, HSD_REFERENCE_ROOT=ref, PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=300)
    assert out.returncode == 0, out.stderr[-1500:]
    lines = out.stdout.strip().splitlines()
    assert lines[0].startswith(ref) and lines[1] == "hsd_b200.tools.hierarchy"
    assert lines[2] == "hsd_b200.tools.rw" and lines[3] == "hsd_b200.model.HSD"


def test_weighted_edge_detection_and_identity_label_fast_path():
    """has_nonunit_weights (the guard in front of the unit-weight Chebyshev kernel) and the two
    label paths of CSRGraph.from_networkx (labels that are the indices / arbitrary labels)."""
    import networkx as nx
    from hsd_b200.graph import CSRGraph, has_nonunit_weights
    g = nx.Graph()
    g.add_edge(0, 1)
    g.add_edge(1, 2, color="red")
    g.add_edge(2, 3, weight=1.0)
    assert not has_nonunit_weights(g) and not has_nonunit_weights(nx.Graph())
    g.add_edge(3, 0, weight=0.5)
    assert has_nonunit_weights(g)
    base = nx.barabasi_albert_graph(200, 3, seed=7)                       # labels 0..n-1 in order: fast path
    a = CSRGraph.from_networkx(base)
    perm = nx.relabel_nodes(base, {v: f"n{v}" for v in base.nodes()})      # same graph, string labels, same order
    b = CSRGraph.from_networkx(perm)
    assert np.array_equal(a.rowptr, b.rowptr) and np.array_equal(a.col, b.col)
    assert a.nodes == list(range(200)) and b.nodes == [f"n{v}" for v in range(200)]
    e = np.array(base.edges(), dtype=np.int64)
    c = CSRGraph.from_edges(200, e)
    assert np.array_equal(a.rowptr, c.rowptr) and np.array_equal(a.col, c.col)


def test_drop_in_import_paths():
    """Every import form the reference's own callers use resolves (ADVICE r1): the package
    re-exports the three classes (model/__init__.py:2-4), the submodules are importable by
    path (tests/robust_test/main.py:11) and `model.GraphWave` is the module
    (tests/graphwave_test/main.py:12,33-34)."""
    import sys
    import types
    from model import HSD, MultiHSD, DynamicHSD
    from model.HSD import HSD as H2
    from model.multiscale_HSD import MultiHSD as M2
    from model.dynamic_HSD import DynamicHSD as D2
    from model import GraphWave
    assert HSD is H2 and MultiHSD is M2 and DynamicHSD is D2
    assert isinstance(GraphWave, types.ModuleType) and isinstance(sys.modules["model.HSD"], types.ModuleType)
    assert isinstance(GraphWave.GraphWave, type) and callable(GraphWave.recommend_scale_range)
    from tools import hierarchy, util, save_vectors_dict   # model/multiscale_HSD.py:12, tools/multiscales.py:11
    from tools.hierarchy import get_hierarchical_representation, read_hierarchy
    assert callable(get_hierarchical_representation) and callable(read_hierarchy) and callable(save_vectors_dict)


def test_calculate_distance_metric_names_and_exceptions():
    """tools/metrics.py:151-192: same exception types as the reference for every metric name."""
    from tools.metrics import calculate_distance
    p, q = [0.2, 0.3, 0.5], [0.5, 0.25, 0.25]
    # values printed by the unmodified reference (tools/metrics.py imported by path) on the same input
    assert abs(calculate_distance(p, q, "l1") - 0.09999999999999998) < 1e-15
    assert abs(calculate_distance(p, q, "kl") - 0.010067756775344432) < 1e-15
    assert abs(calculate_distance(p, q, "symmetric_kl") - 0.010136627702704112) < 1e-15
    assert abs(calculate_distance(p, q, "wasserstein_guass") - 4.7207654837878865e-05) < 1e-18
    assert abs(calculate_distance(p, q, "l2") - (0.05 ** 2 + 0.05 ** 2)) < 1e-12
    ps, qs = np.sort(p), np.sort(q)
    assert abs(calculate_distance(p, q, "kl") - float(np.sum(ps * np.log(ps / qs)))) < 1e-12
    sym = (np.sum(ps * np.log(ps / qs)) + np.sum(qs * np.log(qs / ps))) / 2
    assert abs(calculate_distance(p, q, "symmetric_kl") - sym) < 1e-12
    for m in ("l1", "l2", "kl", "symmetric_kl", "js"):
        with pytest.raises(ValueError):                                  # un-normalised ring signals
            calculate_distance([1.0, 2.0], [3.0], m)
    with pytest.raises(ValueError):                                      # m = p + q sums to 2 (as written, :103-105)
        calculate_distance(p, q, "js")
    with pytest.raises(NotImplementedError):
        calculate_distance(p, q, "dtw")
    with pytest.raises(TypeError):
        calculate_distance(p, q, None)
    assert calculate_distance([], [], "l1") == 0.0


@pytest.mark.parametrize("n,panels,threads", [(1000, [(0, 1000)], 3), (4099, [(0, 256), (256, 768), (1024, 3075)], 8),
                                               (130, [(0, 128), (128, 2)], 1)])
def test_host_mirror_completes_the_symmetric_matrix(n, panels, threads):
    """hsd_mirror_upper_to_lower_host (the opt-in e2e path that ships each unordered pair once):
    panel by panel, D[j][i] = D[i][j] below the panel; entries on and above the diagonal untouched."""
    from hsd_b200._lib import check, lib
    rng = np.random.default_rng(n)
    U = np.triu(rng.random((n, n), dtype=np.float32))
    D = U.copy()
    D[np.tril_indices(n, -1)] = -1.0
    for p0, pr in panels:
        check(lib.hsd_mirror_upper_to_lower_host(D.ctypes.data, n, n, p0, p0 + pr, threads))
    assert np.array_equal(D, U + np.triu(U, 1).T)
    assert lib.hsd_mirror_upper_to_lower_host(D.ctypes.data, n, n, 5, 64, 1) == -1     # panels start on 64-row boundaries


@pytest.mark.parametrize("n,world", [(20000, 8), (2500, 3), (1801, 4), (300, 2), (100000, 8)])
@pytest.mark.parametrize("tile_n", [128, 64])
def test_symmetric_tile_list_covers_every_tile_once(n, world, tile_n):
    """sharded.symmetric_tile_list: over the ranks every upper-triangle tile appears exactly once, is computed
    by the owner of its row block or of its column block, is oriented so that the mirrored store is local,
    and the ranks' shares are balanced."""
    from hsd_b200.sharded import shard_rows, symmetric_tile_list
    per = shard_rows(n, world, 0)[2]
    own = lambda t: min(t * 128 // per, world - 1)
    seen, halves_of, counts = set(), {}, []
    for r in range(world):
        tl = symmetric_tile_list(n, world, per, r, tile_n).numpy()
        counts.append(len(tl))
        for i0, j0, m in tl.tolist():
            assert i0 % 128 == 0 and j0 % tile_n == 0 and i0 < n and j0 < n
            key = (min(i0 // 128, j0 // 128), max(i0 // 128, j0 // 128), (j0 % 128) // 64)
            assert key not in seen
            seen.add(key)
            halves_of.setdefault(key[:2], (j0 // 128, set()))[1].add(key[2])
            assert (m == 1) == (i0 // 128 != j0 // 128)
            assert own(j0 // 128) == r          # the mirrored store (rows of the column block) is local ...
            assert m == 1 or own(i0 // 128) == r   # ... and a diagonal tile is entirely local
    T = (n + 127) // 128
    assert len(halves_of) == T * (T + 1) // 2                       # every unordered pair of 128-blocks, once
    for (a, b), (y, halves) in halves_of.items():                   # with every existing half of its column block
        want = {0} if tile_n == 128 else {h for h in (0, 1) if y * 128 + 64 * h < n}
        assert halves == want
    assert max(counts) <= -(-sum(counts) // world) * 1.03 + 2           # nobody is overloaded (some halves do not exist)


def test_dynamic_update_workspace_buffers():
    """DynamicHSD's grow-only update workspace (host logic, exercised on CPU tensors): the signature tables
    alternate between two buffers so the previous table survives the next update, a few more distinct degrees
    fit without a new allocation, and the K-major table comes back zeroed with room for one chunk of rows."""
    import torch
    from hsd_b200 import engine
    from hsd_b200.model.dynamic_HSD import _UpdateWorkspace
    n, hops, rows = 1001, 3, 64
    ws = _UpdateWorkspace(n, torch.device("cpu"), hops, rows)
    a = ws.next_signature_table(n, 436)
    a.fill_(1.0)
    b = ws.next_signature_table(n, 436)
    b.fill_(2.0)
    assert a.shape == b.shape == (n, 436) and a.is_contiguous() and a.data_ptr() != b.data_ptr()
    assert float(a.min()) == 1.0                       # the previous table is untouched by the next one
    c = ws.next_signature_table(n, 436 + 3 * 15)       # 15 more distinct degrees per hop: same buffer as `a`
    assert c.data_ptr() == a.data_ptr() and c.shape == (n, engine.roundup(436 + 45, 4))
    assert float(b.min()) == 2.0
    d = ws.next_signature_table(n, 2000)               # beyond the slack: a new buffer for this slot only
    assert d.shape == (n, 2000) and d.data_ptr() != b.data_ptr()
    t = ws.k_major_table(436)
    assert t.shape == (engine.roundup(436, engine.PAIR_KCHUNK), engine.roundup(n, 4) + rows) and t.is_contiguous()
    t.fill_(3.0)
    t2 = ws.k_major_table(440)
    assert t2.data_ptr() == t.data_ptr() and float(t2.abs().max()) == 0.0
    assert ws.block.shape == (rows, engine.roundup(n, 4))
    # allocated up front when the signature length is known: the first updates allocate nothing
    ws2 = _UpdateWorkspace(n, torch.device("cpu"), hops, rows, k_used=436)
    ptrs = {ws2._sig[0].data_ptr(), ws2._sig[1].data_ptr()}
    first, second = ws2.next_signature_table(n, 436), ws2.next_signature_table(n, 440)
    assert {first.data_ptr(), second.data_ptr()} == ptrs and ws2.k_major_table(436).data_ptr() == ws2._sigT.data_ptr()
