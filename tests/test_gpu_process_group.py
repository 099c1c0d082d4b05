"""The multi-GPU degree-mode entry points under a real NCCL process group, one process per GPU.

The other sharding tests emulate every rank in one process (no process group: the entry points return
partials and the test merges them) or run the plumbing on CPU tensors over gloo.  Here the code behind
`dist.is_initialized()` runs as users run it: `agree_min`, `agree_all`, `agree_status` and `agree_radius_cap`
as NCCL collectives on device tensors, `gather_csr_parts`, `_knn_table`'s gathered signatures with the
all-gather + `topk_merge` of `_knn_sweep`, the column-split vote and peer memory of `ShardedDegreeHSD`.  Every
rank's output must equal the one-GPU result, computed by the same worker on its own device, bit for bit.

The ranks are made unequal: odd ranks see little free device memory (`torch.cuda.mem_get_info` patched,
no memory taken), so every plan a rank derives from its free memory differs from the even ranks' plans
unless the ranks agree on it.  Each case also records those unagreed plans, so that a test can show its
skew took effect.

One spawn per world size (2, and every visible GPU when there are more) runs all cases in sequence; each
test reads its own case's result.  Skipped with fewer than two GPUs."""
import contextlib
import datetime
import os
import queue
import socket
import time
import traceback

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SMALL_N = 20000          # below 32768 nodes: the row-split ring phase
LARGE_N = 40000          # from 32768 nodes: the column-split ring phase by default
MiB = 1 << 20
KNN_FREE = 32 * MiB      # odd ranks' free memory: below every k-NN panel cap here (128-row panels)
RADIUS_FREE = 96 * MiB   # ... for the radius graph: small panels, yet a default max_pairs above the graphs' nnz
RING_FREE = 96 * MiB     # ... for the ring phase: the dense variant's tables and the column split do not fit
DYN_FREE = 4 * MiB       # ... the same at the 3000-node graph of the update cases
TIMEOUT_S = 1200         # one world size, every case
NCCL_TIMEOUT_S = 300     # a collective that waits longer ends its process (ranks out of step: a failure, not a hang)

KNN_CASES = [(SMALL_N, 3, k) for k in (1, 20, 64)] + [(LARGE_N, 2, k) for k in (1, 20, 64)] + [(SMALL_N, 4, 20)]
MODEL_KNN_CASES = [(SMALL_N, 3, 20), (LARGE_N, 2, 20), (100, 2, 10)]          # 100 < 128 nodes: one panel
RADIUS_CASES = ([(SMALL_N, 3, r) for r in ("zero", "typical", "none")]
                + [(LARGE_N, 2, r) for r in ("zero", "typical", "none")] + [(300, 2, "inf")])
STEP_CASES = [(SMALL_N, 3, peer, True) for peer in (False, True)] + [(LARGE_N, 2, peer, skew)
                                                                     for skew in (True, False) for peer in (False, True)]
EMPTY_CASES = [(peer, empty) for peer in (False, True) for empty in ("raise", "zero")]
DYNAMIC_CASES = [False, True]


def _world_sizes():
    count = torch.cuda.device_count()
    return [2] + ([count] if count > 2 else [])


# ---------------------------------------------------------------------------------------------- worker side
@contextlib.contextmanager
def _skewed(rank, free_bytes):
    """On odd ranks, make engine._free_bytes see `free_bytes` (torch.cuda.mem_get_info reports that much minus
    what torch's allocator caches, after the cache is emptied) and forget the cached dense-ring workspaces, whose
    presence would otherwise decide the ring variant regardless of free memory.  Even ranks see their real
    memory.  Nothing is allocated."""
    if rank % 2 == 0:
        yield
        return
    from hsd_b200 import engine
    real = torch.cuda.mem_get_info

    def fake(device=None):
        torch.cuda.empty_cache()
        cached = torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device)
        return max(free_bytes - cached, 0), real(device)[1]

    engine._DENSE_WS.clear()
    torch.cuda.empty_cache()
    torch.cuda.mem_get_info = fake
    try:
        yield
    finally:
        torch.cuda.mem_get_info = real


def _gather(value):
    import torch.distributed as dist
    out = [None] * dist.get_world_size()
    dist.all_gather_object(out, value)
    return out


def _knn_result(idx, val, ref_idx, ref_val, plans, note=""):
    """ok, the first row that differs from the one-GPU lists, the rows whose list holds an id twice."""
    idx, val = torch.as_tensor(idx).cpu(), torch.as_tensor(val).cpu()
    ref_idx, ref_val = torch.as_tensor(ref_idx).cpu(), torch.as_tensor(ref_val).cpu()
    bad = (idx != ref_idx).any(1) | (val.view(torch.int32) != ref_val.view(torch.int32)).any(1)
    s = idx.sort(1).values
    dups = int(((s[:, 1:] == s[:, :-1]) & (s[:, 1:] >= 0)).any(1).sum())
    rows = torch.nonzero(bad).reshape(-1)
    return dict(ok=not bool(bad.any()) and dups == 0, row=int(rows[0]) if rows.numel() else -1, dups=dups,
                plans=plans, note=note)


def _csr_result(got, want, plans, note=""):
    """ok, and the first row whose entries (ids or distance bits) differ from the one-GPU CSR."""
    gi, gx, gd = (np.asarray(a) for a in got)
    wi, wx, wd = (np.asarray(a) for a in want)
    ok = (np.array_equal(gi, wi) and np.array_equal(gx, wx) and np.array_equal(gd.view(np.uint32), wd.view(np.uint32)))
    row = -1
    if not ok:
        if gi.shape != wi.shape or not np.array_equal(gi, wi):
            diff = np.nonzero(gi[:min(gi.size, wi.size)] != wi[:min(gi.size, wi.size)])[0]
            row = int(diff[0]) - 1 if diff.size else min(gi.size, wi.size) - 1
        else:
            bad = np.nonzero((gx != wx) | (gd.view(np.uint32) != wd.view(np.uint32)))[0]
            row = int(np.searchsorted(wi, bad[0], side="right")) - 1
    return dict(ok=ok, row=row, dups=0, plans=plans, note=note)


class _Inputs:
    """Graphs, models and one-GPU references, built once per worker."""

    def __init__(self):
        self._cache = {}

    def get(self, key, make):
        if key not in self._cache:
            self._cache[key] = make()
        return self._cache[key]

    def device_graph(self, n):
        from hsd_b200 import engine
        from hsd_b200.graph import powerlaw_graph
        return self.get(("dg", n), lambda: engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0)))

    def model(self, n, hops):
        import networkx as nx
        from model import HSD
        return self.get(("model", n, hops), lambda: HSD(nx.barabasi_albert_graph(n, 5, seed=0), f"pl{n}", 0, hops,
                                                       "wasserstein", signal="degree"))


def _case_knn(inp, rank, world, n, hops, k):
    from hsd_b200 import engine
    dg = inp.device_graph(n)
    ref_idx, ref_val = engine.degree_knn(dg, hops, k)
    torch.cuda.synchronize()
    events = []
    with _skewed(rank, KNN_FREE):
        plans = _gather(engine.knn_panel_rows(n, int(engine._free_bytes(dg.rowptr.device) * engine.KNN_BLOCK_FRACTION),
                                              world))
        idx, val = engine.degree_knn(dg, hops, k, rank=rank, world=world, pair_events=events)
    swept = np.zeros(n, np.int64)
    for panels in _gather([(r0, r1) for r0, r1, _, _ in events]):
        for r0, r1 in panels:
            swept[r0:r1] += 1
    note = f"rows swept by no rank: {int((swept == 0).sum())}, by two or more: {int((swept > 1).sum())}"
    res = _knn_result(idx, val, ref_idx, ref_val, plans, note)
    res["ok"] = res["ok"] and bool(np.all(swept == 1))
    return res


def _case_model_knn(inp, rank, world, n, hops, k):
    from hsd_b200 import engine
    m = inp.model(n, hops)
    ref = m.nearest_neighbors(k)
    block_bytes = (1 + rank % 2) * 128 * 4 * engine.roundup(n, 4)       # 128-row panels, 256 on odd ranks
    plans = _gather(engine.knn_panel_rows(n, block_bytes, world))
    got = m.nearest_neighbors_sharded(k, rank, world, block_bytes=block_bytes)
    return _knn_result(got[0], got[1], ref[0], ref[1], plans)


def _radius_plan(n, world, rank, free):
    """(panel rows, default max_pairs) a rank would take from its own free memory, before the ranks agree."""
    from hsd_b200 import engine
    rows = engine.radius_panel_rows(n, int(free * engine.KNN_BLOCK_FRACTION), world)
    mine = engine.knn_deal(n, engine.knn_panels(n, rows), world)[rank]
    return rows, engine.radius_sharded_max_pairs(free - engine.radius_fixed_bytes(n, mine) - 8 * world * (n + 1))


def _radii(inp, n, hops):
    """radius name -> value: 0, the median 10th-neighbour distance, just below the smallest distance, +inf."""
    def make():
        _, val = inp.model(n, hops).nearest_neighbors(10)
        dmin = np.float32(val[:, 0].min())
        return {"zero": 0.0, "typical": float(np.median(val[:, 9])), "inf": float("inf"),
                "none": float(np.nextafter(dmin, np.float32(0))) if dmin > 0 else None}
    return inp.get(("radii", n, hops), make)


def _case_radius(inp, rank, world, n, hops, which):
    m = inp.model(n, hops)
    radius = _radii(inp, n, hops)[which]
    if radius is None:
        return dict(ok=False, row=-1, dups=0, plans=[], note="the graph has distance-0 pairs: no radius is empty")
    want = m.radius_neighbors(radius)
    if which == "none" and want[1].size:
        return dict(ok=False, row=-1, dups=0, plans=[], note="the 'none' radius is not empty on one GPU")
    from hsd_b200 import engine
    with _skewed(rank, RADIUS_FREE):
        plans = _gather(_radius_plan(n, world, rank, engine._free_bytes(torch.cuda.current_device())))
        got = m.radius_neighbors_sharded(radius, rank, world)
    return _csr_result(got, want, plans, note=f"radius {radius!r}, nnz {want[1].size}")


def _case_radius_cap(inp, rank, world):
    """max_pairs differs per rank; the smallest is below the global nnz: every rank raises the same ValueError."""
    m = inp.model(SMALL_N, 3)
    radius = _radii(inp, SMALL_N, 3)["typical"]
    nnz = int(m.radius_neighbors(radius)[1].size)
    max_pairs = nnz // 2 if rank % 2 else 4 * nnz
    try:
        m.radius_neighbors_sharded(radius, rank, world, max_pairs=max_pairs)
    except ValueError as e:
        return dict(ok=f"max_pairs = {nnz // 2}" in str(e), row=-1, dups=0, plans=_gather(max_pairs), note=str(e))
    return dict(ok=False, row=-1, dups=0, plans=_gather(max_pairs), note="no ValueError")


def _ring_plan(plan):
    """The ring phase a rank would pick from its own free memory: the dense or frontier variant of the row split,
    and its vote for the column split (from 32768 nodes)."""
    from hsd_b200 import engine
    dg = plan.dg
    algo = engine.ring_algorithm(dg.n, plan.n_src, plan.hops, dg.rowptr.device)
    return algo, plan._cols_workspace_fits() if dg.n >= 32768 else None


def _case_step(inp, rank, world, n, hops, peer, skew):
    from hsd_b200 import engine
    from hsd_b200.sharded import ShardedDegreeHSD
    dg = inp.device_graph(n)
    D, _ = engine.degree_distance_device(dg, hops)
    with _skewed(rank, RING_FREE) if skew else contextlib.nullcontext():
        plan = ShardedDegreeHSD(dg, hops, rank, world, peer=peer)
        plans = _gather(_ring_plan(plan))
        blk = plan.step()
        plan.check()
        torch.cuda.synchronize()
    ok = torch.equal(blk, D[plan.row0:plan.row0 + plan.n_rows])
    modes = _gather(plan.ring_mode)
    bad = torch.nonzero((blk != D[plan.row0:plan.row0 + plan.n_rows]).any(1)).reshape(-1)
    del D, plan, blk
    torch.cuda.empty_cache()
    return dict(ok=bool(ok) and len(set(modes)) == 1, row=int(bad[0]) if bad.numel() else -1, dups=0, plans=plans,
                note=f"ring phase per rank: {modes}")


def _isolated_graph():
    """A 3000-node power-law graph plus one isolated node, the last id: in the last rank's row block, and
    BFS-ed by one rank only (sources are dealt round-robin)."""
    from hsd_b200.graph import CSRGraph, powerlaw_graph
    g0 = powerlaw_graph(3000, 5, seed=0)
    rows = np.repeat(np.arange(g0.n), np.diff(g0.rowptr))
    return CSRGraph.from_edges(g0.n + 1, np.stack([rows, g0.col], 1)[rows < g0.col])


def _case_empty(inp, rank, world, peer, empty):
    from hsd_b200 import engine
    from hsd_b200.sharded import ShardedDegreeHSD
    dg = inp.get("isolated", lambda: engine.DeviceGraph.upload(_isolated_graph(), include_zero=True))
    hops = 3
    with _skewed(rank, DYN_FREE):
        plan = ShardedDegreeHSD(dg, hops, rank, world, empty=empty, peer=peer)
        plans = _gather(_ring_plan(plan))
        blk = plan.step()
        try:
            plan.check()
        except engine.EmptyRingError:
            return dict(ok=empty == "raise", row=-1, dups=0, plans=plans, note="EmptyRingError")
    if empty == "raise":
        return dict(ok=False, row=-1, dups=0, plans=plans, note="no EmptyRingError")
    D, _ = engine.degree_distance_device(dg, hops, empty="zero")
    ok = torch.equal(blk, D[plan.row0:plan.row0 + plan.n_rows])
    return dict(ok=bool(ok), row=-1, dups=0, plans=plans, note=f"rows {plan.row0}..{plan.row0 + plan.n_rows}")


def _case_dynamic(inp, rank, world, peer):
    """Two updates of DynamicHSD.structural_distance_update_sharded: insertions between low-degree nodes (the
    set of distinct degrees stays: the incremental path), then one more edge at the biggest hub (a new distinct
    degree: the plan is rebuilt).  After each, this rank's block equals its rows of the one-GPU update."""
    import networkx as nx
    from model import DynamicHSD
    n, hop = 3000, 2
    g0 = nx.barabasi_albert_graph(n, 5, seed=0)
    deg = dict(g0.degree())
    low = sorted(v for v in g0 if deg[v] <= 6)
    rng = np.random.default_rng(3)
    batch1 = set()
    while len(batch1) < 5:
        u, v = (int(x) for x in rng.choice(low, 2, replace=False))
        if not g0.has_edge(u, v):
            batch1.add((min(u, v), max(u, v)))
    batch1 = sorted(batch1)
    hub = max(deg, key=lambda v: (deg[v], -v))
    batch2 = [(hub, x) for x in low if not g0.has_edge(hub, x) and (min(hub, x), max(hub, x)) not in batch1][:1]
    one = DynamicHSD(g0.copy(), "ba", hop, 1, "wasserstein", signal="degree")
    refs = [one.structural_distance_update().clone()]
    for batch in (batch1, batch2):
        one.dynamic_add_edges(batch)
        refs.append(one.structural_distance_update().clone())
    del one
    m = DynamicHSD(g0.copy(), "ba", hop, 1, "wasserstein", signal="degree")
    notes, ok, plans = [], True, []
    with _skewed(rank, DYN_FREE):
        for step, batch in enumerate((None, batch1, batch2)):
            before = getattr(m, "_plan", None)
            if batch is not None:
                m.dynamic_add_edges(batch)
            blk = m.structural_distance_update_sharded(rank, world, peer=peer)
            torch.cuda.synchronize()
            p = m._plan
            if step == 0:
                plans = _gather(_ring_plan(p))
            same = torch.equal(blk, refs[step][p.row0:p.row0 + p.n_rows])
            path = "incremental" if p is before else "rebuilt"
            notes.append(f"update {step}: {path}, {int(m.last_affected.numel())} affected, equal {same}")
            ok = ok and same and (step == 0 or path == ("incremental" if step == 1 else "rebuilt"))
    return dict(ok=bool(ok), row=-1, dups=0, plans=plans, note="; ".join(notes))


def _cases():
    """(key, function, args) in the order every rank runs them."""
    out = [(f"knn-{n}-{h}-{k}", _case_knn, (n, h, k)) for n, h, k in KNN_CASES]
    out += [(f"model-knn-{n}-{h}-{k}", _case_model_knn, (n, h, k)) for n, h, k in MODEL_KNN_CASES]
    out += [(f"radius-{n}-{h}-{r}", _case_radius, (n, h, r)) for n, h, r in RADIUS_CASES]
    out += [("radius-cap", _case_radius_cap, ())]
    out += [(f"step-{n}-{h}-{p}-{s}", _case_step, (n, h, p, s)) for n, h, p, s in STEP_CASES]
    out += [(f"empty-{p}-{e}", _case_empty, (p, e)) for p, e in EMPTY_CASES]
    out += [(f"dynamic-{p}", _case_dynamic, (p,)) for p in DYNAMIC_CASES]
    return out


def _worker(rank, world, port, results):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    # the dense ring variant is a candidate at every world size tested here (default: from a fifth of the
    # nodes per rank), so that the skew also moves the choice between the two variants at 8 ranks
    os.environ["HSD_RING_DENSE_MIN_FRAC"] = "0.1"
    try:
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank),
                                timeout=datetime.timedelta(seconds=NCCL_TIMEOUT_S))
        inp = _Inputs()
        for key, fn, args in _cases():
            try:
                res = fn(inp, rank, world, *args)
            except Exception:
                res = dict(ok=False, row=-1, dups=0, plans=[], note=traceback.format_exc()[-3000:])
            results.put((rank, key, res))
        dist.destroy_process_group()
    except Exception:
        results.put((rank, "__error__", traceback.format_exc()[-3000:]))
    finally:
        results.put((rank, "__done__", None))


# ---------------------------------------------------------------------------------------------- test side
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.fixture(scope="module", params=_world_sizes(), ids=lambda w: f"world{w}")
def runs(request):
    """{rank: {case key: result}} of one spawn of `world` ranks, one per GPU."""
    import torch.multiprocessing as mp
    world = request.param
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, {torch.cuda.device_count()} visible")
    ctx = mp.get_context("spawn")
    results = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, results)) for r in range(world)]
    out = {r: {} for r in range(world)}
    done = set()
    try:
        for p in procs:
            p.start()
        deadline = time.monotonic() + TIMEOUT_S
        while len(done) < world and time.monotonic() < deadline:
            try:
                rank, key, res = results.get(timeout=5)
            except queue.Empty:
                if not any(p.is_alive() for p in procs):
                    break
                continue
            if key == "__done__":
                done.add(rank)
            else:
                out[rank][key] = res
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
        for p in procs:
            p.join(30)
            if p.is_alive():
                p.kill()
                p.join()
    return world, out


def _result(runs, key):
    world, out = runs
    for r in range(world):
        assert "__error__" not in out[r], f"rank {r}: {out[r]['__error__']}"
        assert key in out[r], f"rank {r} returned no result for {key} (the run stopped before it)"
    return world, [out[r][key] for r in range(world)]


def _assert_ok(results):
    for r, res in enumerate(results):
        assert res["ok"], (f"rank {r}: first row unlike one GPU {res['row']}, rows with a duplicate id {res['dups']}; "
                           f"{res['note']}")


def _assert_skew_took_effect(results):
    plans = results[0]["plans"]
    assert len(set(map(repr, plans))) > 1, f"every rank derived the same plan from its free memory: {plans}"


@pytest.mark.parametrize("n,hops,k", KNN_CASES)
def test_degree_knn_under_unequal_free_memory(runs, n, hops, k):
    """engine.degree_knn with a process group, odd ranks short of free memory: without an agreed panel height
    the ranks deal different panel lists, some rows are swept by no rank and some twice."""
    _, res = _result(runs, f"knn-{n}-{hops}-{k}")
    _assert_skew_took_effect(res)
    _assert_ok(res)


@pytest.mark.parametrize("n,hops,k", MODEL_KNN_CASES)
def test_model_nearest_neighbors_sharded_with_per_rank_block_bytes(runs, n, hops, k):
    world, res = _result(runs, f"model-knn-{n}-{hops}-{k}")
    if n >= 128 * world:
        _assert_skew_took_effect(res)
    _assert_ok(res)


@pytest.mark.parametrize("n,hops,which", RADIUS_CASES)
def test_model_radius_neighbors_sharded_under_unequal_free_memory(runs, n, hops, which):
    _, res = _result(runs, f"radius-{n}-{hops}-{which}")
    _assert_skew_took_effect(res)
    _assert_ok(res)


def test_model_radius_neighbors_sharded_cap_raises_on_every_rank(runs):
    _, res = _result(runs, "radius-cap")
    _assert_skew_took_effect(res)
    _assert_ok(res)
    assert len({r["note"] for r in res}) == 1, [r["note"] for r in res]


@pytest.mark.parametrize("n,hops,peer,skew", STEP_CASES)
def test_sharded_step_equals_one_gpu_rows(runs, n, hops, peer, skew):
    world, res = _result(runs, f"step-{n}-{hops}-{peer}-{skew}")
    if skew:
        _assert_skew_took_effect(res)
    _assert_ok(res)
    if n >= 32768:     # the column split is taken only when every rank votes for it
        assert res[0]["note"].count("'cols'" if not skew else "'rows'") == world, res[0]["note"]


@pytest.mark.parametrize("peer,empty", EMPTY_CASES)
def test_sharded_step_isolated_node(runs, peer, empty):
    """One isolated node in the last rank's block: with empty='raise' every rank raises EmptyRingError,
    with 'zero' every rank's block equals the one-GPU rows."""
    _, res = _result(runs, f"empty-{peer}-{empty}")
    _assert_skew_took_effect(res)
    _assert_ok(res)


@pytest.mark.parametrize("peer", DYNAMIC_CASES)
def test_dynamic_update_sharded_equals_one_gpu(runs, peer):
    _, res = _result(runs, f"dynamic-{peer}")
    _assert_skew_took_effect(res)
    _assert_ok(res)
