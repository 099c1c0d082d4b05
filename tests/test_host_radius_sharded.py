"""Host-side parts of the radius graph over several ranks (engine.degree_radius with world > 1,
HSD.radius_neighbors_sharded) that need no GPU: the panel plan, the default cap, argument validation of
hsd_radius_merge_parts, and world-2 gloo runs of the variable-size gather and of the cap agreement."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _run_world2(target, *args):
    """Runs target(rank, world, port, *args, ret) in two spawned gloo processes; returns ret (rank -> value).
    Joins with a timeout: a rank left waiting in a collective fails the exit-code check instead of hanging."""
    world = 2
    port = _free_port()
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    procs = [ctx.Process(target=target, args=(r, world, port) + args + (ret,)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
    for p in procs:
        if p.exitcode is None:
            p.kill()
            p.join()
    assert [p.exitcode for p in procs] == [0, 0]
    return dict(ret)


def _init(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)


# ---------------------------------------------------------------- plan and cap
@pytest.mark.parametrize("n", [34, 4099, 20000, 100000, 300000])
@pytest.mark.parametrize("budget", [1, 128 * 4 * 4100, 178 * (1 << 30) // 2])
def test_radius_panel_rows_world_cap(n, budget):
    """world = 1 is the one-GPU plan; with several ranks the panels are capped at about
    N / (KNN_PANELS_PER_RANK x world) rows, like knn_panel_rows, and never grow."""
    from hsd_b200.engine import KNN_PANELS_PER_RANK, knn_panel_rows, radius_panel_rows
    one = radius_panel_rows(n, budget)
    assert radius_panel_rows(n, budget, world=1) == one
    for world in (2, 3, 8):
        r = radius_panel_rows(n, budget, world)
        assert r <= one and (r == n or r % 128 == 0)
        cap = max(128, n // (KNN_PANELS_PER_RANK * world) // 128 * 128)
        assert r == (n if min(one, cap) >= n else min(one, cap))
        assert r <= knn_panel_rows(n, budget, world)


def test_radius_sharded_max_pairs_formula():
    """Each global entry exists as gathered id + dist and as merged id + dist (16 bytes) next to the rank's
    own partial (8 bytes per entry, at most the global count): 24 bytes."""
    from hsd_b200.engine import RADIUS_PAIR_FRACTION, radius_sharded_max_pairs
    free = 10 ** 10
    assert radius_sharded_max_pairs(free) == int(free * RADIUS_PAIR_FRACTION) // 24
    assert radius_sharded_max_pairs(24) == 0 and radius_sharded_max_pairs(-5) == 0


def test_radius_merge_parts_argument_validation_without_gpu():
    from hsd_b200._lib import lib
    b = (ctypes.c_int64 * 256)()
    p = ctypes.addressof(b)
    err = lib.hsd_last_error_string
    f = lib.hsd_radius_merge_parts
    # (n_parts, n_rows, part_indptr, part_base, idx, val, elem_bytes, indptr, idx_out, val_out, stream)
    for k in range(7):
        ptrs = [p] * 7
        ptrs[k] = None
        pi, pb, ix, vl, ip, io, vo = ptrs
        assert f(2, 4, pi, pb, ix, vl, 4, ip, io, vo, None) == -1 and b"null" in err(), k
    assert f(2, 4, p, p, p, p, 2, p, p, p, None) == -1 and b"elem_bytes" in err()
    assert f(2, 4, p, p, p, p, 16, p, p, p, None) == -1 and b"elem_bytes" in err()
    assert f(0, 4, p, p, p, p, 4, p, p, p, None) == -1 and b"n_parts" in err()
    assert f(65, 4, p, p, p, p, 4, p, p, p, None) == -1 and b"n_parts" in err()
    assert f(-1, 4, p, p, p, p, 4, p, p, p, None) == -1 and b"n_parts" in err()
    assert f(2, -1, p, p, p, p, 8, p, p, p, None) == -1 and b"n_rows" in err()
    assert f(64, 0, p, p, p, p, 8, p, p, p, None) == 0                                     # no rows: nothing to do


# ---------------------------------------------------------------- gloo, world 2
def _csr(rng, n, nnz, dtype):
    """A random CSR over n rows with nnz entries: ascending ids per row, values of the given dtype."""
    rows = np.sort(rng.integers(0, n, nnz))
    indptr = np.zeros(n + 1, np.int64)
    np.add.at(indptr, rows + 1, 1)
    indptr = np.cumsum(indptr)
    idx = rng.integers(0, 1 << 20, nnz).astype(np.int32)
    for i in range(n):
        idx[indptr[i]:indptr[i + 1]].sort()
    return indptr, idx, rng.standard_normal(nnz).astype(dtype)


def _gather_worker(rank, world, port, n, sizes, dtype, ret):
    _init(rank, world, port)
    from hsd_b200.sharded import gather_csr_parts
    parts = [_csr(np.random.default_rng(r), n, sizes[r], dtype) for r in range(world)]   # every rank knows all
    indptr, idx, val = (torch.from_numpy(a) for a in parts[rank])
    part_indptr, part_base, idx_all, val_all = gather_csr_parts(indptr, idx, val, world)
    ok = part_indptr.shape == (world, n + 1) and part_base.tolist() == [0, sizes[0]]
    ok = ok and idx_all.dtype == torch.int32 and val_all.dtype == getattr(torch, dtype)
    for r in range(world):
        s = slice(int(part_base[r]), int(part_base[r]) + sizes[r])
        ok = ok and np.array_equal(part_indptr[r].numpy(), parts[r][0])
        ok = ok and np.array_equal(idx_all[s].numpy(), parts[r][1])
        ok = ok and np.array_equal(val_all[s].numpy().view(np.uint8), parts[r][2].view(np.uint8))
    ret[rank] = (bool(ok), int(idx_all.numel()))
    dist.destroy_process_group()


@pytest.mark.parametrize("sizes,dtype", [((1000, 37), "float32"), ((5, 4000), "float64"), ((0, 300), "float32"),
                                         ((300, 0), "float32"), ((0, 0), "float32")])
def test_world2_gather_csr_parts_uneven_and_empty(sizes, dtype):
    """Entry counts differ per rank, one rank (or both) may hold none; every rank gets every part, exact size."""
    ret = _run_world2(_gather_worker, 211, sizes, dtype)
    assert ret[0] == ret[1] == (True, sum(sizes))


def _cap_worker(rank, world, port, nnz, stopped, max_pairs, ret):
    _init(rank, world, port)
    from hsd_b200.sharded import agree_radius_cap
    try:
        ret[rank] = ("ok", agree_radius_cap(nnz[rank], stopped[rank], max_pairs, 0.5))
    except ValueError as e:
        ret[rank] = ("raised", str(e))
    dist.destroy_process_group()


@pytest.mark.parametrize("nnz,stopped,max_pairs,raised", [
    ((120, 4), (True, False), 100, True),      # one rank passed the cap alone and stopped its sweep
    ((4, 120), (False, True), 100, True),
    ((60, 60), (False, False), 100, True),     # neither rank alone, the sum does
    ((60, 40), (False, False), 100, False),    # exactly the cap: allowed
    ((0, 0), (False, False), 0, False),
])
def test_world2_radius_cap_is_agreed(nnz, stopped, max_pairs, raised):
    """Both ranks raise the same ValueError (today's wording) or both return the global nnz; nobody hangs."""
    ret = _run_world2(_cap_worker, nnz, stopped, max_pairs)
    assert ret[0] == ret[1]
    if raised:
        assert ret[0][0] == "raised"
        msg = ret[0][1]
        assert f"at least {sum(nnz)} entries" in msg and f"max_pairs = {max_pairs}" in msg and "radius 0.5" in msg
    else:
        assert ret[0] == ("ok", sum(nnz))
