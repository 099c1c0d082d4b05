"""The multi-GPU ring phase is chosen collectively: the column-split and the row-split phases issue
different collectives, so every rank must take the same one whatever its own free memory says."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _vote_worker(rank, world, port, votes, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from hsd_b200.sharded import agree_all
    ret[rank] = agree_all(votes[rank], world, device="cpu")      # the call ShardedDegreeHSD makes per rank
    dist.destroy_process_group()


@pytest.mark.parametrize("votes", [(True, True), (True, False), (False, True), (False, False)])
def test_world2_ring_mode_vote_is_unanimous(votes):
    """One rank short of memory (another job on its GPU) sends every rank to the row-split phase."""
    world = 2
    port = _free_port()
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    procs = [ctx.Process(target=_vote_worker, args=(r, world, port, votes, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert ret[0] == ret[1] == all(votes)


@pytest.mark.parametrize("n,world", [(32768, 2), (100000, 3), (1000000, 8), (1000003, 7)])
def test_cols_workspace_words_is_the_largest_rank(n, world):
    """Every rank sizes its vote by the rank with the most bitmap pieces, not by its own share."""
    from hsd_b200.engine import ring_cols_range
    from hsd_b200._lib import lib
    from hsd_b200.sharded import agree_all, cols_workspace_words
    per_rank = [int(lib.hsd_ring_cols_workspace_words(n, *ring_cols_range(n, r, world))) for r in range(world)]
    assert cols_workspace_words(n, world) == max(per_rank)
    assert agree_all(False, world) is False and agree_all(True, 1) is True     # no process group: the local vote
