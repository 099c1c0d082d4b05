"""torchrun check: k nearest neighbours of every node over G GPUs (engine.degree_knn with a process
group: dealt signatures, dealt row panels, one all-gather + hsd_topk_merge) equal the one-GPU result
bit for bit on every rank.

  torchrun --nproc_per_node G scripts/check_knn_sharded.py [N] [HOPS] [K]     (default 100000 4 20)

Every rank also computes the one-GPU result on its own device; prints the verdict and both times."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from hsd_b200 import engine
from hsd_b200.graph import powerlaw_graph

rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
n = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
hops = int(sys.argv[2]) if len(sys.argv) > 2 else 4
k = int(sys.argv[3]) if len(sys.argv) > 3 else 20
dg = engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0))     # same deterministic graph on every rank

torch.cuda.synchronize()
t0 = time.perf_counter()
idx1, val1 = engine.degree_knn(dg, hops, k)
torch.cuda.synchronize()
t_one = time.perf_counter() - t0
torch.cuda.empty_cache()
dist.barrier()
t0 = time.perf_counter()
idx, val = engine.degree_knn(dg, hops, k, rank=rank, world=world)
torch.cuda.synchronize()
dist.barrier()
t_sharded = time.perf_counter() - t0
ok = torch.equal(idx, idx1) and torch.equal(val.view(torch.int32), val1.view(torch.int32))
t = torch.tensor([int(ok)], device="cuda")
dist.all_reduce(t, op=dist.ReduceOp.MIN)
if rank == 0:
    print(f"world={world} n={n} hops={hops} k={k} device={torch.cuda.get_device_name()}: every rank bit-equal "
          f"to one GPU: {bool(t.item())}; one GPU {t_one * 1e3:.1f} ms, {world} GPUs {t_sharded * 1e3:.1f} ms "
          f"(host clock, first call of each)", flush=True)
dist.destroy_process_group()
