"""torchrun check: the radius graph of every node over G GPUs (engine.degree_radius with a process group:
dealt signatures, dealt row panels, the partial CSRs gathered and merged by hsd_radius_merge_parts) equals the
one-GPU result bit for bit on every rank — indptr, indices and the distance bits.

  torchrun --nproc_per_node G scripts/check_radius_sharded.py [N] [HOPS] [--profile DIR]   (default 100000 4)

The radius is the median over nodes of the 20th-NN distance (the rule of scripts/time_radius.py), so a node
has about 20 neighbours.  Every rank also computes the one-GPU result on its own device.  Rank 0 prints the
verdict, the device name, power limit and SM clocks, and both times (host clock around each call, ended by a
device synchronise; the first call of each after one warm-up call of each), with the summed event time of
the pairwise launches of this rank's panels.  --profile DIR: one more sharded call under torch.profiler,
whose per-kernel CUDA times rank 0 writes to DIR/radius_sharded_profile_w{G}.json (a run of its own:
tracing slows the host)."""
import json
import os
import subprocess
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
args = [a for i, a in enumerate(sys.argv[1:], 1) if not a.startswith("--") and sys.argv[i - 1] != "--profile"]
n = int(args[0]) if len(args) > 0 else 100000
hops = int(args[1]) if len(args) > 1 else 4
prof_dir = sys.argv[sys.argv.index("--profile") + 1] if "--profile" in sys.argv else None
dg = engine.DeviceGraph.upload(powerlaw_graph(n, 5, seed=0))     # same deterministic graph on every rank
_, kval = engine.degree_knn(dg, hops, 20)
radius = float(kval[:, 19].median())
del kval


def timed(**kw):
    events = []
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    out = engine.degree_radius(dg, hops, radius, pair_events=events, **kw)
    torch.cuda.synchronize()
    t = time.perf_counter() - t0
    pair = sum(e0.elapsed_time(e1) for _, _, e0, e1 in events)
    return out, t, pair, len(events)


timed()                                               # warm-up: module loads, allocator, NCCL communicators
torch.cuda.empty_cache()
timed(rank=rank, world=world)
torch.cuda.empty_cache()
one, t_one, pair_one, panels_one = timed()
torch.cuda.empty_cache()
got, t_sh, pair_sh, panels_sh = timed(rank=rank, world=world)
ok = (torch.equal(got[0], one[0]) and torch.equal(got[1], one[1])
      and torch.equal(got[2].view(torch.int32), one[2].view(torch.int32)))
stats = torch.tensor([int(ok), t_sh * 1e6, pair_sh * 1e3], dtype=torch.float64, device="cuda")
lo, hi = stats.clone(), stats.clone()
dist.all_reduce(lo, op=dist.ReduceOp.MIN)
dist.all_reduce(hi, op=dist.ReduceOp.MAX)
if rank == 0:
    q = subprocess.run(["nvidia-smi", "-i", str(lr), "--query-gpu=power.limit,clocks.sm,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(f"world={world} n={n} hops={hops} radius={radius!r} nnz={one[1].numel()} "
          f"device={torch.cuda.get_device_name()} [power limit, SM clock, max SM clock: {q}]: every rank "
          f"bit-equal to one GPU: {bool(lo[0].item())}; one GPU {t_one * 1e3:.1f} ms ({panels_one} panels, "
          f"pairwise {pair_one:.1f} ms), {world} GPUs {hi[1].item() / 1e3:.1f} ms (slowest rank; pairwise "
          f"{lo[2].item() / 1e3:.1f}-{hi[2].item() / 1e3:.1f} ms per rank over {panels_sh} panels on rank 0)",
          flush=True)
del got, one
torch.cuda.empty_cache()
if prof_dir:
    from torch.profiler import ProfilerActivity, profile
    dist.barrier()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        engine.degree_radius(dg, hops, radius, rank=rank, world=world)
        torch.cuda.synchronize()
    if rank == 0:
        kernels = []
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
            if t and e.device_type.name == "CUDA":
                kernels.append({"name": e.key[:120], "cuda_ms": t / 1e3, "calls": e.count})
        kernels.sort(key=lambda k: -k["cuda_ms"])
        os.makedirs(prof_dir, exist_ok=True)
        with open(os.path.join(prof_dir, f"radius_sharded_profile_w{world}.json"), "w") as f:
            json.dump({"n": n, "hops": hops, "world": world, "rank": 0, "radius": radius,
                       "device": torch.cuda.get_device_name(), "kernels": kernels}, f, indent=1)
dist.destroy_process_group()
