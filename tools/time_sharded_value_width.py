"""A database sharded along M with values of width D = 768 / 1024 / 2048: ms per step of the sharded embed (RANGE+
beta = 0.5, 100 000 queries per step in all, M = 1 M entries) and the time of reduce_route_kernel, the kernel that sums
a query chunk's database-split partials and stores each row into its owner's receive buffer.
    python -m torch.distributed.run --nproc-per-node 8 tools/time_sharded_value_width.py
    python tools/time_sharded_value_width.py          (one GPU: one rank's share, see below)
Environment: M (entries, default 1 000 000), N (queries per step in all, default 100 000), SHARDS (one GPU only: the
ranks whose share it runs, default 8).
Every rank passes N / world queries; the step bound is raised so that a call is one step at every D (the default bound
splits D = 2048 into two steps of 65 536 rows).  Step time: host clock around 10 calls that end in a device synchronise
and a barrier, median of 3 windows after a warm-up.  Kernel time: torch.profiler (CUDA activities) over 3 further calls,
in a run of its own after the timed windows; the sum of reduce_route_kernel launches per call, rank 0.
On one GPU (no torchrun) a one-rank world runs the share of one rank of SHARDS: M / SHARDS entries against all N queries,
through the same routed path into a local receive buffer - the compute of one rank, without NVLink stores or the
other ranks' collectives.  Prints the card and its power limit.
"""
import contextlib
import os
import subprocess
import sys
import time
from argparse import Namespace

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from range_b200 import synthetic                                # noqa: E402
from range_b200.database import DeviceDatabase                 # noqa: E402
from range_b200.distributed import ShardedRetriever            # noqa: E402
from range_b200.range import LocationEncoder                   # noqa: E402

M, N = int(os.environ.get("M", 1_000_000)), int(os.environ.get("N", 100_000))
torchrun = "RANK" in os.environ
rank, world = (int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])) if torchrun else (0, 1)
local = int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if torchrun:
    dist.init_process_group("nccl", device_id=dev)
else:
    dist.init_process_group("nccl", init_method="tcp://127.0.0.1:29561", rank=0, world_size=1, device_id=dev)
shards = world if world > 1 else int(os.environ.get("SHARDS", 8))
card = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit,clocks.max.sm",
                       "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
enc = dict(L=40, dims=[1600, 512, 512, 256], weights=synthetic.siren_init(seed=7))
coords = torch.tensor(synthetic.area_uniform(N // world, np.random.default_rng(11 + rank)), device=dev)


def step_ms(fn, reps=10, windows=3):
    fn(); torch.cuda.synchronize(); dist.barrier()
    ts = []
    for _ in range(windows):
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize(); dist.barrier()
        ts.append((time.perf_counter() - t0) / reps * 1e3)
    return sorted(ts)[windows // 2]


def route_kernel_ms(fn, calls=3):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "reduce_route_kernel" in e.key)
    n = sum(e.count for e in prof.key_averages() if "reduce_route_kernel" in e.key)
    return us / 1e3 / calls, n // calls


if rank == 0:
    print(f"card: {card}")
    what = f"{world} GPUs" if world > 1 else f"one GPU running the share of one rank of {shards}"
    print(f"{what}: M = {M} ({M // shards} per shard), {N} queries per step in all, RANGE+ beta = 0.5")
for D in (768, 1024, 2048):
    db = DeviceDatabase.synthetic(M // shards if world == 1 else M, dev, seed=3, value_dim=D,
                                  shard=None if world == 1 else (rank, world))
    with contextlib.redirect_stdout(sys.stderr):
        model = LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=enc, device=dev, beta=0.5,
                                          range_db=db))
    sr = ShardedRetriever(model.engine, merge="peer")
    slab = (coords.shape[0] + 127) // 128 * 128                                                # one step per call
    sr.MAX_STEP_ROWS = max(ShardedRetriever.MAX_STEP_ROWS, slab * world * max(D, 1024) // 1024)
    model.sharded = sr
    out = torch.empty(coords.shape[0], D + 256, dtype=torch.float32, device=dev)
    call = lambda: model.embed(coords, out=out)                 # noqa: E731
    before = sr.collectives
    call()
    steps = (sr.collectives - before - 1) // 4
    ms = step_ms(call)
    k_ms, k_n = route_kernel_ms(call)
    if rank == 0:
        path = "producer/consumer epilogue" if D == 1024 else f"CTA pairs x {(D + 255) // 256} slices + reduce_route"
        print(f"D = {D:4d}  {ms:8.2f} ms per call ({steps} step{'s' if steps > 1 else ''}, {path}); "
              f"reduce_route_kernel {k_ms:7.3f} ms per call over {k_n} launches; merge '{sr.merge}'")
    sr.close()
    del model, sr, db, out
    torch.cuda.empty_cache()
dist.destroy_process_group()
