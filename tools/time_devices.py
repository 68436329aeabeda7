"""One model on several GPUs of this host (load_model(..., devices=n)): how do model(locs) and embed scale?
RANGE+ beta = 0.5, M = 100 000 entries (H = 512 SIREN, bench.py's synthetic inputs), in ONE process:

  model(locs)  float64 coordinates in page-locked host memory -> numpy float64 (N, 1280)   (end to end)
  embed        float64 coordinates on the primary -> (N, 1280) float32 on the primary       (device-resident)

at n = 1, 2, 4, 8 devices (those visible), for 100 000 queries per device and for TOTAL queries in all.  Wall clock
around each call, every device synchronised before and after; 2 warm-up calls, then REPS calls: median, min and max.
--dup k adds a run of k replicas on GPU 0 alone (devices=[0] * k: the cost of splitting, no speed-up possible).
--trace prints model(locs)'s piece timeline on every replica for the largest n (LocationEncoder.trace).

    python tools/time_devices.py [--total 10000000] [--reps 5] [--dup 3] [--trace] [--json out.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from argparse import Namespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                                    # noqa: E402
from range_b200.database import DeviceDatabase                 # noqa: E402
from range_b200.range import LocationEncoder                   # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--total", type=int, default=10_000_000)
ap.add_argument("--per-device", type=int, default=100_000)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--dup", type=int, default=0)
ap.add_argument("--trace", action="store_true")
ap.add_argument("--json")
opt = ap.parse_args()

count = torch.cuda.device_count()
cards = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
host_mem = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_AVPHYS_PAGES")
print(f"{count} visible GPUs: " + " | ".join(cards))
print(f"host: {os.cpu_count()} cores, {host_mem / 2**30:.0f} GiB free memory")
db, weights, _ = bench.synthetic_inputs(M=100_000)
enc = dict(L=40, dims=[1600, 512, 512, 256], weights=weights)
ddb = DeviceDatabase(db, "cuda:0")


def sync():
    for d in range(count):
        torch.cuda.synchronize(d)


def timed(fn):
    for _ in range(2):
        fn()
    ts = []
    for _ in range(opt.reps):
        sync()
        t = time.perf_counter()
        fn()
        sync()
        ts.append(time.perf_counter() - t)
    return float(np.median(ts)), min(ts), max(ts)


configs = [[i for i in range(n)] for n in (1, 2, 4, 8) if n <= count]
if opt.dup > 1:
    configs.append([0] * opt.dup)
results = dict(cards=cards, M=100_000, model="RANGE+", beta=0.5, rows=[])
for devs in configs:
    model = LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=enc, device="cuda:0", range_db=ddb,
                                      beta=0.5, devices=devs if len(devs) > 1 else None))
    for N in (opt.per_device * len(devs), opt.total):
        rng = np.random.default_rng(N)
        c = torch.tensor(np.stack([rng.uniform(-180, 180, N), np.degrees(np.arcsin(rng.uniform(-1, 1, N)))], 1))
        h, dc = c.pin_memory(), c.to("cuda:0")
        row = dict(devices=devs, N=N, host_threads=model.host_threads)
        t = timed(lambda: model.embed(dc))
        row["embed_s"] = t
        if N * 1280 * 8 * 1.5 < host_mem:
            row["model_s"] = timed(lambda: model(h))
        else:
            row["model_s"] = None                   # the float64 result would not fit this host's free memory
        results["rows"].append(row)
        msg = f"devices {devs}  N {N:>9}  embed {t[0] * 1e3:8.1f} ms [{t[1] * 1e3:.1f}-{t[2] * 1e3:.1f}] " \
              f"= {N / t[0] / 1e6:6.2f} M q/s"
        if row["model_s"] is not None:
            m = row["model_s"]
            msg += f"  model(locs) {m[0] * 1e3:8.1f} ms [{m[1] * 1e3:.1f}-{m[2] * 1e3:.1f}] = {N / m[0] / 1e6:6.2f} M q/s"
        else:
            msg += "  model(locs) not run: float64 result larger than free host memory"
        print(msg, flush=True)
        if opt.trace and devs == configs[-1] and N == opt.per_device * len(devs):
            reps = model.replicas.models if model.replicas is not None else [model]
            for r in reps:
                r.trace = []
            sync()
            w = time.perf_counter()
            model(h)
            sync()
            wall = time.perf_counter() - w
            print(f"  timeline of one model(locs) call (wall {wall * 1e3:.1f} ms), ms from each replica's start:")
            for i, r in enumerate(reps):
                t0 = r.trace[0][1]
                print(f"  replica {i} (cuda:{r.engine.index}): " + " | ".join(
                    f"{rows}: computed {t0.elapsed_time(a):.1f} copied {t0.elapsed_time(b):.1f}" for rows, a, b in r.trace[1:]))
                r.trace = None
        del c, h, dc
    model.close()
    del model
    torch.cuda.empty_cache()
if opt.json:
    with open(opt.json, "w") as f:
        json.dump(results, f, indent=1)
