"""Databases of other value widths: RANGE+ (beta = 0.5) at 100 000 queries x 100 000 entries for D in
{64, 256, 768, 1024, 2048}.  Times the statistics pass, the apply pass (range_retrieve_apply into an (N, D) array) and
LocationEncoder.embed end to end (sort, encode, statistics, apply + concat into an (N, D + 256) fp32 result).
    python tools/time_value_width.py [N] [M]      -> ms per call (CUDA events, median of 10 calls after 3 warm-ups)
Synthetic spatially sorted database (DeviceDatabase.synthetic(value_dim=D): geo-term skipping active), area-uniform
queries sorted spatially like model(locs) does.  D = 1024 runs the producer/consumer apply kernel, every other width the
CTA-pair kernel over ceil(D / 256) value slices.
"""
import os
import subprocess
import sys
from argparse import Namespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from range_b200 import synthetic                                # noqa: E402
from range_b200.database import DeviceDatabase                 # noqa: E402
from range_b200.range import LocationEncoder                   # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 100_000
M = int(sys.argv[2]) if len(sys.argv) > 2 else 100_000
dev = torch.device("cuda", 0)
card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card}")
enc = dict(L=40, dims=[1600, 512, 512, 256], weights=synthetic.siren_init(seed=7))
raw = torch.tensor(synthetic.area_uniform(N, np.random.default_rng(5)), device=dev)


def timed(fn, reps=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return sorted(ts)[reps // 2], min(ts)


print(f"N = {N}, M = {M}, RANGE+ beta = 0.5")
for D in (64, 256, 768, 1024, 2048):
    model = LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=enc, device=dev, beta=0.5,
                                      range_db=DeviceDatabase.synthetic(M, dev, seed=3, value_dim=D)))
    eng, a = model.engine, model.args
    coords, _ = eng.sort_queries(raw)
    _, q16, qxyz = eng.encode(coords)
    sums, maxs = eng.retrieve_stats("RANGE+", q16, qxyz, a.temp, a.geo_temp)
    O = torch.empty(N, D, dtype=torch.float32, device=dev)
    out = torch.empty(N, D + 256, dtype=torch.float32, device=dev)
    s_med, _ = timed(lambda: eng.retrieve_stats("RANGE+", q16, qxyz, a.temp, a.geo_temp))
    a_med, a_lo = timed(lambda: eng.retrieve_apply("RANGE+", q16, qxyz, a.temp, a.geo_temp, 0.5, sums, maxs, O=O))
    e_med, e_lo = timed(lambda: model.embed(raw, out=out))
    kernel = "producer/consumer" if D == 1024 else f"CTA pairs x {(D + 255) // 256} slices"
    print(f"D = {D:4d}  statistics {s_med:7.3f} ms  apply {a_med:7.3f} ms (min {a_lo:7.3f}, {kernel})  "
          f"embed {e_med:7.3f} ms (min {e_lo:7.3f})  {N / e_med / 1e3:5.2f} M queries/s")
    del model, eng, O, out
    torch.cuda.empty_cache()
