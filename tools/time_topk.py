"""Retrieval neighbours: the statistics pass alone against the top-k pass (range_retrieve_topk) at 100 000 queries x
100 000 entries, RANGE and RANGE+ (beta = 0.5), k in {1, 8, 32}.
    python tools/time_topk.py [N] [M]      -> ms per call (CUDA events, median of 20 calls after 3 warm-ups)
Synthetic spatially sorted database (DeviceDatabase.synthetic: geo-term skipping active), area-uniform queries sorted
spatially like model(locs) does.  The keys (M x 512 B = 51 MB at M = 100 000) stay in the 126 MB L2 between calls.
"""
import subprocess
import sys
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from range_b200 import synthetic                                # noqa: E402
from range_b200.database import DeviceDatabase                 # noqa: E402
from range_b200.engine import RangeEngine                      # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 100_000
M = int(sys.argv[2]) if len(sys.argv) > 2 else 100_000
dev = torch.device("cuda", 0)
card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card}")
eng = RangeEngine(dev, encoder=dict(L=40, dims=[1600, 512, 512, 256], weights=synthetic.siren_init(seed=7)),
                  database=DeviceDatabase.synthetic(M, dev, seed=3))
coords, _ = eng.sort_queries(torch.tensor(synthetic.area_uniform(N, np.random.default_rng(5)), device=dev))
_, q16, qxyz = eng.encode(coords)


def timed(fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return sorted(ts)[reps // 2], min(ts)


flop = 2.0 * N * M * 256
print(f"N = {N}, M = {M}: Q.K^T = {flop / 1e12:.2f} TFLOP per pass")
for name, temp, beta in [("RANGE", 15.0, None), ("RANGE+", 12.0, 0.5)]:
    sums, _ = eng.retrieve_stats(name, q16, qxyz, temp, 40.0)
    med, lo = timed(lambda: eng.retrieve_stats(name, q16, qxyz, temp, 40.0))
    print(f"{name:6s} statistics        median {med:7.3f} ms  min {lo:7.3f} ms  ({flop / med / 1e9:6.0f} TFLOP/s)")
    stats_med = med
    for k in (1, 8, 32):
        med, lo = timed(lambda: eng.retrieve_topk(name, q16, qxyz, temp, 40.0, beta, sums, k))
        print(f"{name:6s} top-k k = {k:2d}     median {med:7.3f} ms  min {lo:7.3f} ms  ({flop / med / 1e9:6.0f} TFLOP/s, "
              f"{med / stats_med:.2f}x statistics)")
