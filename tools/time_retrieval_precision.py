"""Split-fp16 retrieval against fp16 operands: RANGE+ (beta = 0.5) at 100 000 queries x 100 000 entries, D = 1024 and 768.
Times the statistics pass, the apply pass (range_retrieve_apply into an (N, D) array) and LocationEncoder.embed end to end
(sort, encode, statistics, apply + concat into an (N, D + 256) fp32 result) for retrieval_precision 'fp16' and 'f16x3'.
    python tools/time_retrieval_precision.py [N] [M] [json_out]   -> ms per call (CUDA events, median of 10 calls after
                                                                     3 warm-ups), the two modes alternating per round
One synthetic spatially sorted database with its lo halves serves both models (an 'fp16' model does not read them).
Also reports, on a 4096-query sample, the relative row difference between the modes.
"""
import json
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
OUT = sys.argv[3] if len(sys.argv) > 3 else None
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
    return sorted(ts)[reps // 2]


results = dict(card=card, N=N, M=M, model="RANGE+", beta=0.5, rows=[])
print(f"N = {N}, M = {M}, RANGE+ beta = 0.5")
for D in (1024, 768):
    ddb = DeviceDatabase.synthetic(M, dev, seed=3, value_dim=D, lo=True)
    models = {p: LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=enc, device=dev, beta=0.5,
                                           range_db=ddb, retrieval_precision=p)) for p in ("fp16", "f16x3")}
    prep = {}
    for p, model in models.items():
        eng, a = model.engine, model.args
        coords, _ = eng.sort_queries(raw)
        _, q16, qxyz = eng.encode(coords)
        sums, maxs = eng.retrieve_stats("RANGE+", q16, qxyz, a.temp, a.geo_temp)
        prep[p] = (eng, a, q16, qxyz, sums, maxs, torch.empty(N, D, dtype=torch.float32, device=dev),
                   torch.empty(N, D + 256, dtype=torch.float32, device=dev))
    t = {p: dict(stats=[], apply=[], embed=[]) for p in models}
    for _ in range(3):                        # the modes alternate: drift of the shared card hits both alike
        for p, model in models.items():
            eng, a, q16, qxyz, sums, maxs, O, out = prep[p]
            t[p]["stats"].append(timed(lambda: eng.retrieve_stats("RANGE+", q16, qxyz, a.temp, a.geo_temp)))
            t[p]["apply"].append(timed(lambda: eng.retrieve_apply("RANGE+", q16, qxyz, a.temp, a.geo_temp, 0.5, sums, maxs,
                                                                  O=O)))
            t[p]["embed"].append(timed(lambda: model.embed(raw, out=out)))
    sample = raw[:4096]
    e16 = models["fp16"].embed(sample, out_dtype=torch.float64)[:, :D]
    e3 = models["f16x3"].embed(sample, out_dtype=torch.float64)[:, :D]
    diff = float(((e3 - e16).norm(dim=1) / e3.norm(dim=1)).max())
    for p in models:
        row = dict(D=D, precision=p, **{k: float(np.median(v)) for k, v in t[p].items()})
        results["rows"].append(row)
        print(f"D = {D:4d} {p:6s} statistics {row['stats']:7.3f} ms  apply {row['apply']:7.3f} ms  "
              f"embed {row['embed']:7.3f} ms  {N / row['embed'] / 1e3:5.2f} M queries/s")
    print(f"D = {D:4d} max relative row difference f16x3 vs fp16 (4096 queries): {diff:.2e}")
    results[f"rel_row_diff_D{D}"] = diff
    del models, prep, ddb
    torch.cuda.empty_cache()
if OUT:
    with open(OUT, "w") as f:
        json.dump(results, f, indent=1)
