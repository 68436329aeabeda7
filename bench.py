"""Headline benchmark: RANGE+ (beta = 0.5) embeddings/s on a range_db_large-shaped synthetic database.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--shard m]

One "step" = the whole hot path (spatial batching -> SH + SIREN encoder -> statistics -> fused apply + concat) over one
batch of 100 000 queries per GPU against a 100 000-entry database (BASELINE.json configs[1]).  `value` times it with the
queries already in HBM and the (N,1280) result left in HBM; `e2e` times `model(locs)` - the reference's public API -
from a pinned host tensor to the numpy float64 array it returns.

N > 1 (torchrun, one rank per GPU): the headline keeps the reference's data-parallel reading - every rank embeds its
own 100 000 queries against a replicated database, no data-path collective: weak scaling.  The same line also carries
`m_sharded`: BASELINE.json configs[3], the database sharded along M over the N ranks (range_b200/distributed.py: the
exp-sums merge by one 8 B/query all-reduce, the partial outputs leave the apply kernel's epilogue into the owner
rank's receive buffer over NVLink), at M = 100 k and 1 M (and 10 M on 8 GPUs), each next to the collective-free
replicated-database run of the same shape.  `--shard m` runs only that section (one JSON line of its own).

--impl reference times the reference's own CPU implementation on the host cores: the UNMODIFIED mvrl/RANGE package
(oracle/_ref/reference, staged by __graft_entry__.build(); oracle/ref_harness.py) when it is there, else the oracle
port, on a bounded sample of the same workload.

--dump-outputs DIR (rank 0) writes what the last timed step returned, so that two builds can be compared output for
output on the same seeded inputs: DIR/embeddings.npy (float32, the step's (N,1280) result) and
DIR/model_embeddings.npy (float64, the (N,1280) array `model(locs)` returns), both as the same fixed sample of
DUMP_ROWS rows (dump_rows()), 47 MB in all.
"""
import argparse
import contextlib
import glob
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_QUERIES = 100_000
M_DB = 100_000
M_MED = 50_000                  # range_db_med shape (BASELINE.md section 3: assumption, parameterised)
H = 512
BETA = 0.5
FLOP_PER_PAIR = 2566.0          # 2*256 + 2*3 + 2*1024 (SURVEY.md 8d, blended-P form)
METRIC = "RANGE+ embeddings/sec"
UNIT = "queries/s"
REF_SAMPLE_QUERIES = 5000       # per step of the reference arm: each N x M fp32 matrix it materialises is 2 GB
WORKLOAD = f"RANGE+ beta={BETA}, M={M_DB} (range_db_large shape), SatCLIP-L40 H={H} random-init"
DUMP_ROWS = 3072                # 3072 x 1280 x (4 + 8) B = 47 MB: the dump stays under 64 MB


def dump_rows():
    """the rows --dump-outputs writes: a fixed seeded sample of the N_QUERIES result rows, in increasing order"""
    return np.sort(np.random.default_rng(0).choice(N_QUERIES, DUMP_ROWS, replace=False))


def synthetic_inputs(rank=0, M=M_DB, n=N_QUERIES):
    from range_b200 import synthetic as S
    db = S.iid_database(M, seed=0)
    weights = S.siren_init(40, H, 2, 256, seed=0)
    coords = S.area_uniform(n, np.random.default_rng(1 + rank))
    return db, weights, coords


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["bf16_tflops_sustained"]), float(d["hbm_gbs"]), "measured"
    return 1400.0, 6650.0, "fallback"


def apply_kernel_traffic():
    """DRAM bytes per launch of the apply kernel from the newest `ncu --set full` summary under profiles/
    (dram__bytes_read.sum + dram__bytes_write.sum of the range_apply_pc_kernel column), or (None, None)"""
    import csv
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_k2_ncu_full_selected.csv")), reverse=True):
        try:
            rows = {r[0]: r for r in csv.reader(open(path)) if r}
            col = next(i for i, v in enumerate(rows["Kernel Name"]) if "range_apply_pc_kernel" in v)
            scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
            total = sum(float(rows[k][col]) * scale[rows[k][1]] for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
            return total, os.path.relpath(path, ROOT)
        except Exception:
            continue
    return None, None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region"""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def __enter__(self):
        if os.environ.get("RANGE_BENCH_NO_SMI") == "1":      # developer switch: run without the sampler process
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for t, r in self.rows if self.t0 is None or (self.t0 - 0.05 <= t <= (self.t1 or 1e30) + 0.1)]
        for r in rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for nm, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# the reference's CPU path
# ------------------------------------------------------------------------------------------------------------------
class ReferenceCpu:
    """the reference's `load_model(...)` / `model(locs)` on the host cores: the unmodified package when it is staged
    (kind 'reference'), else the oracle port (kind 'port')"""

    def __init__(self, want_port=False):
        from oracle import ref_harness as R
        want_port = want_port or os.environ.get("RANGE_BENCH_REFERENCE", "") == "port"      # (tests: force the port)
        self.kind = "reference" if (R.available() and not want_port) else "port"
        self.tmp = tempfile.mkdtemp(prefix="range_ref_")
        import atexit
        import shutil
        atexit.register(shutil.rmtree, self.tmp, ignore_errors=True)       # the fabricated checkpoint / database files
        self._models = {}
        if self.kind == "reference":
            with contextlib.redirect_stdout(sys.stderr):
                self.load_model, module = R.import_reference()
                self.ckpt = os.path.join(self.tmp, "satclip_l40.ckpt")
                R.fabricate_ckpt(module, self.ckpt, H, seed=0)

    def model(self, name, M, beta=BETA, device="cpu"):
        key = (name, M, device)
        if key in self._models:
            return self._models[key]
        db, weights, _ = synthetic_inputs(M=M, n=1)
        if self.kind == "reference":
            path = os.path.join(self.tmp, f"db_{M}.npz")
            if not os.path.exists(path):
                np.savez(path, **db)
            with contextlib.redirect_stdout(sys.stderr):
                m = self.load_model(name, self.ckpt, device=device, db_path=path, beta=beta)

            def run(coords, m=m):
                with torch.no_grad():
                    return m(torch.tensor(coords).to(device))       # the reference expects the locations on its device
        else:
            from oracle import range_oracle as O
            from range_b200.sh_table import load_entries
            orc = O.RangeOracle(name, weights, load_entries(40), db, beta=beta)
            run = orc
        self._models[key] = run
        return run

    def time(self, name, M, n, steps=1, warmup=1, device="cpu"):
        """(queries/s, seconds per call) of `steps` calls of n queries"""
        from range_b200 import synthetic as S
        run = self.model(name, M, device=device)
        coords = S.area_uniform(n, np.random.default_rng(1))
        for _ in range(warmup):
            run(coords[: max(64, n // 8)])
        ts = []
        for _ in range(steps):
            t = time.perf_counter()
            out = run(coords)
            if device != "cpu":
                torch.cuda.synchronize()
            ts.append(time.perf_counter() - t)
        assert out.shape == (n, 1280)
        return n / float(np.mean(ts)), float(np.mean(ts))


def host_description():
    model = ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"cpu_count": os.cpu_count(), "cpu_model": model}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    ref = ReferenceCpu()
    cores = torch.get_num_threads()
    n = REF_SAMPLE_QUERIES
    qps, sec = ref.time("RANGE+", M_DB, n, steps=max(1, args.steps), warmup=min(1, max(0, args.warmup)))
    sample = f"{n} of {N_QUERIES} queries x full {M_DB}-entry DB per step"
    line = {
        "impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 (f64 encoder)", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample, "host": host_description()},
        "cpu_baseline": {"value": qps, "unit": UNIT, "cores": cores, "kind": ref.kind, "sample": sample},
        "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}
    if args.gpus == 1 and not args.quick:
        # BASELINE.json configs[0] (RANGE, range_db_med shape, 10 000 queries in one call) and the port beside the reference
        extras = {}
        try:
            q1, s1 = ref.time("RANGE", M_MED, 10_000, steps=1, warmup=1)
            extras["config1_RANGE_Mmed_N10000"] = {"value": q1, "unit": UNIT, "seconds": s1, "M": M_MED, "kind": ref.kind,
                                                   "cores": cores}
            if ref.kind == "reference":
                port = ReferenceCpu(want_port=True)
                qp, sp = port.time("RANGE+", M_DB, n, steps=1, warmup=1)
                extras["port_same_sample"] = {"value": qp, "unit": UNIT, "seconds": sp, "kind": "port", "cores": cores}
                if torch.cuda.is_available():
                    # same box, library kernels: the reference with device='cuda' (torch eager, TF32 matmuls,
                    # range/location_models/satclip/main_old.py:13; V re-uploaded every call, range/range.py:217,236)
                    qg, sg = ref.time("RANGE+", M_DB, 10_000, steps=3, warmup=1, device="cuda")
                    extras["torch_eager_cuda"] = {"value": qg, "unit": UNIT, "seconds": sg, "queries_per_call": 10_000,
                                                  "note": "unmodified reference, device='cuda'"}
        except Exception as e:                     # the headline above stands on its own
            extras["error"] = repr(e)
        line["extras"] = extras
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# M-sharded database (BASELINE.json configs[3])
# ------------------------------------------------------------------------------------------------------------------
def time_steps(fn, steps, warmup, barrier):
    for _ in range(warmup):
        fn()
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    barrier()
    return t0.elapsed_time(t1) / steps


def run_m_sharded(world, rank, dev, weights, steps, warmup, barrier, sizes):
    """For every database size: N_QUERIES queries per step IN TOTAL (each rank owns N_QUERIES / world of them), once
    with the database sharded along M over the ranks (collectives + NVLink stores) and once replicated (no collective)."""
    import torch.distributed as dist
    from argparse import Namespace
    from range_b200.database import DeviceDatabase
    from range_b200.range import LocationEncoder
    from range_b200 import synthetic as S
    enc = dict(L=40, dims=[1600, H, H, 256], weights=weights)
    n_rank = N_QUERIES // world
    coords = torch.tensor(S.area_uniform(N_QUERIES, np.random.default_rng(7))[rank * n_rank:(rank + 1) * n_rank], device=dev)
    peak_tf, _, _ = peaks()
    out = []
    for M in sizes:
        k = max(2, min(steps, int(2.0e12 * world / (N_QUERIES * M)) + 1))            # about <= 1 s of steps per variant
        row = {"M": M, "queries_per_step": n_rank * world, "steps": k}
        for variant in ("m_sharded", "replicated"):
            shard = (rank, world) if variant == "m_sharded" else None
            with contextlib.redirect_stdout(sys.stderr):
                ddb = DeviceDatabase.synthetic(M, dev, seed=0, shard=shard)
                ns = Namespace(location_model_name="RANGE+", pretrained_path=enc, device=dev, range_db=ddb, beta=BETA)
                if shard is not None:
                    ns.db_shard, ns.db_group = shard, None
                model = LocationEncoder(ns)
            res = torch.empty(n_rank, 1280, dtype=torch.float32, device=dev)
            ms = time_steps(lambda: model.embed(coords, out=res), k, min(warmup, 2), barrier)
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
            pairs = n_rank * world * M / (ms * 1e-3)
            row[variant] = {"ms_per_step": ms, "pairs_per_s": pairs, "queries_per_s": n_rank * world / (ms * 1e-3),
                            "frac_of_tensor_roofline": FLOP_PER_PAIR * pairs / 1e12 / (world * peak_tf)}
            if shard is not None:
                row[variant].update(merge=model.sharded.merge, collectives_per_step=4 if model.sharded.merge == "peer" else 4,
                                    nccl_bytes_per_query=512 + 16 + 8,
                                    nvlink_store_bytes_per_query=4096.0 * (world - 1) / world
                                    if model.sharded.merge == "peer" else 0.0)
                model.sharded.close()
            del model, ddb, res
            torch.cuda.empty_cache()
        row["sharded_vs_replicated"] = row["m_sharded"]["pairs_per_s"] / row["replicated"]["pairs_per_s"]
        out.append(row)
    return out


# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="range_b200", choices=["range_b200", "reference"])
    ap.add_argument("--shard", default="query", choices=["query", "m"], help="m: only the M-sharded section (N > 1)")
    ap.add_argument("--m-sizes", default="", help="comma-separated database sizes of the M-sharded section")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="skip the extras (reference arm: config 1 / port / eager CUDA)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.shard == "m"):
        ap.error("--dump-outputs writes the outputs of the headline path (--impl range_b200 --shard query)")
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    from argparse import Namespace
    from range_b200 import _lib
    from range_b200.range import LocationEncoder

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    warmup = max(3, args.warmup)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    db, weights, coords = synthetic_inputs(rank)
    sizes = [int(x) for x in args.m_sizes.split(",") if x] or ([100_000, 1_000_000] + ([10_000_000] if world >= 8 else []))
    if args.shard == "m":
        if world < 2:
            raise SystemExit("--shard m needs torchrun with at least 2 ranks")
        rows = run_m_sharded(world, rank, dev, weights, args.steps, warmup, barrier, sizes)
        if rank == 0:
            print(json.dumps({"metric": "RANGE+ (query, entry) pairs/sec, database sharded along M", "unit": "pairs/s",
                              "value": rows[-1]["m_sharded"]["pairs_per_s"], "n_gpus": world, "m_sharded": rows,
                              "higher_is_better": True, "data": "synthetic"}))
        dist.destroy_process_group()
        return

    enc = dict(L=40, dims=[1600, H, H, 256], weights=weights)
    with contextlib.redirect_stdout(sys.stderr):      # the reference prints its temperatures; stdout is for the JSON line
        model = LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=enc, device=dev, range_db=db,
                                          beta=BETA))
    eng = model.engine
    d_coords = torch.tensor(coords, device=dev)
    h_coords = torch.tensor(coords).pin_memory()
    out = torch.empty(N_QUERIES, 1280, dtype=torch.float32, device=dev)
    q64 = torch.empty(N_QUERIES, 256, dtype=torch.float64, device=dev)
    q16 = torch.empty(N_QUERIES, 256, dtype=torch.float16, device=dev)
    qxyz = torch.empty(N_QUERIES, 4, dtype=torch.float32, device=dev)

    marks = []

    def step(record=False):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)] if record else None
        if record: ev[5].record()
        s_coords, perm = eng.sort_queries(d_coords)        # spatial batching (geo-term tile skipping)
        if record: ev[0].record()
        eng.encode(s_coords, q64, q16, qxyz)
        if record: ev[1].record()
        sums, maxs = eng.retrieve_stats("RANGE+", q16, qxyz, 12.0, 40.0)
        if record: ev[2].record()
        # apply pass: its epilogue writes the (N,1280) result (rows back in the caller's order); then the location columns
        eng.retrieve_apply_concat("RANGE+", q16, qxyz, 12.0, 40.0, BETA, sums, maxs, q64, out=out, perm=perm)
        if record:
            ev[3].record()
            marks.append(ev)

    with ClockSampler(local) as clocks:       # nvidia-smi needs ~1 s to start: launched before the warm-up
        for _ in range(warmup):
            step()
        barrier()
        launches0 = _lib.launch_count()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks.mark_start()
        t0.record()
        for _ in range(args.steps):
            step(record=True)
        t1.record()
        barrier()
        clocks.mark_end()
    launches = _lib.launch_count() - launches0
    ms = t0.elapsed_time(t1)
    dump = {}
    if args.dump_outputs and rank == 0:
        rows = dump_rows()
        dump["embeddings"] = out[torch.from_numpy(rows).to(dev)].cpu().numpy()
    seg = np.array([[e[i].elapsed_time(e[i + 1]) for i in range(3)] + [0.0, e[5].elapsed_time(e[0])]
                    for e in marks]).mean(0)                                   # enc, stats, apply+concat, -, sort

    # e2e through the public API: pinned host coords -> numpy float64 (N,1280)
    for _ in range(3):
        res = model(h_coords)          # held across iterations like the timed loop (two pinned result buffers)
    barrier()
    e2e_steps = []
    w0 = time.perf_counter()
    for _ in range(args.steps):
        w1 = time.perf_counter()
        res = model(h_coords)
        e2e_steps.append((time.perf_counter() - w1) * 1e3)
    barrier()
    e2e_s = (time.perf_counter() - w0)
    assert res.shape == (N_QUERIES, 1280) and res.dtype == np.float64
    if dump:
        dump["model_embeddings"] = res[rows]
    host_path = model.host_path if model.host_path != "auto" else "copy"
    del res
    # opt-in (NOT the reference's dtype, not the headline): float32 rows halve the device->host bytes
    model.out_dtype = np.dtype(np.float32)
    k32 = max(2, min(args.steps, 5))
    for _ in range(2):
        res = model(h_coords)
    barrier()
    w0 = time.perf_counter()
    for _ in range(k32):
        res = model(h_coords)
    barrier()
    e2e32_s = (time.perf_counter() - w0) / k32
    assert res.dtype == np.float32
    model.out_dtype = np.dtype(np.float64)
    del res

    t = torch.tensor([ms, e2e_s * 1e3, e2e32_s * 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms, e2e32_ms = float(t[0]), float(t[1]), float(t[2])

    sharded = None
    if world > 1:
        del model, eng, out, q64, q16, qxyz
        torch.cuda.empty_cache()
        sharded = run_m_sharded(world, rank, dev, weights, args.steps, warmup, barrier, sizes)

    if rank == 0:
        peak_tf, _, peak_src = peaks()
        t_k2 = (seg[1] + seg[2]) * 1e-3
        achieved_k2 = FLOP_PER_PAIR * N_QUERIES * M_DB / t_k2 / 1e12            # stats + apply
        achieved = FLOP_PER_PAIR * N_QUERIES * M_DB / (seg[2] * 1e-3) / 1e12    # dominant kernel alone
        traffic, traffic_src = apply_kernel_traffic()
        line = {
            "metric": METRIC, "value": world * N_QUERIES * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16 operands / f32 accumulate (retrieval); f64 SH + split-fp16 (f16x3) SIREN (encoder)",
            "data": "synthetic",
            "config": {"workload": f"{WORKLOAD}, {N_QUERIES} queries/GPU", "parallelism": f"query-sharded x{world}, DB replicated"
                       + ("; m_sharded: DB sharded along M" if world > 1 else ""),
                       "l2": "inputs larger than L2 (DB 257 MB fp16 streamed every step; 512 MB output)",
                       "segments_ms": {"sort_queries": seg[4], "encode": seg[0], "retrieve_stats": seg[1], "retrieve_apply_concat": seg[2]},
                       "parity_tolerance": "retrieved columns: relative row error <= 1e-3, 2e-4 on the structured DB (named exception: purely "
                                           "semantic softmax on the iid worst-case DB 2e-3), cosine >= 0.99999; location columns: "
                                           "max-abs <= 3e-5 (|lat| < 60 deg) / 1e-3 (polar) = the reference's own fp64 polynomial "
                                           "noise (tests/test_gpu_parity.py)"},
            # dominant kernel = the apply pass (all 2566 algorithmic flop per pair live there); the stats pass that
            # precedes it is algorithmically redundant work, so the stricter figure over both kernels is given too
            "roofline": {"bound": "tensor", "kernel": "range_apply_pc_kernel (K2b: Q.K^T + softmax blend + P.V)",
                         "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                         "peak_source": f"{peak_src} bf16 dense sustained",
                         "traffic": traffic,
                         "traffic_source": f"ncu --set full, {traffic_src} (dram read + write of the apply kernel)",
                         "algorithmic_flop_per_launch": FLOP_PER_PAIR * N_QUERIES * M_DB,
                         "launch_ms": seg[2],
                         "stats_plus_apply": {"achieved": achieved_k2, "frac": achieved_k2 / peak_tf,
                                              "launch_ms": seg[1] + seg[2]}},
            "e2e": {"value": world * N_QUERIES * args.steps / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": N_QUERIES * 16, "d2h_bytes_per_step": N_QUERIES * 1280 * 8,
                    "host_path": host_path, "ms_per_call_rank0": [round(x, 2) for x in e2e_steps],
                    "float32_opt_in": {"value": world * N_QUERIES / (e2e32_ms * 1e-3), "unit": UNIT,
                                       "d2h_bytes_per_step": N_QUERIES * 1280 * 4,
                                       "note": "load_model(..., out_dtype=np.float32): not the reference's dtype"},
                    "api": "range_b200.load_model(...)(locs) -> numpy float64 (N,1280)"},
            "gpu_launches": int(launches), "clocks": clocks.summary()}
        if sharded is not None:
            line["m_sharded"] = sharded
        if world == 1:
            # BASELINE.json configs[0] on this implementation: RANGE, range_db_med shape, 10 000 queries in one model(locs) call
            with contextlib.redirect_stdout(sys.stderr):
                db1, _, c1 = synthetic_inputs(M=M_MED, n=10_000)
                m1 = LocationEncoder(Namespace(location_model_name="RANGE", pretrained_path=enc, device=dev, range_db=db1))
            h1 = torch.tensor(c1).pin_memory()
            for _ in range(4):
                r1 = m1(h1)          # bound like the timed calls: two page-locked results alive at once, both allocated here
            torch.cuda.synchronize()
            calls1 = []
            for _ in range(10):
                w1 = time.perf_counter()
                r1 = m1(h1)
                calls1.append(time.perf_counter() - w1)
            t1 = sum(calls1) / len(calls1)
            assert r1.shape == (10_000, 1280) and r1.dtype == np.float64
            line["config1_RANGE_Mmed_N10000"] = {"value": 10_000 / t1, "unit": UNIT, "ms_per_call": t1 * 1e3,
                                                 "ms_per_call_min": min(calls1) * 1e3, "M": M_MED,
                                                 "api": "model(locs): pinned host in, numpy float64 out"}
            del m1, r1
        if world == 1 and not args.no_cpu_baseline:
            torch.set_num_threads(os.cpu_count() or 1)
            ref = ReferenceCpu()
            n = REF_SAMPLE_QUERIES
            qps, sec = ref.time("RANGE+", M_DB, n, steps=2, warmup=1)
            line["cpu_baseline"] = {"value": qps, "unit": UNIT, "cores": torch.get_num_threads(), "kind": ref.kind,
                                    "sample": f"{n} of {N_QUERIES} queries x full {M_DB}-entry DB, 2 calls ({sec:.1f} s each)"}
        if dump:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dump.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
