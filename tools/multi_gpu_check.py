"""Run under torchrun on N >= 2 GPUs: the M-sharded database path (range_b200/distributed.py) against the unsharded one.
Every rank owns its own queries (ragged counts, one rank's set clustered in a small region, several steps), the database
is sharded along M; both merges are checked: 'peer' (the apply kernel's epilogue stores partial rows into the owners'
receive buffers over NVLink) and 'reduce_scatter' (NCCL).  Also: query sharding + all_gather == one GPU, and the
M-sharded neighbours(coords, 8) (shard lists exchanged with all_to_all, merged on the owner) against the unsharded one,
the M-sharded embed_sweep (beta 0 .. 1 in 5 steps) against the unsharded sweep, and the M-sharded embed_raster /
forward_raster of every rank's slab of a small raster against the sharded embed of the same points and the unsharded raster.
Environment: M, N (database entries, queries per rank), D (width of the database's values, default 1024; a multiple of 4
on a sharded database), STEP_ROWS.
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/multi_gpu_check.py
"""
import contextlib, os, sys, time
import numpy as np, torch, torch.distributed as dist
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
from argparse import Namespace
from range_b200 import synthetic as S          # seeded input generators
from range_b200.range import LocationEncoder
from range_b200.distributed import shard_rows

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
dev = torch.device("cuda", local)
M, N = int(os.environ.get("M", 200_000)), int(os.environ.get("N", 20_000))
D = int(os.environ.get("D", 1024))
WIDTH = "" if D == 1024 else f", D={D}"                              # named in the printed lines only when not 1024
rng = np.random.default_rng(0)
db = dict(locs=S.area_uniform(M, rng), satclip_embeddings=rng.standard_normal((M, 256), dtype=np.float32),
          image_embeddings=rng.standard_normal((M, D), dtype=np.float32) + 0.5)
enc = dict(L=40, dims=[1600, 512, 512, 256], weights=S.siren_init(40, 512, 2, 256, seed=0))
n_mine = N + 1500 * rank                                            # ragged: the last step of the other ranks is padded
r2 = np.random.default_rng(100 + rank)
mine = S.area_uniform(n_mine, r2)
if rank == world - 1:                                               # a regional query set: thousands of queries per cell
    mine[: n_mine // 2] = np.stack([r2.uniform(10, 12, n_mine // 2), r2.uniform(45, 47, n_mine // 2)], 1)
coords = torch.tensor(mine, device=dev)


def rel(a, b):
    return ((a - b).norm(dim=1) / b.norm(dim=1)).max().item()


def model(**kw):
    with contextlib.redirect_stdout(sys.stderr):
        return LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=enc, device=dev, range_db=db, beta=0.5, **kw))


def timed(fn, reps=3):
    fn(); torch.cuda.synchronize(); dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize(); dist.barrier()
    return (time.perf_counter() - t0) / reps


full = model()
ref = full.embed(coords)                                            # unsharded database, my queries
t_full = timed(lambda: full.embed(coords))
K_NB, TOL = 8, 2e-3
nb_ref = full.neighbours(coords, K_NB)
BETAS = (0.0, 0.25, 0.5, 0.75, 1.0)
sw_ref = full.embed_sweep(coords, BETAS)
RH, RW = 90, 180                                                    # a small raster, every rank its own slab of points
lon_ax, lat_ax = LocationEncoder.coord_grid_axes((RH, RW))
p0, p1 = shard_rows(RH * RW, rank, world)
pts_idx = torch.arange(p0, p1)
raster_pts = torch.stack((lon_ax[pts_idx % RW], lat_ax[pts_idx // RW]), 1).to(dev)
raster_ref = full.embed_raster(lon_ax, lat_ax, rows=(p0, p1))
report, nb_report, nb_out, sw_report, ra_report = {}, {}, {}, {}, {}


def max_all(x):
    x = torch.tensor([float(x)], device=dev)
    dist.all_reduce(x, op=dist.ReduceOp.MAX)
    return float(x[0])


def neighbours_vs_full(got):
    """weights within TOL of the unsharded call position by position; entries only one list holds have weights within
    TOL of the unsharded k-th weight (near-ties at the cut): (max rel weight diff, entries that differ, worst tie gap)"""
    (r_sh, w_sh), (r_un, w_un) = got, nb_ref
    e_w = ((w_sh.double() - w_un.double()).abs() / w_un.double()).max().item() if w_un.numel() else 0.0
    only = ~(r_sh.unsqueeze(2) == r_un.unsqueeze(1)).any(2)
    kth = w_un[:, -1:].double().expand_as(w_un)
    gap = ((w_sh.double() - kth).abs() / kth)[only].max().item() if only.any() else 0.0
    return e_w, int(only.sum()), gap
for merge in ("peer", "reduce_scatter"):
    sh = model(db_shard=(rank, world), db_group=None, db_merge=merge)
    sh.sharded.MAX_STEP_ROWS = int(os.environ.get("STEP_ROWS", 16_384 * world))     # several steps per call
    out = sh.embed(coords)
    err = torch.tensor([rel(out[:, :D], ref[:, :D]), (out[:, D:] - ref[:, D:]).abs().max().item()], device=dev)
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    again = sh.embed(coords)
    same = torch.tensor([float(torch.equal(out, again))], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    t = timed(lambda: sh.embed(coords))
    host = sh(coords.cpu()) if merge == "peer" else None            # the public call, collective
    if host is not None:
        assert host.shape == (n_mine, D + 256) and np.allclose(host[:, :D], out[:, :D].cpu().numpy(), rtol=1e-6, atol=1e-7)
    report[merge] = (sh.sharded.merge, float(err[0]), float(err[1]), bool(same[0] > 0), t)
    nb = sh.neighbours(coords, K_NB)                                 # collective: every rank, the same k
    nb_again = sh.neighbours(coords, K_NB)
    nb_same = max_all(not (torch.equal(nb[0], nb_again[0]) and torch.equal(nb[1], nb_again[1]))) == 0
    e_w, n_diff, gap = neighbours_vs_full(nb)
    t_nb = timed(lambda: sh.neighbours(coords, K_NB))
    sh.sharded.trace = []                                            # CUDA events around the list exchange + owner merge
    sh.neighbours(coords, K_NB)
    torch.cuda.synchronize()
    t_x = sum(a.elapsed_time(b) for a, b in sh.sharded.trace) / 1e3
    sh.sharded.trace = None
    nb_out[merge] = nb
    nb_report[merge] = (max_all(e_w), int(max_all(n_diff)), max_all(gap), nb_same, max_all(t_nb), max_all(t_x), t)
    sw = sh.embed_sweep(coords, BETAS)                               # collective: two routed apply passes per step
    sw_again = sh.embed_sweep(coords, BETAS)
    e_sw = max(rel(a[:, :D], b[:, :D]) for a, b in zip(sw, sw_ref))
    q_sw = max((a[:, D:] - b[:, D:]).abs().max().item() for a, b in zip(sw, sw_ref))
    sw_same = max_all(not all(torch.equal(a, b) for a, b in zip(sw, sw_again))) == 0
    t_sw = timed(lambda: sh.embed_sweep(coords, BETAS))
    sw_report[merge] = (max_all(e_sw), max_all(q_sw), sw_same, max_all(t_sw), t)
    ra = sh.embed_raster(lon_ax, lat_ax, rows=(p0, p1))             # collective: every rank its own points
    ra_eq = torch.equal(ra, sh.embed(raster_pts))
    e_ra = rel(ra[:, :D], raster_ref[:, :D])
    q_ra = (ra[:, D:] - raster_ref[:, D:]).abs().max().item()
    host = np.empty((p1 - p0, D + 256))
    sh.forward_raster(lon_ax, lat_ax, rows=(p0, p1), out=host)
    host_eq = np.array_equal(host, sh.embed_raster(lon_ax, lat_ax, rows=(p0, p1), out_dtype=torch.float64).cpu().numpy())
    t_ra = timed(lambda: sh.embed_raster(lon_ax, lat_ax, rows=(p0, p1)))
    ra_report[merge] = (max_all(e_ra), max_all(q_ra), max_all(not ra_eq) == 0, max_all(not host_eq) == 0, max_all(t_ra))
    sh.sharded.close()
    del sh
lo, hi = shard_rows(N, rank, world)                                # query sharding: my slab of a common set, then gather
common = torch.tensor(S.area_uniform(N, np.random.default_rng(1)), device=dev)
part = full.embed(common[lo:hi].contiguous())
parts = [torch.empty(shard_rows(N, r, world)[1] - shard_rows(N, r, world)[0], D + 256, device=dev) for r in range(world)]
dist.all_gather(parts, part)
e2 = rel(torch.cat(parts)[:, :D], full.embed(common)[:, :D])
if rank == 0:
    for merge, (used, e_o, e_q, same, t) in report.items():
        print(f"world {world}: M-sharded [{merge} -> ran {used}] vs unsharded: max rel-row err {e_o:.2e}, location columns {e_q:.1e}, "
              f"repeatable {same}; {t*1e3:.1f} ms per call vs {t_full*1e3:.1f} ms with the database replicated "
              f"(N={N}+1500 r per rank, M={M}{WIDTH})")
        assert e_o < 1e-3 and e_q == 0.0 and same
    print(f"query-sharded + all_gather vs one GPU {e2:.2e}")
    assert e2 < 1e-3
across = max_all(not all(torch.equal(a, b) for a, b in zip(nb_out["peer"], nb_out["reduce_scatter"]))) == 0
if rank == 0:
    for merge, (e_w, n_diff, gap, same, t_nb, t_x, t) in nb_report.items():
        print(f"M-sharded neighbours k={K_NB} [{merge}] vs unsharded: max rel weight diff {e_w:.2e}, {n_diff} entries differ "
              f"(weights within {gap:.1e} of the k-th), repeatable {same}, same under both merges {across}; "
              f"{t_nb*1e3:.1f} ms per call (list exchange + owner merge {t_x*1e3:.2f} ms, {100 * t_x / t_nb:.1f} %) "
              f"vs {t*1e3:.1f} ms for the sharded embed (world {world}, N={N}+1500 r per rank, M={M}{WIDTH})")
        assert e_w < TOL and gap < TOL and same and across
    for merge, (e_o, e_q, same, t_sw, t) in sw_report.items():
        print(f"M-sharded sweep beta={BETAS} [{merge}] vs unsharded sweep: max rel-row err {e_o:.2e}, location columns "
              f"{e_q:.1e}, repeatable {same}; {t_sw*1e3:.1f} ms per call vs {len(BETAS)} x {t*1e3:.1f} = "
              f"{len(BETAS)*t*1e3:.1f} ms for {len(BETAS)} sharded embed calls (world {world}, N={N}+1500 r per rank, M={M}{WIDTH})")
        assert e_o < 1e-3 and e_q == 0.0 and same
    for merge, (e_o, e_q, eq, host_eq, t_ra) in ra_report.items():
        print(f"M-sharded raster {RH}x{RW} [{merge}], a slab of points per rank: equal to the sharded embed of the same "
              f"coordinates {eq}, vs unsharded embed_raster max rel-row err {e_o:.2e} (location columns {e_q:.1e}), "
              f"forward_raster(out=) equal to the float64 rows {host_eq}; {t_ra*1e3:.1f} ms per call (world {world}, M={M}{WIDTH})")
        assert eq and host_eq and e_o < 1e-3 and e_q < 1e-3
dist.destroy_process_group()
