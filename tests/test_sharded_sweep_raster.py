"""Beta sweeps and rasters on a database sharded along M: ShardedRetriever.embed_sweep (two routed apply passes per step,
range_sweep_concat over the 2 P slots of the receive buffer) and the collective LocationEncoder.embed_raster /
forward_raster (the sharded embed of the raster points' coordinates).

CPU: the host pipeline on gloo (world size 2) through a torch stand-in engine in fp64, against the unsharded linear blend
(1 - beta) P_g V + beta P_s V; the façade's raster calls around the same stand-in.  GPU: range_sweep_concat against fp64
and against range_combine_concat; P = 3 shards emulated one after the other on one device against the unsharded
embed_sweep and the exact oracle; a world of one rank over NCCL through the real peer path.  2 GPUs:
tools/multi_gpu_check.py under torchrun.
"""
import ctypes
import os
import subprocess
import sys
from argparse import Namespace
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import range_oracle as O
from tests.test_distributed import TorchEngine, _database, _encode

DEV = "cuda:0"
TS, TG, D = 12.0, 40.0, 1024


# ---------------------------------------------------------------------------------------------------- CPU: stand-in
class SweepEngine(TorchEngine):
    """TorchEngine with the semantic end of a sweep (mode 'RANGE' with RANGE+'s sums), weighted parts and sweep_concat,
    in fp64; no separable raster encoder"""

    def __init__(self, K, V, X):
        super().__init__(K, V, X)
        self.db = SimpleNamespace(caps=True)             # a spatially sorted database: the façade sorts RANGE+ queries

    def raster_supported(self):
        return False

    def retrieve_apply(self, mode, q16, qxyz, temp, geo_temp, beta, sums, maxs):
        s, g = self._logits(q16, qxyz)
        P = torch.exp(temp * (s - 1)) / sums[:, :1]
        if mode == "RANGE+":
            P = beta * P + (1 - beta) * torch.exp(geo_temp * (g - 1)) / sums[:, 1:]
        return (P @ self.V).contiguous()

    @staticmethod
    def _store(rows, out, perm):
        if perm is None:
            out.copy_(rows)
        else:
            out[perm.long()] = rows.to(out.dtype)

    def combine_concat(self, parts, weights, q64, out=None, dtype=torch.float64, perm=None):
        w = [1.0] * len(parts) if weights is None else weights
        out = torch.empty(q64.shape[0], 1280, dtype=dtype) if out is None else out
        self._store(torch.cat([sum(wk * p for wk, p in zip(w, parts)), q64], 1), out, perm)
        return out

    def sweep_concat(self, geo_parts, sem_parts, betas, q64, out_dtype=torch.float32, perm=None, outs=None):
        G, S = sum(geo_parts), sum(sem_parts)
        outs = [torch.empty(q64.shape[0], 1280, dtype=out_dtype) for _ in betas] if outs is None else outs
        for b, o in zip(betas, outs):
            self._store(torch.cat([(1 - b) * G + b * S, q64], 1), o, perm)
        return outs


def _blend(coords, K, V, X, beta):
    """(1 - beta) P_g V + beta P_s V over the whole database, fp64"""
    q, xyz = _encode(coords)
    s, g = q.half().double() @ K.t(), xyz.float().double() @ X.t()
    return (1 - beta) * torch.softmax(TG * g, 1) @ V + beta * torch.softmax(TS * s, 1) @ V, q


def _coords(n, seed):
    rng = np.random.default_rng(seed)
    return torch.tensor(np.stack([rng.uniform(-180, 180, n), rng.uniform(-90, 90, n)], 1))


def _spawn(fn, base):
    world = 2
    port = base + os.getpid() % 2000
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(fn, args=(world, port, ret), nprocs=world, join=True)
    assert [ret[r] for r in range(world)] == [[], []]


def _init(rank, world, port):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)


def _sweep_worker(rank, world, port, ret):
    _init(rank, world, port)
    from range_b200.distributed import ShardedRetriever, shard_rows
    fails = []
    M = 1001
    K, V, X = _database(M)
    lo, hi = shard_rows(M, rank, world)
    sr = ShardedRetriever(SweepEngine(K[lo:hi], V[lo:hi], X[lo:hi]), merge="reduce_scatter")
    sr.MAX_STEP_ROWS = 256 * world                      # sweep slab 128: rank 0 takes 3 steps, rank 1 one and pads
    n = [300, 77][rank]
    coords = _coords(n, 30 + rank)
    betas = [0.0, 0.3, 1.0]
    for sort in (False, True):
        before = sr.collectives
        got = sr.embed_sweep(coords, TS, TG, sort, betas, out_dtype=torch.float64)
        if sr.collectives - before != 1 + 5 * 3:                              # n, then 3 steps of 5 collectives
            fails.append(("collectives", sort, sr.collectives - before))
        if len(got) != len(betas):
            fails.append(("count", sort, len(got)))
        for beta, o in zip(betas, got):
            ref, q = _blend(coords, K, V, X, beta)
            if o.shape != (n, 1280) or o.dtype != torch.float64:
                fails.append(("shape", sort, beta, tuple(o.shape), o.dtype))
            elif not (torch.allclose(o[:, :D], ref, rtol=1e-9, atol=1e-11) and torch.equal(o[:, D:], q)):
                fails.append(("rows", sort, beta, float((o[:, :D] - ref).abs().max())))
    # the ranks pass different beta lists; one of them an empty list: every rank still takes every step
    mine = [[0.3, 1.0, 0.0], []][rank]
    before = sr.collectives
    got = sr.embed_sweep(coords, TS, TG, True, mine)
    if sr.collectives - before != 1 + 5 * 3:
        fails.append(("collectives, own betas", sr.collectives - before))
    if len(got) != len(mine):
        fails.append(("own betas", len(got)))
    for beta, o in zip(mine, got):
        ref, q = _blend(coords, K, V, X, beta)
        if not (o.dtype == torch.float32 and torch.allclose(o[:, :D].double(), ref, rtol=1e-5, atol=1e-6)):
            fails.append(("own betas rows", beta))
    empty = sr.embed_sweep(coords[:0], TS, TG, True, [0.5, 1.0])               # every rank: no rows
    if [tuple(e.shape) for e in empty] != [(0, 1280), (0, 1280)]:
        fails.append(("empty", [tuple(e.shape) for e in empty]))
    assert sr.buffers is None
    ret[rank] = fails
    dist.destroy_process_group()


def test_sharded_sweep_pipeline_gloo():
    _spawn(_sweep_worker, 33500)


def _facade(rank, world, engine):
    from range_b200.distributed import ShardedRetriever
    from range_b200.range import LocationEncoder
    m = LocationEncoder.__new__(LocationEncoder)
    torch.nn.Module.__init__(m)
    m.args = Namespace(temp=TS, geo_temp=TG, beta=0.3)
    m.location_model_name = "RANGE+"
    m.engine = engine
    m.sharded = ShardedRetriever(engine, merge="reduce_scatter")
    m.out_dtype, m.host_path, m.pinned_limit = np.dtype(np.float64), "auto", 0
    return m


def _raster_worker(rank, world, port, ret):
    _init(rank, world, port)
    from range_b200.distributed import shard_rows
    from range_b200.range import LocationEncoder
    fails = []
    M = 700
    K, V, X = _database(M)
    lo, hi = shard_rows(M, rank, world)
    m = _facade(rank, world, SweepEngine(K[lo:hi], V[lo:hi], X[lo:hi]))
    m.sharded.MAX_STEP_ROWS = 256 * world                # several steps
    H, W = 13, 29
    lon, lat = LocationEncoder.coord_grid_axes((H, W))
    p0, p1 = [(5, 300), (300, 377)][rank]               # different rows on every rank
    got = m.embed_raster(lon, lat, rows=(p0, p1), out_dtype=torch.float64)
    p = torch.arange(p0, p1)
    pts = torch.stack((lon[p % W], lat[p // W]), 1)
    same = m.sharded.embed("RANGE+", pts, TS, TG, 0.3, True, out_dtype=torch.float64)
    if not (got.shape == (p1 - p0, 1280) and torch.equal(got, same)):
        fails.append("embed_raster != sharded embed of the same coordinates")
    ref, q = _blend(pts, K, V, X, 0.3)
    if not (torch.allclose(got[:, :D], ref, rtol=1e-9, atol=1e-11) and torch.equal(got[:, D:], q)):
        fails.append("embed_raster rows")
    host = m.forward_raster(lon, lat, rows=(p0, p1))
    out = np.full((p1 - p0, 1280), np.nan)
    back = m.forward_raster(lon, lat, rows=(p0, p1), out=out)
    if not (back is out and np.array_equal(out, host) and np.array_equal(host, got.numpy())):
        fails.append("forward_raster with and without out=")
    # a rank with no points still takes part
    none = m.embed_raster(lon, lat, rows=(0, 0) if rank else (0, 50), out_dtype=torch.float64)
    if none.shape != ((0, 1280) if rank else (50, 1280)):
        fails.append(("no points", tuple(none.shape)))
    sweep = m.embed_sweep(pts, [0.0, 1.0], out_dtype=torch.float64)           # the façade's sweep is collective too
    for beta, o in zip([0.0, 1.0], sweep):
        if not torch.allclose(o[:, :D], _blend(pts, K, V, X, beta)[0], rtol=1e-9, atol=1e-11):
            fails.append(("façade sweep", beta))
    ret[rank] = fails
    dist.destroy_process_group()


def test_sharded_raster_facade_gloo():
    _spawn(_raster_worker, 35500)


def test_sweep_of_range_model_raises():
    from range_b200.range import LocationEncoder
    m = LocationEncoder.__new__(LocationEncoder)
    torch.nn.Module.__init__(m)
    m.location_model_name = "RANGE"
    with pytest.raises(NotImplementedError, match="RANGE\\+"):
        m.embed_sweep(torch.zeros(3, 2, dtype=torch.float64), [0.5])


def test_sweep_concat_symbol_in_prototypes():
    from range_b200 import _lib
    assert "range_sweep_concat" in _lib.PROTOTYPES and _lib.RANGE_SWEEP_MAX_BETAS == 8


# ---------------------------------------------------------------------------------------------------- GPU: the kernel
def _slots(n, N, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return [torch.randn(N, 1024, generator=g, device=DEV) for _ in range(n)]


@pytest.fixture(scope="module")
def bare():
    from range_b200.engine import RangeEngine
    return RangeEngine(DEV, L=40)


@pytest.mark.gpu
@pytest.mark.parametrize("n_slots", [1, 3, 8])
@pytest.mark.parametrize("n_betas", [1, 8])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("with_perm", [False, True])
def test_sweep_concat_vs_fp64(bare, n_slots, n_betas, dtype, with_perm):
    N = 777
    geo, sem = _slots(n_slots, N, 1 + n_slots), _slots(n_slots, N, 100 + n_slots)
    q64 = torch.randn(N, 256, dtype=torch.float64, device=DEV)
    perm = torch.randperm(N, device=DEV).to(torch.int32) if with_perm else None
    betas = list(np.linspace(0, 1, n_betas)) if n_betas > 1 else [0.3]
    outs = bare.sweep_concat(geo, sem, betas, q64, out_dtype=dtype, perm=perm)
    G, S = sum(p.double() for p in geo), sum(p.double() for p in sem)
    for b, o in zip(betas, outs):
        assert o.dtype == dtype and o.shape == (N, 1280)
        ref = torch.cat([(1 - b) * G + b * S, q64], 1)
        got = o.double() if perm is None else o.double()[perm.long()]
        rel = (got[:, :1024] - ref[:, :1024]).norm(dim=1) / ref[:, :1024].norm(dim=1)
        assert rel.max().item() <= 1e-6, (b, rel.max().item())
        assert torch.equal(got[:, 1024:], q64.to(dtype).double())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_sweep_concat_one_slot_is_combine_concat(bare, dtype):
    """n_slots = 1: bit for bit the blend the unsharded embed_sweep runs (combine_concat of (G, S) with (1 - beta, beta)),
    also past RANGE_SWEEP_MAX_BETAS beta (two launches)"""
    N = 1000
    (G,), (S,) = _slots(1, N, 7), _slots(1, N, 8)
    q64 = torch.randn(N, 256, dtype=torch.float64, device=DEV)
    perm = torch.randperm(N, device=DEV).to(torch.int32)
    betas = [0.0, 0.1, 0.25, 1 / 3, 0.5, 0.6, 0.75, 0.9, 0.99, 1.0, 0.7]
    for p in (None, perm):
        outs = bare.sweep_concat([G], [S], betas, q64, out_dtype=dtype, perm=p)
        for b, o in zip(betas, outs):
            ref = bare.combine_concat([G, S], [1.0 - b, b], q64, dtype=dtype, perm=p)
            assert torch.equal(o, ref), b


@pytest.mark.gpu
def test_sweep_concat_argument_errors(bare):
    from range_b200 import _lib
    N = 256
    slots = _slots(9, N, 3)
    q64 = torch.zeros(N, 256, dtype=torch.float64, device=DEV)
    outs = [torch.empty(N, 1280, device=DEV) for _ in range(9)]
    packed = torch.empty(N, 6144, dtype=torch.uint8, device=DEV)
    lib = bare.lib

    def call(n_slots, n_betas, dtype=_lib.RANGE_OUT_F32, null_slot=False, out_ptrs=None):
        ptrs = [s.data_ptr() for s in slots[:max(n_slots, 1)]]
        if null_slot:
            ptrs[-1] = 0
        P = (ctypes.c_void_p * len(ptrs))(*ptrs)
        nb = max(n_betas, 1)
        Wt = (ctypes.c_float * nb)(*([0.5] * nb))
        Op = (ctypes.c_void_p * nb)(*(out_ptrs or [o.data_ptr() for o in outs[:nb]]))
        return lib.range_sweep_concat(bare.ctx, N, n_slots, P, P, n_betas, Wt, Wt, ctypes.c_void_p(q64.data_ptr()), None,
                                      Op, dtype, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))

    assert call(2, 2) == 0
    torch.cuda.synchronize()
    invalid = -1                                                     # RANGE_ERR_INVALID
    for args in ((0, 1), (9, 1), (1, 0), (1, 9)):
        assert call(*args) == invalid, args
    assert call(2, 1, dtype=_lib.RANGE_OUT_PACKED, out_ptrs=[packed.data_ptr()]) == invalid
    assert call(3, 1, dtype=7) == invalid
    assert call(3, 1, null_slot=True) == invalid
    with pytest.raises(_lib.RangeError):                             # through the engine: a null slot address
        bare.sweep_concat([slots[0].data_ptr(), 0], slots[:2], [0.5], q64)
    with pytest.raises(_lib.RangeError):                             # packed rows
        bare.sweep_concat(slots[:1], slots[:1], [0.5], q64, outs=[packed])
    with pytest.raises(ValueError):
        bare.sweep_concat(slots[:2], slots[:1], [0.5], q64)


# ---------------------------------------------------------------------------------------------------- GPU: P emulated
@pytest.mark.gpu
@pytest.mark.parametrize("slab", [256, 4224])
def test_m_sharded_sweep_emulated(slab, sh_entries):
    """ShardedRetriever.embed_sweep's step with its P = 3 ranks emulated one after the other on one GPU: both routed ends
    (geographic: RANGE+ at beta 0; semantic: RANGE at temp with RANGE+'s sums) stored through PeerBuffers.route into the
    two halves of NaN-filled receive buffers, then every owner's range_sweep_concat over its 2 P slots (PeerBuffers.slots).
    slab 256: single-role kernels + row router; slab 4224: the producer/consumer epilogue routes the rows itself."""
    from range_b200.database import DeviceDatabase
    from range_b200.distributed import PeerBuffers
    from range_b200.engine import RangeEngine
    from range_b200.range import LocationEncoder
    from tests.test_gpu_parity import rel_rows, tol_o
    P, M, temp, geo_temp = 3, 5000, 12.0, 40.0
    betas = [0.0, 0.25, 0.5, 0.75, 1.0]
    ws = O.siren_init(40, 64, 2, 256, seed=2)
    helper = O.RangeOracle.__new__(O.RangeOracle)
    helper.L, helper.entries, helper.weights = 40, sh_entries, ws
    db = O.synthetic_db(M, seed=4, kind="structured", encoder=helper.encode)
    enc = dict(L=40, dims=[1600, 64, 64, 256], weights=ws)
    whole = LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=enc, device=DEV, range_db=db, beta=0.5))
    shards = [RangeEngine(DEV, encoder=enc, database=DeviceDatabase(db, DEV, shard=(r, P))) for r in range(P)]
    coords = [torch.tensor(O.area_uniform(slab, np.random.default_rng(50 + r)), device=DEV) for r in range(P)]
    own = [shards[r].sort_queries(coords[r]) for r in range(P)]
    encd = [shards[r].encode(own[r][0]) for r in range(P)]
    q16_all = torch.cat([e[1] for e in encd]).contiguous()
    qxyz_all = torch.cat([e[2] for e in encd]).contiguous()
    recv = [torch.full((2 * P, slab, 1024), float("nan"), device=DEV) for _ in range(P)]
    bufs = []
    for r in range(P):                                   # what PeerBuffers holds on rank r: every rank's buffer mapped
        b = PeerBuffers.__new__(PeerBuffers)
        b.world, b.rank, b.slab = P, r, 2 * slab
        b.ptrs, b.local = [x.data_ptr() for x in recv], ctypes.c_void_p(recv[r].data_ptr())
        bufs.append(b)
    stats = [s.retrieve_stats("RANGE+", q16_all, qxyz_all, temp, geo_temp) for s in shards]
    sums = torch.stack([a for a, _ in stats]).sum(0)
    for r in range(P):
        shards[r].retrieve_apply_routed("RANGE+", q16_all, qxyz_all, temp, geo_temp, 0.0, sums, stats[r][1],
                                        bufs[r].route(slab, 0))
        shards[r].retrieve_apply_routed("RANGE", q16_all, qxyz_all, temp, 0.0, None, sums, stats[r][1],
                                        bufs[r].route(slab, 1))
    sample = np.arange(0, slab, 1 if slab <= 256 else 33)
    for r in range(P):
        assert torch.isfinite(recv[r]).all()                         # every slot of both halves was written
        got = shards[r].sweep_concat(bufs[r].slots(slab, 0), bufs[r].slots(slab, 1), betas, encd[r][0],
                                     out_dtype=torch.float64, perm=own[r][1])
        ref = whole.embed_sweep(coords[r], betas, out_dtype=torch.float64)
        exact = {b: O.RangeOracle("RANGE+", ws, sh_entries, db, beta=b, exact=True)(coords[r].cpu().numpy()[sample])
                 for b in betas}
        for b, g, u in zip(betas, got, ref):
            assert torch.equal(g[:, 1024:], u[:, 1024:]), (r, b)
            rel = rel_rows(g[:, :1024].cpu().numpy(), u[:, :1024].cpu().numpy())
            assert rel.max() <= 3e-4, (r, b, rel.max())
            rel_x = rel_rows(g[sample, :1024].cpu().numpy(), exact[b][:, :1024])
            assert rel_x.max() <= tol_o("RANGE+", b), (r, b, rel_x.max())


@pytest.mark.gpu
def test_sharded_sweep_and_raster_one_rank_nccl():
    """the real peer path on one GPU: a world of one rank over NCCL (receive buffer from range_peer_alloc, routed ends in
    its two halves, the barrier, several steps) for embed_sweep and the façade's raster calls, against the unsharded calls"""
    from range_b200.distributed import ShardedRetriever
    from range_b200.range import LocationEncoder
    from tests.test_gpu_parity import rel_rows
    port = 37500 + os.getpid() % 2000
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1,
                            device_id=torch.device(DEV))
    try:
        ws = O.siren_init(40, 256, 2, 256, seed=1)
        db = O.synthetic_db(6000, seed=5, kind="iid")
        m = LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=dict(L=40, dims=[1600, 256, 256, 256],
                                      weights=ws), device=DEV, range_db=db, beta=0.5))
        c = torch.tensor(O.area_uniform(3000, np.random.default_rng(9)), device=DEV)
        betas = [0.0, 0.25, 0.5, 0.75, 1.0]
        ref = m.embed_sweep(c, betas, out_dtype=torch.float64)
        lon, lat = m.coord_grid_axes((40, 60))
        ref_raster = m.embed_raster(lon, lat, rows=(100, 2100), out_dtype=torch.float64)
        sr = ShardedRetriever(m.engine, merge="peer")
        sr.MAX_STEP_ROWS = 2048                          # sweep slab 1024: 3 steps
        got = sr.embed_sweep(c, 12.0, 40.0, True, betas, out_dtype=torch.float64)
        assert sr.merge == "peer" and sr.buffers is not None and sr.buffers.slab == 2048
        assert sr.collectives == 1 + 4 * 3
        for b, g, u in zip(betas, got, ref):
            assert torch.equal(g[:, 1024:], u[:, 1024:]), b
            # other step boundaries -> other query tiles: the fp16 rounding of the weights differs in the last bit
            assert rel_rows(g[:, :1024].cpu().numpy(), u[:, :1024].cpu().numpy()).max() <= 5e-4, b
        m.sharded = sr                                   # the façade's collective branches
        r = m.embed_raster(lon, lat, rows=(100, 2100), out_dtype=torch.float64)
        assert (r[:, 1024:] - ref_raster[:, 1024:]).abs().max().item() <= 1e-12
        assert rel_rows(r[:, :1024].cpu().numpy(), ref_raster[:, :1024].cpu().numpy()).max() <= 5e-4
        host = np.full((2000, 1280), np.nan)
        assert m.forward_raster(lon, lat, rows=(100, 2100), out=host) is host
        assert np.array_equal(host, r.cpu().numpy())
        sweep = m.embed_sweep(c, [0.3])                  # the façade's sweep
        assert len(sweep) == 1 and sweep[0].dtype == torch.float32 and sweep[0].shape == (3000, 1280)
        sr.close()
    finally:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------- 2 GPUs
@pytest.mark.gpu
def test_m_sharded_sweep_and_raster_on_two_gpus():
    """tools/multi_gpu_check.py under torchrun on 2 GPUs (skipped on a one-GPU box): the sharded sweep and raster calls
    against the unsharded ones, under both merge settings"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29537", os.path.join(root, "tools", "multi_gpu_check.py")],
                       capture_output=True, text=True, timeout=900, cwd=root, env=dict(os.environ, M="60000", N="9000"))
    assert p.returncode == 0, (p.stdout[-2000:], p.stderr[-3000:])
    assert "M-sharded sweep" in p.stdout and "M-sharded raster" in p.stdout, p.stdout[-2000:]
