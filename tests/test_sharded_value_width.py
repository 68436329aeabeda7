"""Databases sharded along M whose values have a width D other than 1024: every shard's partial rows (D floats) reach
their owners through range_retrieve_apply_routed_values - on the CTA-pair path one fused kernel per query chunk sums the
database splits' partials and stores each row once into the owner's receive buffer (csrc/merge.cu: reduce_route_kernel)
- then the owner's any-width merge kernels.

CPU: the host pipeline on gloo (world size 2) through a torch stand-in engine of width D, in fp64; PeerBuffers' size and
offsets; the step bound that keeps the receive buffer at 512 MB for wide values; the façade's width rule.  GPU: P = 3
shards emulated one after the other on one device (NaN-filled receive buffers, several query chunks, chunks spanning two
owners) against the unsharded model and the exact oracle; a world of one rank over NCCL through the real peer path and
every public entry point.  2 GPUs: tools/multi_gpu_check.py with D=768 under torchrun.
"""
import ctypes
import os
import subprocess
import sys
from argparse import Namespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import range_oracle as O
from tests.test_distributed import _database, _encode
from tests.test_neighbours_sharded import TopkEngine
from tests.test_sharded_sweep_raster import SweepEngine

DEV = "cuda:0"
TS, TG, BETA = 12.0, 40.0, 0.3


# ---------------------------------------------------------------------------------------------------- CPU: stand-in
class WidthEngine(SweepEngine, TopkEngine):
    """the stand-in engines of the 1024-wide tests (sweep ends, top-k lists) over values of width D: results D + 256
    columns wide, in fp64"""

    def __init__(self, K, V, X, lo, M_total):
        TopkEngine.__init__(self, K, V, X, lo, M_total)
        self.db.caps = True
        self.value_dim = V.shape[1]

    def combine_concat(self, parts, weights, q64, out=None, dtype=torch.float64, perm=None):
        out = torch.empty(q64.shape[0], self.value_dim + 256, dtype=dtype) if out is None else out
        return super().combine_concat(parts, weights, q64, out=out, perm=perm)

    def sweep_concat(self, geo_parts, sem_parts, betas, q64, out_dtype=torch.float32, perm=None, outs=None):
        outs = [torch.empty(q64.shape[0], self.value_dim + 256, dtype=out_dtype) for _ in betas] if outs is None else outs
        return super().sweep_concat(geo_parts, sem_parts, betas, q64, perm=perm, outs=outs)


def _values(M, D):
    return torch.randn(M, D, generator=torch.Generator().manual_seed(D), dtype=torch.float64)


def _gloo_worker(rank, world, port, D, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from range_b200.distributed import ShardedRetriever, shard_rows
    fails = []
    M = 1001
    K, V1024, X = _database(M)
    V = _values(M, D)
    lo, hi = shard_rows(M, rank, world)
    sr = ShardedRetriever(WidthEngine(K[lo:hi], V[lo:hi], X[lo:hi], lo, M), merge="reduce_scatter")
    sr.MAX_STEP_ROWS = 256 * world * max(1, D // 1024)  # 256 rows per rank and step for every D: rank 0 takes 2 steps
    n = [300, 77][rank]
    rng = np.random.default_rng(40 + rank)
    coords = torch.tensor(np.stack([rng.uniform(-180, 180, n), rng.uniform(-90, 90, n)], 1))
    q, xyz = _encode(coords)
    s, g = q.half().double() @ K.t(), xyz.float().double() @ X.t()
    Ps, Pg = torch.softmax(TS * s, 1), torch.softmax(TG * g, 1)
    for sort in (False, True):
        before = sr.collectives
        got = sr.embed("RANGE+", coords, TS, TG, BETA, sort, out_dtype=torch.float64)
        if sr.collectives - before != 1 + 4 * 2:                                  # n, then 2 steps of 4 collectives
            fails.append(("embed collectives", sort, sr.collectives - before))
        ref = (BETA * Ps + (1 - BETA) * Pg) @ V
        if got.shape != (n, D + 256):
            fails.append(("embed shape", sort, tuple(got.shape)))
        elif not (torch.allclose(got[:, :D], ref, rtol=1e-9, atol=1e-11) and torch.equal(got[:, D:], q)):
            fails.append(("embed rows", sort, float((got[:, :D] - ref).abs().max())))
        betas = [0.0, 0.3, 1.0]
        before = sr.collectives
        sweep = sr.embed_sweep(coords, TS, TG, sort, betas, out_dtype=torch.float64)
        if sr.collectives - before != 1 + 5 * 3:                                  # half the slab: 3 steps of 5
            fails.append(("sweep collectives", sort, sr.collectives - before))
        for b, o in zip(betas, sweep):
            ref = ((1 - b) * Pg + b * Ps) @ V
            if o.shape != (n, D + 256):
                fails.append(("sweep shape", sort, b, tuple(o.shape)))
            elif not (torch.allclose(o[:, :D], ref, rtol=1e-9, atol=1e-11) and torch.equal(o[:, D:], q)):
                fails.append(("sweep rows", sort, b))
        # neighbours do not read the values: the same lists as a 1024-wide database's
        wide = ShardedRetriever(WidthEngine(K[lo:hi], V1024[lo:hi], X[lo:hi], lo, M), merge="reduce_scatter")
        wide.MAX_STEP_ROWS = sr.MAX_STEP_ROWS
        a = sr.neighbours("RANGE+", coords, TS, TG, BETA, sort, 8)
        b = wide.neighbours("RANGE+", coords, TS, TG, BETA, sort, 8)
        if not (torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])):
            fails.append(("neighbours", sort))
    empty = sr.embed("RANGE+", coords[:0], TS, TG, BETA, True, out_dtype=torch.float64)
    if empty.shape != (0, D + 256):
        fails.append(("empty", tuple(empty.shape)))
    if sr.buffers is not None:
        fails.append("peer buffers under reduce_scatter")
    ret[rank] = fails
    dist.destroy_process_group()


@pytest.mark.parametrize("D", [12, 768, 2048])
def test_sharded_pipeline_of_another_width_gloo(D):
    world = 2
    port = 39500 + os.getpid() % 2000 + D % 97
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_gloo_worker, args=(world, port, D, ret), nprocs=world, join=True)
    assert [ret[r] for r in range(world)] == [[], []]


class _FakeLib:
    """range_peer_alloc / range_peer_free of a one-rank world without a device: records the bytes asked for"""

    def __init__(self):
        self.nbytes = None

    def range_peer_alloc(self, nbytes, local, handle):
        self.nbytes = nbytes
        local._obj.value = 1 << 20
        return 0

    def range_peer_free(self, p):
        return 0


@pytest.mark.parametrize("D", [768, 4096])
def test_peer_buffers_size_and_offsets(D):
    from range_b200.distributed import PeerBuffers
    port = 41500 + os.getpid() % 2000 + D % 89
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1)
    try:
        lib = _FakeLib()
        b = PeerBuffers(lib, -1, 512, None, D)
        assert b.width == D and lib.nbytes == 1 * 512 * D * 4
    finally:
        dist.destroy_process_group()
    # a buffer of P = 3 ranks as rank 1 sees it
    b = PeerBuffers.__new__(PeerBuffers)
    b.world, b.rank, b.slab, b.width = 3, 1, 1024, D
    b.ptrs, b.local = [1 << 32, 2 << 32, 3 << 32], ctypes.c_void_p(2 << 32)
    r0, r1 = b.route(256), b.route(256, 1)
    assert (r0.n_ranks, r0.rank, r0.slab_rows) == (3, 1, 256)
    assert list(r0.peer[:3]) == b.ptrs and list(r1.peer[:3]) == [p + 3 * 256 * D * 4 for p in b.ptrs]
    assert b.slots(256) == [(2 << 32) + k * 256 * D * 4 for k in range(3)]
    assert b.slots(256, 1) == [(2 << 32) + (3 + k) * 256 * D * 4 for k in range(3)]
    old = PeerBuffers.__new__(PeerBuffers)               # built without a width (the 1024-wide tests): 4096-byte rows
    old.world, old.rank, old.slab, old.ptrs, old.local = 2, 0, 512, [1 << 32, 2 << 32], ctypes.c_void_p(1 << 32)
    assert old.width == 1024 and old.slots(128, 1) == [(1 << 32) + 2 * 128 * 4096, (1 << 32) + 3 * 128 * 4096]


def _retriever(world, D, step_rows=None):
    from range_b200.distributed import ShardedRetriever
    sr = ShardedRetriever.__new__(ShardedRetriever)
    sr.world, sr.width = world, D
    if step_rows is not None:
        sr.MAX_STEP_ROWS = step_rows
    return sr


@pytest.mark.parametrize("world", [1, 3, 8])
def test_step_rows_keep_the_receive_buffer_bounded(world):
    n_max = 10 ** 7
    base = _retriever(world, 1024)._slab_for(n_max)
    for D in (4, 768, 1024):
        assert _retriever(world, D)._slab_for(n_max) == base
    for D in (1028, 2048, 4096):
        slab = _retriever(world, D)._slab_for(n_max)
        assert world * slab * D * 4 <= 512 << 20, (D, slab)
        assert world * 2 * (slab // 2 // 128 * 128) * D * 4 <= 512 << 20          # the sweep's two halves
    assert _retriever(8, 4096)._step_rows() == 32768 and _retriever(8, 4096)._slab_for(n_max) == 4096
    assert _retriever(2, 2048, step_rows=2048)._step_rows() == 1024                # on top of a MAX_STEP_ROWS override
    assert _retriever(2, 768, step_rows=2048)._step_rows() == 2048


def _args(D, **kw):
    rng = np.random.default_rng(D)
    db = dict(locs=O.area_uniform(200, rng), satclip_embeddings=rng.standard_normal((200, 256)),
              image_embeddings=rng.standard_normal((200, D)))
    return Namespace(location_model_name="RANGE+", pretrained_path=dict(L=40), device="cpu", range_db=db, beta=0.5,
                     db_shard=(0, 2), **kw)


@pytest.mark.parametrize("D", [1, 10, 257])
def test_sharded_width_not_a_multiple_of_4_raises(D, monkeypatch):
    from range_b200 import range as R
    monkeypatch.setattr(R, "RangeEngine", lambda *a, **k: pytest.fail("an engine was created"))
    with pytest.raises(NotImplementedError, match="multiple of 4") as e:
        R.LocationEncoder(_args(D))
    assert "1024" in str(e.value) and "unsharded" in str(e.value)


def test_sharded_width_768_is_accepted():
    """no width error: construction goes on to the engine, which needs a CUDA device"""
    from range_b200 import range as R
    from range_b200._lib import RangeError
    with pytest.raises(RangeError, match="CUDA"):
        R.LocationEncoder(_args(768))


def test_routed_values_symbol_in_prototypes():
    from range_b200 import _lib
    assert "range_retrieve_apply_routed_values" in _lib.PROTOTYPES
    assert _lib.PROTOTYPES["range_retrieve_apply_routed_values"] == _lib.PROTOTYPES["range_retrieve_apply_routed"]


# ---------------------------------------------------------------------------------------------------- GPU: P emulated
@pytest.fixture
def chunk_bytes():
    """set(bytes) replaces the apply pass's query-chunk bound for one test; the default is back afterwards"""
    from range_b200 import _lib
    lib = _lib.load()
    lib.range_debug_set_apply_chunk_bytes.argtypes = [ctypes.c_size_t]
    lib.range_debug_set_apply_chunk_bytes.restype = ctypes.c_size_t
    yield lib.range_debug_set_apply_chunk_bytes
    lib.range_debug_set_apply_chunk_bytes(0)


def _wide_db(M, D, sh_entries, ws, seed=4):
    helper = O.RangeOracle.__new__(O.RangeOracle)
    helper.L, helper.entries, helper.weights = 40, sh_entries, ws
    db = O.synthetic_db(M, seed=seed, kind="structured", encoder=helper.encode)
    return dict(db, image_embeddings=np.random.default_rng(D).standard_normal((M, D)) + 0.5)


def _emulated(db, enc, P, slab, D):
    """P shard engines and every rank's queries, sorted and encoded; the receive buffers [2P][slab][D] of every rank,
    NaN-filled, and what PeerBuffers holds on each rank"""
    from range_b200.database import DeviceDatabase
    from range_b200.distributed import PeerBuffers
    from range_b200.engine import RangeEngine
    shards = [RangeEngine(DEV, encoder=enc, database=DeviceDatabase(db, DEV, shard=(r, P))) for r in range(P)]
    assert all(s.value_dim == D for s in shards)
    coords = [torch.tensor(O.area_uniform(slab, np.random.default_rng(60 + r)), device=DEV) for r in range(P)]
    own = [shards[r].sort_queries(coords[r]) for r in range(P)]
    encd = [shards[r].encode(own[r][0]) for r in range(P)]
    recv = [torch.full((2 * P, slab, D), float("nan"), device=DEV) for _ in range(P)]
    bufs = []
    for r in range(P):
        b = PeerBuffers.__new__(PeerBuffers)
        b.world, b.rank, b.slab, b.width = P, r, 2 * slab, D
        b.ptrs, b.local = [x.data_ptr() for x in recv], ctypes.c_void_p(recv[r].data_ptr())
        bufs.append(b)
    return shards, coords, own, encd, recv, bufs


@pytest.mark.gpu
@pytest.mark.parametrize("D", [4, 768, 1028, 2048, 4096])
def test_m_sharded_routed_values_emulated(D, sh_entries, chunk_bytes):
    """ShardedRetriever's embed and embed_sweep steps with P = 3 ranks emulated on one GPU, values of width D: every
    shard's routed apply pass (range_retrieve_apply_routed_values) into NaN-filled [2P][slab][D] receive buffers, then
    every owner's range_combine_concat / range_sweep_concat over its slots, against the unsharded model and the exact
    oracle.  1028: the last 256-column value slice partly filled.  4096: 256-row query chunks (the chunk bound shrunk),
    so the chunk [256, 512) spans owners 0 and 1 of 384-row slabs."""
    from range_b200.range import LocationEncoder
    from tests.test_gpu_parity import rel_rows, tol_o
    P, M, slab = 3, 12_000, 384
    ws = O.siren_init(40, 64, 2, 256, seed=2)
    db = _wide_db(M, D, sh_entries, ws)
    enc = dict(L=40, dims=[1600, 64, 64, 256], weights=ws)
    if D == 4096:
        chunk_bytes(1)                                   # the smallest chunk: one CTA pair of query tiles, 256 rows
    whole = LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=enc, device=DEV, range_db=db, beta=0.5))
    whole_r = LocationEncoder(Namespace(location_model_name="RANGE", pretrained_path=enc, device=DEV, range_db=db))
    shards, coords, own, encd, recv, bufs = _emulated(db, enc, P, slab, D)
    q16_all = torch.cat([e[1] for e in encd]).contiguous()
    qxyz_all = torch.cat([e[2] for e in encd]).contiguous()
    sample = np.arange(0, slab, 29)
    for name, beta, temp in (("RANGE", None, 15.0), ("RANGE+", 0.0, 12.0), ("RANGE+", 0.5, 12.0), ("RANGE+", 1.0, 12.0)):
        model = whole_r if name == "RANGE" else whole
        model.args.beta = beta
        stats = [s.retrieve_stats(name, q16_all, qxyz_all, temp, 40.0) for s in shards]
        sums = torch.stack([a for a, _ in stats]).sum(0)
        for x in recv:
            x.fill_(float("nan"))
        for r in range(P):
            shards[r].retrieve_apply_routed(name, q16_all, qxyz_all, temp, 40.0, beta, sums, stats[r][1],
                                            bufs[r].route(slab))
        oracle = O.RangeOracle(name, ws, sh_entries, db, beta=beta, exact=True)
        for r in range(P):
            assert torch.isfinite(recv[r][:P]).all(), (D, name, beta, r)        # every slot of every owner was written
            assert torch.isnan(recv[r][P:]).all()                               # and nothing past them
            got = shards[r].combine_concat(bufs[r].slots(slab), None, encd[r][0], perm=own[r][1], dtype=torch.float64)
            ref = model.embed(coords[r], out_dtype=torch.float64)
            assert got.shape == (slab, D + 256) and torch.equal(got[:, D:], ref[:, D:])
            rel = rel_rows(got[:, :D].cpu().numpy(), ref[:, :D].cpu().numpy())
            assert rel.max() <= 3e-4, (D, name, beta, r, rel.max())
            exact = oracle(coords[r].cpu().numpy()[sample])
            rel_x = rel_rows(got[sample, :D].cpu().numpy(), exact[:, :D])
            assert rel_x.max() <= tol_o(name, beta), (D, name, beta, r, rel_x.max())
    # a beta sweep: both ends routed into the two halves, then every owner's sweep_concat over its 2 P slots
    betas = [0.0, 0.5, 1.0]
    stats = [s.retrieve_stats("RANGE+", q16_all, qxyz_all, 12.0, 40.0) for s in shards]
    sums = torch.stack([a for a, _ in stats]).sum(0)
    for x in recv:
        x.fill_(float("nan"))
    for r in range(P):
        shards[r].retrieve_apply_routed("RANGE+", q16_all, qxyz_all, 12.0, 40.0, 0.0, sums, stats[r][1],
                                        bufs[r].route(slab, 0))
        shards[r].retrieve_apply_routed("RANGE", q16_all, qxyz_all, 12.0, 0.0, None, sums, stats[r][1],
                                        bufs[r].route(slab, 1))
    for r in range(P):
        assert torch.isfinite(recv[r]).all()
        got = shards[r].sweep_concat(bufs[r].slots(slab, 0), bufs[r].slots(slab, 1), betas, encd[r][0],
                                     out_dtype=torch.float64, perm=own[r][1])
        ref = whole.embed_sweep(coords[r], betas, out_dtype=torch.float64)
        for b, g, u in zip(betas, got, ref):
            assert g.shape == (slab, D + 256) and torch.equal(g[:, D:], u[:, D:]), (D, b, r)
            rel = rel_rows(g[:, :D].cpu().numpy(), u[:, :D].cpu().numpy())
            assert rel.max() <= 3e-4, (D, b, r, rel.max())


@pytest.mark.gpu
@pytest.mark.parametrize("slab", [256, 4224])
def test_routed_values_at_1024_is_routed(slab, sh_entries):
    """a 1024-wide database: range_retrieve_apply_routed_values stores the same bits as range_retrieve_apply_routed,
    on the CTA-pair path (slab 256) and the producer/consumer path (slab 4224)"""
    from range_b200 import _lib
    from range_b200.engine import MODE, _ptr, _stream
    P = 3
    ws = O.siren_init(40, 64, 2, 256, seed=2)
    db = _wide_db(12_000, 1024, sh_entries, ws)
    enc = dict(L=40, dims=[1600, 64, 64, 256], weights=ws)
    shards, _, _, encd, recv, bufs = _emulated(db, enc, P, slab, 1024)
    q16_all = torch.cat([e[1] for e in encd]).contiguous()
    qxyz_all = torch.cat([e[2] for e in encd]).contiguous()
    stats = [s.retrieve_stats("RANGE+", q16_all, qxyz_all, 12.0, 40.0) for s in shards]
    sums = torch.stack([a for a, _ in stats]).sum(0)
    for r, s in enumerate(shards):
        ws_ = s._ret_ws(P * slab)
        for half, fn in ((0, s.lib.range_retrieve_apply_routed), (1, s.lib.range_retrieve_apply_routed_values)):
            with torch.cuda.device(s.index):
                assert fn(s.ctx, MODE["RANGE+"], P * slab, _ptr(q16_all), _ptr(qxyz_all), 12.0, 40.0, 0.5, _ptr(sums),
                          _ptr(stats[r][1]), ctypes.byref(bufs[r].route(slab, half)), _ptr(ws_), ws_.numel(),
                          _stream()) == 0, _lib.load().range_last_error()
    for r in range(P):
        assert torch.isfinite(recv[r]).all() and torch.equal(recv[r][:P], recv[r][P:])


@pytest.mark.gpu
def test_routed_values_needs_a_multiple_of_4():
    from range_b200 import _lib
    from range_b200.database import DeviceDatabase
    from range_b200.engine import RangeEngine, _ptr, _stream
    rng = np.random.default_rng(1)
    db = dict(locs=O.area_uniform(3000, rng), satclip_embeddings=rng.standard_normal((3000, 256)),
              image_embeddings=rng.standard_normal((3000, 258)))
    eng = RangeEngine(DEV, L=40, database=DeviceDatabase(db, DEV))
    N = 512
    q16 = torch.randn(N, 256, device=DEV).half()
    qxyz = torch.zeros(N, 4, device=DEV)
    sums, maxs = eng.retrieve_stats("RANGE", q16, qxyz, 15.0, 0.0)
    ws = eng._ret_ws(N)
    buf = torch.full((N, 258), float("nan"), device=DEV)
    route = _lib.Route(1, 0, 512, (ctypes.c_void_p * _lib.RANGE_MAX_RANKS)(buf.data_ptr()))
    for fn in (eng.lib.range_retrieve_apply_routed_values, eng.lib.range_retrieve_apply_routed):
        assert fn(eng.ctx, 0, N, _ptr(q16), _ptr(qxyz), 15.0, 0.0, 0.0, _ptr(sums), _ptr(maxs), ctypes.byref(route),
                  _ptr(ws), ws.numel(), _stream()) == -4                        # RANGE_ERR_UNSUPPORTED
    with pytest.raises(_lib.RangeError, match="multiple of 4"):
        eng.retrieve_apply_routed("RANGE", q16, qxyz, 15.0, 0.0, None, sums, maxs, route)
    torch.cuda.synchronize()
    assert torch.isnan(buf).all()


# ---------------------------------------------------------------------------------------------------- GPU: one rank
@pytest.mark.gpu
def test_sharded_768_one_rank_nccl(tmp_path):
    """the real peer path of a 768-wide database on one GPU: a world of one rank over NCCL (receive buffer from
    range_peer_alloc, several steps), every public entry point of the façade against the unsharded model"""
    from range_b200.distributed import ShardedRetriever
    from range_b200.range import LocationEncoder
    from range_b200.save import embed_to_npy
    from tests.test_gpu_parity import rel_rows
    D = 768
    port = 43500 + os.getpid() % 2000
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1,
                            device_id=torch.device(DEV))
    try:
        ws = O.siren_init(40, 256, 2, 256, seed=1)
        rng = np.random.default_rng(5)
        db = dict(locs=O.area_uniform(6000, rng), satclip_embeddings=rng.standard_normal((6000, 256)),
                  image_embeddings=rng.standard_normal((6000, D)))
        enc = dict(L=40, dims=[1600, 256, 256, 256], weights=ws)

        def model(**kw):
            return LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=enc, device=DEV, range_db=db,
                                             beta=0.5, **kw))

        full = model()
        cache = str(tmp_path / "db.npz")
        model(db_cache=cache)
        m = model(db_cache=cache)                        # the prepared layout read back from the cache
        assert full.location_feature_dim == m.location_feature_dim == D + 256
        sr = ShardedRetriever(m.engine, merge="peer")
        sr.MAX_STEP_ROWS = 1024                          # embed: 3 steps of 1024 rows; sweep: 6 of 512
        m.sharded = sr
        n = 3000
        c = O.area_uniform(n, np.random.default_rng(9))
        dc = torch.tensor(c, device=DEV)

        def close(got, ref, what):
            got, ref = torch.as_tensor(got).double().cpu(), torch.as_tensor(ref).double().cpu()
            assert got.shape == ref.shape == (ref.shape[0], D + 256), what
            assert (got[:, D:] - ref[:, D:]).abs().max().item() <= 1e-12, what
            # other step boundaries -> other query tiles: the fp16 rounding of the weights differs in the last bit
            assert rel_rows(got[:, :D].numpy(), ref[:, :D].numpy()).max() <= 5e-4, what

        ref = full.embed(dc, out_dtype=torch.float64)
        before = sr.collectives
        got = m.embed(dc, out_dtype=torch.float64)
        assert sr.merge == "peer" and sr.buffers is not None and sr.buffers.width == D
        assert sr.collectives - before == 1 + 4 * 3
        close(got, ref, "embed")
        for path in ("copy", "packed"):
            m.host_path = path
            host = m(c)
            assert host.dtype == np.float64 and np.array_equal(host, got.cpu().numpy()), path
        m.host_path = "auto"
        into = np.full((n, D + 256), np.nan)
        assert m.embed_into(c, into) is into and np.array_equal(into, got.cpu().numpy())
        npy = embed_to_npy(m, c, str(tmp_path / "e.npy"))
        assert npy.shape == (n, D + 256) and np.array_equal(np.load(tmp_path / "e.npy"), got.cpu().numpy())
        betas = [0.0, 0.5, 1.0]
        for b, g, u in zip(betas, m.embed_sweep(dc, betas, out_dtype=torch.float64),
                           full.embed_sweep(dc, betas, out_dtype=torch.float64)):
            close(g, u, ("sweep", b))
        a, b = m.neighbours(dc, 8), full.neighbours(dc, 8)
        assert a[0].shape == (n, 8) and torch.allclose(a[1], b[1], rtol=2e-3, atol=0)
        assert (a[0] != b[0]).double().mean().item() <= 1e-3                   # near-ties at the cut may swap
        lon, lat = m.coord_grid_axes((40, 60))
        ras = m.forward_raster(lon, lat, rows=(100, 2100))
        close(ras, full.forward_raster(lon, lat, rows=(100, 2100)), "forward_raster")
        assert np.array_equal(ras, m.embed_raster(lon, lat, rows=(100, 2100), out_dtype=torch.float64).cpu().numpy())
        sr.close()
    finally:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------- 2 GPUs
@pytest.mark.gpu
def test_m_sharded_768_on_two_gpus():
    """tools/multi_gpu_check.py with D=768 under torchrun on 2 GPUs (skipped on a one-GPU box)"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29547", os.path.join(root, "tools", "multi_gpu_check.py")],
                       capture_output=True, text=True, timeout=900, cwd=root,
                       env=dict(os.environ, M="60000", N="9000", D="768"))
    assert p.returncode == 0, (p.stdout[-2000:], p.stderr[-3000:])
    assert "D=768" in p.stdout and "M-sharded sweep" in p.stdout and "M-sharded raster" in p.stdout, p.stdout[-2000:]
