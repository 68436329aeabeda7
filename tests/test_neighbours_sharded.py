"""Retrieval neighbours of a database sharded along M: every shard's top-k lists in rows of the whole database
(range_retrieve_topk_rows), the lists exchanged, merged on the owner of the query (range_topk_merge), rows of the sorted
layout mapped to file rows (DeviceDatabase.file_rows_global).

CPU: the host pipeline of ShardedRetriever.neighbours on gloo (world size 2) through a torch stand-in engine, exactly
against the unsharded fp64 top-k; file_rows_global.  GPU: P = 3 shards emulated one after the other on one device, every
row against the exact fp64 weights (the contract of tests/test_neighbours.py), and the same against the unsharded pass.
2 GPUs: tools/multi_gpu_check.py under torchrun.
"""
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import range_oracle as O
from range_b200.database import DeviceDatabase
from tests.test_distributed import TorchEngine, _database, _encode
from tests.test_neighbours import ATOL, GEO_TEMP, KS, MODES, TEMP, TOL, check_rows, exact_weights, make_engine

DEV = "cuda:0"


# ---------------------------------------------------------------------------------------------------- CPU: gloo pipeline
def _top(w, rows, k):
    """per query row: the k largest w, equal weights by the smaller row; rows -1 (empty slots) never chosen; slots
    beyond the available entries are (-1, 0)"""
    key = torch.where(rows >= 0, w, torch.full_like(w, -float("inf")))
    o = torch.argsort(rows, dim=1, stable=True)                              # secondary key first: the row ...
    o = o.gather(1, torch.argsort(key.gather(1, o), dim=1, descending=True, stable=True))    # ... then the weight
    o = o[:, :k]
    kw, r, ww = key.gather(1, o), rows.gather(1, o), w.gather(1, o)
    empty = kw == -float("inf")
    r, ww = torch.where(empty, -1, r).to(torch.int32), torch.where(empty, 0.0, ww)
    if r.shape[1] < k:
        pad = k - r.shape[1]
        r = torch.cat([r, torch.full((r.shape[0], pad), -1, dtype=r.dtype)], 1)
        ww = torch.cat([ww, torch.zeros(ww.shape[0], pad, dtype=ww.dtype)], 1)
    return r, ww


class TopkEngine(TorchEngine):
    """TorchEngine with the two top-k entry points, in fp64, over database rows [lo, lo + M) of M_total"""

    def __init__(self, K, V, X, lo, M_total):
        super().__init__(K, V, X)
        self.db = SimpleNamespace(row_range=(lo, lo + K.shape[0]), M_total=M_total)

    def weights(self, mode, q16, qxyz, temp, geo_temp, beta, sums):
        s, g = self._logits(q16, qxyz)
        ws = torch.exp(temp * (s - 1)) / sums[:, :1]
        if mode == "RANGE":
            return ws
        return beta * ws + (1 - beta) * torch.exp(geo_temp * (g - 1)) / sums[:, 1:]

    def retrieve_topk_rows(self, mode, q16, qxyz, temp, geo_temp, beta, sums, k, row0):
        W = self.weights(mode, q16, qxyz, temp, geo_temp, beta, sums)
        return _top(W, torch.arange(row0, row0 + W.shape[1]).expand_as(W), k)

    def topk_merge(self, part_w, part_idx, perm=None):
        parts, N, k = part_w.shape
        idx, w = _top(part_w.permute(1, 0, 2).reshape(N, parts * k), part_idx.permute(1, 0, 2).reshape(N, parts * k), k)
        if perm is None:
            return idx, w
        oi, ow = torch.empty_like(idx), torch.empty_like(w)
        oi[perm.long()], ow[perm.long()] = idx, w
        return oi, ow


def _gloo_worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from range_b200.distributed import ShardedRetriever, shard_rows
    fails = []
    n = [300, 77][rank]                                 # ragged: rank 0 takes two steps of 256, rank 1 one, padded
    rng = np.random.default_rng(20 + rank)
    coords = torch.tensor(np.stack([rng.uniform(-180, 180, n), rng.uniform(-90, 90, n)], 1))
    for M, ks in ((1001, (1, 8, 32)), (40, (8, 32))):   # M = 40: k = 32 > 20 entries per shard
        K, V, X = _database(M)
        lo, hi = shard_rows(M, rank, world)
        full = TopkEngine(K, V, X, 0, M)
        sr = ShardedRetriever(TopkEngine(K[lo:hi], V[lo:hi], X[lo:hi], lo, M), merge="reduce_scatter")
        sr.MAX_STEP_ROWS = 256 * world
        q, q16, qxyz = full.encode(coords)
        for name, beta in MODES:
            temp = TEMP[name]
            sums, _ = full.retrieve_stats(name, q16, qxyz, temp, GEO_TEMP)
            for k in ks:
                ref_idx, ref_w = full.retrieve_topk_rows(name, q16, qxyz, temp, GEO_TEMP, beta, sums, k, 0)
                for sort in (False, True):
                    before = sr.collectives
                    idx, w = sr.neighbours(name, coords, temp, GEO_TEMP, beta, sort, k)
                    what = (M, name, beta, k, sort)
                    if not (idx.dtype == torch.int32 and idx.shape == w.shape == (n, k)):
                        fails.append(("shape", what))
                    elif not (torch.equal(idx, ref_idx) and torch.allclose(w, ref_w, rtol=1e-12, atol=0)):
                        fails.append(("rows", what, int((idx != ref_idx).sum())))
                    if sr.collectives - before != 1 + 5 * 2:              # n / k, then 2 steps of 5 collectives
                        fails.append(("collectives", what, sr.collectives - before))
        assert sr.buffers is None                                            # no peer buffers
    # the ranks disagree on k: ValueError on every rank, before any list is computed
    try:
        sr.neighbours("RANGE", coords, 15.0, GEO_TEMP, None, False, 4 + rank)
        fails.append("mismatched k accepted")
    except ValueError:
        pass
    idx, w = sr.neighbours("RANGE+", coords[:0], 12.0, GEO_TEMP, 0.5, True, 8)   # every rank: no rows
    if not (idx.shape == w.shape == (0, 8)):
        fails.append(("empty", tuple(idx.shape)))
    ret[rank] = fails
    dist.destroy_process_group()


def test_sharded_neighbours_pipeline_gloo():
    world = 2
    port = 31500 + os.getpid() % 2000
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_gloo_worker, args=(world, port, ret), nprocs=world, join=True)
    assert [ret[r] for r in range(world)] == [[], []]


def test_stand_in_top_orders_ties_by_row():
    w = torch.tensor([[1.0, 2.0, 2.0, 0.5]], dtype=torch.float64)
    rows = torch.tensor([[7, 9, 3, -1]])
    idx, ww = _top(w, rows, 5)
    assert idx.tolist() == [[3, 9, 7, -1, -1]] and ww.tolist() == [[2.0, 2.0, 1.0, 0.0, 0.0]]


# ---------------------------------------------------------------------------------------------------- CPU: file rows
@pytest.mark.parametrize("kw", [dict(), dict(spatial_sort=False)], ids=["sorted", "unsorted"])
def test_file_rows_global(kw, tmp_path):
    db = O.synthetic_db(700, seed=9, kind="iid")
    P = 3
    shards = [DeviceDatabase(db, "cpu", shard=(r, P), **kw) for r in range(P)]
    for s in shards:
        s.save_cache(tmp_path / "db", fingerprint="x")
    cached = [DeviceDatabase.from_cache(tmp_path / "db", "cpu", shard=(r, P)) for r in range(P)]
    whole = DeviceDatabase(db, "cpu", **kw)
    for group in ([whole], shards, cached):
        union = []
        for d in group:
            i = torch.arange(d.M)
            lo = d.row_range[0]
            assert torch.equal(d.file_rows_global(lo + i), d.file_rows(i))
            assert torch.equal(d.file_rows_global(torch.arange(700)), whole.file_rows(torch.arange(700)))
            union.append(d.file_rows(i))
        assert torch.equal(torch.cat(union).sort().values, torch.arange(700))
    two_d = torch.tensor([[0, 699], [5, 1]], dtype=torch.int32)
    assert shards[1].file_rows_global(two_d).dtype == torch.int64
    assert torch.equal(shards[1].file_rows_global(two_d), whole.file_rows(two_d))


def test_file_rows_global_synthetic_shards():
    P, M = 3, 500
    shards = [DeviceDatabase.synthetic(M, "cpu", seed=3, shard=(r, P)) for r in range(P)]
    union = torch.cat([d.file_rows_global(torch.arange(*d.row_range)) for d in shards])
    assert torch.equal(union.sort().values, torch.arange(M))
    assert torch.equal(union, torch.from_numpy(shards[0].order))


def test_sharded_topk_symbols_in_prototypes():
    from range_b200 import _lib
    assert "range_retrieve_topk_rows" in _lib.PROTOTYPES and "range_topk_merge" in _lib.PROTOTYPES


# ---------------------------------------------------------------------------------------------------- GPU: P emulated
def _emulate(shards, coords, name, beta, k, sort=True):
    """ShardedRetriever.neighbours with its P ranks run one after the other on one device: (file rows, weight) of every
    owner's queries in the owner's row order.  coords: one (slab, 2) tensor per rank."""
    P, slab = len(shards), coords[0].shape[0]
    own = [shards[r].sort_queries(coords[r]) if sort else (coords[r], None) for r in range(P)]
    encd = [shards[r].encode(own[r][0]) for r in range(P)]
    q16_all = torch.cat([e[1] for e in encd]).contiguous()
    qxyz_all = torch.cat([e[2] for e in encd]).contiguous()
    temp = TEMP[name]
    sums = torch.stack([s.retrieve_stats(name, q16_all, qxyz_all, temp, GEO_TEMP)[0] for s in shards]).sum(0)
    lists = [s.retrieve_topk_rows(name, q16_all, qxyz_all, temp, GEO_TEMP, beta, sums, k, s.db.row_range[0])
             for s in shards]
    out = []
    for r in range(P):
        part_w = torch.stack([w[r * slab:(r + 1) * slab] for _, w in lists]).contiguous()
        part_idx = torch.stack([i[r * slab:(r + 1) * slab] for i, _ in lists]).contiguous()
        idx, w = shards[r].topk_merge(part_w, part_idx, perm=own[r][1])
        assert idx.dtype == torch.int32 and idx.shape == w.shape == (slab, k)
        out.append((shards[r].db.file_rows_global(idx), w))
    return out


def _check_against_unsharded(whole, wddb, ref, coords, got, name, beta, k):
    """the unsharded pass on the same queries: weights within TOL position by position, and the two lists hold the same
    entries except where their exact weights are within TOL of the k-th largest"""
    q64, q16, qxyz = whole.encode(coords)
    sums, _ = whole.retrieve_stats(name, q16, qxyz, TEMP[name], GEO_TEMP)
    idx, w = whole.retrieve_topk(name, q16, qxyz, TEMP[name], GEO_TEMP, beta, sums, k)
    rows_un = wddb.file_rows(idx)
    rows_sh, w_sh = got
    assert ((w_sh.double() - w.double()).abs() <= TOL * w.double() + ATOL).all(), (name, beta, k)
    W = exact_weights(ref, q64, qxyz, name, beta)
    kth = W.topk(k, dim=1).values[:, -1:]
    for a, b in ((rows_sh, rows_un), (rows_un, rows_sh)):
        only = ~(a.unsqueeze(2) == b.unsqueeze(1)).any(2)
        err = (W.gather(1, a) - kth).abs() - (TOL * kth + ATOL)
        assert (err[only] <= 0).all(), (name, beta, k, int(only.sum()))


def _run(db, ws, slab, modes=MODES, ks=KS, sample=None, sort=True, **kw):
    P = 3
    whole, wddb, ref = make_engine(db, ws, **kw)
    shards = [make_engine(db, ws, shard=(r, P), **kw)[0] for r in range(P)]
    coords = [torch.tensor(O.area_uniform(slab, np.random.default_rng(40 + r)), device=DEV) for r in range(P)]
    rows = torch.arange(slab, device=DEV) if sample is None else torch.as_tensor(sample, device=DEV)
    for name, beta in modes:
        for k in ks:
            got = _emulate(shards, coords, name, beta, k, sort=sort)
            for r in range(P):
                q64, _, qxyz = whole.encode(coords[r][rows])
                W = exact_weights(ref, q64, qxyz, name, beta)
                check_rows(got[r][0][rows], got[r][1][rows], W, k, (name, beta, k, db["locs"].shape[0], r))
                if k <= wddb.M:
                    _check_against_unsharded(whole, wddb, ref, coords[r][rows],
                                             (got[r][0][rows], got[r][1][rows]), name, beta, k)
    return whole, shards, coords


@pytest.fixture(scope="module")
def ws():
    return O.siren_init(40, 64, 2, 256, seed=5)


@pytest.mark.gpu
def test_sharded_topk_tiny_db(ws):
    """M = 50 over 3 shards of 16-17 entries: k = 32 exceeds every shard (lists end in -1 entries before the merge)"""
    db = O.synthetic_db(50, seed=8, kind="iid")
    _, shards, coords = _run(db, ws, 256)
    eng = shards[0]
    _, q16, qxyz = eng.encode(coords[0])
    sums, _ = eng.retrieve_stats("RANGE", q16, qxyz, 15.0, GEO_TEMP)
    i, w = eng.retrieve_topk_rows("RANGE", q16, qxyz, 15.0, GEO_TEMP, None, sums, 32, 1000)
    m = eng.db.M
    assert (i[:, m:] == -1).all() and (w[:, m:] == 0).all()
    assert ((i[:, :m] >= 1000) & (i[:, :m] < 1000 + m)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(), dict(spatial_sort=False)], ids=["sorted", "unsorted"])
def test_sharded_topk_exact(ws, kw):
    db = O.synthetic_db(20077, seed=6, kind="iid")
    _run(db, ws, 256, **kw)


@pytest.mark.gpu
def test_sharded_topk_large_slab_and_geo_mask(ws):
    """4 224 rows per rank: 12 672 gathered queries, so the statistics come from the CTA-pair kernel; spatially sorted
    queries on a sorted database, so the geo mask skips tiles; a sample of every owner's rows is checked"""
    db = O.synthetic_db(20077, seed=6, kind="iid")
    whole, shards, coords = _run(db, ws, 4224, modes=[("RANGE", None), ("RANGE+", 0.5)], ks=(8, 32),
                                 sample=np.arange(0, 4224, 33))
    encd = [s.encode(s.sort_queries(c)[0]) for s, c in zip(shards, coords)]
    q16 = torch.cat([e[1] for e in encd]).contiguous()
    qxyz = torch.cat([e[2] for e in encd]).contiguous()
    sums = torch.stack([s.retrieve_stats("RANGE+", q16, qxyz, 12.0, GEO_TEMP)[0] for s in shards]).sum(0)
    assert all(s.geo_mask(qxyz, GEO_TEMP, sums).any() for s in shards)


@pytest.mark.gpu
def test_sharded_topk_deterministic(ws):
    db = O.synthetic_db(20077, seed=6, kind="iid")
    shards = [make_engine(db, ws, shard=(r, 3))[0] for r in range(3)]
    coords = [torch.tensor(O.area_uniform(512, np.random.default_rng(60 + r)), device=DEV) for r in range(3)]
    for name, beta in (("RANGE", None), ("RANGE+", 0.5)):
        a = _emulate(shards, coords, name, beta, 16)
        b = _emulate(shards, coords, name, beta, 16)
        assert all(torch.equal(x[0], y[0]) and torch.equal(x[1], y[1]) for x, y in zip(a, b))


@pytest.mark.gpu
def test_sharded_topk_merge_argument_errors(ws):
    from range_b200 import _lib
    db = O.synthetic_db(300, seed=8, kind="iid")
    eng = make_engine(db, ws, shard=(0, 2))[0]
    w = torch.zeros(9, 4, 8, device=DEV)
    with pytest.raises(_lib.RangeError):                              # more parts than RANGE_MAX_RANKS
        eng.topk_merge(w, torch.zeros(9, 4, 8, dtype=torch.int32, device=DEV))
    with pytest.raises(ValueError):
        eng.topk_merge(w[:2], torch.zeros(2, 4, 8, dtype=torch.int64, device=DEV))
    _, q16, qxyz = eng.encode(torch.zeros(4, 2, dtype=torch.float64, device=DEV))
    sums, _ = eng.retrieve_stats("RANGE", q16, qxyz, 15.0, GEO_TEMP)
    for k, row0 in ((33, 0), (8, -1), (8, 2**31 - 100)):
        with pytest.raises(_lib.RangeError):
            eng.retrieve_topk_rows("RANGE", q16, qxyz, 15.0, GEO_TEMP, None, sums, k, row0)


# ---------------------------------------------------------------------------------------------------- 2 GPUs
@pytest.mark.gpu
def test_m_sharded_neighbours_on_two_gpus():
    """tools/multi_gpu_check.py under torchrun on 2 GPUs (skipped on a one-GPU box): the sharded neighbours call against
    the unsharded one, repeatable, identical under both merge settings"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(root, "tools", "multi_gpu_check.py")],
                       capture_output=True, text=True, timeout=900, cwd=root, env=dict(os.environ, M="60000", N="9000"))
    assert p.returncode == 0, (p.stdout[-2000:], p.stderr[-3000:])
    assert "M-sharded neighbours" in p.stdout, p.stdout[-2000:]
