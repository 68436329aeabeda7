"""Split-fp16 retrieval (retrieval_precision='f16x3'): Q.K^T and P'.V with every operand as hi + lo fp16 and three
tensor-core products per term, against fp16 operands and the fp64 restatement of the reference (oracle/).

CPU: load_model's validation; the retrieval plan of a split-fp16 ctx (single-role kernels, query chunks); the lo halves
of the device database (Kh / Vt unchanged, hi + lo reconstructs the fp32 source) and its cache; the M-sharded pipeline
on gloo with 512-wide query rows.  GPU: accuracy on iid, structured and offset databases; every entry point and value
width; neighbours; three shards emulated on one device; the C ABI's errors.
"""
import ctypes
import os
from argparse import Namespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import range_oracle as O
from tests.test_distributed import TorchEngine

DEV = "cuda:0"
FIELDS = ("splits", "tiles_per_split", "stats_splits", "stats_tiles_per_split", "pc", "stats_pc", "chunk_rows", "total")


def rel_rows(a, b, center=0.0):
    """relative row error ||a - b|| / ||b - center|| (center: the database mean for offset values)"""
    return np.linalg.norm(a - b, axis=1) / np.linalg.norm(b - center, axis=1)


# ---------------------------------------------------------------------------------------------------- CPU
def test_load_model_rejects_unknown_precision():
    from range_b200.engine import check_retrieval_precision
    from range_b200.load_model import load_model
    assert check_retrieval_precision("fp16") == "fp16" and check_retrieval_precision("f16x3") == "f16x3"
    for bad in ("bf16", "fp32", "F16X3", None):
        with pytest.raises(ValueError, match="retrieval_precision"):
            load_model("RANGE+", pretrained_path="unused.ckpt", db_path="unused.npz", retrieval_precision=bad)


def _plan(lib, sm, M, D, caps, precision, N):
    out = (ctypes.c_int64 * 8)()
    lib.range_debug_retrieval_plan_precision(sm, M, D, int(caps), precision, N, out)
    return dict(zip(FIELDS, out))


@pytest.fixture(scope="module")
def lib():
    from range_b200 import _lib
    lib = _lib.load()
    for name, extra in (("range_debug_retrieval_plan", []), ("range_debug_retrieval_plan_precision", [ctypes.c_int])):
        getattr(lib, name).argtypes = [ctypes.c_int, ctypes.c_int64, ctypes.c_int, ctypes.c_int] + extra + \
            [ctypes.c_int64, ctypes.POINTER(ctypes.c_int64)]
        getattr(lib, name).restype = None
    return lib


@pytest.mark.parametrize("N", [100, 12_288, 100_000])
@pytest.mark.parametrize("D", [768, 1024])
def test_split_plan_runs_the_single_role_kernels_in_chunks(lib, N, D):
    """f16x3: never the producer/consumer kernels, the apply pass in query chunks whose split partials and scratch rows
    stay within 1 GiB; the fp16 plan is the one range_debug_retrieval_plan describes"""
    from range_b200 import _lib
    M = 100_000
    f16 = _plan(lib, 148, M, D, True, _lib.RANGE_RET_F16, N)
    old = (ctypes.c_int64 * 8)()
    lib.range_debug_retrieval_plan(148, M, D, 1, N, old)
    assert f16 == dict(zip(FIELDS, old))
    x3 = _plan(lib, 148, M, D, True, _lib.RANGE_RET_F16X3, N)
    assert x3["pc"] == 0 and x3["stats_pc"] == 0
    assert x3["chunk_rows"] <= N and (x3["chunk_rows"] == N or x3["chunk_rows"] % 256 == 0)
    arrays = x3["splits"] + 1 if x3["splits"] > 1 else 1
    assert x3["chunk_rows"] == 256 or arrays * x3["chunk_rows"] * D * 4 <= 1 << 30
    if f16["pc"]:       # large batches: the workspace of the split mode is not the fp16 one
        assert x3["total"] != f16["total"]


def _small_db(M, D, offset=0.0, seed=3):
    rng = np.random.default_rng(seed)
    return dict(locs=O.area_uniform(M, rng), satclip_embeddings=rng.standard_normal((M, 256), dtype=np.float32),
                image_embeddings=(offset + rng.standard_normal((M, D))).astype(np.float32))


def _lo_bound(x, hi):
    """|hi + lo - x| for lo = rn_f16(x - hi): half an fp16 ulp of the residual (2^-11 relative) where lo is normal,
    2^-25 where it is subnormal"""
    return 2.0 ** -11 * np.abs(x - hi) + 2.0 ** -25


@pytest.mark.parametrize("D", [100, 1024])
def test_lo_halves_reconstruct_the_fp32_source(D):
    from range_b200.database import DeviceDatabase
    db = _small_db(1000, D, offset=100.0)
    plain = DeviceDatabase(db, "cpu")
    split = DeviceDatabase(db, "cpu", lo=True)
    assert plain.Kl is None and plain.Vtl is None and not plain.has_lo and split.has_lo
    assert torch.equal(split.Kh, plain.Kh) and torch.equal(split.Vt, plain.Vt)       # the fp16 path reads the same bits
    assert split.Kl.shape == split.Kh.shape and split.Vtl.shape == split.Vt.shape
    assert split.nbytes() == plain.nbytes() + split.Kl.numel() * 2 + split.Vtl.numel() * 2
    rows = split.order[: split.M]
    K = db["satclip_embeddings"][rows].astype(np.float32)
    K = K / np.linalg.norm(K, axis=1, keepdims=True)
    kh, kl = split.Kh[: split.M].double().numpy(), split.Kl[: split.M].double().numpy()
    assert (np.abs(kh + kl - K) <= _lo_bound(K, kh)).all()
    V = db["image_embeddings"][rows].astype(np.float64) * split.vscale
    vh, vl = split.Vt[:D, : split.M].double().numpy().T, split.Vtl[:D, : split.M].double().numpy().T
    assert (np.abs(vh + vl - V) <= _lo_bound(V, vh)).all()
    # the split keeps 22 significant bits of the offset values: far below fp16's 2^-11 of the row
    assert np.abs(vh + vl - V).max() <= 2.0 ** -22 * np.abs(V).max()
    assert np.abs(vh - V).max() >= 2.0 ** -14 * np.abs(V).max()
    assert not split.Kl[split.M:].any() and not split.Vtl[:, split.M:].any() and not split.Vtl[D:].any()


def test_synthetic_lo_halves():
    from range_b200.database import DeviceDatabase
    a = DeviceDatabase.synthetic(3000, "cpu", seed=2, value_dim=300)
    b = DeviceDatabase.synthetic(3000, "cpu", seed=2, value_dim=300, lo=True)
    assert torch.equal(a.Kh, b.Kh) and torch.equal(a.Vt, b.Vt) and a.Kl is None
    assert b.Kl.abs().max() <= 2.0 ** -11 and b.Vtl[300:].abs().max() == 0


def test_cache_without_lo_is_rebuilt_for_a_split_model(tmp_path):
    """a cache written without lo halves does not satisfy f16x3 (from_cache -> None: the caller rebuilds and rewrites
    it); one with them serves both precisions"""
    from range_b200.database import DeviceDatabase
    db = _small_db(700, 64)
    fp = DeviceDatabase.source_fingerprint(db)
    path = str(tmp_path / "db.npz")
    DeviceDatabase(db, "cpu").save_cache(path, fingerprint=fp)
    assert DeviceDatabase.from_cache(path, "cpu", fingerprint=fp, lo=True) is None
    old = DeviceDatabase.from_cache(path, "cpu", fingerprint=fp)
    assert old is not None and old.Kl is None
    split = DeviceDatabase(db, "cpu", lo=True)
    split.save_cache(path, fingerprint=fp)
    back = DeviceDatabase.from_cache(path, "cpu", fingerprint=fp, lo=True)
    assert torch.equal(back.Kl, split.Kl) and torch.equal(back.Vtl, split.Vtl) and torch.equal(back.Kh, split.Kh)
    plain = DeviceDatabase.from_cache(path, "cpu", fingerprint=fp)          # an fp16 model reads the same file
    assert plain.Kl is None and torch.equal(plain.Vt, split.Vt)
    assert DeviceDatabase.from_cache(path, "cpu", fingerprint="other", lo=True) is None


class SplitEngine(TorchEngine):
    """the stand-in engine of tests/test_distributed.py with split-fp16 query rows: encode returns (N,512) [hi | lo],
    the logits use hi + lo"""
    q_cols = 512

    def encode(self, c):
        q, q16, qxyz = super().encode(c)
        return q, torch.cat([q16, (q - q16.double()).half()], 1), qxyz

    def _logits(self, q16, qxyz):
        assert q16.shape[1] == 512
        return (q16[:, :256].double() + q16[:, 256:].double()) @ self.K.t(), qxyz[:, :3].double() @ self.X.t()


def _gloo_worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from range_b200.distributed import ShardedRetriever, shard_rows
    from tests.test_distributed import TS, TG, BETA, D, _database, _encode
    M = 1001
    K, V, X = _database(M)
    lo, hi = shard_rows(M, rank, world)
    sr = ShardedRetriever(SplitEngine(K[lo:hi], V[lo:hi], X[lo:hi]), merge="reduce_scatter")
    sr.MAX_STEP_ROWS = 256 * world
    n = [300, 77][rank]
    rng = np.random.default_rng(10 + rank)
    coords = torch.tensor(np.stack([rng.uniform(-180, 180, n), rng.uniform(-90, 90, n)], 1))
    got = sr.embed("RANGE+", coords, TS, TG, BETA, True, out_dtype=torch.float64)
    q, xyz = _encode(coords)
    q2 = q.half().double() + (q - q.half().double()).half().double()          # hi + lo: what the split kernels see
    s, g = q2 @ K.t(), xyz.float().double() @ X.t()
    ref = (BETA * torch.softmax(TS * s, 1) + (1 - BETA) * torch.softmax(TG * g, 1)) @ V
    ok = got.shape == (n, D + 256) and torch.allclose(got[:, :D], ref, rtol=1e-9, atol=1e-11)
    ok = ok and torch.equal(got[:, D:], q)
    ret[rank] = bool(ok)
    dist.destroy_process_group()


def test_m_sharded_pipeline_gathers_split_rows_gloo():
    """ShardedRetriever gathers the engine's (N,512) [hi | lo] query rows (1 024 B per query) and hands them to every
    pass; the result matches the unsharded softmax of the hi + lo queries"""
    world = 2
    port = 31500 + os.getpid() % 2000
    ret = mp.Manager().dict()
    mp.spawn(_gloo_worker, args=(world, port, ret), nprocs=world, join=True)
    assert all(ret[r] for r in range(world))


# ---------------------------------------------------------------------------------------------------- GPU
MODELS = (("RANGE", None, 15.0), ("RANGE+", 0.0, 12.0), ("RANGE+", 0.5, 12.0), ("RANGE+", 1.0, 12.0))


def _enc(seed=1):
    ws = O.siren_init(40, 64, 2, 256, seed=seed)
    return ws, dict(L=40, dims=[1600, 64, 64, 256], weights=ws)


def _db(kind, M, ws, sh_entries, D=1024, seed=3):
    if kind == "structured":
        helper = O.RangeOracle.__new__(O.RangeOracle)
        helper.L, helper.entries, helper.weights = 40, sh_entries, ws
        db = O.synthetic_db(M, seed=seed, kind="structured", encoder=helper.encode)
    else:
        db = O.synthetic_db(M, seed=seed, kind="iid")
    if kind == "offset":
        db = dict(db, image_embeddings=(100.0 + np.random.default_rng(seed).standard_normal((M, D))).astype(np.float32))
    elif D != 1024:
        db = dict(db, image_embeddings=np.random.default_rng(D).standard_normal((M, D)).astype(np.float32))
    return db


def _engines(db, enc):
    from range_b200.database import DeviceDatabase
    from range_b200.engine import RangeEngine
    return (RangeEngine(DEV, encoder=enc, database=DeviceDatabase(db, DEV)),
            RangeEngine(DEV, encoder=enc, database=DeviceDatabase(db, DEV, lo=True), retrieval_precision="f16x3"))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["iid", "structured", "offset"])
def test_accuracy_against_fp64(kind, sh_entries):
    """relative row error <= 5e-5 against range/range.py:213-238 in fp64 on the same (fp64-encoded) queries, for RANGE
    and RANGE+ at beta 0, 0.5, 1 (the queries are the engine's: the reference's harmonics carry their own ~1e-5 noise,
    DESIGN.md section 2, which would hide the retrieval's error); the location columns are bit-identical to fp16 mode.
    Offset database (V = 100 + N(0,1)): the error of the part a probe sees (the rows minus the database mean) exceeds
    1e-2 with fp16 operands (measured on the B200: 1.7e-1) and is at most half that with split operands (measured 5.2e-2,
    not the 1e-4 a CPU emulation without the accumulator's truncation predicts: the split rows are within 4.2e-6 of fp64,
    the floor of the truncating tensor-core accumulation of positive values, DESIGN.md section 2, and centring these
    near-flat rows amplifies that ~1e4 times)"""
    N, M = 256, 20_000
    ws, enc = _enc()
    db = _db(kind, M, ws, sh_entries)
    e16, e3 = _engines(db, enc)
    c = O.area_uniform(N, np.random.default_rng(11))
    q64, q16, qxyz = e16.encode(torch.tensor(c))
    q64b, q16x2, qxyzb = e3.encode(torch.tensor(c))
    assert torch.equal(q64, q64b) and torch.equal(q16x2[:, :256], q16) and torch.equal(qxyz, qxyzb)
    center = np.asarray(db["image_embeddings"], np.float64).mean(0) if kind == "offset" else 0.0
    report = []
    for name, beta, temp in MODELS:
        ref = _fp64_retrieval(db, e3.db, q64.cpu().numpy(), c, name, beta, temp)
        o3 = e3.retrieve_concat(name, q16x2, qxyz, temp, 40.0, beta, q64)
        o16 = e16.retrieve_concat(name, q16, qxyz, temp, 40.0, beta, q64)
        assert torch.equal(o3[:, 1024:], o16[:, 1024:])
        r3 = rel_rows(o3[:, :1024].cpu().numpy(), ref).max()
        r16 = rel_rows(o16[:, :1024].cpu().numpy(), ref).max()
        report.append((name, beta, r16, r3))
        assert r3 <= 5e-5, report
        if kind == "offset":
            c3 = rel_rows(o3[:, :1024].cpu().numpy(), ref, center).max()
            c16 = rel_rows(o16[:, :1024].cpu().numpy(), ref, center).max()
            report.append(("centred", name, beta, c16, c3))
            assert c16 > 1e-2 and c3 <= 0.5 * c16, report
    print(kind, report)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [64, 100, 768, 1024, 2048])
def test_entry_points_agree(D, sh_entries):
    """model(locs), embed_into, embed_sweep, embed_raster / forward_raster and embed in f16x3 mode on the same
    coordinates agree; embed is within 5e-5 of the fp64 restatement"""
    from range_b200.range import LocationEncoder
    ws, enc = _enc(2)
    M = 6000
    db = _db("structured", M, ws, sh_entries, D=D)
    m = LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=enc, device=DEV, range_db=db, beta=0.5,
                                  retrieval_precision="f16x3"))
    assert m.args.retrieval_precision == "f16x3" and m.engine.q_cols == 512
    lon, lat = m.coord_grid_axes((12, 24))
    grid = torch.stack(torch.meshgrid(lat, lon, indexing="ij")[::-1], -1).reshape(-1, 2)
    emb = m.embed(grid.to(DEV), out_dtype=torch.float64).cpu().numpy()
    assert emb.shape == (grid.shape[0], D + 256)
    c = grid.numpy()[::7]
    ref = _fp64_retrieval(db, m.engine.db, emb[::7, D:], c, "RANGE+", 0.5, 12.0)
    assert rel_rows(emb[::7, :D], ref).max() <= 5e-5
    tol = 1e-5                                             # other batches: other query tiles, other geo-skip masks
    assert rel_rows(m(grid.numpy())[:, :D], emb[:, :D]).max() <= tol
    into = np.empty_like(emb)
    m.embed_into(grid.numpy(), into)
    assert rel_rows(into[:, :D], emb[:, :D]).max() <= tol
    ras = m.embed_raster(lon, lat, out_dtype=torch.float64).cpu().numpy()
    assert rel_rows(ras[:, :D], emb[:, :D]).max() <= tol and np.array_equal(ras[:, D:], emb[:, D:])
    assert rel_rows(m.forward_raster(lon, lat)[:, :D], emb[:, :D]).max() <= tol
    sweep = m.embed_sweep(grid.to(DEV), [0.5], out_dtype=torch.float64)[0].cpu().numpy()
    assert rel_rows(sweep[:, :D], emb[:, :D]).max() <= 1e-4


@pytest.mark.gpu
def test_several_accumulation_windows_keep_the_mass(sh_entries):
    """a database of 313 tiles (longer than one 256-tile accumulation window) with V = 1: every retrieved value is 1; the
    split mode's deficit is no worse than fp16 mode's"""
    ws, enc = _enc()
    M = 40_000
    db = dict(_db("iid", M, ws, sh_entries), image_embeddings=np.ones((M, 1024), np.float32))
    e16, e3 = _engines(db, enc)
    c = torch.tensor(O.area_uniform(1000, np.random.default_rng(5)))
    q64, q16, qxyz = e16.encode(c)
    _, q16x2, _ = e3.encode(c)
    for name, beta, temp in MODELS:
        d16 = (1.0 - e16.retrieve(name, q16, qxyz, temp, 40.0, beta)).abs().max().item()
        d3 = (1.0 - e3.retrieve(name, q16x2, qxyz, temp, 40.0, beta)).abs().max().item()
        assert d3 <= max(d16, 1e-6), (name, beta, d16, d3)


def _fp64_retrieval(db, ddb, q64, c, name, beta, temp):
    """range/range.py:213-238 in fp64 for the queries q64 (N,256) at coordinates c: the retrieved (N, D) rows"""
    rows = ddb.order[: ddb.M]
    return _fp64_weights(db, ddb, q64, c, name, beta, temp) @ np.asarray(db["image_embeddings"], np.float64)[rows]


def _fp64_weights(db, ddb, q64, c, name, beta, temp):
    """(N, M) fp64 retrieval weights of range/range.py:213-238 over the device rows of ddb"""
    from range_b200.utils import rad_to_cart
    rows = ddb.order[: ddb.M]
    K = db["satclip_embeddings"][rows].astype(np.float32)
    K = (K / np.linalg.norm(K, axis=1, keepdims=True)).astype(np.float64)
    s = q64 @ K.T
    ws = np.exp(temp * (s - s.max(1, keepdims=True)))
    ws /= ws.sum(1, keepdims=True)
    if name == "RANGE":
        return ws
    X = rad_to_cart(db["locs"][rows].astype(np.float32) * np.float32(np.pi / 180)).astype(np.float64)
    Q = rad_to_cart(c.astype(np.float32) * np.float32(np.pi / 180)).astype(np.float64)
    g = Q @ X.T
    wg = np.exp(40.0 * (g - g.max(1, keepdims=True)))
    wg /= wg.sum(1, keepdims=True)
    return beta * ws + (1 - beta) * wg


@pytest.mark.gpu
def test_neighbours_against_fp64(sh_entries):
    """neighbour weights within 2e-5 relative of the fp64 weights (measured on the B200: 1.2e-5 for RANGE; a bound of
    1e-6 is out of reach - every logit is the sum of 48 truncating tensor-core accumulator updates, 16 in fp16 mode,
    DESIGN.md section 2).  The index sets are the fp64 ones wherever the k-th and (k+1)-th fp64 weights differ by more
    than 1e-5 relative."""
    ws, enc = _enc()
    M, N, k = 8000, 256, 8
    db = _db("structured", M, ws, sh_entries)
    _, e3 = _engines(db, enc)
    c = O.area_uniform(N, np.random.default_rng(7))
    q64, q16x2, qxyz = e3.encode(torch.tensor(c))
    for name, beta, temp in MODELS:
        sums, _ = e3.retrieve_stats(name, q16x2, qxyz, temp, 40.0)
        idx, w = e3.retrieve_topk(name, q16x2, qxyz, temp, 40.0, beta, sums, k)
        W = _fp64_weights(db, e3.db, q64.cpu().numpy(), c, name, beta, temp)
        idx, w = idx.cpu().numpy(), w.cpu().numpy().astype(np.float64)
        got = np.take_along_axis(W, idx, 1)
        assert (np.abs(w - got) <= 2e-5 * got).all(), (name, beta, np.abs(w / got - 1).max())
        print(name, beta, "max relative weight error", np.abs(w / got - 1).max())
        top = -np.sort(-W, 1)[:, : k + 1]
        clear = top[:, k - 1] - top[:, k] > 1e-5 * top[:, k - 1]
        want = np.argsort(-W, 1, kind="stable")[:, :k]
        for n in np.flatnonzero(clear):
            assert set(idx[n]) == set(want[n]), (name, beta, n)


@pytest.mark.gpu
def test_three_shards_emulated_match_unsharded(sh_entries):
    """three shards in f16x3 mode on one device: summed statistics, summed apply passes (embed and both ends of a beta
    sweep), shard top-k lists in global rows merged - against the unsharded f16x3 model"""
    from range_b200.database import DeviceDatabase
    from range_b200.engine import RangeEngine
    ws, enc = _enc(2)
    M = 9000
    db = _db("structured", M, ws, sh_entries)
    whole = RangeEngine(DEV, encoder=enc, database=DeviceDatabase(db, DEV, lo=True), retrieval_precision="f16x3")
    shards = [RangeEngine(DEV, encoder=enc, database=DeviceDatabase(db, DEV, shard=(r, 3), lo=True),
                          retrieval_precision="f16x3") for r in range(3)]
    c = torch.tensor(O.area_uniform(700, np.random.default_rng(9)))
    q64, q16x2, qxyz = whole.encode(c)
    for name, beta, temp in (("RANGE+", 0.5, 12.0), ("RANGE+", 0.0, 12.0), ("RANGE", None, 12.0)):
        stats = [s.retrieve_stats(name, q16x2, qxyz, temp, 40.0) for s in shards]
        sums = torch.stack([a for a, _ in stats]).sum(0)
        merged = sum(s.retrieve_apply(name, q16x2, qxyz, temp, 40.0, beta, sums, m)
                     for s, (_, m) in zip(shards, stats)).cpu().numpy()
        full = whole.retrieve(name, q16x2, qxyz, temp, 40.0, beta).cpu().numpy()
        assert rel_rows(merged, full).max() <= 1e-5, (name, beta)
        parts = [s.retrieve_topk_rows(name, q16x2, qxyz, temp, 40.0, beta, sums, 8, s.db.row_range[0]) for s in shards]
        mi, mw = whole.topk_merge(torch.stack([w for _, w in parts]).contiguous(),
                                  torch.stack([i for i, _ in parts]).contiguous())
        wsum, _ = whole.retrieve_stats(name, q16x2, qxyz, temp, 40.0)
        wi, ww = whole.retrieve_topk(name, q16x2, qxyz, temp, 40.0, beta, wsum, 8)
        assert torch.allclose(mw, ww, rtol=1e-5, atol=0)
        same = (mi == wi).float().mean().item()
        assert same >= 0.99, (name, beta, same)


@pytest.mark.gpu
def test_c_abi_errors_and_query_split(sh_entries):
    from range_b200 import _lib
    from range_b200.database import DeviceDatabase
    from range_b200.engine import RangeEngine
    ws, enc = _enc()
    db = _db("iid", 3000, ws, sh_entries)
    eng = RangeEngine(DEV, encoder=enc, database=DeviceDatabase(db, DEV))
    lib = eng.lib
    assert lib.range_ctx_set_retrieval_precision(eng.ctx, _lib.RANGE_RET_F16X3) == -1       # RANGE_ERR_INVALID
    assert b"range_ctx_set_db_lo" in lib.range_last_error()
    assert lib.range_ctx_set_retrieval_precision(eng.ctx, 7) != 0
    with pytest.raises(ValueError, match="lo halves"):
        RangeEngine(DEV, encoder=enc, database=DeviceDatabase(db, DEV), retrieval_precision="f16x3")
    e3 = RangeEngine(DEV, encoder=enc, database=DeviceDatabase(db, DEV, lo=True), retrieval_precision="f16x3")
    c = torch.tensor(O.area_uniform(300, np.random.default_rng(1)))
    q64, q16, qxyz = eng.encode(c)
    with pytest.raises(ValueError, match=r"\(N,512\)"):
        e3.retrieve_stats("RANGE", q16, qxyz, 15.0, 0.0)                 # fp16 rows handed to a split ctx
    with pytest.raises(ValueError, match=r"\(N,256\)"):
        eng.retrieve_stats("RANGE", e3.split_queries(q64), qxyz, 15.0, 0.0)
    # the workspace functions size for the mode: a large batch runs the chunked single-role apply in f16x3
    N = 30_000
    ws16 = lib.range_retrieve_workspace_bytes(eng.ctx, N)
    ws3 = lib.range_retrieve_workspace_bytes(e3.ctx, N)
    assert ws16 > 0 and ws3 > 0 and ws16 != ws3
    # range_split_queries: the hi half is range_encode's q16 bit for bit, hi + lo within 2^-11 of the residual
    x2 = e3.split_queries(q64)
    assert torch.equal(x2[:, :256], q16)
    q = q64.cpu().numpy()
    hi, lo = x2[:, :256].double().cpu().numpy(), x2[:, 256:].double().cpu().numpy()
    assert (np.abs(hi + lo - q) <= 2.0 ** -11 * np.abs(q - hi) + 2.0 ** -25).all()
    # clearing the lo halves returns the ctx to fp16
    assert lib.range_ctx_set_db_lo(e3.ctx, None, None) == 0
    assert lib.range_ctx_set_retrieval_precision(e3.ctx, _lib.RANGE_RET_F16X3) != 0
