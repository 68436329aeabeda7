"""One model on several GPUs of a host (load_model(..., devices=...)): the rows of every call split into slabs over
database replicas, each slab computed by the unchanged single-device code.

CPU: the slab planner, argument errors raised before any CUDA call.  GPU, one B200: three replicas on GPU 0
(devices=[0, 0, 0]) against single-device calls on the planner's slabs, byte for byte, for every entry point.  GPU, two
or more B200: devices=[0, 1]."""
from argparse import Namespace

import numpy as np
import pytest
import torch

from oracle import range_oracle as O

ROUND = 24 * 256


# ------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("n_devices", [1, 2, 3, 8])
@pytest.mark.parametrize("N", [0, 1, 2 * ROUND - 1, 2 * ROUND, 3 * ROUND + 17, 40_000, 100_003, 10_000_000])
def test_split_rows(N, n_devices):
    from range_b200.devices import split_rows
    from range_b200.range import ROUND_ROWS
    assert ROUND_ROWS == ROUND
    cuts = split_rows(N, n_devices)
    assert cuts[0][0] == 0 and cuts[-1][1] == N
    assert all(a[1] == b[0] for a, b in zip(cuts, cuts[1:]))                # contiguous, in order
    assert all(hi > lo for lo, hi in cuts) or cuts == [(0, 0)]
    sizes = [hi - lo for lo, hi in cuts]
    if N < 2 * ROUND or n_devices == 1:
        assert cuts == [(0, N)]
        return
    assert len(cuts) == min(n_devices, N // ROUND)
    assert all(s % ROUND == 0 for s in sizes[1:])                          # whole rounds but the first
    assert sizes[0] - N % ROUND == sizes[0] // ROUND * ROUND                # the ragged rows go to the first slab
    rounds = [s // ROUND for s in sizes]
    assert max(rounds) - min(rounds) <= 1 and max(sizes) - min(sizes) <= ROUND


def test_split_rows_examples():
    from range_b200.devices import split_rows
    assert split_rows(100_003, 8) == [(0, 2 * ROUND + 1699)] + [(2 * ROUND + 1699 + i * 2 * ROUND,
                                                                  2 * ROUND + 1699 + (i + 1) * 2 * ROUND) for i in range(7)]
    assert split_rows(100_003, 3) == [(0, 5 * ROUND + 1699), (5 * ROUND + 1699, 10 * ROUND + 1699),
                                      (10 * ROUND + 1699, 100_003)]
    assert split_rows(3 * ROUND + 17, 8) == [(0, ROUND + 17), (ROUND + 17, 2 * ROUND + 17), (2 * ROUND + 17, 3 * ROUND + 17)]


@pytest.fixture
def no_cuda(monkeypatch):
    """every way the constructor could reach a device or read the checkpoint / database fails the test"""
    import range_b200.range as R

    def boom(*a, **k):
        raise AssertionError("reached CUDA or the model's files before rejecting its arguments")
    for name in ("device_count", "is_available", "current_device", "init"):
        monkeypatch.setattr(torch.cuda, name, boom)
    for name in ("RangeEngine", "load_satclip_location_encoder", "open_npz"):
        monkeypatch.setattr(R, name, boom)
    for name in ("__init__", "from_cache", "synthetic"):
        monkeypatch.setattr(R.DeviceDatabase, name, boom)


@pytest.mark.parametrize("kw", [dict(devices=[0], db_shard=(0, 2)), dict(devices=2, db_shard=(1, 2)),
                                dict(devices=[]), dict(devices=["cpu"]), dict(devices=[0, "cpu"]),
                                dict(devices=0), dict(devices="cuda:0")])
def test_device_argument_errors(kw, no_cuda):
    from range_b200.load_model import load_model
    from range_b200.range import LocationEncoder
    with pytest.raises(ValueError, match="devices"):
        load_model("RANGE+", pretrained_path="unused.ckpt", db_path="unused.npz", **kw)
    with pytest.raises(ValueError, match="devices"):
        LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path="unused.ckpt", device="cuda",
                                  range_db="unused.npz", beta=0.5, **kw))


# ------------------------------------------------------------------------------------------------------------- GPU
M = 20_077
SIZES = [0, 1, ROUND - 1, 3 * ROUND + 17, 40_000]
DUP = [0, 0, 0]


def _enc(seed=0):
    return dict(L=40, dims=[1600, 256, 256, 256], weights=O.siren_init(40, 256, 2, 256, seed=seed))


@pytest.fixture(scope="module")
def setup():
    from range_b200.database import DeviceDatabase
    enc = _enc()
    ddb = DeviceDatabase.synthetic(M, "cuda:0", seed=5)
    models = {}

    def model(devices=None, db=ddb, **kw):
        key = (tuple(devices or ()), id(db), tuple(sorted(kw.items())))
        if key not in models:
            from range_b200.range import LocationEncoder
            models[key] = LocationEncoder(Namespace(location_model_name="RANGE+", pretrained_path=enc, device="cuda:0",
                                                    range_db=db, beta=0.5, devices=devices, **kw))
        return models[key]
    yield model
    for m in models.values():
        m.close()


def _coords(N, seed=0):
    return torch.tensor(O.area_uniform(N, np.random.default_rng(1000 + N + seed)))


def _slabs(N, n):
    from range_b200.devices import split_rows
    return split_rows(N, n)


def _same(a, b):
    a, b = (x.cpu().numpy() if torch.is_tensor(x) else x for x in (a, b))
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("N", SIZES)
def test_model_call_host_paths(setup, N, tmp_path):
    from range_b200.save import embed_to_npy
    c = _coords(N)
    slabs = _slabs(N, len(DUP))
    for kw in (dict(), dict(pinned_limit=0), dict(out_dtype=np.float32)):
        multi, single = setup(DUP, **kw), setup(None, **kw)
        got = multi(c)
        want = np.concatenate([single(c[lo:hi]) for lo, hi in slabs])
        assert _same(got, want), kw
    multi, single = setup(DUP), setup(None)
    got = np.full((N, 1280), np.nan)
    multi.embed_into(c, got)
    want = np.full((N, 1280), np.nan)
    for lo, hi in slabs:
        single.embed_into(c[lo:hi], want[lo:hi])
    assert _same(got, want)
    if N:
        assert _same(np.asarray(embed_to_npy(multi, c, str(tmp_path / "e.npy"))), want)
    # against one single-device call on the whole batch: the location columns are the same bits, the retrieved ones
    # agree to test_gpu_parity's bound for this path (the spatial batching groups other queries into tiles)
    whole = single(c)
    assert _same(got[:, 1024:], whole[:, 1024:])
    if N:
        r = np.linalg.norm(got[:, :1024] - whole[:, :1024], axis=1) / np.linalg.norm(whole[:, :1024], axis=1)
        assert r.max() <= 1e-3, r.max()


def _outcome(fn):
    """fn()'s result, or the type of the exception it raised"""
    try:
        return fn()
    except Exception as e:                      # noqa: BLE001 - compared, not swallowed
        return type(e)


@pytest.mark.gpu
def test_zero_rows_behave_like_one_device(setup):
    """a call of 0 rows runs on the primary alone: what it returns, or raises, is what the single-device call does"""
    multi, single = setup(DUP), setup(None)
    c = _coords(0).to("cuda:0")
    lon, lat = multi.coord_grid_axes((20, 40))
    calls = [lambda m: m(c.cpu()), lambda m: m.embed(c), lambda m: m.embed_sweep(c, [0.0, 1.0]),
             lambda m: m.neighbours(c, k=8), lambda m: m.embed_raster(lon, lat, rows=(5, 5)),
             lambda m: m.forward_raster(lon, lat, rows=(5, 5))]
    for call in calls:
        a, b = _outcome(lambda: call(multi)), _outcome(lambda: call(single))
        if isinstance(a, type) or isinstance(b, type):
            assert a is b
        else:
            a, b = (x if isinstance(x, (list, tuple)) else [x] for x in (a, b))
            assert len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))


@pytest.mark.gpu
@pytest.mark.parametrize("N", SIZES[1:])
def test_device_entry_points(setup, N):
    multi, single = setup(DUP), setup(None)
    c = _coords(N, seed=1).to("cuda:0")
    slabs = _slabs(N, len(DUP))
    got = multi.embed(c)
    assert got.device == torch.device("cuda:0") and got.dtype == torch.float32
    assert _same(got, torch.cat([single.embed(c[lo:hi]) for lo, hi in slabs]))
    out = torch.full((N, 1280), float("nan"), dtype=torch.float64, device="cuda:0")
    assert multi.embed(c, out=out) is out
    assert _same(out, torch.cat([single.embed(c[lo:hi], out_dtype=torch.float64) for lo, hi in slabs]))
    whole = single.embed(c)
    assert _same(got[:, 1024:], whole[:, 1024:])
    betas = [0.0, 0.5, 1.0]
    sweep = multi.embed_sweep(c, betas)
    parts = [single.embed_sweep(c[lo:hi], betas) for lo, hi in slabs]
    assert len(sweep) == 3 and all(s.device == torch.device("cuda:0") for s in sweep)
    for b in range(3):
        assert _same(sweep[b], torch.cat([p[b] for p in parts])), betas[b]
    idx, w = multi.neighbours(c, k=8)
    ref = [single.neighbours(c[lo:hi], k=8) for lo, hi in slabs]
    assert idx.device == torch.device("cuda:0") and idx.dtype == torch.int64
    assert _same(idx, torch.cat([r[0] for r in ref])) and _same(w, torch.cat([r[1] for r in ref]))


@pytest.mark.gpu
@pytest.mark.parametrize("N", SIZES[1:])
def test_raster_entry_points(setup, N):
    multi, single = setup(DUP), setup(None)
    lon, lat = multi.coord_grid_axes((200, 400))
    p0 = 1234
    slabs = _slabs(N, len(DUP))
    got = multi.embed_raster(lon, lat, rows=(p0, p0 + N))
    assert _same(got, torch.cat([single.embed_raster(lon, lat, rows=(p0 + lo, p0 + hi)) for lo, hi in slabs]))
    host = multi.forward_raster(lon, lat, rows=(p0, p0 + N))
    assert _same(host, np.concatenate([single.forward_raster(lon, lat, rows=(p0 + lo, p0 + hi)) for lo, hi in slabs]))
    out = np.full((N, 1280), np.nan)
    multi.forward_raster(lon, lat, rows=(p0, p0 + N), out=out)
    assert _same(out, host)


@pytest.mark.gpu
def test_other_value_width_and_split_precision(setup):
    from range_b200.database import DeviceDatabase
    N = 3 * ROUND + 17
    c = _coords(N, seed=2)
    slabs = _slabs(N, len(DUP))
    for db, kw in ((DeviceDatabase.synthetic(M, "cuda:0", seed=6, value_dim=768), dict()),
                   (DeviceDatabase.synthetic(M, "cuda:0", seed=7, lo=True), dict(retrieval_precision="f16x3"))):
        multi, single = setup(DUP, db=db, **kw), setup(None, db=db, **kw)
        W = db.value_dim + 256
        got = multi(c)
        assert got.shape == (N, W)
        assert _same(got, np.concatenate([single(c[lo:hi]) for lo, hi in slabs]))
        dc = c.to("cuda:0")
        assert _same(multi.embed(dc), torch.cat([single.embed(dc[lo:hi]) for lo, hi in slabs]))


@pytest.mark.gpu
def test_replicas_hold_the_primary_bytes(setup):
    from range_b200.database import DeviceDatabase
    db = DeviceDatabase.synthetic(M, "cuda:0", seed=7, lo=True)
    multi = setup(DUP, db=db, retrieval_precision="f16x3")
    reps = multi.replicas.models
    assert len(reps) == 3 and reps[0].engine is multi.engine
    for r in reps[1:]:
        rdb = r.engine.db
        assert rdb is not db and r.engine is not multi.engine
        for name in ("Kh", "Vt", "xyz", "caps", "Kl", "Vtl"):
            a, b = getattr(db, name), getattr(rdb, name)
            assert a.data_ptr() != b.data_ptr() and _same(a, b), name
        assert rdb.order is db.order and (rdb.M, rdb.Mpad, rdb.M_total, rdb.vscale, rdb.value_dim, rdb.row_range) == \
            (db.M, db.Mpad, db.M_total, db.vscale, db.value_dim, db.row_range)


@pytest.mark.gpu
def test_small_batches_and_close_run_on_the_primary(setup):
    from range_b200 import _lib
    from range_b200.database import DeviceDatabase
    db = DeviceDatabase.synthetic(M, "cuda:0", seed=8)
    multi, single = setup(DUP, db=db), setup(None, db=db)
    c = _coords(2 * ROUND - 1, seed=3).to("cuda:0")
    before = _lib.launch_count()
    a = multi.embed(c)
    launches = _lib.launch_count() - before
    before = _lib.launch_count()
    b = single.embed(c)
    assert _lib.launch_count() - before == launches and _same(a, b)
    multi.close()
    assert multi.replicas is None
    big = _coords(3 * ROUND, seed=4).to("cuda:0")
    assert _same(multi.embed(big), single.embed(big))


@pytest.mark.gpu
def test_an_error_on_one_replica_is_raised_after_the_others(setup):
    import threading
    from range_b200.database import DeviceDatabase
    multi = setup(DUP, db=DeviceDatabase.synthetic(M, "cuda:0", seed=9))
    slabs = _slabs(3 * ROUND, len(DUP))
    ran = []

    def work(i, m, lo, hi):
        ran.append(i)
        if i == 1:
            raise RuntimeError(f"slab {i}")
        return hi - lo
    threads = threading.active_count()
    with pytest.raises(RuntimeError, match="slab 1"):
        multi.replicas.run(slabs, work)
    assert ran == [0, 1] and threading.active_count() == threads
    with pytest.raises(ValueError, match="k="):
        multi.neighbours(_coords(3 * ROUND).to("cuda:0"), k=0)
    assert multi.replicas.run(slabs, lambda i, m, lo, hi: (i, m.engine.device)) == \
        [(i, torch.device("cuda:0")) for i in range(3)]


two_gpus = pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2,
                              reason="needs two GPUs")


@pytest.mark.gpu
@two_gpus
@pytest.mark.parametrize("N", [3 * ROUND + 17, 40_000])
def test_two_gpus(setup, N):
    import threading
    multi, single = setup([0, 1]), setup(None)
    c = _coords(N, seed=5)
    slabs = _slabs(N, 2)
    assert len(slabs) == 2
    assert _same(multi(c), np.concatenate([single(c[lo:hi]) for lo, hi in slabs]))
    dc = c.to("cuda:0")
    got = multi.embed(dc)
    assert got.device == torch.device("cuda:0")
    assert _same(got, torch.cat([single.embed(dc[lo:hi]) for lo, hi in slabs]))
    threads = threading.active_count()
    assert _same(multi.embed(dc), got)                                      # a repeat call: the same bits
    assert threading.active_count() == threads                              # no worker outlives the call
    idx, w = multi.neighbours(dc, k=8)
    ref = [single.neighbours(dc[lo:hi], k=8) for lo, hi in slabs]
    assert idx.device == torch.device("cuda:0")
    assert _same(idx, torch.cat([r[0] for r in ref])) and _same(w, torch.cat([r[1] for r in ref]))
