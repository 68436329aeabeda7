"""Databases whose values have a width D other than SatMAE's 1024 columns (range/range.py:213-240 is width-agnostic:
softmax(...) @ V, then np.concatenate): results are (N, D + 256) rows on every unsharded path.

CPU: the device layout (Vt padded to whole 256-row value slices), argument errors, the disk cache's width, the host
unpack of packed rows, the sharded-width error.  GPU: every public path against the exact oracle and against each other,
the padding rows never showing, the query chunking that bounds the apply workspace, C ABI errors."""
import ctypes
from argparse import Namespace

import numpy as np
import pytest
import torch

from oracle import range_oracle as O

DEV = "cuda:0"


def _db(M, D, seed=3, probabilities=False):
    """iid N(0,1) keys and values; probabilities=True: values are a class-probability table (rows of non-negative
    values summing to 1)"""
    rng = np.random.default_rng(seed)
    V = rng.standard_normal((M, D))
    if probabilities:
        V = np.exp(V) / np.exp(V).sum(1, keepdims=True)
    return dict(locs=O.area_uniform(M, rng), satclip_embeddings=rng.standard_normal((M, 256)), image_embeddings=V)


def _round256(D):
    return (D + 255) // 256 * 256


# ------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("D", [1, 10, 257, 768, 2048])
def test_layout_of_any_value_width(D):
    from range_b200.database import DeviceDatabase, prepare_reference_arrays
    M = 700
    db = _db(M, D)
    V = prepare_reference_arrays(db)[1]
    for kw in (dict(), dict(spatial_sort=False), dict(shard=(1, 3))):
        d = DeviceDatabase(db, "cpu", **kw)
        lo, hi = d.row_range
        rows = d.order[lo:hi] if d.order is not None else np.arange(lo, hi)
        assert d.value_dim == D and d.Vt.shape == (_round256(D), d.Mpad) and d.Vt.dtype == torch.float16
        assert not d.Vt[D:].any() and not d.Vt[:, d.M:].any()                  # padding rows and columns are zero
        assert torch.equal(d.Vt[:D, :d.M].t().contiguous(), (torch.from_numpy(V[rows]) * d.vscale).half())


def test_value_width_errors():
    from range_b200.database import DeviceDatabase
    for bad in (np.zeros((50, 0)), np.zeros((50, 4097)), np.zeros((50, 4, 4))):
        db = _db(50, 8)
        db["image_embeddings"] = bad
        with pytest.raises(ValueError, match="4096"):
            DeviceDatabase(db, "cpu")
    with pytest.raises(ValueError, match="4096"):
        DeviceDatabase.synthetic(100, "cpu", value_dim=4097)


def test_cache_records_the_width(tmp_path):
    from range_b200.database import DeviceDatabase
    d = DeviceDatabase(_db(300, 257), "cpu")
    path = d.save_cache(tmp_path / "c.npz", fingerprint="x")
    back = DeviceDatabase.from_cache(path, "cpu", fingerprint="x", value_dim=257)
    assert back.value_dim == 257 and torch.equal(back.Vt, d.Vt) and torch.equal(back.Kh, d.Kh)
    assert DeviceDatabase.from_cache(path, "cpu", fingerprint="x").value_dim == 257
    assert DeviceDatabase.from_cache(path, "cpu", fingerprint="x", value_dim=1024) is None     # another width: rebuilt
    # a cache written before the width was recorded holds 1024-wide values and still loads
    d1 = DeviceDatabase(_db(300, 1024), "cpu")
    p1 = d1.save_cache(tmp_path / "old.npz")
    z = dict(np.load(p1))
    del z["value_dim"]
    np.savez(p1, **z)
    old = DeviceDatabase.from_cache(p1, "cpu", value_dim=1024)
    assert old.value_dim == 1024 and torch.equal(old.Vt, d1.Vt)
    assert DeviceDatabase.from_cache(p1, "cpu", value_dim=768) is None


def _packed(f, q):
    """packed rows (include/range_b200.h: RANGE_OUT_PACKED): D fp32 padded to a multiple of 4, then 256 fp64"""
    N, D = f.shape
    Dr = (D + 3) // 4 * 4
    p = np.zeros((N, 4 * Dr + 2048), np.uint8)
    p[:, :4 * D] = f.view(np.uint8).reshape(N, 4 * D)
    p[:, 4 * Dr:] = q.view(np.uint8).reshape(N, 2048)
    return p


@pytest.mark.parametrize("D", [10, 257, 768, 1024])
def test_host_unpack_rows(D):
    """range_host_unpack_rows is a HOST entry point: exact, any thread count, aligned (AVX2 when D % 4 == 0) or not"""
    from range_b200 import _lib
    from range_b200.engine import packed_row_bytes
    lib = _lib.load()
    rng = np.random.default_rng(D)
    for N in (0, 1, 300, 1000):
        f = rng.standard_normal((N, D)).astype(np.float32)
        q = rng.standard_normal((N, 256))
        packed = _packed(f, q)
        assert packed.shape[1] == packed_row_bytes(D)
        want = np.concatenate([f.astype(np.float64), q], axis=1)
        for threads in (1, 3):
            for off in (0, 1):
                buf = np.full(N * (D + 256) + 1, np.nan)
                out = buf[off:off + N * (D + 256)].reshape(N, D + 256)
                assert lib.range_host_unpack_rows(packed.ctypes.data if N else None, N, D,
                                                  out.ctypes.data if N else None, threads) == 0
                assert np.array_equal(out, want)
                if D == 1024:
                    old = np.full_like(out, np.nan)
                    assert lib.range_host_unpack(packed.ctypes.data if N else None, N, old.ctypes.data if N else None,
                                                 threads) == 0
                    assert np.array_equal(old, out)
    assert packed_row_bytes(1024) == 6144
    for bad in (0, 4097):
        assert lib.range_host_unpack_rows(None, 0, bad, None, 1) == _lib_err("INVALID")


def test_sharded_model_of_another_width_raises():
    from range_b200.range import LocationEncoder
    args = Namespace(location_model_name="RANGE+", pretrained_path=dict(L=40), device="cpu", range_db=_db(200, 10),
                     beta=0.5, db_shard=(0, 2))
    with pytest.raises(NotImplementedError, match="1024"):
        LocationEncoder(args)


def test_new_symbols_in_prototypes():
    from range_b200 import _lib
    assert "range_ctx_set_db_values" in _lib.PROTOTYPES and "range_host_unpack_rows" in _lib.PROTOTYPES
    assert _lib.RANGE_MAX_VALUE_DIM == 4096


# ------------------------------------------------------------------------------------------------------------- GPU
def _tol():
    from tests.test_gpu_parity import TOL_Q, TOL_Q_POLAR, cos_rows, rel_rows, tol_o
    return tol_o, rel_rows, cos_rows, TOL_Q, TOL_Q_POLAR


def _model(name, ddb, ws, beta=0.5, **kw):
    from range_b200.range import LocationEncoder
    H = ws[0][0].shape[0]
    enc = dict(L=40, dims=[1600, H, H, 256], weights=ws)
    return LocationEncoder(Namespace(location_model_name=name, pretrained_path=enc, device=DEV, range_db=ddb,
                                     beta=beta, **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1_000, 20_077])
@pytest.mark.parametrize("D", [10, 257, 768, 2048])
def test_embed_vs_exact_oracle(D, M, sh_entries):
    """embed for RANGE and RANGE+ at beta 0 / 0.5 / 1, N 1 / 300 / 20 000 (a 1024-wide database takes the
    producer/consumer kernel there), sorted and unsorted database rows, against the fp64 oracle.  D = 10 is a
    class-probability table: with iid zero-mean values over only 10 columns a row's relative error is a ratio of 10-d
    norms, whose tail exceeds the bound measured over 1024 columns (2.4e-3 for RANGE's flat semantic softmax)"""
    from range_b200.database import DeviceDatabase
    tol_o, rel_rows, cos_rows, TOL_Q, TOL_Q_POLAR = _tol()
    db = _db(M, D, seed=D, probabilities=D == 10)
    ws = O.siren_init(40, 64, 2, 256, seed=1)
    cases = [("RANGE", None), ("RANGE+", 0.0), ("RANGE+", 0.5), ("RANGE+", 1.0)]
    coords = {N: O.area_uniform(N, np.random.default_rng(N)) for N in (1, 300, 20_000)}
    sub = {N: np.arange(N) if N <= 300 else np.linspace(0, N - 1, 96).astype(np.int64) for N in coords}
    refs = {(name, beta, N): O.RangeOracle(name, ws, sh_entries, db, beta=beta, exact=True)(coords[N][sub[N]])
            for name, beta in cases for N in coords}
    for sort in (True, False):
        ddb = DeviceDatabase(db, DEV, spatial_sort=sort)
        models = {name: _model(name, ddb, ws) for name in ("RANGE", "RANGE+")}
        assert all(m.location_feature_dim == D + 256 for m in models.values())
        for N, c in coords.items():
            dc = torch.tensor(c, device=DEV)
            q64 = models["RANGE"].engine.encode(dc)[0]
            for name, beta in cases:
                m = models[name]
                m.args.beta = beta
                out = m.embed(dc, out_dtype=torch.float64)
                assert out.shape == (N, D + 256) and torch.isfinite(out).all()
                assert torch.equal(out[:, D:], q64), (D, M, sort, N, name, beta)
                got = out[torch.from_numpy(sub[N]).to(DEV)].cpu().numpy()
                ref = refs[(name, beta, N)]
                r = rel_rows(got[:, :D], ref[:, :D])
                assert r.max() <= tol_o(name, beta) and cos_rows(got[:, :D], ref[:, :D]).min() >= 0.99999, \
                    (D, M, sort, N, name, beta, r.max())
                lat = np.abs(coords[N][sub[N], 1])
                dq = np.abs(got[:, D:] - ref[:, D:])
                assert dq[lat < 60].max(initial=0) <= TOL_Q and dq.max() <= TOL_Q_POLAR
        del models


@pytest.mark.gpu
@pytest.mark.parametrize("D", [10, 257, 768])
def test_every_public_path_returns_the_same_rows(D, tmp_path):
    """model(locs) on both host paths, out_dtype float32, embed_into a memory-mapped .npy, embed_raster / forward_raster:
    the rows of embed, bit for bit; two calls give the same bits"""
    from range_b200.database import DeviceDatabase
    from range_b200.range import LocationEncoder
    from range_b200.save import embed_to_npy
    db = _db(20_077, D, seed=7)
    ws = O.siren_init(40, 256, 2, 256, seed=0)          # tensor-core encoder: the separable raster encoder runs
    ddb = DeviceDatabase(db, DEV)
    N = 3000
    c = O.area_uniform(N, np.random.default_rng(3))
    m = _model("RANGE+", ddb, ws)
    ref = m.embed(torch.tensor(c, device=DEV), out_dtype=torch.float64).cpu().numpy()
    assert np.array_equal(ref, m.embed(torch.tensor(c, device=DEV), out_dtype=torch.float64).cpu().numpy())
    for path in ("copy", "packed"):
        mp = _model("RANGE+", ddb, ws, host_path=path)
        got = mp(c)
        assert got.dtype == np.float64 and got.shape == (N, D + 256) and np.array_equal(got, ref), path
        assert np.array_equal(mp(c), got)
    m32 = _model("RANGE+", ddb, ws, out_dtype=np.float32)
    assert np.array_equal(m32(c), ref.astype(np.float32))
    npy = embed_to_npy(m, c, str(tmp_path / "e.npy"))
    assert npy.shape == (N, D + 256) and np.array_equal(np.load(tmp_path / "e.npy"), ref)
    with pytest.raises(ValueError, match=str(D + 256)):
        m.embed_into(c, np.empty((N, 1280)))
    # rasters: the same rows as embed / model(locs) on the grid's coordinates
    H, W = 30, 61
    lon, lat = LocationEncoder.coord_grid_axes((H, W))
    assert m.engine.raster_supported()
    p = np.arange(H * W)
    pts = np.stack((lon.numpy()[p % W], lat.numpy()[p // W]), axis=1)
    want = m.embed(torch.tensor(pts, device=DEV), out_dtype=torch.float64)
    assert torch.equal(m.embed_raster(lon, lat, out_dtype=torch.float64), want)
    host = m.forward_raster(lon, lat)
    assert host.shape == (H * W, D + 256) and np.array_equal(host, m(pts))
    out = np.full((H * W, D + 256), np.nan)
    assert m.forward_raster(lon, lat, out=out) is out and np.array_equal(out, host)


@pytest.mark.gpu
def test_embed_sweep_of_another_width(sh_entries):
    from range_b200.database import DeviceDatabase
    tol_o, rel_rows, _, _, _ = _tol()
    D = 768
    db = _db(20_077, D, seed=11)
    ws = O.siren_init(40, 64, 2, 256, seed=1)
    m = _model("RANGE+", DeviceDatabase(db, DEV), ws)
    c = O.area_uniform(3000, np.random.default_rng(4))
    dc = torch.tensor(c, device=DEV)
    betas = [0.0, 0.3, 1.0]
    sweep = m.embed_sweep(dc, betas, out_dtype=torch.float64)
    sub = np.linspace(0, len(c) - 1, 64).astype(np.int64)
    for beta, o in zip(betas, sweep):
        assert o.shape == (len(c), D + 256)
        m.args.beta = beta
        one = m.embed(dc, out_dtype=torch.float64)
        assert torch.equal(o[:, D:], one[:, D:])
        assert rel_rows(o[:, :D].cpu().numpy(), one[:, :D].cpu().numpy()).max() <= 1e-3, beta
        ref = O.RangeOracle("RANGE+", ws, sh_entries, db, beta=beta, exact=True)(c[sub])
        assert rel_rows(o[torch.from_numpy(sub).to(DEV)][:, :D].cpu().numpy(), ref[:, :D]).max() <= tol_o("RANGE+", beta)


@pytest.mark.gpu
def test_neighbours_do_not_read_the_values():
    from range_b200.database import DeviceDatabase
    db = _db(5_000, 257, seed=5)
    wide = dict(db, image_embeddings=np.random.default_rng(1).standard_normal((5_000, 1024)))
    ws = O.siren_init(40, 64, 2, 256, seed=1)
    c = torch.tensor(O.area_uniform(2000, np.random.default_rng(6)), device=DEV)
    for name in ("RANGE", "RANGE+"):
        a = _model(name, DeviceDatabase(db, DEV), ws).neighbours(c, k=8)
        b = _model(name, DeviceDatabase(wide, DEV), ws).neighbours(c, k=8)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
@pytest.mark.parametrize("D", [257, 4096])
def test_no_mass_loss_and_no_padding_of_another_width(D):
    """V = 1 on the D real rows of Vt, padding rows zero, 300 000 entries: every output column stays 1 within the bound
    of test_gpu_parity.test_no_mass_loss_over_a_long_database_axis; D = 4096 runs the apply pass in query chunks (the
    split partials would be 3.3 GB in one piece)"""
    from range_b200 import _lib
    from range_b200.database import DeviceDatabase
    from range_b200.engine import RangeEngine
    M, N = 300_000, 20_000
    d = DeviceDatabase.synthetic(M, DEV, seed=3, value_dim=D)
    d.Vt.fill_(0)
    d.Vt[:D, :M] = d.vscale
    eng = RangeEngine(DEV, L=40, database=d)
    g = torch.Generator(device="cpu").manual_seed(1)
    q = torch.randn(N, 256, generator=g); q = (q / q.norm(dim=1, keepdim=True)).half().to(DEV)
    c = eng.sort_queries(torch.tensor(O.area_uniform(N, np.random.default_rng(1))))[0].cpu()
    xyz = torch.zeros(N, 4); xyz[:, :3] = torch.tensor(O.rad_to_cart(c.numpy() * np.pi / 180)).float(); xyz = xyz.to(DEV)
    q64 = torch.randn(N, 256, dtype=torch.float64, device=DEV)
    ws_bytes = eng.lib.range_retrieve_workspace_bytes(eng.ctx, N)
    assert ws_bytes <= (1 << 30) + N * 1024, ws_bytes
    for mode, beta, t in (("RANGE", None, 15.0), ("RANGE+", 0.5, 12.0)):
        O_ = eng.retrieve(mode, q, xyz, t, 40.0, beta)
        assert O_.shape == (N, D)
        dev = O_.double() - 1.0
        assert abs(dev.mean().item()) < 1e-4 and dev.abs().max().item() < 5e-4, (mode, dev.mean().item(), dev.abs().max().item())
        out = eng.retrieve_concat(mode, q, xyz, t, 40.0, beta, q64)
        assert out.shape == (N, D + 256) and torch.equal(out[:, :D].float(), O_) and torch.equal(out[:, D:], q64)
    assert _lib.RANGE_MAX_VALUE_DIM >= D


@pytest.mark.gpu
def test_capi_errors_of_another_width():
    from range_b200 import _lib
    from range_b200.database import DeviceDatabase
    from range_b200.engine import RangeEngine, _ptr, _stream
    d = DeviceDatabase(_db(3000, 257), DEV)
    eng = RangeEngine(DEV, L=40, database=d)
    lib = eng.lib
    for bad in (0, -1, 4097):
        assert lib.range_ctx_set_db_values(eng.ctx, d.M, d.Mpad, bad, _ptr(d.Kh), _ptr(d.Vt), _ptr(d.xyz),
                                           float(d.vscale)) == _lib_err("INVALID")
    N = 500
    q16 = torch.randn(N, 256, device=DEV).half()
    qxyz = torch.zeros(N, 4, device=DEV)
    sums, maxs = eng.retrieve_stats("RANGE", q16, qxyz, 15.0, 0.0)
    ws = eng._ret_ws(N)
    buf = torch.empty(N * 257, device=DEV)
    route = _lib.Route(1, 0, 512, (ctypes.c_void_p * _lib.RANGE_MAX_RANKS)(buf.data_ptr()))
    assert lib.range_retrieve_apply_routed(eng.ctx, 0, N, _ptr(q16), _ptr(qxyz), 15.0, 0.0, 0.0, _ptr(sums), _ptr(maxs),
                                           ctypes.byref(route), _ptr(ws), ws.numel(), _stream()) == _lib_err("UNSUPPORTED")
    assert b"1024" in lib.range_last_error()
    O_ = torch.empty(N, 257, device=DEV)
    need = lib.range_retrieve_workspace_bytes(eng.ctx, N)
    assert lib.range_retrieve_apply(eng.ctx, 0, N, _ptr(q16), _ptr(qxyz), 15.0, 0.0, 0.0, _ptr(sums), _ptr(maxs), _ptr(O_),
                                    _ptr(ws), need - 1, _stream()) == _lib_err("WORKSPACE")
    with pytest.raises(ValueError, match="257"):
        eng.combine_concat([torch.zeros(N, 1024, device=DEV)], None, torch.zeros(N, 256, dtype=torch.float64, device=DEV))


def _lib_err(name):
    return {"INVALID": -1, "CUDA": -2, "WORKSPACE": -3, "UNSUPPORTED": -4}[name]


@pytest.mark.gpu
def test_load_model_on_a_768_wide_npz(tmp_path, sh_entries):
    """the drop-in boundary with CLIP-width features: load_model(db_path=<768-wide .npz>) / model(locs) ->
    numpy float64 (N, 1024) rows matching the oracle; with db_cache the second load reads the prepared layout"""
    from range_b200.load_model import load_model
    tol_o, rel_rows, _, _, TOL_Q_POLAR = _tol()
    ws = O.siren_init(40, 64, 2, 256, seed=4)
    sd = {}
    for (W, b), nm in zip(ws, ["layers.0", "layers.1", "last_layer"]):
        sd[f"model.location.nnet.{nm}.weight"], sd[f"model.location.nnet.{nm}.bias"] = W, b
    hp = dict(embed_dim=256, legendre_polys=40, le_type="sphericalharmonics", pe_type="siren",
              harmonics_calculation="analytic", num_hidden_layers=2, capacity=64, eval_downstream=False,
              air_temp_data_path=None, election_data_path=None)
    ckpt = tmp_path / "satclip.ckpt"
    torch.save({"hyper_parameters": hp, "state_dict": sd}, ckpt)
    db = _db(6_000, 768, seed=8)
    np.savez(tmp_path / "clip_db.npz", **db)
    c = O.area_uniform(500, np.random.default_rng(8))
    ref = O.RangeOracle("RANGE+", ws, sh_entries, db, beta=0.5, exact=True)(c)
    outs = []
    for _ in range(2):
        model = load_model("RANGE+", str(ckpt), device="cuda", db_path=str(tmp_path / "clip_db.npz"), beta=0.5,
                           db_cache=str(tmp_path / "cache.npz"))
        assert model.location_feature_dim == 1024
        out = model(c)
        assert isinstance(out, np.ndarray) and out.dtype == np.float64 and out.shape == (500, 1024)
        assert rel_rows(out[:, :768], ref[:, :768]).max() <= tol_o("RANGE+", 0.5)
        assert np.abs(out[:, 768:] - ref[:, 768:]).max() <= TOL_Q_POLAR
        outs.append(out)
    assert np.array_equal(outs[0], outs[1])
