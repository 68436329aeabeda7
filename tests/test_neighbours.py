"""Retrieval neighbours: the k database entries with the largest retrieval weight per query (range_retrieve_topk,
DeviceDatabase.file_rows, LocationEncoder.neighbours).

The GPU checks compare against the exact weights in fp64, computed with torch from prepare_reference_arrays(db) and the
GPU's own q64 / qxyz, so they test the retrieval alone.  The kernels' semantic logits carry the fp16 rounding of q and K
(temperature x 2.5e-5, DESIGN.md section 2): weights within TOL relative (+ ATOL absolute) of the exact weight of the same
entry, and a valid top-k up to that tolerance - entries whose exact weights differ by less may come in either order.
"""
import math

import numpy as np
import pytest
import torch

from oracle import range_oracle as O
from range_b200.database import DeviceDatabase, prepare_reference_arrays
from range_b200.utils import rad_to_cart

DEV = "cuda:0"
TOL, ATOL = 2e-3, 1e-7
MODES = [("RANGE", None), ("RANGE+", 0.0), ("RANGE+", 0.5), ("RANGE+", 1.0)]
KS = (1, 8, 32)
TEMP = {"RANGE": 15.0, "RANGE+": 12.0}
GEO_TEMP = 40.0


# ---------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("kw", [dict(), dict(spatial_sort=False), dict(shard=(1, 3))], ids=["sorted", "unsorted", "shard"])
def test_file_rows_map_device_rows_to_file_rows(kw, tmp_path):
    db = O.synthetic_db(700, seed=9, kind="iid")
    ddb = DeviceDatabase(db, "cpu", **kw)
    lo, hi = ddb.row_range
    dev_rows = torch.arange(ddb.M, dtype=torch.int32)
    rows = ddb.file_rows(dev_rows)
    assert rows.dtype == torch.int64 and rows.shape == (ddb.M,)
    # the device layout's row r holds the entry of file row rows[r]: its location and its key
    xyz = rad_to_cart(np.asarray(db["locs"]).astype(np.float32) * math.pi / 180)
    assert np.array_equal(ddb.xyz[:ddb.M, :3].numpy(), xyz[rows.numpy()])
    K, _, _ = prepare_reference_arrays(db)
    assert np.abs(ddb.Kh[:ddb.M].float().numpy() - K[rows.numpy()]).max() < 1e-3
    assert len(np.unique(rows.numpy())) == ddb.M
    if "shard" not in kw and ddb.order is None:
        assert np.array_equal(rows.numpy(), np.arange(lo, hi))
    # any shape; the same answer from a database loaded from its cache
    two_d = torch.tensor([[0, ddb.M - 1], [3, 1]])
    assert torch.equal(ddb.file_rows(two_d), rows[two_d])
    ddb.save_cache(tmp_path / "db", fingerprint="x")
    again = DeviceDatabase.from_cache(tmp_path / "db", "cpu", shard=kw.get("shard"))
    assert torch.equal(again.file_rows(dev_rows), rows)


def test_topk_symbols_in_prototypes():
    from range_b200 import _lib
    assert "range_retrieve_topk" in _lib.PROTOTYPES and "range_topk_workspace_bytes" in _lib.PROTOTYPES
    assert _lib.RANGE_TOPK_MAX == 32


# ---------------------------------------------------------------------------------------------------- GPU helpers
def exact_weights(ref, q64, qxyz, name, beta):
    """(n, M) fp64 weights over the file rows: softmax(15 S), or (1-beta) softmax(40 G) + beta softmax(12 S)"""
    K, xyz = ref
    S = q64.double() @ K.T
    ws = torch.softmax(TEMP[name] * S, dim=1)
    if name == "RANGE":
        return ws
    G = qxyz[:, :3].double() @ xyz.T
    return (1.0 - beta) * torch.softmax(GEO_TEMP * G, dim=1) + beta * ws


def check_rows(rows_file, w, W, k, what):
    """per-row contract: in range, distinct, non-increasing, weights of the same entries, a top-k up to TOL"""
    M = W.shape[1]
    assert rows_file.shape == w.shape == (W.shape[0], k), what
    assert int(rows_file.min()) >= 0 and int(rows_file.max()) < M, what
    s = rows_file.sort(1).values
    assert (s[:, 1:] != s[:, :-1]).all(), what
    assert (w[:, 1:] <= w[:, :-1]).all(), what
    we = W.gather(1, rows_file)
    err = (w.double() - we).abs() - (TOL * we + ATOL)
    assert (err <= 0).all(), (what, float(err.max()))
    wmin = we.min(1).values
    kth = W.topk(k, dim=1).values[:, -1]
    assert (wmin >= (1 - TOL) * kth - ATOL).all(), (what, float((kth - wmin).max()))
    if k < M:
        omitted = W.scatter(1, rows_file, -1.0).max(1).values
        assert (omitted <= (1 + TOL) * wmin + ATOL).all(), (what, float((omitted - wmin).max()))


def make_engine(db, ws, **kw):
    from range_b200.engine import RangeEngine
    ddb = DeviceDatabase(db, DEV, **kw)
    eng = RangeEngine(DEV, encoder=dict(L=40, dims=[1600, 64, 64, 256], weights=ws), database=ddb)
    K, _, xyz = prepare_reference_arrays(db)
    ref = (torch.from_numpy(K).to(DEV, torch.float64), torch.from_numpy(np.asarray(xyz)).to(DEV, torch.float64))
    return eng, ddb, ref


def run_all(eng, ddb, ref, coords, sample=None, modes=MODES, ks=KS):
    """every mode and k on these queries; rows `sample` (default all) checked against the exact weights"""
    q64, q16, qxyz = eng.encode(torch.as_tensor(coords).to(DEV))
    rows = torch.arange(q64.shape[0], device=DEV) if sample is None else torch.as_tensor(sample, device=DEV)
    for name, beta in modes:
        sums, _ = eng.retrieve_stats(name, q16, qxyz, TEMP[name], GEO_TEMP)
        W_all = [exact_weights(ref, q64[r], qxyz[r], name, beta) for r in rows.split(512)]
        for k in ks:
            if k > ddb.M:
                continue
            idx, w = eng.retrieve_topk(name, q16, qxyz, TEMP[name], GEO_TEMP, beta, sums, k)
            assert idx.dtype == torch.int32 and w.dtype == torch.float32
            for r, W in zip(rows.split(512), W_all):
                check_rows(ddb.file_rows(idx[r]), w[r], W, k, (name, beta, k, ddb.M))


@pytest.fixture(scope="module")
def ws():
    return O.siren_init(40, 64, 2, 256, seed=5)


@pytest.fixture(scope="module")
def sorted20k(ws):
    """a spatially sorted (geo-skipping) iid database of a ragged size"""
    db = O.synthetic_db(20077, seed=6, kind="iid")
    return (db,) + make_engine(db, ws)


# ---------------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 127, 129])
def test_topk_exact_sorted_db(sorted20k, N):
    _, eng, ddb, ref = sorted20k
    run_all(eng, ddb, ref, O.area_uniform(N, np.random.default_rng(N)))


@pytest.mark.gpu
def test_topk_exact_unsorted_db(ws):
    db = O.synthetic_db(20077, seed=7, kind="iid")
    eng, ddb, ref = make_engine(db, ws, spatial_sort=False)
    assert ddb.order is None and ddb.caps is None
    run_all(eng, ddb, ref, O.area_uniform(3000, np.random.default_rng(3)))


@pytest.mark.gpu
def test_topk_exact_small_db(ws):
    """M < 128: one partial database tile"""
    db = O.synthetic_db(100, seed=8, kind="iid")
    eng, ddb, ref = make_engine(db, ws)
    run_all(eng, ddb, ref, O.area_uniform(127, np.random.default_rng(4)))


@pytest.mark.gpu
def test_topk_exact_many_splits(ws):
    """one query over 100 000 entries: the database is split over many CTAs (the statistics plan's split count)"""
    db = O.synthetic_db(100_000, seed=10, kind="iid")
    eng, ddb, ref = make_engine(db, ws)
    run_all(eng, ddb, ref, O.area_uniform(1, np.random.default_rng(5)))
    run_all(eng, ddb, ref, O.area_uniform(1500, np.random.default_rng(6)), sample=np.arange(0, 1500, 7))


@pytest.mark.gpu
def test_topk_exact_structured_db(ws, sh_entries):
    """peaky weights: keys near the encoder's own embedding of the entry's location"""
    helper = O.RangeOracle.__new__(O.RangeOracle)
    helper.L, helper.entries, helper.weights = 40, sh_entries, ws
    db = O.synthetic_db(6000, seed=11, kind="structured", encoder=helper.encode)
    eng, ddb, ref = make_engine(db, ws)
    run_all(eng, ddb, ref, O.area_uniform(129, np.random.default_rng(7)))


@pytest.mark.gpu
def test_topk_geo_skip_and_perm(sorted20k):
    """spatially sorted queries on a sorted database: the apply-pass mask skips tiles; rows through perm"""
    _, eng, ddb, ref = sorted20k
    c = torch.tensor(O.area_uniform(3000, np.random.default_rng(8)), device=DEV)
    cs, perm = eng.sort_queries(c)
    q64, q16, qxyz = eng.encode(cs)
    sums, _ = eng.retrieve_stats("RANGE+", q16, qxyz, 12.0, GEO_TEMP)
    assert eng.geo_mask(qxyz, GEO_TEMP, sums).any()
    run_all(eng, ddb, ref, cs, modes=[("RANGE+", 0.0), ("RANGE+", 0.5)])
    idx, w = eng.retrieve_topk("RANGE+", q16, qxyz, 12.0, GEO_TEMP, 0.5, sums, 8)
    idx_p, w_p = eng.retrieve_topk("RANGE+", q16, qxyz, 12.0, GEO_TEMP, 0.5, sums, 8, perm=perm)
    assert torch.equal(idx_p[perm.long()], idx) and torch.equal(w_p[perm.long()], w)


@pytest.mark.gpu
def test_topk_exact_large_batch(sorted20k):
    """N >= 6144: the normalisers come from the CTA-pair statistics kernel; a sample of rows is checked"""
    _, eng, ddb, ref = sorted20k
    run_all(eng, ddb, ref, O.area_uniform(8192, np.random.default_rng(9)), sample=np.arange(0, 8192, 16))


@pytest.mark.gpu
def test_topk_known_answer_and_determinism(sorted20k):
    """RANGE+ at beta = 0 with queries on database locations: the top entry is that location's file row"""
    db, eng, ddb, _ = sorted20k
    file_rows = np.random.default_rng(10).choice(ddb.M, 300, replace=False)
    c = torch.tensor(np.asarray(db["locs"])[file_rows], device=DEV)
    q64, q16, qxyz = eng.encode(c)
    sums, _ = eng.retrieve_stats("RANGE+", q16, qxyz, 12.0, GEO_TEMP)
    idx, w = eng.retrieve_topk("RANGE+", q16, qxyz, 12.0, GEO_TEMP, 0.0, sums, 4)
    assert np.array_equal(ddb.file_rows(idx[:, 0]).cpu().numpy(), file_rows)
    idx2, w2 = eng.retrieve_topk("RANGE+", q16, qxyz, 12.0, GEO_TEMP, 0.0, sums, 4)
    assert torch.equal(idx, idx2) and torch.equal(w, w2)


def _checkpoint(tmp_path, ws):
    sd = {}
    for (W, b), nm in zip(ws, ["layers.0", "layers.1", "last_layer"]):
        sd[f"model.location.nnet.{nm}.weight"] = W
        sd[f"model.location.nnet.{nm}.bias"] = b
    hp = dict(embed_dim=256, legendre_polys=40, le_type="sphericalharmonics", pe_type="siren",
              harmonics_calculation="analytic", num_hidden_layers=2, capacity=64, eval_downstream=False,
              air_temp_data_path=None, election_data_path=None)
    path = tmp_path / "satclip.ckpt"
    torch.save({"hyper_parameters": hp, "state_dict": sd}, path)
    return str(path)


@pytest.mark.gpu
def test_neighbours_api(tmp_path, ws):
    from range_b200.load_model import load_model
    M = 20
    db = O.synthetic_db(M, seed=12, kind="iid")
    dbfile = tmp_path / "db.npz"
    np.savez(dbfile, **db)
    ckpt = _checkpoint(tmp_path, ws)
    model = load_model("RANGE+", ckpt, device="cuda", db_path=str(dbfile), beta=0.0)
    shuffle = np.random.default_rng(13).permutation(M)
    coords = torch.tensor(np.asarray(db["locs"])[shuffle], device=DEV)
    before = model.embed(coords)
    idx, w = model.neighbours(coords, k=5)
    assert idx.dtype == torch.int64 and w.dtype == torch.float32 and idx.shape == w.shape == (M, 5)
    assert np.array_equal(idx[:, 0].cpu().numpy(), shuffle)           # caller's row order, file rows
    assert (w[:, 1:] <= w[:, :-1]).all()
    idx2, w2 = model.neighbours(coords, k=5)
    assert torch.equal(idx, idx2) and torch.equal(w, w2)
    assert torch.equal(model.embed(coords), before)
    assert model.neighbours(coords, k=M)[0].shape == (M, M)
    for bad in (0, 33, M + 1):
        with pytest.raises(ValueError):
            model.neighbours(coords, k=bad)
    # RANGE: the semantic softmax alone; the weights of the full list sum to 1
    m2 = load_model("RANGE", ckpt, device="cuda", db_path=str(dbfile))
    idx3, w3 = m2.neighbours(coords, k=M)
    assert torch.allclose(w3.double().sum(1), torch.ones(M, dtype=torch.float64, device=DEV), atol=2e-3)
    assert (idx3.sort(1).values == torch.arange(M, device=DEV)).all()
