"""RANGE database: the reference's preparation (range/range.py:78-100) and the device-resident layout the
retrieval kernels stream.

Device layout (what include/range_b200.h:range_ctx_set_db takes):
  Kh  (Mpad, 256)  fp16  row-normalised SatCLIP keys, row-major  -> TMA boxes [128 entries x 64 dims]
  Vt  (1024, Mpad) fp16  values TRANSPOSED (entries contiguous) x vscale -> TMA boxes [256 dims x 64 entries];
                         K-major B operand of the P.V tensor-core product, same descriptor as the keys
  xyz (Mpad, 4)    fp32  unit vectors of the entry locations (x, y, z, 0)
  caps (Mpad/128, 4) fp32 bounding cap of every 128-entry tile: (unit centre, angular radius [rad])
Mpad = M rounded up to 128; padding is zero and masked in-kernel.

Row order: the reference's results do not depend on the order of the database rows (softmax-weighted sums,
range/range.py:213-238), so the rows are stored sorted along a cube-map Hilbert curve.  Consecutive 128-entry
tiles are then spatially compact, which lets the RANGE+ kernels skip the geographic term for tiles far from a
query tile (include/range_b200.h: range_ctx_set_db_caps).
"""
import hashlib
import math
import os
import struct
import zipfile

import numpy as np
import torch

from .utils import rad_to_cart

BLOCK = 128


def prepare_reference_arrays(db):
    """Exactly range/range.py:79-95, on the host in numpy fp32 (bit-identical to the reference's tensors)."""
    locs = np.asarray(db["locs"]).astype(np.float32)                                  # :79
    K = np.asarray(db["satclip_embeddings"]).astype(np.float32)                       # :85
    K = K / np.linalg.norm(K, ord=2, axis=1, keepdims=True)                           # :89
    V = np.asarray(db["image_embeddings"]).astype(np.float32)                         # :90
    xyz = rad_to_cart(locs * math.pi / 180)                                           # :93-95 (fp32)
    return K, V, xyz


def open_npz(path):
    """{name: array} of a RANGE database file (range/range.py:78 reads it with np.load).  generate_db.py:209-214 writes
    it with np.savez, i.e. uncompressed: such members are memory-mapped in place instead of read, so the (M, 1024)
    float64 value matrix of a 10 M-entry database (82 GB) is never resident at once - DeviceDatabase converts it block
    by block.  Compressed, object-typed or empty members are read the way np.load reads them."""
    from numpy.lib import format as npf
    out, loaded = {}, None
    with zipfile.ZipFile(path) as zf, open(path, "rb") as f:
        for info in zf.infolist():
            name = info.filename[:-4] if info.filename.endswith(".npy") else info.filename
            arr = None
            if info.compress_type == zipfile.ZIP_STORED and info.filename.endswith(".npy"):
                f.seek(info.header_offset)
                local = f.read(30)                         # local file header: name / extra lengths at bytes 26..30
                if len(local) == 30 and local[:4] == b"PK\x03\x04":
                    nlen, elen = struct.unpack("<HH", local[26:30])
                    f.seek(info.header_offset + 30 + nlen + elen)
                    try:
                        version = npf.read_magic(f)
                        read_header = {(1, 0): npf.read_array_header_1_0, (2, 0): npf.read_array_header_2_0}.get(version)
                        if read_header is not None:
                            shape, fortran, dtype = read_header(f)
                            if not dtype.hasobject and len(shape) > 0 and int(np.prod(shape)) > 0:
                                arr = np.memmap(path, dtype=dtype, mode="r", offset=f.tell(), shape=shape,
                                                order="F" if fortran else "C")
                    except ValueError:
                        arr = None
            if arr is None:
                loaded = np.load(path, allow_pickle=True) if loaded is None else loaded
                arr = loaded[name]
            out[name] = arr
    return out


def _abs_max_fp32(V, step=1 << 16):
    """float(np.abs(V.astype(np.float32)).max()) without materialising the fp32 copy (NaN propagates like there)"""
    m = np.float32(0.0)
    for lo in range(0, V.shape[0], step):
        m = np.maximum(m, np.abs(np.asarray(V[lo:lo + step]).astype(np.float32)).max())
    return float(m)


def _hilbert_index(ix, iy, bits):
    """position of grid cell (ix, iy) of a 2^bits x 2^bits grid along the Hilbert curve (vectorised xy2d)"""
    x, y = ix.astype(np.int64).copy(), iy.astype(np.int64).copy()
    d = np.zeros_like(x)
    n = 1 << bits
    s = n >> 1
    while s > 0:
        rx, ry = ((x & s) > 0).astype(np.int64), ((y & s) > 0).astype(np.int64)
        d += s * s * ((3 * rx) ^ ry)
        flip = (ry == 0) & (rx == 1)
        x, y = np.where(flip, n - 1 - x, x), np.where(flip, n - 1 - y, y)
        x, y = np.where(ry == 0, y, x), np.where(ry == 0, x, y)
        s >>= 1
    return d


def hilbert_order(xyz, bits=12):
    """stable argsort of unit vectors along a per-face Hilbert curve of the equal-angle cube map: consecutive rows
    are neighbours on the sphere (bounding caps of 128-row tiles ~1.5x the ideal disc; a Morton curve: ~2.7x)"""
    x, y, z = (np.asarray(xyz[:, i], dtype=np.float64) for i in range(3))
    ax, ay, az = np.abs(x), np.abs(y), np.abs(z)
    fx = (ax >= ay) & (ax >= az)
    fy = ~fx & (ay >= az)
    fz = ~fx & ~fy
    face = np.where(fx, np.where(x >= 0, 0, 1), np.where(fy, np.where(y >= 0, 2, 3), np.where(z >= 0, 4, 5)))
    m = np.maximum(np.where(fx, ax, np.where(fy, ay, az)), 1e-30)
    u = np.where(fx, y, x) / m
    v = np.where(fz, y, z) / m
    g = 1 << bits
    iu = np.clip(((np.arctan(u) * (4 / np.pi) + 1) * 0.5 * g).astype(np.int64), 0, g - 1)
    iv = np.clip(((np.arctan(v) * (4 / np.pi) + 1) * 0.5 * g).astype(np.int64), 0, g - 1)
    key = (face.astype(np.int64) << (2 * bits)) | _hilbert_index(iu, iv, bits)
    return np.argsort(key, kind="stable")


def tile_caps(xyz, block=BLOCK):
    """(ceil(M/block), 4) fp32: unit mean direction and the largest angle to it, per tile of `block` rows"""
    M = xyz.shape[0]
    T = (M + block - 1) // block
    pad = T * block - M
    p = np.asarray(xyz, dtype=np.float64)
    if pad:
        p = np.concatenate([p, np.repeat(p[-1:], pad, axis=0)], axis=0)     # repeat a real entry: caps unchanged
    p = p.reshape(T, block, 3)
    c = p.sum(1)
    n = np.linalg.norm(c, axis=1, keepdims=True)
    c = np.where(n > 1e-9, c / np.maximum(n, 1e-30), np.array([0.0, 0.0, 1.0]))
    cosang = np.clip(np.einsum("tbi,ti->tb", p, c) / np.maximum(np.linalg.norm(p, axis=2), 1e-30), -1.0, 1.0)
    r = np.arccos(cosang).max(1)
    r = np.where(n[:, 0] > 1e-9, r, np.pi)                                    # degenerate tile: covers the sphere
    return np.concatenate([c, r[:, None]], axis=1).astype(np.float32)


class DeviceDatabase:
    STAGING_ROWS = 1 << 18          # rows converted / uploaded at a time (1.3 GB of fp32 staging)

    def __init__(self, db, device, shard=None, spatial_sort=True):
        """db: mapping with locs / satclip_embeddings / image_embeddings (an opened .npz works).
        shard=(rank, world): keep rows [rank*M/world, (rank+1)*M/world) of the (sorted) database only (M-sharding).
        spatial_sort: store the rows along a Hilbert curve and build the tile caps (geo-term skipping)."""
        # keys and values stay what they are (ndarrays, or memory maps from open_npz): range.py:85-90's .astype(float32)
        # and row normalisation are applied block by block on the way to the device, in the reference's arithmetic
        locs = np.asarray(db["locs"]).astype(np.float32)                                  # range.py:79
        xyz = rad_to_cart(locs * math.pi / 180)                                           # range.py:93-95 (fp32)
        Kraw, V = (a if isinstance(a, np.ndarray) else np.asarray(a)
                   for a in (db["satclip_embeddings"], db["image_embeddings"]))
        self.M_total = xyz.shape[0]
        if Kraw.ndim != 2 or Kraw.shape[1] != 256 or V.ndim != 2 or V.shape[1] != 1024:
            raise ValueError(f"RANGE database must have 256-d keys and 1024-d values, got {Kraw.shape[1:]}, {V.shape[1:]}")
        if Kraw.shape[0] != self.M_total or V.shape[0] != self.M_total:
            raise ValueError(f"RANGE database arrays disagree on the number of entries: locs {self.M_total}, "
                             f"keys {Kraw.shape[0]}, values {V.shape[0]}")
        self.order = hilbert_order(xyz) if spatial_sort and self.M_total > 0 else None
        lo, hi = (0, self.M_total) if shard is None else ((self.M_total * shard[0]) // shard[1],
                                                          (self.M_total * (shard[0] + 1)) // shard[1])
        self.row_range = (lo, hi)
        self.shard = None if shard is None else (int(shard[0]), int(shard[1]))
        rows_of = np.arange(lo, hi) if self.order is None else self.order[lo:hi]      # file rows of this layout's rows
        xyz = xyz[rows_of]
        M = hi - lo
        if M == 0:
            raise ValueError("empty database (shard)")
        Mpad = (M + BLOCK - 1) // BLOCK * BLOCK
        dev = torch.device(device)
        self.M, self.Mpad = M, Mpad
        # the value scale: over this shard's rows when the file order is kept, over the whole file when the rows are
        # spread by the spatial sort
        vmax = _abs_max_fp32(V[lo:hi] if self.order is None else V)
        self.vscale = 1.0 if vmax == 0.0 or not math.isfinite(vmax) else 2.0 ** math.floor(math.log2(256.0 / vmax))
        self.Kh = torch.zeros(Mpad, 256, dtype=torch.float16, device=dev)
        self.Vt = torch.zeros(1024, Mpad, dtype=torch.float16, device=dev)
        step = self.STAGING_ROWS
        for b0 in range(0, M, step):                       # bounded staging memory for 10M-entry databases
            b1 = min(M, b0 + step)
            want = rows_of[b0:b1]
            idx = np.sort(want)                            # gather in file order (sequential reads of a memory map) ...
            back = np.searchsorted(idx, want)              # ... then permute into layout order
            k = np.asarray(Kraw[idx]).astype(np.float32)                                  # range.py:85
            k = (k / np.linalg.norm(k, ord=2, axis=1, keepdims=True))[back]               # range.py:89
            self.Kh[b0:b1] = torch.from_numpy(np.ascontiguousarray(k)).to(dev).half()
            v = np.asarray(V[idx]).astype(np.float32)[back]                               # range.py:90
            self.Vt[:, b0:b1] = (torch.from_numpy(np.ascontiguousarray(v)).to(dev) * self.vscale).half().t()
        self.xyz = torch.zeros(Mpad, 4, dtype=torch.float32, device=dev)
        self.xyz[:M, :3] = torch.from_numpy(np.ascontiguousarray(xyz)).to(dev)
        self.caps = torch.from_numpy(tile_caps(xyz)).to(dev) if self.order is not None else None

    # ---- device-resident format on disk (SURVEY.md section 8f-1): skips normalisation / sorting / transposition at start-up
    CACHE_VERSION = 2

    @staticmethod
    def source_fingerprint(source):
        """identifies the database a cache was built from: (path, size, mtime) of a file, or the entry count and a
        digest of the locations of an in-memory mapping"""
        if isinstance(source, (str, os.PathLike)):
            st = os.stat(source)
            return f"file:{os.path.abspath(source)}:{st.st_size}:{st.st_mtime_ns}"
        locs = np.ascontiguousarray(np.asarray(source["locs"]))
        return f"mem:{locs.shape[0]}:{locs.dtype}:{hashlib.sha1(locs.tobytes()).hexdigest()}"

    @staticmethod
    def cache_path(path, shard=None):
        """the file save_cache / from_cache use: always '.npz' (np.savez would append it silently), one file per shard"""
        path = os.fspath(path)
        stem = path[:-4] if path.endswith(".npz") else path
        if shard is not None:
            stem += f".shard{int(shard[0])}of{int(shard[1])}"
        return stem + ".npz"

    def save_cache(self, path, fingerprint=""):
        """write the prepared layout (fp16 keys / transposed values, xyz, tile caps, row order) as an .npz; the file
        appears atomically (temporary file + rename), so a concurrent reader never sees a partial cache"""
        path = self.cache_path(path, self.shard)
        tmp = f"{path}.{os.getpid()}.tmp.npz"
        shard = (-1, -1) if self.shard is None else self.shard
        try:
            with open(tmp, "wb") as f:
                np.savez(f, version=self.CACHE_VERSION, M=self.M, Mpad=self.Mpad, M_total=self.M_total,
                         row_range=np.asarray(self.row_range), vscale=self.vscale, shard=np.asarray(shard),
                         fingerprint=np.asarray(fingerprint),
                         Kh=self.Kh.cpu().numpy(), Vt=self.Vt.cpu().numpy(), xyz=self.xyz.cpu().numpy(),
                         caps=np.zeros((0, 4), np.float32) if self.caps is None else self.caps.cpu().numpy(),
                         order=np.zeros(0, np.int64) if self.order is None else self.order)
            os.replace(tmp, path)
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
        return path

    @classmethod
    def from_cache(cls, path, device, shard=None, fingerprint=None, spatial_sort=None):
        """load a cache written by save_cache.  Returns None (the caller rebuilds) when the file is missing or was built
        for another shard, another source (fingerprint, when given) or another row order; raises on a malformed file."""
        path = cls.cache_path(path, shard)
        if not os.path.exists(path):
            return None
        z = np.load(path)
        if "version" not in z or int(z["version"]) != cls.CACHE_VERSION:
            return None
        want = (-1, -1) if shard is None else (int(shard[0]), int(shard[1]))
        if tuple(int(v) for v in z["shard"]) != want:
            return None
        if fingerprint is not None and str(z["fingerprint"]) != fingerprint:
            return None
        if spatial_sort is not None and bool(z["order"].shape[0]) != bool(spatial_sort):
            return None
        self = cls.__new__(cls)
        dev = torch.device(device)
        self.M, self.Mpad, self.M_total = int(z["M"]), int(z["Mpad"]), int(z["M_total"])
        self.row_range = tuple(int(v) for v in z["row_range"])
        self.shard = None if want == (-1, -1) else want
        if self.shard is not None:
            lo, hi = (self.M_total * want[0]) // want[1], (self.M_total * (want[0] + 1)) // want[1]
            if self.row_range != (lo, hi):
                raise ValueError(f"{path}: rows {self.row_range} do not match shard {want} of {self.M_total} entries")
        self.vscale = float(z["vscale"])
        self.Kh = torch.from_numpy(z["Kh"]).to(dev)
        self.Vt = torch.from_numpy(z["Vt"]).to(dev)
        self.xyz = torch.from_numpy(z["xyz"]).to(dev)
        self.caps = torch.from_numpy(z["caps"]).to(dev) if z["caps"].shape[0] else None
        self.order = z["order"] if z["order"].shape[0] else None
        if self.Kh.shape != (self.Mpad, 256) or self.Vt.shape != (1024, self.Mpad) or self.Kh.dtype != torch.float16 \
                or self.M != self.row_range[1] - self.row_range[0]:
            raise ValueError(f"{path}: malformed database cache")
        return self

    @classmethod
    def synthetic(cls, M, device, seed=0, shard=None):
        """Benchmark-only: an iid synthetic database (area-uniform locations, N(0,1) keys and values - the worst case
        for the fp16 operands, SURVEY.md 8d) generated block by block straight into the device layout, so 10 M-entry
        databases (25.7 GB in fp16) do not need their 51 GB of fp32 source arrays on the host.
        shard=(rank, world): rows [rank*M/world, (rank+1)*M/world) of the spatially sorted database only - every rank
        draws the same M locations (same seed) and sorts them the same way, keys / values are iid per entry."""
        self = cls.__new__(cls)
        dev = torch.device(device)
        rng = np.random.default_rng(seed)
        lon = rng.uniform(-180.0, 180.0, M)
        lat = np.degrees(np.arcsin(rng.uniform(-1.0, 1.0, M)))
        locs = np.stack([lon, lat], 1).astype(np.float32)
        xyz = rad_to_cart(locs * math.pi / 180)                                       # range.py:93-95 (fp32)
        self.order = hilbert_order(xyz)
        self.M_total = M
        lo, hi = (0, M) if shard is None else ((M * shard[0]) // shard[1], (M * (shard[0] + 1)) // shard[1])
        self.shard = None if shard is None else (int(shard[0]), int(shard[1]))
        self.row_range = (lo, hi)
        xyz = xyz[self.order[lo:hi]]
        self.M = m = hi - lo
        self.Mpad = (m + BLOCK - 1) // BLOCK * BLOCK
        self.vscale = 2.0 ** math.floor(math.log2(256.0 / 6.0))                      # |N(0,1)| < 6
        self.Kh = torch.zeros(self.Mpad, 256, dtype=torch.float16, device=dev)
        self.Vt = torch.zeros(1024, self.Mpad, dtype=torch.float16, device=dev)
        g = torch.Generator(device=dev).manual_seed(seed if shard is None else seed * 1000003 + 1 + int(shard[0]))
        step = 1 << 18
        for b0 in range(0, m, step):
            b1 = min(m, b0 + step)
            k = torch.randn(b1 - b0, 256, device=dev, generator=g)
            self.Kh[b0:b1] = (k / k.norm(dim=1, keepdim=True)).half()                 # range.py:89
            v = torch.randn(b1 - b0, 1024, device=dev, generator=g).clamp_(-6.0, 6.0)
            self.Vt[:, b0:b1] = (v * self.vscale).half().t()
        self.xyz = torch.zeros(self.Mpad, 4, dtype=torch.float32, device=dev)
        self.xyz[:m, :3] = torch.from_numpy(np.ascontiguousarray(xyz)).to(dev)
        self.caps = torch.from_numpy(tile_caps(xyz)).to(dev)
        return self

    def file_rows(self, idx):
        """device rows (e.g. the entries RangeEngine.retrieve_topk returns) -> rows of the database file, so that
        db['locs'][rows] are the entries' locations: order[row_range[0] + idx], or row_range[0] + idx when the rows keep
        the file order.  idx: integer tensor on any device; returns int64 on the same device."""
        idx = torch.as_tensor(idx)
        return self.file_rows_global(idx.long() + self.row_range[0])

    def file_rows_global(self, rows):
        """rows of the WHOLE sorted layout (e.g. what an M-sharded neighbours call returns; every shard holds the full
        row order) -> rows of the database file: order[rows], or rows when the file order is kept.  rows: integer
        tensor on any device; returns int64 on the same device."""
        rows = torch.as_tensor(rows).long()
        if self.order is None:
            return rows
        cached = getattr(self, "_order_t", None)
        if cached is None or cached.device != rows.device:
            cached = self._order_t = torch.from_numpy(np.asarray(self.order, dtype=np.int64)).to(rows.device)
        return cached[rows]

    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in (self.Kh, self.Vt, self.xyz))
