"""`LocationEncoder` for 'RANGE' / 'RANGE+' - the B200-native counterpart of range/range.py:69-278.

Same constructor contract (an argparse-style namespace with location_model_name, pretrained_path, device,
range_db, beta), same attributes other code reads (location_feature_dim, args.temp, args.geo_temp,
args.beta), same forward contract: `model(locs)` with locs (N,2) float64 (lon, lat) degrees returns a
numpy float64 (N, 1280) array = [retrieved visual feature (1024) | L2-normalised SatCLIP embedding (256)].
Only the RANGE branches exist here; every other encoder name raises like the reference's final `else`.
"""
import os

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .checkpoint import load_satclip_location_encoder
from .database import DeviceDatabase, open_npz
from .engine import RangeEngine

# one round of the producer/consumer apply kernel on 148 SMs: 24 units x 2 query tiles of 128
ROUND_ROWS = 24 * 256
DEFAULT_CHUNK = 4 * ROUND_ROWS   # largest piece of model(locs)'s pipeline (two device buffers of chunk x 10 KB)
DEFAULT_TAIL = ROUND_ROWS        # the last piece: its device->host copy (63-94 MB) is the only one not overlapped
DEFAULT_TAPER = 0.5


class LocationEncoder(nn.Module):
    def __init__(self, args):
        super().__init__()
        self.args = args
        self.location_model_name = args.location_model_name
        if 'RANGE' not in self.location_model_name:
            raise NotImplementedError(f'{self.location_model_name} not implemented')      # range.py:200
        if self.location_model_name == 'RANGE':
            self.args.temp = 15.0                                                          # range.py:103
            print(f'Using RANGE with temperature {self.args.temp}')
        elif self.location_model_name == 'RANGE+':
            self.args.geo_temp = 40.0                                                      # range.py:109
            self.args.temp = 12.0                                                          # range.py:108
            print(f'Using RANGE+ with temperatures {self.args.temp} and {self.args.geo_temp}')
        else:
            raise ValueError('Unimplemented RANGE model')                                  # range.py:114
        shard = getattr(args, 'db_shard', None)
        enc = load_satclip_location_encoder(args.pretrained_path) if isinstance(args.pretrained_path, str) \
            else args.pretrained_path
        self.location_feature_dim = 1024 + 256                                             # range.py:86
        cache = getattr(args, 'db_cache', None)        # optional: prepared device layout on disk (database.py)
        ddb = None
        if isinstance(args.range_db, DeviceDatabase):   # an already prepared device layout (its own shard, if any)
            ddb = args.range_db
            if shard is not None and tuple(shard) != ddb.shard:
                raise ValueError(f'db_shard={tuple(shard)} but the prepared database holds shard {ddb.shard}')
            shard = ddb.shard
        elif cache is not None:
            # the cache is only used when it was built from this source, for this shard (one file per shard)
            fp = DeviceDatabase.source_fingerprint(args.range_db)
            ddb = DeviceDatabase.from_cache(cache, args.device, shard=shard, fingerprint=fp)
        if ddb is None:
            db = open_npz(args.range_db) if isinstance(args.range_db, str) else args.range_db      # range.py:78
            ddb = DeviceDatabase(db, args.device, shard=shard)
            if cache is not None:
                ddb.save_cache(cache, fingerprint=fp)
        self.engine = RangeEngine(args.device, encoder=enc, database=ddb)
        self.chunk = int(getattr(args, 'chunk', DEFAULT_CHUNK))
        self.tail = max(1, min(self.chunk, int(getattr(args, 'tail', DEFAULT_TAIL))))
        self.super_batch = max(self.chunk, int(getattr(args, 'super_batch', 1 << 20)) // self.chunk * self.chunk)
        self.taper = float(getattr(args, 'taper', DEFAULT_TAPER))
        # numpy dtype of model(locs)'s result: float64 is what the reference returns (range.py:222,240 - its feature
        # columns are fp32 values widened by np.concatenate); 'float32' is an opt-in that halves the bytes crossing PCIe
        # and landing in host memory - the e2e ceiling when several GPUs share one host (profiles/r2_d2h_wall.md)
        self.out_dtype = np.dtype(getattr(args, 'out_dtype', np.float64))
        if self.out_dtype not in (np.dtype(np.float64), np.dtype(np.float32)):
            raise ValueError(f'out_dtype={self.out_dtype}: expected float64 (the reference\'s) or float32')
        # how model(locs) hands the (N,1280) float64 result to the host (see _forward_host)
        self.host_path = getattr(args, 'host_path', 'auto')
        if self.host_path not in ('auto', 'copy', 'packed'):
            raise ValueError(f"host_path={self.host_path!r}: expected 'auto', 'copy' or 'packed'")
        self.pinned_limit = int(getattr(args, 'pinned_limit', 8 << 30))       # largest page-locked result, bytes
        local_ranks = max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1')))      # torchrun: ranks sharing this host
        self.host_threads = int(getattr(args, 'host_threads', 0)) or max(1, min(16, (os.cpu_count() or 1) // local_ranks))
        self.group = getattr(args, 'db_group', None)       # torch.distributed group when the DB is M-sharded
        self.sharded = None
        if shard is not None and shard[1] > 1:
            from .distributed import ShardedRetriever
            self.sharded = ShardedRetriever(self.engine, self.group, merge=getattr(args, 'db_merge', 'peer'))
        self._copy_stream = None
        self.trace = None           # developer timeline of _forward_host: a list collects (rows, computed, copied) events
        self.eval()

    def close(self):
        """release the peer receive buffers of an M-sharded model (a collective call: every rank closes)"""
        if self.sharded is not None:
            self.sharded.close()

    # the reference calls model.to(device) after construction (load_model.py:50); tensors live in the engine
    def _apply(self, fn, recurse=True):
        return self

    def _sorts(self):
        eng = self.engine
        return self.location_model_name == 'RANGE+' and eng.db is not None and eng.db.caps is not None

    def _retrieve_concat(self, q16, qxyz, q64, out, out_dtype, perm):
        """statistics, apply and concat: (N,1280) = [retrieved feature | q64] with row n at out[perm[n]]"""
        eng, a = self.engine, self.args
        name = self.location_model_name
        beta = getattr(a, 'beta', None)
        geo_temp = float(getattr(a, 'geo_temp', 0.0))
        return eng.retrieve_concat(name, q16, qxyz, a.temp, geo_temp, beta, q64, out=out, dtype=out_dtype, perm=perm)

    @torch.no_grad()
    def embed(self, coords, out=None, out_dtype=torch.float32):
        """Device-resident path: coords (N,2) fp64 on the device -> (N,1280) device tensor.
        With an M-sharded database (db_shard / db_group) this is a COLLECTIVE call: every rank passes its own
        queries and gets its own rows (distributed.py)."""
        eng, a = self.engine, self.args
        if self.sharded is not None:
            coords = coords.to(eng.device, torch.float64).contiguous()
            return self.sharded.embed(self.location_model_name, coords, a.temp, float(getattr(a, 'geo_temp', 0.0)),
                                      getattr(a, 'beta', None), self._sorts(), out=out, out_dtype=out_dtype)
        perm = None
        if self._sorts():
            # spatial batching: the geo softmax is local, tiles of nearby queries skip far database tiles
            coords, perm = eng.sort_queries(coords)
        q64, q16, qxyz = eng.encode(coords)
        return self._retrieve_concat(q16, qxyz, q64, out, out_dtype, perm)

    @torch.no_grad()
    def embed_sweep(self, coords, betas, out_dtype=torch.float32):
        """RANGE+ for several beta on the same queries (multi-resolution use, Readme.md:27-31).  range/range.py:238 is
        linear in beta - O(beta) = (1 - beta) O_geo + beta O_sem - so the encoder, the statistics pass and TWO apply
        passes (the geographic and the semantic end) serve any number of beta; each beta then costs one memory-bound
        blend + concat kernel.  Returns a list of (N,1280) device tensors.
        With an M-sharded database (db_shard / db_group) this is a COLLECTIVE call: every rank passes its own queries
        and its own beta list (the lists may differ; every rank takes every step) and gets its own rows for each of its
        beta (distributed.py: two routed apply passes per step, one merge kernel for all beta)."""
        if self.location_model_name != 'RANGE+':
            raise NotImplementedError('embed_sweep: only RANGE+ has a beta to sweep')
        eng, a = self.engine, self.args
        if self.sharded is not None:
            coords = torch.as_tensor(coords).to(eng.device, torch.float64).contiguous()
            return self.sharded.embed_sweep(coords, a.temp, a.geo_temp, self._sorts(), betas, out_dtype=out_dtype)
        perm = None
        if self._sorts():
            coords, perm = eng.sort_queries(coords)
        q64, q16, qxyz = eng.encode(coords)
        sums, maxs = eng.retrieve_stats('RANGE+', q16, qxyz, a.temp, a.geo_temp)
        O_geo = eng.retrieve_apply('RANGE+', q16, qxyz, a.temp, a.geo_temp, 0.0, sums, maxs)
        # the semantic end is the one-softmax retrieval at RANGE+'s temperature: no geographic work at all
        O_sem = eng.retrieve_apply('RANGE', q16, qxyz, a.temp, 0.0, None, sums, maxs)
        return [eng.combine_concat([O_geo, O_sem], [1.0 - float(b), float(b)], q64, dtype=out_dtype, perm=perm)
                for b in betas]

    @torch.no_grad()
    def neighbours(self, coords, k=8):
        """Which database entries each embedding is made of: coords (N,2) fp64 (lon, lat) degrees -> (index (N,k) int64,
        weight (N,k) float32) device tensors in the caller's row order.  index holds rows of the database file
        (db['locs'][index] are the neighbours' locations), weight the coefficient the retrieved feature gives each of
        them (range/range.py:213-238 with this model's temp, geo_temp and beta), largest first.
        With an M-sharded database (db_shard / db_group) this is a COLLECTIVE call: every rank passes its own queries
        and the same k, and gets the neighbours of its own rows over the whole database (distributed.py)."""
        eng, a = self.engine, self.args
        k = int(k)
        k_max = min(_lib.RANGE_TOPK_MAX, eng.db.M_total)       # the whole database: the same bound on every rank
        if not 1 <= k <= k_max:
            raise ValueError(f'k={k}: expected 1 <= k <= {k_max} (database of {eng.db.M_total} entries)')
        coords = coords.to(eng.device, torch.float64).contiguous()
        name = self.location_model_name
        geo_temp = float(getattr(a, 'geo_temp', 0.0))
        if self.sharded is not None:
            rows, weight = self.sharded.neighbours(name, coords, a.temp, geo_temp, getattr(a, 'beta', None),
                                                   self._sorts(), k)
            return eng.db.file_rows_global(rows), weight
        perm = None
        if self._sorts():
            coords, perm = eng.sort_queries(coords)
        _, q16, qxyz = eng.encode(coords)
        sums, _ = eng.retrieve_stats(name, q16, qxyz, a.temp, geo_temp)
        idx, weight = eng.retrieve_topk(name, q16, qxyz, a.temp, geo_temp, getattr(a, 'beta', None), sums, k, perm=perm)
        return eng.db.file_rows(idx), weight

    @staticmethod
    def _chunks(N, chunk, tail, taper=DEFAULT_TAPER):
        """[lo, hi) pieces of one super-batch.  Every piece's device->host copy overlaps the computation of the pieces
        after it, except the last one's: full chunks while more than two chunks' worth of rows remain, then every piece
        takes the fraction `taper` of what is left (whole rounds of the producer/consumer apply kernel - 24 units x 256
        rows on 148 SMs - while it is at least one round, else whole 128-row tiles), down to a last piece of about
        `tail` rows.  taper <= 0.64 keeps a piece's copy (5.6 M rows/s over PCIe) shorter than the computation that
        follows it (3.2 M rows/s).  No piece is longer than chunk + ROUND_ROWS - 1 rows."""
        cuts, lo = [], 0
        tail = max(1, tail)
        # The rows beyond whole rounds go into the FIRST piece: the apply kernel spreads such leftover tile pairs over
        # database ranges wherever they are, but at the end they would lengthen the one copy nothing overlaps
        # (100 000 rows: last piece 6 144 instead of 7 840 rows).
        ragged = N % ROUND_ROWS
        if ragged and chunk % ROUND_ROWS == 0 and tail % ROUND_ROWS == 0 and N - ragged >= chunk + tail:
            cuts.append((0, chunk + ragged)); lo = chunk + ragged
        while N - lo > 2 * chunk:
            cuts.append((lo, lo + chunk)); lo += chunk
        while N - lo > tail + tail // 2:
            rem = N - lo
            piece = int(rem * taper)
            if piece >= ROUND_ROWS:
                piece = piece // ROUND_ROWS * ROUND_ROWS
            elif piece >= 128:
                piece = piece // 128 * 128
            piece = min(chunk, max(piece, min(tail, rem)))
            if rem - piece < max(1, tail // 2):          # do not leave a sliver behind
                break
            cuts.append((lo, lo + piece)); lo += piece
        cuts.append((lo, N))
        return cuts

    @classmethod
    def _pieces(cls, N, chunk, tail, super_batch, taper=DEFAULT_TAPER):
        """(super-batches [s0, s1), their pieces [lo, hi) relative to s0, rows of the largest piece).  Buffers are sized
        for the largest piece of ANY super-batch: a short last super-batch can end in a longer piece than the first."""
        batches = [(s0, min(N, s0 + super_batch)) for s0 in range(0, N, super_batch)]
        plan = [cls._chunks(s1 - s0, chunk, tail, taper) for s0, s1 in batches]
        rows = max(hi - lo for cuts in plan for lo, hi in cuts)
        return batches, plan, rows

    @torch.no_grad()
    def forward(self, coords):
        """range.py:206-242.  Returns numpy float64 (N, 1280).  Per super-batch (<= 1M queries): every chunk is
        batched spatially, the encoder runs once over the whole super-batch (full-width launches), then chunk after
        chunk is retrieved on the current stream while the previous chunk's rows travel to pinned host memory on a
        copy stream."""
        if 'RANGE' not in self.location_model_name:
            raise NotImplementedError(f'{self.location_model_name} not implemented')
        coords = torch.as_tensor(coords)
        if coords.dim() != 2 or coords.shape[1] != 2:
            raise ValueError(f'coords must be (N, 2) (lon, lat) degrees, got {tuple(coords.shape)}')
        return self._forward_host(coords.shape[0], coords=coords)

    @torch.no_grad()
    def embed_into(self, coords, out):
        """forward() writing into the caller's float64 (N,1280) array - e.g. rows of a memory-mapped .npy
        (save.embed_to_npy): the rows cross PCIe packed into small page-locked staging buffers and a host thread team
        widens them straight into `out` while the GPU works on the next chunks ('packed' path of _forward_host)."""
        coords = torch.as_tensor(coords)
        if coords.dim() != 2 or coords.shape[1] != 2:
            raise ValueError(f'coords must be (N, 2) (lon, lat) degrees, got {tuple(coords.shape)}')
        if not (isinstance(out, np.ndarray) and out.dtype == np.float64 and out.shape == (coords.shape[0], 1280)
                and out.flags['C_CONTIGUOUS'] and out.flags['WRITEABLE']):
            raise ValueError('out must be a writable C-contiguous float64 (N, 1280) array')
        return self._forward_host(coords.shape[0], coords=coords, result=out)

    # ------------------------------------------------------------------ dense lat/lon rasters
    @staticmethod
    def coord_grid_axes(grid_size):
        """(lon_axis (W,), lat_axis (H,)) of the reference's coord_grid(grid_size=(H, W))
        (evaluation/visualize_embeddings.py:29-39): linspace(-180, 180, W) / linspace(90, -90, H) stored in a float32
        array and later promoted with .double().  Raster point p = i * W + j is (lon_axis[j], lat_axis[i])."""
        H, W = grid_size
        lon = np.linspace(-180, 180, W).astype(np.float32).astype(np.float64)
        lat = np.linspace(90, -90, H).astype(np.float32).astype(np.float64)
        return torch.from_numpy(lon), torch.from_numpy(lat)

    def _raster_ij(self, W, p0, p1):
        p = torch.arange(p0, p1, device=self.engine.device, dtype=torch.int64)
        return torch.stack((p // W, p % W), dim=1).to(torch.int32)

    @staticmethod
    def _raster_coords(tables, ij):
        return torch.stack((tables['lon'][ij[:, 1].long()], tables['lat'][ij[:, 0].long()]), dim=1)

    def raster_tables(self, lon_axis, lat_axis):
        """per-axis harmonics tables for embed_raster / forward_raster (build once per raster)"""
        eng = self.engine
        if eng.raster_supported():
            return eng.raster_tables(lon_axis, lat_axis)
        # closed-form harmonics / fp64 encoder: no separable evaluation, the per-point encoder runs on the coordinates
        lon = torch.as_tensor(lon_axis).to(eng.device, torch.float64).contiguous()
        lat = torch.as_tensor(lat_axis).to(eng.device, torch.float64).contiguous()
        return dict(H=lat.numel(), W=lon.numel(), buf=None, lon=lon, lat=lat)

    def _raster_lonlat(self, tables, p0, n):
        """(n,2) fp64 device coordinates of the raster points [p0, p0 + n), built on the device"""
        eng = self.engine
        if n == 0:
            return torch.empty(0, 2, dtype=torch.float64, device=eng.device)
        if tables['buf'] is None:
            return self._raster_coords(tables, self._raster_ij(tables['W'], p0, p0 + n)).contiguous()
        lonlat = torch.empty(n, 2, dtype=torch.float64, device=eng.device)
        eng.raster_points(tables, p0, n, lonlat=lonlat)
        return lonlat

    def _encode_raster(self, tables, ij):
        eng = self.engine
        if tables['buf'] is None:
            return eng.encode(self._raster_coords(tables, ij))
        return eng.encode_raster(tables, ij)[1:]

    @torch.no_grad()
    def embed_raster(self, lon_axis, lat_axis, rows=None, out=None, out_dtype=torch.float32, tables=None):
        """Device-resident dense-grid path (BASELINE config 5): the points [rows[0], rows[1]) of the lat-major raster
        lat_axis x lon_axis (point p = i * W + j, like coord_grid) -> (n, 1280) device tensor in raster order.  The
        harmonics are evaluated separably (once per distinct latitude / longitude, csrc/encoder_raster.cu); results
        are bit-identical to embed() on the same coordinates.
        With an M-sharded database (db_shard / db_group) this is a COLLECTIVE call: every rank passes the same axes and
        its own rows (e.g. its slab of the raster) and gets those points' rows over the whole database - the sharded
        embed() of the points' coordinates, built on the device (the per-point encoder: the separable one is no faster
        there and gives the same bits)."""
        eng = self.engine
        tables = self.raster_tables(lon_axis, lat_axis) if tables is None else tables
        p0, p1 = (0, tables['H'] * tables['W']) if rows is None else rows
        n = p1 - p0
        if self.sharded is not None:
            return self.embed(self._raster_lonlat(tables, p0, n), out=out, out_dtype=out_dtype)
        perm = None
        if tables['buf'] is None:              # no separable evaluation: the per-point encoder on the materialised coordinates
            ij = self._raster_ij(tables['W'], p0, p1)
            if self._sorts():
                _, perm = eng.sort_queries(self._raster_coords(tables, ij))
                ij = ij[perm.long()]
        else:                                  # index / coordinate rows come from the device (range_raster_points)
            if self._sorts():
                lonlat = torch.empty(n, 2, dtype=torch.float64, device=eng.device)
                eng.raster_points(tables, p0, n, lonlat=lonlat)
                _, perm = eng.sort_queries(lonlat)
            ij = torch.empty(n, 2, dtype=torch.int32, device=eng.device)
            eng.raster_points(tables, p0, n, perm=perm, ij=ij)
        q64, q16, qxyz = self._encode_raster(tables, ij)
        return self._retrieve_concat(q16, qxyz, q64, out, out_dtype, perm)

    @torch.no_grad()
    def forward_raster(self, lon_axis, lat_axis, rows=None, out=None):
        """model(coord_grid(...)) without building the coordinate list on the host: numpy float64 (H * W, 1280).
        rows=(p0, p1): only those raster points (a rank's slab); out: the caller's float64 (p1 - p0, 1280) array, e.g.
        rows of a memory-mapped .npy (filled through the packed path with bounded page-locked memory).
        With an M-sharded database (db_shard / db_group) this is a COLLECTIVE call like embed_raster: every rank passes
        the same axes and its own rows; its points' rows are computed on the device, then copied to the host."""
        tables = self.raster_tables(lon_axis, lat_axis)
        p0, p1 = (0, tables['H'] * tables['W']) if rows is None else rows
        if out is not None and not (isinstance(out, np.ndarray) and out.dtype == np.float64 and out.shape == (p1 - p0, 1280)
                                    and out.flags['C_CONTIGUOUS'] and out.flags['WRITEABLE']):
            raise ValueError('out must be a writable C-contiguous float64 (rows, 1280) array')
        return self._forward_host(p1 - p0, raster=tables, result=out, raster_p0=p0)

    def _forward_host(self, N, coords=None, raster=None, result=None, raster_p0=0):
        """model(locs) -> numpy float64 (N,1280) (range/range.py:222,240).  Two ways to hand the rows to the host:

        'copy'    chunk by chunk into device buffers; every chunk's float64 rows travel to the page-locked result on a
                  copy stream while the next chunk is computed (pieces get smaller towards the end: only the last
                  piece's copy is exposed).  Result page-locked: N * 10 KB.
        'packed'  the rows cross PCIe packed (6 KB: fp32 feature columns + fp64 location columns, RANGE_OUT_PACKED)
                  into small page-locked staging buffers and are widened into an ordinary (pageable) numpy array - or
                  the caller's array, embed_into - by a host thread team (range_host_unpack): bounded page-locked
                  memory for any N, 40 % fewer PCIe bytes, but the host cores must keep up (measured on the 16-core
                  1-GPU box: 6.3 M rows/s with 16 threads, 2.2 M queries/s end to end against 2.9 M for 'copy').
        'auto'    'copy' while the result fits `pinned_limit` (8 GB), else 'packed'.
        (Measured and dropped: letting the apply kernel's epilogue store straight into the mapped page-locked result -
        stores from the SMs to host memory run at ~6 GB/s and stall the consumers: 170 ms per 100 000 queries.)"""
        eng = self.engine
        path = self.host_path
        tdtype = torch.float32 if self.out_dtype == np.dtype(np.float32) and result is None else torch.float64
        row_bytes = 1280 * (4 if tdtype == torch.float32 else 8)
        if result is not None:
            path = 'packed'
        elif tdtype == torch.float32:
            path = 'copy'                          # nothing to widen: the rows are copied as they are
        elif path == 'auto':
            path = 'copy' if N * row_bytes <= self.pinned_limit else 'packed'
        if self.sharded is not None:            # collective: distributed.py chunks (every rank must take the same steps)
            if raster is None:
                dev = coords.to(eng.device, torch.float64, non_blocking=True)
            else:
                dev = self._raster_lonlat(raster, raster_p0, N)
            res = self.embed(dev, out_dtype=tdtype)
            host = torch.empty((N, 1280), dtype=tdtype, pin_memory=N * row_bytes <= self.pinned_limit)
            host.copy_(res)
            if result is None:
                return host.numpy()
            result[...] = host.numpy()
            return result
        if path == 'packed':
            result = np.empty((N, 1280), dtype=np.float64) if result is None else result
        else:
            host = torch.empty((N, 1280), dtype=tdtype, pin_memory=True)
            result = host.numpy()
        if N == 0:
            return result
        with torch.cuda.device(eng.index):
            if raster is None:
                dev_coords = coords.to(eng.device, torch.float64, non_blocking=True)
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(device=eng.device)
            chunk = min(self.chunk, N)
            batches, plan, rows = self._pieces(N, chunk, self.tail, self.super_batch, self.taper)
            n_pieces = sum(len(cuts) for cuts in plan)
            if path == 'copy':
                # three buffers: with two, piece i + 2 waits for the copy of piece i, which is still running when the
                # pieces shrink faster than their copies (measured: 0.9 ms stall before the fifth piece of 100 000 rows)
                bufs = [torch.empty(rows, 1280, dtype=tdtype, device=eng.device) for _ in range(min(3, n_pieces))]
            elif path == 'packed':
                depth = min(3, n_pieces)
                bufs = [torch.empty(rows, 6144, dtype=torch.uint8, device=eng.device) for _ in range(depth)]
                stage = [torch.empty(rows, 6144, dtype=torch.uint8, pin_memory=True) for _ in range(depth)]
                landed = [None] * depth          # (event, result rows, staging rows) of the piece in each slot
            freed = [None] * len(bufs)
            cur = torch.cuda.current_stream()
            if self.trace is not None:
                t0 = torch.cuda.Event(enable_timing=True)
                t0.record(cur)
                self.trace.append((0, t0, t0))

            def unpack(slot):
                ev, r0, r1 = landed[slot]
                ev.synchronize()
                _check_unpack(eng.lib.range_host_unpack(stage[slot].data_ptr(), r1 - r0, result[r0:r1].ctypes.data,
                                                        self.host_threads))
                landed[slot] = None

            i = 0
            for (s0, s1), cuts in zip(batches, plan):
                sort_cuts = cuts
                ij, perms = None, None
                if raster is not None and raster['buf'] is not None:
                    # dense raster: index / coordinate rows are produced on the device, chunk by chunk, straight into
                    # one (n,2) index array in batched order
                    n = s1 - s0
                    ij = torch.empty(n, 2, dtype=torch.int32, device=eng.device)
                    if self._sorts():
                        lonlat = torch.empty(n, 2, dtype=torch.float64, device=eng.device)
                        eng.raster_points(raster, raster_p0 + s0, n, lonlat=lonlat)
                        perms = []
                        for lo, hi in sort_cuts:
                            perms.append(eng.sort_queries(lonlat[lo:hi])[1])
                            eng.raster_points(raster, raster_p0 + s0 + lo, hi - lo, perm=perms[-1], ij=ij[lo:hi])
                    else:
                        eng.raster_points(raster, raster_p0 + s0, n, ij=ij)
                else:
                    if raster is None:
                        sub = dev_coords[s0:s1]
                    else:
                        ij = self._raster_ij(raster['W'], raster_p0 + s0, raster_p0 + s1)
                        sub = self._raster_coords(raster, ij)
                    if self._sorts():
                        # spatial batching chunk by chunk (a tile's 128 queries should be neighbours; the order of the
                        # chunks does not matter)
                        parts = [eng.sort_queries(sub[lo:hi]) for lo, hi in sort_cuts]
                        sub = torch.cat([p[0] for p in parts]) if len(parts) > 1 else parts[0][0]
                        perms = [p[1] for p in parts]
                        if ij is not None:
                            ij = torch.cat([ij[lo:hi][p.long()] for (lo, hi), p in zip(sort_cuts, perms)])
                q64, q16, qxyz = eng.encode(sub) if ij is None else self._encode_raster(raster, ij)
                for c, (lo, hi) in enumerate(cuts):
                    perm = None if perms is None else perms[c]
                    k = i % len(bufs)
                    i += 1
                    if path == 'packed' and landed[k] is not None:
                        unpack(k)                              # the slot's previous piece: wait for its copy, widen it
                    if freed[k] is not None:
                        cur.wait_event(freed[k])
                    buf = bufs[k][: hi - lo]
                    assert buf.shape[0] == hi - lo
                    self._retrieve_concat(q16[lo:hi], qxyz[lo:hi], q64[lo:hi], buf, buf.dtype, perm)
                    timed = self.trace is not None            # developer timeline (tools/time_e2e.py)
                    ready = torch.cuda.Event(enable_timing=timed)
                    ready.record(cur)
                    self._copy_stream.wait_event(ready)
                    with torch.cuda.stream(self._copy_stream):
                        if path == 'copy':
                            host[s0 + lo:s0 + hi].copy_(buf, non_blocking=True)
                        else:
                            stage[k][: hi - lo].copy_(buf, non_blocking=True)
                        freed[k] = torch.cuda.Event(enable_timing=timed)
                        freed[k].record(self._copy_stream)
                    if timed:
                        self.trace.append((hi - lo, ready, freed[k]))
                    if path == 'packed':
                        landed[k] = (freed[k], s0 + lo, s0 + hi)
            if path == 'packed':
                for k in sorted((k for k in range(len(bufs)) if landed[k] is not None), key=lambda k: landed[k][1]):
                    unpack(k)
            else:
                self._copy_stream.synchronize()
        return result                                                                     # range.py:222,240


def _check_unpack(code):
    if code != 0:
        raise RuntimeError(f'range_host_unpack failed ({code})')
