"""Device-side engine: owns a range_ctx (C ABI) and the torch tensors it borrows.

PyTorch is plumbing here (device memory, streams); every computation is a kernel of librange_b200.so.
"""
import ctypes
from ctypes import c_int32, c_void_p

import numpy as np
import torch

from . import _lib
from .sh_table import build_table, closed_form_norms

MODE = {"RANGE": _lib.RANGE_MODE_RANGE, "RANGE+": _lib.RANGE_MODE_RANGE_PLUS}


def _ptr(t):
    return c_void_p(t.data_ptr())


def _stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


# result layouts of the concat step: numpy float64 (what the reference returns), float32, or packed rows of 6144 bytes
# (1024 fp32 + 256 fp64, include/range_b200.h: RANGE_OUT_PACKED) held in a uint8 tensor
PACKED_ROW_BYTES = 6144


def _out_code(t):
    if t.dtype == torch.float64:
        return _lib.RANGE_OUT_F64
    if t.dtype == torch.float32:
        return _lib.RANGE_OUT_F32
    if t.dtype == torch.uint8 and t.shape[-1] == PACKED_ROW_BYTES:
        return _lib.RANGE_OUT_PACKED
    raise ValueError(f"result tensor must be float64 / float32 (N,1280) or uint8 (N,{PACKED_ROW_BYTES}), got "
                     f"{t.dtype} {tuple(t.shape)}")


def _new_out(N, dtype, device):
    if dtype == torch.uint8:
        return torch.empty(N, PACKED_ROW_BYTES, dtype=torch.uint8, device=device)
    return torch.empty(N, 1280, dtype=dtype, device=device)


class RangeEngine:
    def __init__(self, device, encoder=None, database=None, L=None, encoder_precision="auto", harmonics=None):
        """encoder: dict from checkpoint.load_satclip_location_encoder (or None: SH only with `L`);
        database: database.DeviceDatabase or None;
        encoder_precision: 'fp64' (the reference's arithmetic, DMMA), 'f16x3' (tensor cores, split fp16 operands,
        fp32-class accuracy; 'tf32x3' is accepted as an alias) or 'auto' (= f16x3 when the layer widths allow it, else fp64)."""
        self.encoder_precision = encoder_precision
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.RangeError(f"range_b200 runs on CUDA (sm_100a) devices only, got device={device!r}; "
                                  "there is no CPU path")
        if not torch.cuda.is_available():
            raise _lib.RangeError("no CUDA device is available; range_b200 has no CPU path")
        self.lib = _lib.load()
        self.index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", self.index)
        ctx = c_void_p()
        with torch.cuda.device(self.index):
            _lib.check(self.lib.range_ctx_create(self.index, ctypes.byref(ctx)))
        self.ctx = ctx
        self._ws = {}
        self.db = None
        self.L = int(encoder["L"]) if encoder is not None else int(L)
        # spherical harmonics: the generated polynomials ('analytic', the SatCLIP-L40 checkpoint) or the recurrence
        self.harmonics = harmonics or (encoder or {}).get("harmonics_calculation", "analytic")
        if self.harmonics == "analytic":
            t = build_table(self.L)
            self._tab = dict(pref=torch.from_numpy(t["pref"]).to(self.device),
                             off=torch.from_numpy(t["off"]).to(self.device),
                             coef=torch.from_numpy(t["coef"]).to(self.device),
                             par=torch.from_numpy(t["par"]).to(self.device))
            _lib.check(self.lib.range_ctx_set_sh_table(self.ctx, self.L, len(t["pref"]), _ptr(self._tab["pref"]),
                                                       _ptr(self._tab["off"]), _ptr(self._tab["coef"]),
                                                       _ptr(self._tab["par"])))
        elif self.harmonics == "closed-form":
            self._tab = dict(norm=torch.from_numpy(closed_form_norms(self.L)).to(self.device))
            _lib.check(self.lib.range_ctx_set_sh_closed_form(self.ctx, self.L, self._tab["norm"].numel(),
                                                             _ptr(self._tab["norm"])))
        else:
            raise ValueError(f"harmonics_calculation={self.harmonics!r}: expected 'analytic' or 'closed-form'")
        self.dims = None
        if encoder is not None:
            self.set_encoder(encoder)
        if database is not None:
            self.set_database(database)

    def __del__(self):
        try:
            if getattr(self, "ctx", None):
                self.lib.range_ctx_destroy(self.ctx)
                self.ctx = None
        except Exception:
            pass

    # ------------------------------------------------------------------ setup
    def set_encoder(self, enc, w0_first=30.0, w0_hidden=1.0):
        self._weights = [(w.to(self.device, torch.float64).contiguous(), b.to(self.device, torch.float64).contiguous())
                         for w, b in enc["weights"]]
        enc_dims = [int(d) for d in enc["dims"]]
        if enc_dims[0] % 16:            # e.g. SatCLIP-L10: 100 features -> zero-padded input columns (fp64 encoder)
            pad = 16 - enc_dims[0] % 16
            w0, b0 = self._weights[0]
            self._weights[0] = (torch.nn.functional.pad(w0, (0, pad)).contiguous(), b0)
            enc_dims[0] += pad
        n = len(self._weights)
        dims = (c_int32 * (n + 1))(*enc_dims)
        W = (c_void_p * n)(*[w.data_ptr() for w, _ in self._weights])
        B = (c_void_p * n)(*[b.data_ptr() for _, b in self._weights])
        _lib.check(self.lib.range_ctx_set_encoder(self.ctx, n, dims, W, B, w0_first, w0_hidden))
        self.dims = enc_dims
        self._prepared = None
        self.precision = "fp64"
        want = "f16x3" if self.encoder_precision == "tf32x3" else self.encoder_precision
        nbytes = self.lib.range_encoder_prepared_bytes(self.ctx)
        if want == "f16x3" and nbytes == 0:
            raise _lib.RangeError("encoder_precision='f16x3' needs every SIREN width to be a multiple of 256")
        if want in ("auto", "f16x3") and nbytes > 0:
            self._prepared = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
            with torch.cuda.device(self.index):
                _lib.check(self.lib.range_ctx_prepare_encoder(self.ctx, _ptr(self._prepared), int(nbytes), _stream()))
            self.precision = "f16x3"

    def set_database(self, db):
        _lib.check(self.lib.range_ctx_set_db(self.ctx, db.M, db.Mpad, _ptr(db.Kh), _ptr(db.Vt), _ptr(db.xyz),
                                             float(db.vscale)))
        if getattr(db, "caps", None) is not None:
            _lib.check(self.lib.range_ctx_set_db_caps(self.ctx, db.caps.shape[0], _ptr(db.caps), db.M_total))
        self.db = db

    def _workspace(self, key, nbytes):
        buf = self._ws.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
            self._ws[key] = buf
        return buf

    # ------------------------------------------------------------------ kernels
    def sh_features(self, lonlat):
        """(N,2) fp64 device tensor -> (N, L*L) fp64 (a transposed view of the feature-major buffer)"""
        lonlat = lonlat.to(self.device, torch.float64).contiguous()
        N = lonlat.shape[0]
        ld = (N + 127) // 128 * 128
        Yt = torch.empty(self.L * self.L, ld, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.range_sh_features(self.ctx, N, _ptr(lonlat), _ptr(Yt), ld, _stream()))
        return Yt[:, :N].t()

    def sort_queries(self, lonlat):
        """(N,2) fp64 device tensor -> (lonlat_sorted (N,2), perm (N,) int32): spatial batching for RANGE+.
        perm[i] is the caller's row of sorted row i; hand it to concat()."""
        lonlat = lonlat.to(self.device, torch.float64).contiguous()
        N = lonlat.shape[0]
        out = torch.empty_like(lonlat)
        perm = torch.empty(N, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.index):
            ws = self._workspace("sort", self.lib.range_sort_workspace_bytes(self.ctx, N))
            _lib.check(self.lib.range_sort_queries(self.ctx, N, _ptr(lonlat), _ptr(out), _ptr(perm), _ptr(ws),
                                                   ws.numel(), _stream()))
        return out, perm

    def geo_mask(self, qxyz, geo_temp, sums=None):
        """diagnostic: (query tiles, database tiles) bool tensor, True = the geo term of that tile pair is skipped;
        sums (from retrieve_stats) selects the tighter mask of the apply pass"""
        N = qxyz.shape[0]
        rows, words = c_int32(), c_int32()
        _lib.check(self.lib.range_geo_mask_shape(self.ctx, N, ctypes.byref(rows), ctypes.byref(words)))
        mask = torch.zeros(rows.value, words.value, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.range_geo_mask(self.ctx, N, _ptr(qxyz), float(geo_temp),
                                               c_void_p(None) if sums is None else _ptr(sums), _ptr(mask), _stream()))
        bits = (mask.unsqueeze(-1) >> torch.arange(32, device=self.device, dtype=torch.int32)) & 1
        return bits.reshape(rows.value, -1)[: (N + 127) // 128, : self.db.Mpad // 128].bool()

    def encode(self, lonlat, q64=None, q16=None, qxyz=None):
        lonlat = lonlat.to(self.device, torch.float64).contiguous()
        N = lonlat.shape[0]
        q64 = torch.empty(N, 256, dtype=torch.float64, device=self.device) if q64 is None else q64
        q16 = torch.empty(N, 256, dtype=torch.float16, device=self.device) if q16 is None else q16
        qxyz = torch.empty(N, 4, dtype=torch.float32, device=self.device) if qxyz is None else qxyz
        with torch.cuda.device(self.index):
            nbytes = self.lib.range_encode_workspace_bytes(self.ctx, N)
            ws = self._workspace("enc", nbytes)
            _lib.check(self.lib.range_encode(self.ctx, N, _ptr(lonlat), _ptr(q64), _ptr(q16), _ptr(qxyz), _ptr(ws),
                                             ws.numel(), _stream()))
        return q64, q16, qxyz

    def raster_tables(self, lon_axis, lat_axis):
        """Per-axis tables of a lat/lon raster (encoder_raster.cu): the latitude factor of every harmonic for each
        distinct latitude, cos/sin(m phi) for each distinct longitude.  Returns an opaque handle for encode_raster."""
        lon = torch.as_tensor(lon_axis).to(self.device, torch.float64).contiguous()
        lat = torch.as_tensor(lat_axis).to(self.device, torch.float64).contiguous()
        H, W = lat.numel(), lon.numel()
        with torch.cuda.device(self.index):
            nbytes = self.lib.range_raster_tables_bytes(self.ctx, H, W)
            buf = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            _lib.check(self.lib.range_raster_tables(self.ctx, H, _ptr(lat), W, _ptr(lon), _ptr(buf), buf.numel(),
                                                    _stream()))
        return dict(H=H, W=W, buf=buf, lon=lon, lat=lat)

    def raster_points(self, tables, p0, n, perm=None, ij=None, lonlat=None):
        """rows of the raster points p0 + (perm[k] if perm is given else k), k < n, written into the given tensors:
        ij (n,2) int32 (latitude index, longitude index) and / or lonlat (n,2) fp64 - built on the device"""
        with torch.cuda.device(self.index):
            _lib.check(self.lib.range_raster_points(
                self.ctx, tables["H"], tables["W"], _ptr(tables["buf"]), int(p0), int(n),
                c_void_p(None) if perm is None else _ptr(perm), c_void_p(None) if ij is None else _ptr(ij),
                c_void_p(None) if lonlat is None else _ptr(lonlat), _stream()))
        return ij, lonlat

    def encode_raster(self, tables, ij):
        """ij (N,2) int32 = (latitude index, longitude index) -> (lonlat (N,2) fp64, q64, q16, qxyz); bit-identical to
        encode() on those coordinates, without re-evaluating the harmonics' latitude / longitude factors per point."""
        ij = ij.to(self.device, torch.int32).contiguous()
        N = ij.shape[0]
        lonlat = torch.empty(N, 2, dtype=torch.float64, device=self.device)
        q64 = torch.empty(N, 256, dtype=torch.float64, device=self.device)
        q16 = torch.empty(N, 256, dtype=torch.float16, device=self.device)
        qxyz = torch.empty(N, 4, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.index):
            ws = self._workspace("enc", self.lib.range_encode_workspace_bytes(self.ctx, N))
            _lib.check(self.lib.range_encode_raster(self.ctx, tables["H"], tables["W"], _ptr(tables["buf"]), N, _ptr(ij),
                                                    _ptr(lonlat), _ptr(q64), _ptr(q16), _ptr(qxyz), _ptr(ws), ws.numel(),
                                                    _stream()))
        return lonlat, q64, q16, qxyz

    def raster_supported(self):
        """the separable raster encoder needs the analytic harmonics and the tensor-core SIREN"""
        return self.harmonics == "analytic" and getattr(self, "precision", None) == "f16x3"

    def _ret_ws(self, N):
        return self._workspace("ret", self.lib.range_retrieve_workspace_bytes(self.ctx, N))

    def retrieve(self, mode, q16, qxyz, temp, geo_temp, beta, O=None):
        N = q16.shape[0]
        O = torch.empty(N, 1024, dtype=torch.float32, device=self.device) if O is None else O
        with torch.cuda.device(self.index):
            ws = self._ret_ws(N)
            _lib.check(self.lib.range_retrieve(self.ctx, MODE[mode], N, _ptr(q16), _ptr(qxyz), temp, geo_temp,
                                               0.0 if beta is None else float(beta), _ptr(O), _ptr(ws), ws.numel(),
                                               _stream()))
        return O

    def retrieve_stats(self, mode, q16, qxyz, temp, geo_temp):
        N = q16.shape[0]
        sums = torch.empty(N, 2, dtype=torch.float32, device=self.device)
        maxs = torch.empty(N, 2, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.index):
            ws = self._ret_ws(N)
            _lib.check(self.lib.range_retrieve_stats(self.ctx, MODE[mode], N, _ptr(q16), _ptr(qxyz), temp, geo_temp,
                                                     _ptr(sums), _ptr(maxs), _ptr(ws), ws.numel(), _stream()))
        return sums, maxs

    def retrieve_topk(self, mode, q16, qxyz, temp, geo_temp, beta, sums, k, perm=None):
        """the k largest retrieval weights of every query (sums from retrieve_stats): (idx (N,k) int32 device database
        rows, weight (N,k) fp32), descending; row n of the result at row perm[n] (perm from sort_queries)"""
        N = q16.shape[0]
        idx = torch.empty(N, k, dtype=torch.int32, device=self.device)
        weight = torch.empty(N, k, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.index):
            ws = self._workspace("topk", max(1, self.lib.range_topk_workspace_bytes(self.ctx, N, k)))
            _lib.check(self.lib.range_retrieve_topk(
                self.ctx, MODE[mode], N, _ptr(q16), _ptr(qxyz), temp, geo_temp, 0.0 if beta is None else float(beta),
                _ptr(sums), k, c_void_p(None) if perm is None else _ptr(perm), _ptr(idx), _ptr(weight), _ptr(ws),
                ws.numel(), _stream()))
        return idx, weight

    def retrieve_topk_rows(self, mode, q16, qxyz, temp, geo_temp, beta, sums, k, row0):
        """retrieve_topk as one shard of an M-sharded database (sums: the global ones): entries are row0 + device row
        (rows of the whole sorted database with row0 = db.row_range[0]), k may exceed this shard's M (unfilled slots:
        entry -1, weight 0), row n of the result is query n"""
        N = q16.shape[0]
        idx = torch.empty(N, k, dtype=torch.int32, device=self.device)
        weight = torch.empty(N, k, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.index):
            ws = self._workspace("topk", max(1, self.lib.range_topk_workspace_bytes(self.ctx, N, k)))
            _lib.check(self.lib.range_retrieve_topk_rows(
                self.ctx, MODE[mode], N, _ptr(q16), _ptr(qxyz), temp, geo_temp, 0.0 if beta is None else float(beta),
                _ptr(sums), k, int(row0), _ptr(idx), _ptr(weight), _ptr(ws), ws.numel(), _stream()))
        return idx, weight

    def topk_merge(self, part_w, part_idx, perm=None):
        """(parts, N, k) fp32 / int32 lists (each sorted by weight descending, then entry; -1 entries last) -> the merged
        (idx (N,k) int32, weight (N,k) fp32), row n at row perm[n]"""
        parts, N, k = part_w.shape
        if part_idx.shape != part_w.shape or part_w.dtype != torch.float32 or part_idx.dtype != torch.int32 \
                or not (part_w.is_contiguous() and part_idx.is_contiguous()):
            raise ValueError(f"part_w / part_idx must be contiguous (parts, N, k) float32 / int32, got "
                             f"{part_w.dtype} {tuple(part_w.shape)}, {part_idx.dtype} {tuple(part_idx.shape)}")
        idx = torch.empty(N, k, dtype=torch.int32, device=self.device)
        weight = torch.empty(N, k, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.range_topk_merge(self.ctx, parts, N, k, _ptr(part_w), _ptr(part_idx),
                                                 c_void_p(None) if perm is None else _ptr(perm), _ptr(idx),
                                                 _ptr(weight), _stream()))
        return idx, weight

    def retrieve_apply(self, mode, q16, qxyz, temp, geo_temp, beta, sums, maxs, O=None):
        N = q16.shape[0]
        O = torch.empty(N, 1024, dtype=torch.float32, device=self.device) if O is None else O
        with torch.cuda.device(self.index):
            ws = self._ret_ws(N)
            _lib.check(self.lib.range_retrieve_apply(self.ctx, MODE[mode], N, _ptr(q16), _ptr(qxyz), temp, geo_temp,
                                                     0.0 if beta is None else float(beta), _ptr(sums), _ptr(maxs),
                                                     _ptr(O), _ptr(ws), ws.numel(), _stream()))
        return O

    def retrieve_apply_concat(self, mode, q16, qxyz, temp, geo_temp, beta, sums, maxs, q64, out=None,
                              dtype=torch.float64, perm=None):
        """apply pass + concat in one call: (N,1280) = [retrieved feature | q64], row n at out[perm[n]]"""
        N = q16.shape[0]
        out = _new_out(N, dtype, self.device) if out is None else out
        code = _out_code(out)
        with torch.cuda.device(self.index):
            ws = self._ret_ws(N)
            _lib.check(self.lib.range_retrieve_apply_concat(
                self.ctx, MODE[mode], N, _ptr(q16), _ptr(qxyz), temp, geo_temp, 0.0 if beta is None else float(beta),
                _ptr(sums), _ptr(maxs), _ptr(q64), c_void_p(None) if perm is None else _ptr(perm), _ptr(out), code,
                _ptr(ws), ws.numel(), _stream()))
        return out

    def retrieve_concat(self, mode, q16, qxyz, temp, geo_temp, beta, q64, out=None, dtype=torch.float64, perm=None):
        """statistics + apply + concat in one call (unsharded database): (N,1280) = [retrieved feature | q64], row n at
        out[perm[n]]"""
        N = q16.shape[0]
        out = _new_out(N, dtype, self.device) if out is None else out
        with torch.cuda.device(self.index):
            ws = self._ret_ws(N)
            _lib.check(self.lib.range_retrieve_concat(
                self.ctx, MODE[mode], N, _ptr(q16), _ptr(qxyz), temp, geo_temp, 0.0 if beta is None else float(beta),
                _ptr(q64), c_void_p(None) if perm is None else _ptr(perm), _ptr(out), _out_code(out), _ptr(ws), ws.numel(),
                _stream()))
        return out

    def concat(self, O, q64, out=None, dtype=torch.float64, perm=None):
        """[O | q64] -> (N,1280); with perm (from sort_queries) row n is written to out[perm[n]]"""
        N = O.shape[0]
        out = _new_out(N, dtype, self.device) if out is None else out
        code = _out_code(out)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.range_concat_scatter(self.ctx, N, _ptr(O), _ptr(q64),
                                                     c_void_p(None) if perm is None else _ptr(perm), _ptr(out), code,
                                                     _stream()))
        return out

    def retrieve_apply_routed(self, mode, q16, qxyz, temp, geo_temp, beta, sums, maxs, route):
        """apply pass of an M-sharded database: this shard's partial rows leave from the kernel's epilogue into the
        owner ranks' receive buffers (route: _lib.Route with the mapped peer pointers)"""
        N = q16.shape[0]
        with torch.cuda.device(self.index):
            ws = self._ret_ws(N)
            _lib.check(self.lib.range_retrieve_apply_routed(
                self.ctx, MODE[mode], N, _ptr(q16), _ptr(qxyz), temp, geo_temp, 0.0 if beta is None else float(beta),
                _ptr(sums), _ptr(maxs), ctypes.byref(route), _ptr(ws), ws.numel(), _stream()))

    def combine_concat(self, parts, weights, q64, out=None, dtype=torch.float64, perm=None):
        """out[perm[n]] = [sum_k weights[k] parts[k][n] | q64[n]]: the slots of an M-sharded receive buffer
        (weights None = 1) or the two ends of a beta sweep, (1 - beta) O(0) + beta O(1)"""
        N = q64.shape[0]
        n = len(parts)
        ptrs = []
        for p in parts:                       # tensors, or raw device addresses (slots of a peer receive buffer)
            if isinstance(p, int):
                ptrs.append(p)
                continue
            if p.dtype != torch.float32 or p.shape != (N, 1024) or not p.is_contiguous():
                raise ValueError(f"parts must be contiguous (N,1024) float32, got {p.dtype} {tuple(p.shape)}")
            ptrs.append(p.data_ptr())
        out = _new_out(N, dtype, self.device) if out is None else out
        P = (c_void_p * n)(*ptrs)
        W = None if weights is None else (ctypes.c_float * n)(*[float(w) for w in weights])
        with torch.cuda.device(self.index):
            _lib.check(self.lib.range_combine_concat(self.ctx, N, n, P, W, _ptr(q64),
                                                     c_void_p(None) if perm is None else _ptr(perm), _ptr(out),
                                                     _out_code(out), _stream()))
        return out

    def sweep_concat(self, geo_parts, sem_parts, betas, q64, out_dtype=torch.float32, perm=None, outs=None):
        """[(1 - beta) G[n] + beta S[n] | q64[n]] at row perm[n] for every beta: G / S = the sum of the slots geo_parts /
        sem_parts (the geographic and semantic ends of a beta sweep; tensors or raw device addresses, (N,1024) fp32),
        each slot read once per RANGE_SWEEP_MAX_BETAS beta.  Returns a list of (N,1280) tensors in out_dtype (float64 or
        float32), or fills `outs` (one per beta)."""
        N = q64.shape[0]
        if len(geo_parts) != len(sem_parts):
            raise ValueError(f"{len(geo_parts)} geo slots but {len(sem_parts)} sem slots")

        def addresses(parts):
            ptrs = []
            for p in parts:
                if isinstance(p, int):
                    ptrs.append(p)
                    continue
                if p.dtype != torch.float32 or p.shape != (N, 1024) or not p.is_contiguous():
                    raise ValueError(f"slots must be contiguous (N,1024) float32, got {p.dtype} {tuple(p.shape)}")
                ptrs.append(p.data_ptr())
            return (c_void_p * len(ptrs))(*ptrs)

        G, S = addresses(geo_parts), addresses(sem_parts)
        betas = [float(b) for b in betas]
        if outs is None:
            if out_dtype not in (torch.float64, torch.float32):
                raise ValueError(f"out_dtype={out_dtype}: expected torch.float64 or torch.float32")
            outs = [_new_out(N, out_dtype, self.device) for _ in betas]
        if len(outs) != len(betas):
            raise ValueError(f"{len(outs)} outputs for {len(betas)} beta")
        codes = {_out_code(o) for o in outs}
        if len(codes) > 1:
            raise ValueError("every output of a sweep must have the same dtype")
        for o in outs:
            width = PACKED_ROW_BYTES if _out_code(o) == _lib.RANGE_OUT_PACKED else 1280
            if o.shape != (N, width) or not o.is_contiguous():
                raise ValueError(f"outputs must be contiguous ({N}, {width}), got {tuple(o.shape)}")
        if N == 0:
            return outs
        step = _lib.RANGE_SWEEP_MAX_BETAS              # the kernel's limit: longer lists in groups
        with torch.cuda.device(self.index):
            for b0 in range(0, len(betas), step):
                bs, group = betas[b0:b0 + step], outs[b0:b0 + step]
                n = len(bs)
                # the weights are rounded to fp32 here, like combine_concat's (1 - beta, beta) in the unsharded sweep
                _lib.check(self.lib.range_sweep_concat(
                    self.ctx, N, len(geo_parts), G, S, n, (ctypes.c_float * n)(*[1.0 - b for b in bs]),
                    (ctypes.c_float * n)(*bs), _ptr(q64), c_void_p(None) if perm is None else _ptr(perm),
                    (c_void_p * n)(*[o.data_ptr() for o in group]), _out_code(group[0]), _stream()))
        return outs
