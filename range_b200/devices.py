"""Queries split over database replicas on the GPUs of one process (`load_model(..., devices=...)`).

The database is prepared once on the primary device (the first entry of `devices`) and copied device to device to the
others (DeviceDatabase.replicate); every device gets its own RangeEngine.  A call splits its rows into contiguous slabs
(split_rows) and every replica runs the unchanged single-device code on its slab, so the rows of a multi-device call are
bit for bit the rows the same single-device call returns for each slab.  Device-resident results are gathered on the
primary (or wherever the caller's `out=` lives), host results are written by each device into its own rows of one array.

Execution: one thread per physical device, the primary's being the calling thread.  Replicas that share a physical
device (duplicate entries: a way to test the path on one GPU, no faster than one replica) run one after the other in the
same thread: the producer/consumer apply kernel needs every CTA pair of its GPU resident, so two of its launches must
never be in flight on one GPU at once.  Every thread works on the streams that are current on the calling thread, so a
result is ordered on the caller's stream exactly like a single-device one.
"""
import copy
import threading

import torch

from .engine import RangeEngine, _new_out
from .range import ROUND_ROWS


def split_rows(N, n_devices):
    """[(lo, hi), ...]: contiguous slabs covering [0, N) in device order.  Every slab but the first is whole rounds of the
    apply kernel (ROUND_ROWS), the rounds are spread to within one, and the rows beyond whole rounds go to the first slab
    (as in LocationEncoder._chunks); the extra rounds go to the last slabs, so no two slabs differ by more than a round
    of rows.  Fewer than two rounds run as one slab: splitting them costs launches and gains nothing."""
    rounds = N // ROUND_ROWS
    n = max(1, min(int(n_devices), rounds))
    if N < 2 * ROUND_ROWS or n == 1:
        return [(0, N)]
    base, extra = divmod(rounds, n)
    sizes = [(base + (i >= n - extra)) * ROUND_ROWS for i in range(n)]
    sizes[0] += N - rounds * ROUND_ROWS
    cuts, lo = [], 0
    for s in sizes:
        cuts.append((lo, lo + s))
        lo += s
    return cuts


def check_devices(devices):
    """`devices` of load_model -> list of CUDA torch.device with their indices; ValueError for an empty list, a device
    that is not CUDA (both before any CUDA call) or one that is not visible.  An int n is the first n visible GPUs, 'all'
    every visible GPU; a list holds indices or 'cuda:i' strings."""
    if isinstance(devices, str) and devices == 'all':
        n = torch.cuda.device_count()
        if n == 0:
            raise ValueError("devices='all': no CUDA device is visible")
        return [torch.device('cuda', i) for i in range(n)]
    if isinstance(devices, int) and not isinstance(devices, bool):
        if devices < 1:
            raise ValueError(f'devices={devices}: expected at least one device')
        devices = list(range(devices))
    if isinstance(devices, (str, torch.device)) or not hasattr(devices, '__iter__'):
        raise ValueError(f"devices={devices!r}: expected an int, 'all' or a list of device indices / 'cuda:i' strings")
    out = []
    for d in devices:
        dev = torch.device('cuda', d) if isinstance(d, int) and not isinstance(d, bool) else torch.device(d)
        if dev.type != 'cuda':
            raise ValueError(f'devices: {d!r} is not a CUDA device (range_b200 runs on CUDA devices only)')
        out.append(dev)
    if not out:
        raise ValueError('devices: empty list; expected at least one device')
    count = torch.cuda.device_count()
    for i, dev in enumerate(out):
        out[i] = dev = torch.device('cuda', torch.cuda.current_device() if dev.index is None else dev.index)
        if dev.index >= count:
            raise ValueError(f'devices: {dev} is not visible ({count} CUDA devices)')
    return out


def _single(model, engine):
    """a single-device LocationEncoder over `engine` with model's settings (its own copy stream and trace)"""
    rep = copy.copy(model)
    rep.engine, rep.replicas, rep._copy_stream, rep.trace = engine, None, None, None
    return rep


class Replicas:
    """The single-device models of a multi-device LocationEncoder, one per entry of `devices`: models[0] runs on the
    primary's engine, the others on engines of their own over replicas of its database."""

    def __init__(self, model, encoder, devices):
        db = model.engine.db
        self.models = [_single(model, model.engine)]
        for dev in devices[1:]:
            eng = RangeEngine(dev, encoder=encoder, database=db.replicate(dev),
                              retrieval_precision=model.args.retrieval_precision)
            self.models.append(_single(model, eng))

    def close(self):
        self.models = []

    def slabs(self, N):
        """the slabs of an N-row call, or None when it runs on the primary alone"""
        cuts = split_rows(N, len(self.models))
        return cuts if len(cuts) > 1 else None

    def run(self, slabs, work):
        """[work(i, model i, lo, hi) for slab i = (lo, hi)] with slab i on replica i: the physical devices in parallel, the
        replicas of one device one after the other.  If one raises, the others finish first, then the first error is
        raised again."""
        out = [None] * len(slabs)
        groups = {}
        for i in range(len(slabs)):
            groups.setdefault(self.models[i].engine.index, []).append(i)
        streams = {d: torch.cuda.current_stream(d) for d in groups}
        errors = []

        def drain(d):
            try:
                with torch.cuda.device(d), torch.cuda.stream(streams[d]), torch.no_grad():
                    for i in groups[d]:
                        out[i] = work(i, self.models[i], *slabs[i])
            except BaseException as e:          # noqa: B036 - re-raised on the calling thread
                errors.append(e)

        primary = self.models[0].engine.index
        threads = [threading.Thread(target=drain, args=(d,)) for d in groups if d != primary]
        for t in threads:
            t.start()
        try:
            drain(primary)
        finally:
            for t in threads:
                t.join()
        if errors:
            raise errors[0]
        return out

    def _inputs(self, x, slabs):
        """slab i of x for replica i: host rows stay where they are (the replica copies them itself), device rows on
        another GPU are copied here, on the calling thread's streams, before any slab's work is queued"""
        parts = []
        for i, (lo, hi) in enumerate(slabs):
            part = x[lo:hi]
            dev = self.models[i].engine.device
            parts.append(part.to(dev) if part.is_cuda and part.device != dev else part)
        return parts

    @staticmethod
    def _gather(dst, slabs, pieces):
        """dst[lo:hi] = piece for the pieces not written in place (None); device to device on the calling thread"""
        for (lo, hi), piece in zip(slabs, pieces):
            if piece is not None:
                dst[lo:hi].copy_(piece)
        return dst

    def _raster_tables(self, tables, slabs):
        """raster_tables of each slab's replica, built on the calling thread (the caller's tables where they live)"""
        return [tables if m.engine.device == tables['lon'].device else m.raster_tables(tables['lon'], tables['lat'])
                for m in self.models[:len(slabs)]]

    # ------------------------------------------------------------------ entry points (LocationEncoder's)
    def embed(self, coords, slabs, out, out_dtype):
        eng = self.models[0].engine
        out = _new_out(coords.shape[0], out_dtype, eng.device, eng.value_dim) if out is None else out
        xs = self._inputs(coords, slabs)

        def work(i, m, lo, hi):
            if m.engine.device == out.device:
                m.embed(xs[i], out=out[lo:hi])
                return None
            return m.embed(xs[i], out_dtype=out.dtype)
        return self._gather(out, slabs, self.run(slabs, work))

    def embed_raster(self, tables, p0, slabs, out, out_dtype):
        eng = self.models[0].engine
        n = slabs[-1][1]
        out = _new_out(n, out_dtype, eng.device, eng.value_dim) if out is None else out
        tabs = self._raster_tables(tables, slabs)

        def work(i, m, lo, hi):
            if m.engine.device == out.device:
                m.embed_raster(None, None, rows=(p0 + lo, p0 + hi), out=out[lo:hi], tables=tabs[i])
                return None
            return m.embed_raster(None, None, rows=(p0 + lo, p0 + hi), out_dtype=out.dtype, tables=tabs[i])
        return self._gather(out, slabs, self.run(slabs, work))

    def embed_sweep(self, coords, slabs, betas, out_dtype):
        eng = self.models[0].engine
        xs = self._inputs(coords, slabs)
        pieces = self.run(slabs, lambda i, m, lo, hi: m.embed_sweep(xs[i], betas, out_dtype=out_dtype))
        N = coords.shape[0]
        outs = [_new_out(N, out_dtype, eng.device, eng.value_dim) for _ in betas]
        for b, o in enumerate(outs):
            self._gather(o, slabs, [p[b] for p in pieces])
        return outs

    def neighbours(self, coords, slabs, k):
        eng = self.models[0].engine
        xs = self._inputs(coords, slabs)
        pieces = self.run(slabs, lambda i, m, lo, hi: m.neighbours(xs[i], k))
        N = coords.shape[0]
        idx = self._gather(torch.empty(N, k, dtype=torch.int64, device=eng.device), slabs, [p[0] for p in pieces])
        weight = self._gather(torch.empty(N, k, dtype=torch.float32, device=eng.device), slabs, [p[1] for p in pieces])
        return idx, weight

    def forward_host(self, slabs, coords, raster, raster_p0, result, host):
        """LocationEncoder._forward_host over the slabs: each replica writes its rows of `result` (the 'packed' path's
        array) or of `host` (the 'copy' path's page-locked tensor)"""
        xs = None if coords is None else self._inputs(coords, slabs)
        tabs = None if raster is None else self._raster_tables(raster, slabs)

        def work(i, m, lo, hi):
            m._forward_host(hi - lo, coords=None if xs is None else xs[i], raster=None if tabs is None else tabs[i],
                            raster_p0=raster_p0 + lo, result=None if result is None else result[lo:hi],
                            host=None if host is None else host[lo:hi])
        self.run(slabs, work)
