"""Multi-GPU: one process per GPU, torch.distributed (NCCL over NVLink) for the plumbing.

Queries shard trivially (rows are independent, range/range.py:213-240): every rank embeds its own rows against a
replicated database, no collective.

A database sharded along M (rank r holds rows [r M/P, (r+1) M/P) of the spatially sorted database) merges per-rank
partial softmax state.  Every logit is bounded (|s|,|g| <= 1), so the kernels use the fixed offset "-1" instead of a
running max and the merge needs no rescaling:

    every rank          sorts + encodes ITS OWN queries (a slab of `slab` rows per step)
    all_gather          the compact queries: fp16 embedding (512 B) + unit vector (16 B) per query
    every rank          row statistics of all P * slab queries over its shard       (range_retrieve_stats)
    all_reduce(SUM)     the exp-sums, 8 B per query; the maxima stay local (they only scale the fp16 weights)
    every rank          apply pass over its shard with the global sums; the kernel's epilogue stores row n of the
                        partial result straight into the receive buffer of its owner, rank n / slab, over NVLink
                        (range_retrieve_apply_routed) - no collective moves the (N,1024) partial outputs
    barrier             a 4-byte all_reduce: every rank's stores have landed
    every rank          sums its P slots in rank order and appends the location columns (range_combine_concat)

merge='reduce_scatter' replaces the routed epilogue + barrier by a local (N,1024) result and NCCL's reduce_scatter
(the comparison baseline; also what runs if the peers' buffers cannot be mapped).

neighbours() shares the steps up to the SUM of the exp-sums, then:
    every rank          top-k lists of all P * slab queries over its shard, entries as rows of the whole database
                        (range_retrieve_topk_rows)
    all_to_all          the lists, k x 8 B per query and rank: rank r receives its own queries' lists from every shard
    every rank          merges its P lists by weight, then row (range_topk_merge)

embed_sweep() (RANGE+ for several beta) shares the steps up to the SUM of the exp-sums, then:
    every rank          apply passes of the geographic end (beta 0) and the semantic end (beta 1), routed into the two
                        halves of the owners' receive buffers
    barrier             one for both ends
    every rank          sums its P slots of each end and writes (1 - beta) G + beta S for every beta (range_sweep_concat)
"""
import ctypes

import torch
import torch.distributed as dist

from . import _lib
from .engine import _new_out


def shard_rows(n, rank, world):
    """contiguous slab [lo, hi) of n rows for `rank` of `world` (query sharding)"""
    return (n * rank) // world, (n * (rank + 1)) // world


def merge_sums(sums, group=None):
    """all-reduce the per-shard exp-sums in place (the softmax denominators of range/range.py:215,234)"""
    dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    return sums


def _reduce_scatter(O_all, world, rank, group):
    """(P * slab, 1024) partial rows of every rank -> this rank's (slab, 1024) summed rows"""
    slab = O_all.shape[0] // world
    mine = torch.empty(slab, O_all.shape[1], dtype=O_all.dtype, device=O_all.device)
    try:
        dist.reduce_scatter_tensor(mine, O_all, op=dist.ReduceOp.SUM, group=group)
    except RuntimeError:                      # backends without reduce_scatter (gloo, the CPU tests)
        dist.all_reduce(O_all, op=dist.ReduceOp.SUM, group=group)
        mine.copy_(O_all[rank * slab:(rank + 1) * slab])
    return mine


class PeerBuffers:
    """Receive buffers [P][slab][1024] fp32, one per rank, each mapped into every rank's process (CUDA IPC through
    the C ABI: range_peer_alloc / range_peer_open)."""

    def __init__(self, lib, device_index, slab, group):
        self.lib, self.slab, self.group = lib, int(slab), group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.index = device_index
        nbytes = self.world * self.slab * 1024 * 4
        self.local = ctypes.c_void_p()
        handle = (ctypes.c_ubyte * 64)()
        with torch.cuda.device(device_index):
            code = lib.range_peer_alloc(nbytes, ctypes.byref(self.local), handle)
        why = None if code == 0 else lib.range_last_error().decode()
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle) if code == 0 else None, group=group)    # every rank gets here
        self.ptrs, self._opened = [], []
        if any(h is None for h in handles):
            if code == 0:
                with torch.cuda.device(device_index):
                    lib.range_peer_free(self.local)
            self.local = None
            raise _lib.RangeError(f"a rank could not allocate its receive buffer ({why or 'another rank'})")
        with torch.cuda.device(device_index):
            for r, h in enumerate(handles):
                if r == self.rank:
                    self.ptrs.append(self.local.value)
                    continue
                p = ctypes.c_void_p()
                _lib.check(lib.range_peer_open((ctypes.c_ubyte * 64).from_buffer_copy(h), ctypes.byref(p)))
                self._opened.append(p)
                self.ptrs.append(p.value)

    def route(self, slab, half=0):
        """range_route of a step of `slab` rows per rank: slot r of a buffer starts at r * slab rows.  half=1 (a beta
        sweep: the two ends of a step, each `slab` <= self.slab / 2 rows per rank): slot r of half h starts at
        (h * P + r) * slab rows"""
        assert (half + 1) * slab <= self.slab
        base = half * self.world * int(slab) * 4096
        return _lib.Route(self.world, self.rank, int(slab),
                          (ctypes.c_void_p * _lib.RANGE_MAX_RANKS)(*[p + base for p in self.ptrs]))

    def slots(self, slab, half=0):
        """device addresses of this rank's P slots for a step of `slab` rows per rank (in `half`, see route)"""
        return [self.local.value + (half * self.world + r) * int(slab) * 4096 for r in range(self.world)]

    def close(self):
        if getattr(self, "local", None) is None:
            return
        try:
            torch.cuda.synchronize(self.index)
            dist.barrier(group=self.group)           # no rank unmaps while a peer may still store into its buffer
        except Exception:
            pass
        with torch.cuda.device(self.index):
            for p in self._opened:
                self.lib.range_peer_close(p)
            self.lib.range_peer_free(self.local)
        self.local, self._opened = None, []


class ShardedRetriever:
    """embed() of a model whose database is sharded along M over the ranks of `group`.  A COLLECTIVE call: every rank
    passes its own queries (the counts may differ) and gets its own rows back."""

    MAX_STEP_ROWS = 131072          # P * slab rows per apply launch (receive buffer: 4 KB per row and rank)
    TOPK_WORKSPACE_BYTES = 1 << 30  # bound of the top-k workspace of a neighbours step (_topk_step_rows)

    def __init__(self, engine, group=None, merge="peer"):
        if merge not in ("peer", "reduce_scatter"):
            raise ValueError(f"merge={merge!r}: expected 'peer' or 'reduce_scatter'")
        self.engine, self.group, self.merge = engine, group, merge
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > _lib.RANGE_MAX_RANKS:
            raise ValueError(f"at most {_lib.RANGE_MAX_RANKS} ranks share a database, got {self.world}")
        self.buffers = None
        self._token = None
        self.collectives = 0            # NCCL calls issued (bench.py reports them)
        self.trace = None               # developer timing: a list collects CUDA events around neighbours' exchange + merge

    def _slab_for(self, n_max, step_rows=None):
        cap = max(128, (step_rows or self.MAX_STEP_ROWS) // self.world // 128 * 128)
        return min(cap, (n_max + 127) // 128 * 128)

    def _ensure_buffers(self, slab):
        if self.merge != "peer":
            return
        if self.buffers is not None and self.buffers.slab >= slab:
            return
        if self.buffers is not None:
            self.buffers.close()
        try:
            self.buffers = PeerBuffers(self.engine.lib, self.engine.index, slab, self.group)
            ok = torch.ones(1, device=self.engine.device)
        except _lib.RangeError as e:
            print(f"range_b200: rank {self.rank}: peer buffers unavailable ({e}); merging with reduce_scatter")
            ok = torch.zeros(1, device=self.engine.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)      # all ranks take the same path
        if ok.item() < 1:
            if self.buffers is not None:
                self.buffers.close()
            self.buffers, self.merge = None, "reduce_scatter"

    def close(self):
        if self.buffers is not None:
            self.buffers.close()
            self.buffers = None

    def _steps(self, mode, coords, temp, geo_temp, sort, n_max, slab):
        """the step loop of embed and neighbours: per step of `slab` rows per rank, this rank's rows (padded) sorted and
        encoded, every rank's compact queries gathered, their statistics over this shard and the SUM of the exp-sums.
        Yields (lo, rows, perm, q64, q16_all, qxyz_all, sums, maxs): this rank's rows [lo, lo + rows) of the step."""
        eng, P = self.engine, self.world
        dev = eng.device
        n = coords.shape[0]
        q16_all = torch.empty(P * slab, 256, dtype=torch.float16, device=dev)
        qxyz_all = torch.empty(P * slab, 4, dtype=torch.float32, device=dev)
        for lo in range(0, n_max, slab):
            mine = coords[lo:min(n, lo + slab)] if lo < n else coords[:0]
            rows = mine.shape[0]
            step = torch.zeros(slab, 2, dtype=torch.float64, device=dev)          # padding rows: (0, 0), results dropped
            step[:rows] = mine
            perm = None
            if sort:
                step, perm = eng.sort_queries(step)
            q64, q16, qxyz = eng.encode(step)
            dist.all_gather_into_tensor(q16_all, q16, group=self.group)
            dist.all_gather_into_tensor(qxyz_all, qxyz, group=self.group)
            sums, maxs = eng.retrieve_stats(mode, q16_all, qxyz_all, temp, geo_temp)
            merge_sums(sums, self.group)
            self.collectives += 3
            yield lo, rows, perm, q64, q16_all, qxyz_all, sums, maxs

    def embed(self, mode, coords, temp, geo_temp, beta, sort, out=None, out_dtype=torch.float32):
        """coords (n,2) fp64 on the device (this rank's queries) -> (n,1280) device tensor (this rank's rows)"""
        eng, P, me = self.engine, self.world, self.rank
        dev = eng.device
        n = coords.shape[0]
        n_max = torch.tensor([n], device=dev, dtype=torch.int64)
        dist.all_reduce(n_max, op=dist.ReduceOp.MAX, group=self.group)
        n_max = int(n_max.item())
        self.collectives += 1
        out = _new_out(n, out_dtype, dev) if out is None else out
        if n_max == 0:
            return out
        slab = self._slab_for(n_max)
        self._ensure_buffers(slab)
        if self._token is None:
            self._token = torch.zeros(1, device=dev)
        for lo, rows, perm, q64, q16_all, qxyz_all, sums, maxs in self._steps(mode, coords, temp, geo_temp, sort, n_max,
                                                                              slab):
            whole = rows == slab
            dst = out[lo:lo + slab] if whole else torch.empty((slab,) + tuple(out.shape[1:]), dtype=out.dtype, device=dev)
            if self.merge == "peer":
                bufs = self.buffers
                eng.retrieve_apply_routed(mode, q16_all, qxyz_all, temp, geo_temp, beta, sums, maxs, bufs.route(slab))
                dist.all_reduce(self._token, group=self.group)                    # barrier: all partial rows have landed
                self.collectives += 1
                eng.combine_concat(bufs.slots(slab), None, q64, out=dst, perm=perm)
            else:
                O_all = eng.retrieve_apply(mode, q16_all, qxyz_all, temp, geo_temp, beta, sums, maxs)
                O_mine = _reduce_scatter(O_all, P, me, self.group)
                self.collectives += 1
                eng.combine_concat([O_mine], None, q64, out=dst, perm=perm)
            if not whole and rows > 0:
                out[lo:lo + rows] = dst[:rows]
        return out

    def embed_sweep(self, coords, temp, geo_temp, sort, betas, out_dtype=torch.float32):
        """RANGE+ for several beta on this rank's queries: coords (n,2) fp64 on the device -> a list of (n,1280) device
        tensors, one per beta, in this rank's row order.  A COLLECTIVE call: every rank takes every step, whatever its
        own n and its own beta list (the lists may differ between ranks; an empty one returns []).

        The steps of embed (RANGE+ statistics, SUM of the exp-sums), then TWO apply passes per step whatever the number
        of beta, as in the unsharded LocationEncoder.embed_sweep: the geographic end (beta 0) and the semantic end (the
        one-softmax retrieval at temp, with RANGE+'s sums).  Peer merge: the two ends are routed into the two halves of
        the receive buffer (slot r of half h at row (h P + r) slab, PeerBuffers.route / slots; slab <= MAX_STEP_ROWS / 2P,
        so the buffer is the one embed allocates), one barrier, then range_sweep_concat over this rank's 2 P slots writes
        every beta.  The buffer is reused across steps for the same reason as embed's: a rank's apply passes of step i + 1
        follow its all_gathers of step i + 1 on its stream, which cannot complete before every rank has enqueued - and so,
        in stream order, finished - its sweep_concat of step i.  merge='reduce_scatter': both ends computed locally, two
        reduce_scatters, then range_sweep_concat with one slot per end.  Collectives: 1 + 4 per step (peer), 1 + 5
        (reduce_scatter)."""
        eng, P, me = self.engine, self.world, self.rank
        dev = eng.device
        n = coords.shape[0]
        betas = [float(b) for b in betas]
        if out_dtype not in (torch.float64, torch.float32):
            raise ValueError(f"out_dtype={out_dtype}: expected torch.float64 or torch.float32")
        n_max = torch.tensor([n], device=dev, dtype=torch.int64)
        dist.all_reduce(n_max, op=dist.ReduceOp.MAX, group=self.group)
        n_max = int(n_max.item())
        self.collectives += 1
        outs = [_new_out(n, out_dtype, dev) for _ in betas]
        if n_max == 0:
            return outs
        slab = self._slab_for(n_max, self.MAX_STEP_ROWS // 2)
        self._ensure_buffers(2 * slab)
        if self._token is None:
            self._token = torch.zeros(1, device=dev)
        for lo, rows, perm, q64, q16_all, qxyz_all, sums, maxs in self._steps("RANGE+", coords, temp, geo_temp, sort,
                                                                              n_max, slab):
            if self.merge == "peer":
                bufs = self.buffers
                eng.retrieve_apply_routed("RANGE+", q16_all, qxyz_all, temp, geo_temp, 0.0, sums, maxs, bufs.route(slab, 0))
                eng.retrieve_apply_routed("RANGE", q16_all, qxyz_all, temp, 0.0, None, sums, maxs, bufs.route(slab, 1))
                dist.all_reduce(self._token, group=self.group)                    # barrier: all partial rows have landed
                self.collectives += 1
                geo, sem = bufs.slots(slab, 0), bufs.slots(slab, 1)
            else:
                O_geo = eng.retrieve_apply("RANGE+", q16_all, qxyz_all, temp, geo_temp, 0.0, sums, maxs)
                O_sem = eng.retrieve_apply("RANGE", q16_all, qxyz_all, temp, 0.0, None, sums, maxs)
                geo, sem = [_reduce_scatter(O_geo, P, me, self.group)], [_reduce_scatter(O_sem, P, me, self.group)]
                self.collectives += 2
            if not betas:
                continue
            whole = rows == slab
            dst = [o[lo:lo + slab] if whole else torch.empty(slab, 1280, dtype=o.dtype, device=dev) for o in outs]
            eng.sweep_concat(geo, sem, betas, q64, perm=perm, outs=dst)
            if not whole and rows > 0:
                for o, d in zip(outs, dst):
                    o[lo:lo + rows] = d[:rows]
        return outs

    def _topk_step_rows(self, k):
        """P * slab rows per neighbours step: the top-k pass's workspace is 2 * splits * rows * k * 8 B.  The statistics
        plan it follows (csrc/capi.cu: plan_retrieval) takes at most 16 database splits from ~6 144 rows up (64 below,
        at most 0.2 GB), so rows <= 2^30 / (2 * 16 * 8 * k) keeps it within TOPK_WORKSPACE_BYTES (1 GB)."""
        return min(self.MAX_STEP_ROWS, self.TOPK_WORKSPACE_BYTES // (2 * 16 * 8 * k))

    def neighbours(self, mode, coords, temp, geo_temp, beta, sort, k):
        """coords (n,2) fp64 on the device (this rank's queries) -> (rows (n,k) int32, weight (n,k)) device tensors in
        this rank's row order: the k entries of the WHOLE database with the largest retrieval weight, descending, equal
        weights by the smaller row; rows of the database's sorted layout (DeviceDatabase.file_rows_global maps them to
        file rows).  A COLLECTIVE call; every rank must pass the same k, 1 <= k <= min(RANGE_TOPK_MAX, entries of the
        database) (ValueError on every rank when they differ).

        Per step, after embed's statistics and SUM of the exp-sums: this shard's top-k lists of all P * slab gathered
        queries (entries as global rows), all_to_all of the lists - they are rank-major by owner, so rank r receives
        [P][slab][k] - and the owner's merge of its P lists.  At most 256 B per query and rank cross the links: no peer
        buffers, the same path for both merge settings."""
        eng, P = self.engine, self.world
        dev = eng.device
        n, k = coords.shape[0], int(k)
        head = torch.tensor([n, k, -k], device=dev, dtype=torch.int64)     # max n, and max / min k: the ranks agree?
        dist.all_reduce(head, op=dist.ReduceOp.MAX, group=self.group)
        self.collectives += 1
        n_max, k_max, k_min = int(head[0]), int(head[1]), -int(head[2])
        if k_max != k_min:
            raise ValueError(f"neighbours: every rank must pass the same k, got k from {k_min} to {k_max}")
        if n_max == 0:
            return (torch.empty(0, k, dtype=torch.int32, device=dev), torch.empty(0, k, dtype=torch.float32, device=dev))
        slab = self._slab_for(n_max, self._topk_step_rows(k))
        row0 = eng.db.row_range[0]
        got_idx, got_w = [], []
        for lo, rows, perm, _, q16_all, qxyz_all, sums, _ in self._steps(mode, coords, temp, geo_temp, sort, n_max, slab):
            idx, w = eng.retrieve_topk_rows(mode, q16_all, qxyz_all, temp, geo_temp, beta, sums, k, row0)
            if self.trace is not None:
                t0 = torch.cuda.Event(enable_timing=True)
                t0.record()
            recv_w, recv_idx = torch.empty_like(w), torch.empty_like(idx)
            dist.all_to_all_single(recv_w, w, group=self.group)
            dist.all_to_all_single(recv_idx, idx, group=self.group)
            self.collectives += 2
            mi, mw = eng.topk_merge(recv_w.view(P, slab, k), recv_idx.view(P, slab, k), perm=perm)
            if self.trace is not None:
                t1 = torch.cuda.Event(enable_timing=True)
                t1.record()
                self.trace.append((t0, t1))
            got_idx.append(mi[:rows])
            got_w.append(mw[:rows])
        return torch.cat(got_idx), torch.cat(got_w)

