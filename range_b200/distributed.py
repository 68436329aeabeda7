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

    def route(self, slab):
        """range_route of a step of `slab` (<= self.slab) rows per rank: slot r of a buffer starts at r * slab rows"""
        assert slab <= self.slab
        return _lib.Route(self.world, self.rank, int(slab), (ctypes.c_void_p * _lib.RANGE_MAX_RANKS)(*self.ptrs))

    def slots(self, slab):
        """device addresses of this rank's P slots for a step of `slab` rows per rank"""
        return [self.local.value + r * int(slab) * 4096 for r in range(self.world)]

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

