"""B200-native mirror of the reference's ``cache_manager.py`` (lkp411/cDLRM) plus the
GPU-resident look-ahead planner/mover that replaces its CPU worker pool.

Reference API kept: ``Prefetcher(args, emb_tables_cpu, batch_fifo, eviction_fifo,
finish_event, cache_ld)`` with ``start/join/run`` and the statics
``process_batch_slice``, ``eviction_manager``, ``pin_pool`` (cache_manager.py:8-115).

New (B200-first): ``WindowPlanner`` -- plans window w+1 on a side stream while window w
trains (tags in HBM, bitmap-unique, ballot probe, bit-exact victim choice from the
torch-compatible mt19937 stream) and installs it at the boundary with zero-copy evict /
fill kernels over the pinned master tables.  All arithmetic is in libcdlrm_b200.so.
"""
import ctypes
import math
import os
import threading
import time

import numpy as np
import torch

from . import _lib
from ._lib import check, lib

_vp = ctypes.c_void_p


def _sp(stream):
    return _vp(stream.cuda_stream)


# ------------------------------------------------------------------------------------
# victim-way random stream (main_no_ddp.py:183-185)
# ------------------------------------------------------------------------------------


class VictimRng:
    """Host mt19937 stream bit-identical to ``torch.manual_seed(seed)`` followed by
    ``torch.empty(n).exponential_(1)`` (what Categorical.sample() consumes), produced by
    cdlrm_rng_exponential with a multi-threaded log1p transform."""

    def __init__(self, seed, threads=None):
        self._h = _vp()
        check(lib.cdlrm_rng_create(ctypes.byref(self._h), int(seed)))
        self.threads = threads or max(1, min(16, (os.cpu_count() or 2) - 1))

    def exponential(self, n, pin=True):
        out = torch.empty(max(int(n), 1), dtype=torch.float32, pin_memory=pin and torch.cuda.is_available())
        if n:
            check(lib.cdlrm_rng_exponential(self._h, _vp(out.data_ptr()), int(n), self.threads))
        return out[:n]

    @property
    def draws(self):
        return int(lib.cdlrm_rng_draws(self._h))

    def __del__(self):
        try:
            lib.cdlrm_rng_destroy(self._h)
        except Exception:
            pass


class VictimRngDevice:
    """The same stream as ``VictimRng`` generated on the GPU (cdlrm_rngdev_*): one CTA refreshes
    the mt19937 state in three parallel phases, the select kernel applies the exponential
    transform.  No host work and no PCIe traffic for the draws; every rank of a data-parallel
    job evolves an identical copy."""

    on_device = True

    def __init__(self, seed, device):
        self.device = torch.device(device)
        self._h = _vp()
        check(lib.cdlrm_rngdev_create(ctypes.byref(self._h), self.device.index, int(seed)))

    def exponential(self, n, stream=None):
        """float32 [n] device tensor of draws (tests / tools; the planner consumes raw words)."""
        s = stream or torch.cuda.current_stream(self.device)
        with torch.cuda.stream(s):
            out = torch.empty(max(int(n), 1), dtype=torch.float32, device=self.device)
            raw = torch.empty(2 * max(int(n), 1), dtype=torch.int32, device=self.device)
            check(lib.cdlrm_rngdev_exponential(self._h, _vp(out.data_ptr()), int(n), _vp(raw.data_ptr()), _sp(s)))
        return out[:n]

    @property
    def draws(self):
        return int(lib.cdlrm_rngdev_draws(self._h))

    def snapshot(self, stream):
        """(pinned int32 [625] state {x[624], pos}, draws, event): the state in the order of ``stream`` -- the state
        tensor holds it once ``event`` has completed -- and the number of draws enqueued so far."""
        state = torch.empty(625, dtype=torch.int32, pin_memory=True)
        draws = ctypes.c_uint64()
        check(lib.cdlrm_rngdev_get_state(self._h, _vp(state.data_ptr()), ctypes.byref(draws), _sp(stream)))
        ev = torch.cuda.Event()
        ev.record(stream)
        return state, int(draws.value), ev

    def get_state(self, stream=None):
        """(uint32 numpy [625], draws) after everything enqueued on ``stream`` (default: current)."""
        state, draws, ev = self.snapshot(stream or torch.cuda.current_stream(self.device))
        ev.synchronize()
        return state.numpy().view(np.uint32).copy(), draws

    def set_state(self, state, draws, stream=None):
        s = stream or torch.cuda.current_stream(self.device)
        h = np.ascontiguousarray(np.asarray(state, dtype=np.uint32))
        if h.shape != (625,):
            raise ValueError("victim-stream state must hold 625 words, got shape %s" % (h.shape,))
        check(lib.cdlrm_rngdev_set_state(self._h, _vp(h.ctypes.data), int(draws), _sp(s)))
        s.synchronize()          # the host array may go away after the call

    def __del__(self):
        try:
            lib.cdlrm_rngdev_destroy(self._h)
        except Exception:
            pass


class TorchGlobalRng:
    """Draws from torch's global CPU generator -- literally what the reference's
    ``Categorical(...).sample()`` does, so interleaving with any other consumer of the
    global generator stays identical.  Used by the drop-in ``CacheEmbeddings``."""

    def exponential(self, n, pin=True):
        q = torch.empty(int(n), dtype=torch.float32).exponential_(1) if n else torch.empty(0)
        return q.pin_memory() if (pin and n and torch.cuda.is_available()) else q


# ------------------------------------------------------------------------------------
# planner + mover
# ------------------------------------------------------------------------------------


def wb_share_range(E, r, W):
    """(first entry, count) of rank r's share of an eviction list of E entries written back by W ranks: contiguous,
    disjoint, covering [0, E), sizes differing by at most one."""
    lo, hi = (E * r) // W, (E * (r + 1)) // W
    return lo, hi - lo


class PlanRecord:
    """Decisions for one window (all device tensors are concatenated over tables; the
    lists of table k start at ``off[k]``)."""
    __slots__ = ("uniq", "hits", "dropped", "rows", "E", "F", "off", "evict_ids", "evict_slots",
                 "evict_primary", "fill_ids", "fill_slots", "event",
                 # look-ahead staging (WindowPlanner.stage / install_staged)
                 "L", "loser_off", "loser_soff", "loser_ids", "loser_stage", "fill_stage", "fill_soff", "evict_stage",
                 "staged", "wb_done", "stage_begin", "stage_bytes", "loser_shard", "loser_peers",
                 "marks", "wb_lo", "wb_n", "fill_peers")

    def loser_list(self, k):
        o, n = self.loser_off[k], self.L[k]
        return self.loser_ids[o:o + n]

    def evict_list(self, k):
        o, e = self.off[k], self.E[k]
        return self.evict_ids[o:o + e], self.evict_slots[o:o + e], self.evict_primary[o:o + e]

    def fill_list(self, k):
        o, f = self.off[k], self.F[k]
        return self.fill_ids[o:o + f], self.fill_slots[o:o + f]


class WindowPlanner:
    def __init__(self, cache_group, emb_tables, window_len, rng=None, stream=None, lookahead_tags=False):
        self.cg = cache_group
        self.emb_tables = emb_tables
        self.ctx = cache_group._ensure_ctx(emb_tables)
        self.dev = cache_group.device
        self.T = len(cache_group.emb_l)
        self.ways = cache_group.num_ways
        self.dim = cache_group.dim
        self.rng = rng if rng is not None else TorchGlobalRng()
        self.stream = stream or torch.cuda.current_stream(self.dev)
        self.window_len = int(window_len)
        nbytes = lib.cdlrm_plan_workspace_bytes(self.ctx, self.window_len)
        if nbytes < 0:
            raise _lib.CdlrmError("cdlrm_plan_workspace_bytes failed")
        self._ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.dev)
        base = (self._ws.data_ptr() + 255) // 256 * 256
        check(lib.cdlrm_plan_bind_workspace(self.ctx, _vp(base), nbytes, self.window_len))
        self._h_counts = torch.zeros(self.T * 4, dtype=torch.int64).pin_memory()
        self._h_counts2 = torch.zeros(self.T * 2, dtype=torch.int64).pin_memory()
        self._h_counts3 = torch.zeros(self.T, dtype=torch.int64).pin_memory()
        self.collect_losers = False      # also list the window's un-cached ids (for the HBM loser store)
        # eviction lists with one entry per replaced (set, way) -- its winner -- instead of one per claimant: all the
        # write-back needs; the reference-shaped callers (CacheEmbeddings: eviction_data) keep the full lists
        self.primary_evictions_only = False
        self._bufs = {}                  # persistent grow-only staging buffers (no cudaMalloc per window)
        self._stage_no = 0
        # how master rows cross PCIe: "sm" = zero-copy gather / scatter kernels (move.cu), "ce" = host threads gather
        # into / scatter out of pinned chunks that cudaMemcpyAsync moves (hostio.cu): ~10x gentler on the training
        # step that runs beside it (bench.py --ce-probe-gb), at the price of host cores
        self.pcie_mode = "sm"
        self.host_threads = max(1, min(4, (os.cpu_count() or 2) - 2))
        self._pin = {}                   # pinned host buffers (grow-only)
        self._ce_no = 0
        self._ce_ev = None
        self._pending_wb = None          # ce: (record, average) of the boundary whose evicted rows are not yet written back
        # --evict-victim-cache: the loser store of the installed window is trained in place (cdlrm_embed_victim_update);
        # at the next boundary its rows are carried into the next window's prefetched rows and written back to the master
        self.evict_victim_cache = False
        self._bound = None               # record whose loser store is bound (installed window)
        self._pending_store = None       # ce: record whose store rows are not yet written back
        self._shard = None               # (rank, world, host process group): loser store sharded over the node
        self._fill_shard = None          # (rank, world, host process group): fill prefetch sharded over the node
        self._peer_bufs = {}             # name -> (capacity rows, [device address of every rank's shard buffer])
        self.plan_tags = None
        if lookahead_tags:
            self.enable_lookahead_tags()

    @property
    def loser_cap_rows(self):
        """HBM budget (rows) of ONE loser store; two alternate.  ``CDLRM_LOSER_STORE_GB`` fixes it; otherwise it is
        sized once, at the first plan, from the HBM that is free then: half of (free - 70 GB), within [8, 32] GB.
        The 70 GB are what a Terabyte-shape window still allocates afterwards (fill / evict staging up to the
        cache size, plan records, the next window's inputs).  1-4 GPUs: the whole store fits (5 / 13 / 25 GB); at
        8 GPUs (14 M un-cacheable ids per big table, 42 GB) about half of it does."""
        cap = getattr(self, "_loser_cap_rows", None)
        if cap is None:
            env = os.environ.get("CDLRM_LOSER_STORE_GB")
            if env:
                gb = float(env)
            else:
                free, _total = torch.cuda.mem_get_info(self.dev)
                cached = torch.cuda.memory_reserved(self.dev) - torch.cuda.memory_allocated(self.dev)
                gb = min(32.0, max(8.0, ((free + cached) / 1e9 - 70.0) / 2))
            cap = self._loser_cap_rows = int(gb * 1e9 / (4 * self.dim))
        return cap

    # -- window scan sharded over the ranks of a node ------------------------------------------------------
    def enable_sharded_scan(self, rank, world, group):
        """Let every rank of a ``world``-GPU node mark only ITS share of a window (``scan_shard``) and OR the other
        ranks' id bitmaps into its own over NVLink (``merge_marks``) instead of scanning the whole global window on
        every rank.  The planner workspace moves into a peer-readable allocation (same carve-up on every rank).
        Collective over ``group`` (host-side, gloo): call it on every rank, from the same point of the program."""
        if world <= 1:
            return
        import torch.distributed as dist
        dev = self.dev.index
        nbytes = lib.cdlrm_plan_workspace_bytes(self.ctx, self.window_len)
        mine, handle = _vp(), ctypes.create_string_buffer(64)
        check(lib.cdlrm_peer_alloc(dev, nbytes, ctypes.byref(mine), handle))
        check(lib.cdlrm_plan_bind_workspace(self.ctx, mine, nbytes, self.window_len))
        self._ws = None                   # the torch-allocated workspace is no longer bound
        handles = [None] * world
        dist.all_gather_object(handles, handle.raw, group=group)
        ptrs = []
        for r in range(world):
            if r == rank:
                ptrs.append(mine.value)
            else:
                p = _vp()
                check(lib.cdlrm_peer_open(dev, ctypes.create_string_buffer(handles[r], 64), ctypes.byref(p)))
                ptrs.append(p.value)
        self._scan = (int(rank), int(world), group, ptrs)

    @property
    def scan_shard(self):
        """(rank, world) of the sharded window scan; (0, 1): this rank marks the whole window."""
        sc = getattr(self, "_scan", None)
        return (sc[0], sc[1]) if sc else (0, 1)

    def merge_marks(self):
        """After this rank's ``mark_ids`` calls: wait until every rank has marked its share, OR the others' bitmaps
        into this rank's (NVLink reads), and hold every rank until all have done so (phase A clears the bitmaps)."""
        sc = getattr(self, "_scan", None)
        if not sc:
            return
        import torch.distributed as dist
        rank, world, group, ptrs = sc
        self.stream.synchronize()
        dist.barrier(group=group)
        check(lib.cdlrm_plan_or_peer_bitmaps(self.ctx, _lib.ptr_array(ptrs), world, rank, _sp(self.stream)))
        self.stream.synchronize()
        dist.barrier(group=group)

    def _agreed_loser_cap(self):
        """Rows one window's loser store may hold: ``loser_cap_rows`` on one rank; sharded, ``world`` times the
        smallest per-rank budget (agreed once over the host group, the plans must stay identical)."""
        if self._shard is None:
            return self.loser_cap_rows
        cap = getattr(self, "_loser_cap_agreed", None)
        if cap is None:
            import torch.distributed as dist
            _rank, world, group = self._shard
            caps = [int(self.loser_cap_rows)] * world
            if group != "local":
                dist.all_gather_object(caps, int(self.loser_cap_rows), group=group)
            cap = self._loser_cap_agreed = min(caps) * world
        return cap

    def enable_sharded_losers(self, rank, world, group):
        """Shard the loser store over the ``world`` ranks of ONE node (peer.cu): every rank runs the same plan, so
        the un-cached ids of a window are the same everywhere; rank r prefetches rows [r * shard, (r + 1) * shard) of
        each table's ascending loser list over its own PCIe link into a buffer its peers can read over NVLink, and
        the forward reads a missing row from the rank that holds it.  ``group``: a host-side (gloo) process group
        used to exchange the IPC handles and to agree on sizes; calls that touch it come from the plan thread of
        every rank in the same order."""
        if world > 1:
            if world > 8:
                raise _lib.CdlrmError("the sharded loser store spans the (at most 8) GPUs of one node")
            self._shard = (int(rank), int(world), group)      # group "local": single-process emulation (tests)

    def enable_sharded_fills(self, rank, world, group):
        """Shard the FILL prefetch over the ``world`` ranks of one node: the replicas run the same plan, so the rows
        that enter the cache at a boundary are the same everywhere; rank r pulls the r-th of ``world`` equal shares of
        every table's fill list over its own PCIe link into a peer-readable staging buffer, and at the boundary every
        rank fills its cache from all ``world`` buffers (its own share from local HBM, the others over NVLink): 1/world
        of the PCIe traffic and of the host-memory reads per rank for those rows.  ``group`` as in
        ``enable_sharded_losers`` ("local": single-process emulation for tests)."""
        if world > 1:
            if world > 8:
                raise _lib.CdlrmError("the sharded fill prefetch spans the (at most 8) GPUs of one node")
            self._fill_shard = (int(rank), int(world), group)

    def _peer_buf(self, name, rows, shard=None):
        """Peer-readable [rows, dim] fp32 buffer ``name`` of this rank plus the addresses of the same-named buffers
        of every other rank (collective over the host group: every rank asks for the same ``rows``).  Grown (x1.25)
        only when a window needs more."""
        import torch.distributed as dist
        rank, world, group = shard if shard is not None else self._shard
        ent = self._peer_bufs.get(name)
        if ent is not None and ent[0] >= rows:
            return ent
        if group == "local":
            # in-process emulation (tests on a one-GPU box): the shards of all `world` ranks live on this device
            cap = int(rows) + 16
            keep = [torch.empty(cap, self.dim, dtype=torch.float32, device=self.dev) for _ in range(world)]
            ent = self._peer_bufs[name] = (cap, [t.data_ptr() for t in keep], keep)
            return ent
        dev = self.dev.index
        if ent is not None:
            # nobody reads this buffer any more (it served window w-1; every rank has installed window w: the plan
            # barrier precedes the staging of window w+1): unmap the peers' copies everywhere, then free
            for r, p in enumerate(ent[1]):
                if r != rank:
                    check(lib.cdlrm_peer_close(dev, _vp(p)))
            dist.barrier(group=group)
            check(lib.cdlrm_peer_free(dev, _vp(ent[1][rank])))
        cap = int(rows) + min(int(rows * 0.25), (1 << 30) // (4 * self.dim)) + 16
        mine = _vp()
        handle = ctypes.create_string_buffer(64)
        check(lib.cdlrm_peer_alloc(dev, cap * self.dim * 4, ctypes.byref(mine), handle))
        handles = [None] * world
        dist.all_gather_object(handles, handle.raw, group=group)
        ptrs = []
        for r in range(world):
            if r == rank:
                ptrs.append(mine.value)
            else:
                p = _vp()
                check(lib.cdlrm_peer_open(dev, ctypes.create_string_buffer(handles[r], 64), ctypes.byref(p)))
                ptrs.append(p.value)
        ent = self._peer_bufs[name] = (cap, ptrs)
        return ent

    def enable_lookahead_tags(self):
        """Give the planner its own evolving copy of the tags so that it can run one or more
        windows ahead of the live tags (which are patched by ``install``)."""
        self.plan_tags = [t.clone() for t in self.cg.occupancy_tables]
        self.cg._plan_tags = self.plan_tags     # kept bound across re-binds of the cache group (_ensure_ctx)
        check(lib.cdlrm_ctx_bind_plan_tags(self.ctx, _lib.ptr_array([t.data_ptr() for t in self.plan_tags])))

    def unique_ptr(self, k):
        return lib.cdlrm_plan_unique_ptr(self.ctx, k)

    def unique_tensor(self, k, n):
        """Copy of the ascending unique ids of table k found by the last plan (device)."""
        out = torch.empty(n, dtype=torch.int64, device=self.dev)
        check(lib.cdlrm_plan_copy_unique(self.ctx, k, _vp(out.data_ptr()), n,
                                         _sp(torch.cuda.current_stream(self.dev))))
        return out

    # -- plan -----------------------------------------------------------------------------
    def mark_ids(self, ids):
        """Chunked window scan: OR a chunk of window ids (int64 device tensor [T, n]) into the planner's id
        bitmaps on the planner's stream; finish with ``plan(marked=total ids per table)``."""
        assert ids.is_cuda and ids.dtype == torch.int64 and ids.stride(1) == 1 and ids.shape[0] == self.T
        check(lib.cdlrm_plan_mark_ids(self.ctx, _vp(ids.data_ptr()), ids.stride(0), ids.shape[1], _sp(self.stream)))

    def mark_own_ids(self, ids):
        """Data-parallel ranks: the ids (int64 device tensor [T, n], any number of chunks) of THIS rank's own batches
        of the window about to be planned.  With ``collect_losers`` the plan then lists only the un-cached ids among
        them -- the misses this rank's forwards will actually have -- so the loser store stays as small as on one GPU."""
        assert ids.is_cuda and ids.dtype == torch.int64 and ids.stride(1) == 1 and ids.shape[0] == self.T
        check(lib.cdlrm_plan_mark_own_ids(self.ctx, _vp(ids.data_ptr()), ids.stride(0), ids.shape[1], _sp(self.stream)))

    def plan(self, win_ids=None, uniq_lists=None, marked=None):
        """win_ids: int64 device tensor [T, n] (raw window ids), or uniq_lists: list of T
        ascending-unique int64 tensors (the reference-API path), or marked: the number of ids per table
        already scanned chunk by chunk with ``mark_ids``."""
        s = self.stream
        rec = PlanRecord()
        rec.marks = {}                   # phase name -> timing event on the planner's stream (bench.py: timeline)

        def mark(name):
            e = rec.marks[name] = torch.cuda.Event(enable_timing=True)
            e.record(s)

        t_a = time.perf_counter()
        with torch.cuda.stream(s):
            mark("plan_begin")
            if uniq_lists is not None:
                lens = [int(u.numel()) for u in uniq_lists]
                ld = max(max(lens), 1)
                if ld > self.window_len:
                    raise _lib.CdlrmError("unique list longer than the planner workspace window")
                buf = torch.zeros(self.T, ld, dtype=torch.int64, device=self.dev)
                for k, u in enumerate(uniq_lists):
                    if lens[k]:
                        buf[k, :lens[k]].copy_(u.to(self.dev, non_blocking=True))
                check(lib.cdlrm_plan_phase_a(self.ctx, _vp(buf.data_ptr()), buf.stride(0), ld,
                                             _lib.i64_array(lens), _vp(self._h_counts.data_ptr()), _sp(s)))
            elif marked is not None:
                check(lib.cdlrm_plan_phase_a(self.ctx, None, 0, min(int(marked), self.window_len), None,
                                             _vp(self._h_counts.data_ptr()), _sp(s)))
            else:
                assert win_ids.is_cuda and win_ids.dtype == torch.int64 and win_ids.stride(1) == 1
                check(lib.cdlrm_plan_phase_a(self.ctx, _vp(win_ids.data_ptr()), win_ids.stride(0),
                                             win_ids.shape[1], None, _vp(self._h_counts.data_ptr()), _sp(s)))
            mark("phase_a_done")
            s.synchronize()
            cnt = self._h_counts.view(self.T, 4).clone()
            rec.uniq = cnt[:, 0].tolist()
            rec.hits = cnt[:, 1].tolist()
            rec.dropped = cnt[:, 2].tolist()
            rec.rows = cnt[:, 3].tolist()
            total = int(sum(rec.rows))
            rec.off = [0] * self.T
            for k in range(1, self.T):
                rec.off[k] = rec.off[k - 1] + rec.rows[k - 1]
            # q for table 0..T-1 in one draw: the stream is split-invariant
            t_b = time.perf_counter()
            dev_rng = getattr(self.rng, "on_device", False)
            q_host = None if dev_rng else self.rng.exponential(total * self.ways)
            t_c = time.perf_counter()
            if not dev_rng:
                q = q_host.to(self.dev, non_blocking=True) if total else torch.empty(0, device=self.dev)
            n = max(total, 1)
            # the lists of a window live in one of two alternating sets of grow-only buffers (window w's are read
            # until its write-back, while window w+1 is planned): no per-window allocation beside training
            self._plan_no = getattr(self, "_plan_no", 0) + 1
            par = self._plan_no & 1
            rec.evict_ids = self._list_buf("evict_ids%d" % par, n, torch.int64)
            rec.evict_slots = self._list_buf("evict_slots%d" % par, n, torch.int32)
            rec.evict_primary = self._list_buf("evict_primary%d" % par, n, torch.uint8)
            rec.fill_ids = self._list_buf("fill_ids%d" % par, n, torch.int64)
            rec.fill_slots = self._list_buf("fill_slots%d" % par, n, torch.int32)
            outs = (_vp(rec.evict_ids.data_ptr()), _vp(rec.evict_slots.data_ptr()),
                    _vp(rec.evict_primary.data_ptr()), _vp(rec.fill_ids.data_ptr()),
                    _vp(rec.fill_slots.data_ptr()), _vp(self._h_counts2.data_ptr()), _sp(s))
            check(lib.cdlrm_plan_set_primary_evictions(self.ctx, int(self.primary_evictions_only)))
            if dev_rng:
                cap = max(max(rec.rows) * self.ways, 1)          # draws of the largest table
                raw = self._list_buf("rng_raw", 2 * cap, torch.int32)
                check(lib.cdlrm_plan_phase_b_dev(self.ctx, self.rng._h, _vp(raw.data_ptr()), cap,
                                                 _lib.i64_array(rec.rows), *outs))
            else:
                check(lib.cdlrm_plan_phase_b(self.ctx, _vp(q.data_ptr()) if total else None,
                                             _lib.i64_array(rec.rows), *outs))
            mark("phase_b_done")
            s.synchronize()
            c2 = self._h_counts2.view(self.T, 2).clone()
            rec.E = c2[:, 0].tolist()
            rec.F = c2[:, 1].tolist()
            del q_host
            rec.L = rec.loser_ids = rec.loser_off = None
            if self.collect_losers:
                cap = [rec.dropped[k] + rec.rows[k] for k in range(self.T)]
                rec.loser_off = [0] * self.T
                for k in range(1, self.T):
                    rec.loser_off[k] = rec.loser_off[k - 1] + cap[k - 1]
                rec.loser_ids = self._list_buf("loser_ids%d" % par, max(sum(cap), 1), torch.int64)
                check(lib.cdlrm_plan_losers(self.ctx, _lib.i64_array(rec.uniq), _lib.i64_array(rec.loser_off),
                                            _vp(rec.loser_ids.data_ptr()), _vp(self._h_counts3.data_ptr()), _sp(s)))
                s.synchronize()
                rec.L = self._h_counts3.clone().tolist()
                # HBM budget of the loser store (two of them alternate): beyond the cap only a prefix of each
                # table's ascending loser ids is staged; the forward serves the others zero-copy from the host
                # master (fwd_miss_kernel falls back when the binary search misses) -- same rows either way
                tot = sum(rec.L)
                cap_rows = self._agreed_loser_cap()
                if tot > cap_rows and self.evict_victim_cache:
                    # the misses served from the master would be trained nowhere, and race with the next prefetch
                    raise _lib.CdlrmError(
                        "--evict-victim-cache needs the whole loser store of a window in HBM: this window needs %.2f GB, "
                        "the budget is %.2f GB (raise CDLRM_LOSER_STORE_GB, or shrink --lookahead)"
                        % (tot * 4 * self.dim / 1e9, cap_rows * 4 * self.dim / 1e9))
                if tot > cap_rows:
                    rec.L = [int(x * cap_rows // tot) for x in rec.L]
            self.last_timing = {"phase_a_s": round(t_b - t_a, 4), "rng_s": round(t_c - t_b, 4),
                                "phase_b_s": round(time.perf_counter() - t_c, 4)}
        rec.event = None
        rec.staged = rec.wb_done = rec.fill_stage = rec.loser_stage = rec.evict_stage = None
        rec.loser_shard = rec.loser_peers = rec.fill_peers = None
        rec.stage_begin, rec.stage_bytes = None, 0
        return rec

    def _list_buf(self, name, n, dtype):
        """Persistent 1-D device buffer of at least n elements (grown x1.25 when a window needs more)."""
        b = self._bufs.get(name)
        if b is None or b.numel() < n or b.dtype != dtype:
            self._bufs[name] = None
            b = self._bufs[name] = torch.empty(int(n * 1.25) + 16, dtype=dtype, device=self.dev)
        return b[:n]

    def _buf(self, name, rows):
        """Persistent [rows, dim] fp32 staging buffer, grown (x1.25) only when a window needs more:
        allocation inside the steady state would synchronise the device."""
        b = self._bufs.get(name)
        if b is None or b.shape[0] < rows:
            b = None
            self._bufs[name] = None
            # head-room so that the next, slightly larger window does not re-allocate: 25 %, at most 1 GB
            extra = min(int(rows * 0.25), (1 << 30) // (4 * self.dim))
            b = torch.empty(int(rows) + extra + 16, self.dim, dtype=torch.float32, device=self.dev)
            self._bufs[name] = b
        return b

    # -- copy-engine transfers (pcie_mode "ce") -------------------------------------------------
    # staging chunk: small, because a copy engine does not interleave a chunk with the training step's own copies
    # (inputs in, loss out): with 128 MB chunks single steps stalled 2.5-3 ms behind a chunk, and cutting the chunk into
    # 4 MB cudaMemcpyAsync pieces within one stream did not change that; 8 MB = 0.15 ms of link time
    CE_CHUNK_BYTES = 8 << 20

    def _pinned(self, name, nbytes):
        b = self._pin.get(name)
        if b is None or b.numel() < nbytes:
            self._pin[name] = None
            b = self._pin[name] = torch.empty(int(nbytes * 1.5) + 256, dtype=torch.uint8, pin_memory=True)
        return b

    def _ce_chunks(self):
        """Two pinned staging chunks [rows, dim] that alternate, and the events that tell when the copy engine has
        finished with each."""
        rows = max(1, self.CE_CHUNK_BYTES // (4 * self.dim))
        bufs = [self._pinned("ce%d" % i, rows * 4 * self.dim)[:rows * 4 * self.dim].view(torch.float32).view(rows, self.dim)
                for i in range(2)]
        if self._ce_ev is None:
            self._ce_ev = [torch.cuda.Event(), torch.cuda.Event()]
        return rows, bufs, self._ce_ev

    def _ids_to_host(self, name, dev_ids, segments):
        """Copy the id segments [(offset, count)] of a device int64 list into one packed pinned array; returns the
        host tensor and the packed offsets.  Synchronises the planner's stream."""
        tot = sum(n for _o, n in segments)
        h = self._pinned(name, 8 * max(tot, 1))[:8 * max(tot, 1)].view(torch.int64)
        offs, o = [], 0
        with torch.cuda.stream(self.stream):
            for so, n in segments:
                offs.append(o)
                if n:
                    h[o:o + n].copy_(dev_ids[so:so + n], non_blocking=True)
                o += n
        self.stream.synchronize()
        return h, offs

    def _ce_gather(self, segs):
        """segs: [(table k, host int64 ids, device address of the destination rows)]: rows of the host master gathered
        by host threads into a pinned chunk while the copy engine moves the previous chunk into HBM -- the whole list in
        ONE native call (cdlrm_host_prefetch_rows: no interpreter lock between chunks)."""
        segs = [(k, hid, dst) for k, hid, dst in segs if int(hid.numel())]
        if not segs:
            return
        rows_per, bufs, _evs = self._ce_chunks()
        Ws = [self.emb_tables.emb_l[k].weight.data for k, _h, _d in segs]
        check(lib.cdlrm_host_prefetch_rows(
            self.dev.index, len(segs), _lib.ptr_array([W.data_ptr() for W in Ws]), _lib.i64_array([W.shape[0] for W in Ws]),
            self.dim, _lib.ptr_array([hid.data_ptr() for _k, hid, _d in segs]),
            _lib.i64_array([int(hid.numel()) for _k, hid, _d in segs]), _lib.ptr_array([dst for _k, _h, dst in segs]),
            _vp(bufs[0].data_ptr()), _vp(bufs[1].data_ptr()), rows_per, self.host_threads, _sp(self.stream)))

    def flush_writeback(self):
        """ce mode: write the evicted rows of the last installed window back into the host master (device -> pinned
        chunk by the copy engine, chunk -> master rows by host threads).  Called from the thread that plans the next
        window, before anything of that window reads the master; a no-op when nothing is pending."""
        store, self._pending_store = self._pending_store, None
        if store is not None:
            self._write_store(store, ce=True)
        pend, self._pending_wb = self._pending_wb, None
        if pend is None:
            return
        rec, average = pend
        s, d, dev = self.stream, self.dim, self.dev.index
        wlo, wn = rec.wb_lo, rec.wb_n                  # this rank's share of every table's eviction list
        segs = [(rec.off[k] + wlo[k], wn[k]) for k in range(self.T)]
        hid, offs = self._ids_to_host("wb_ids", rec.evict_ids, segs)
        tot = sum(wn)
        hpr = self._pinned("wb_prim", max(tot, 1))[:max(tot, 1)]
        with torch.cuda.stream(s):
            for k in range(self.T):
                if wn[k]:
                    o = rec.off[k] + wlo[k]
                    hpr[offs[k]:offs[k] + wn[k]].copy_(rec.evict_primary[o:o + wn[k]], non_blocking=True)
        s.synchronize()
        rows_per, bufs, _evs = self._ce_chunks()
        eoff = [0] * self.T
        for k in range(1, self.T):
            eoff[k] = eoff[k - 1] + rec.E[k - 1]
        ks = [k for k in range(self.T) if wn[k]]
        if ks:
            Ws = [self.emb_tables.emb_l[k].weight.data for k in ks]
            # device -> pinned chunk by the copy engine, chunk -> master rows by the pooled host threads, the copy of
            # chunk c beside the scatter of chunk c-1: one native call for the whole write-back
            check(lib.cdlrm_host_writeback_rows(
                dev, len(ks), _lib.ptr_array([W.data_ptr() for W in Ws]), _lib.i64_array([W.shape[0] for W in Ws]), d,
                _lib.ptr_array([hid.data_ptr() + 8 * offs[k] for k in ks]),
                _lib.ptr_array([hpr.data_ptr() + offs[k] for k in ks]), _lib.i64_array([wn[k] for k in ks]),
                _lib.ptr_array([rec.evict_stage[eoff[k] + wlo[k]:].data_ptr() for k in ks]),
                _vp(bufs[0].data_ptr()), _vp(bufs[1].data_ptr()), rows_per, int(average), self.host_threads, _sp(s)))
        rec.wb_done = torch.cuda.Event(enable_timing=True)
        rec.wb_done.record(s)

    def _write_store(self, rec, ce):
        """master[k][id] = the store row of id, for every id of the loser store of ``rec``: a plain write (the row is the
        master row plus this window's updates), on the planner's stream.  ``ce``: copy engine + host threads
        (cdlrm_host_writeback_rows, returns when the rows are in the master); else zero-copy scatter kernels."""
        ks = [k for k in range(self.T) if rec.L[k]]
        if not ks:
            return
        s = self.stream
        if not ce:
            with torch.cuda.stream(s):
                for k in ks:
                    check(lib.cdlrm_move_scatter_master2(self.ctx, k, _vp(rec.loser_ids[rec.loser_off[k]:].data_ptr()), None,
                                                         rec.L[k], _vp(rec.loser_stage[rec.loser_soff[k]:].data_ptr()), 0,
                                                         _sp(s)))
            return
        hid, offs = self._ids_to_host("store_ids", rec.loser_ids, [(rec.loser_off[k], rec.L[k]) for k in ks])
        rows_per, bufs, _evs = self._ce_chunks()
        Ws = [self.emb_tables.emb_l[k].weight.data for k in ks]
        check(lib.cdlrm_host_writeback_rows(
            self.dev.index, len(ks), _lib.ptr_array([W.data_ptr() for W in Ws]), _lib.i64_array([W.shape[0] for W in Ws]),
            self.dim, _lib.ptr_array([hid.data_ptr() + 8 * o for o in offs]), None, _lib.i64_array([rec.L[k] for k in ks]),
            _lib.ptr_array([rec.loser_stage[rec.loser_soff[k]:].data_ptr() for k in ks]),
            _vp(bufs[0].data_ptr()), _vp(bufs[1].data_ptr()), rows_per, 0, self.host_threads, _sp(s)))

    def write_store_to_master(self):
        """--evict-victim-cache: write the rows of the installed window's loser store into the master now (they are
        also the rows its next boundary carries and writes back, so this changes nothing that follows).  Runs after
        the current stream's work; returns when the rows are in the master."""
        if not self.evict_victim_cache or self._bound is None:
            return
        self.stream.wait_stream(torch.cuda.current_stream(self.dev))
        self._write_store(self._bound, ce=self.pcie_mode == "ce" and not self.emb_tables.emb_l[0].weight.is_cuda)
        self.stream.synchronize()

    # -- export of the cached rows into the master ----------------------------------------------------
    # HBM staging of a copy-engine export, in rows of the grow-only "evict" buffer: the list is packed and written back
    # in pieces of at most this many bytes
    EXPORT_STAGE_BYTES = 2 << 30

    def collect_valid(self, share=(0, 1)):
        """Valid cache lines of every table whose set is in share r of W of the sets (cdlrm_cache_collect_valid), on the
        planner's stream: (slots int32, ids int64 device tensors, offsets, counts); table k's list is
        [off[k], off[k] + counts[k]), ascending by slot."""
        s = self.stream
        caps = [self.ways * int(S) for S in self.cg.cache_sizes]
        off = [0] * self.T
        for k in range(1, self.T):
            off[k] = off[k - 1] + caps[k - 1]
        h = torch.zeros(self.T, dtype=torch.int64).pin_memory()
        with torch.cuda.stream(s):
            slots = torch.empty(max(sum(caps), 1), dtype=torch.int32, device=self.dev)
            ids = torch.empty(max(sum(caps), 1), dtype=torch.int64, device=self.dev)
            check(lib.cdlrm_cache_collect_valid(self.ctx, int(share[0]), int(share[1]), _vp(slots.data_ptr()),
                                                _vp(ids.data_ptr()), _lib.i64_array(off), _vp(h.data_ptr()), _sp(s)))
        s.synchronize()
        return slots, ids, off, h.tolist()

    def write_cached_to_master(self, share=(0, 1)):
        """master[k][id] = weight[k][slot] for every valid cache line of share r of W of the sets (what the eviction of
        every cached row would write back); returns the number of rows.  ``pcie_mode`` "sm": the evict kernel writes the
        master zero-copy (its PCIe-throttled grid).  "ce": the same kernel packs the rows into the HBM staging buffer
        (at most EXPORT_STAGE_BYTES at a time) and cdlrm_host_writeback_rows scatters them into the master.  Runs on
        the planner's stream after the current stream's work; returns when the rows are in the master."""
        s = self.stream
        s.wait_stream(torch.cuda.current_stream(self.dev))
        slots, ids, off, cnt = self.collect_valid(share)
        total = sum(cnt)
        ce = self.pcie_mode == "ce" and not self.emb_tables.emb_l[0].weight.is_cuda
        if not ce:
            with torch.cuda.stream(s):
                for k in range(self.T):
                    if cnt[k]:
                        check(lib.cdlrm_move_evict(self.ctx, k, _vp(ids[off[k]:].data_ptr()), _vp(slots[off[k]:].data_ptr()),
                                                   None, cnt[k], None, 1, 0, _sp(s)))
            s.synchronize()
            return total
        hid, hoff = self._ids_to_host("export_ids", ids, [(off[k], cnt[k]) for k in range(self.T)])
        cap = max(1, min(total, self.EXPORT_STAGE_BYTES // (4 * self.dim)))
        stage = self._buf("evict", cap)
        rows_per, bufs, _evs = self._ce_chunks()

        def flush(pieces):              # pieces: (table, offset in the table's list, rows, first staging row)
            with torch.cuda.stream(s):
                for k, o, n, r in pieces:
                    check(lib.cdlrm_move_evict(self.ctx, k, _vp(ids[off[k] + o:].data_ptr()),
                                               _vp(slots[off[k] + o:].data_ptr()), None, n, _vp(stage[r:].data_ptr()),
                                               0, 0, _sp(s)))
            Ws = [self.emb_tables.emb_l[k].weight.data for k, _o, _n, _r in pieces]
            check(lib.cdlrm_host_writeback_rows(
                self.dev.index, len(pieces), _lib.ptr_array([W.data_ptr() for W in Ws]),
                _lib.i64_array([W.shape[0] for W in Ws]), self.dim,
                _lib.ptr_array([hid.data_ptr() + 8 * (hoff[k] + o) for k, o, _n, _r in pieces]), None,
                _lib.i64_array([n for _k, _o, n, _r in pieces]), _lib.ptr_array([stage[r:].data_ptr() for *_x, r in pieces]),
                _vp(bufs[0].data_ptr()), _vp(bufs[1].data_ptr()), rows_per, 0, self.host_threads, _sp(s)))

        pieces, used = [], 0
        for k in range(self.T):
            o = 0
            while o < cnt[k]:
                n = min(cnt[k] - o, cap - used)
                pieces.append((k, o, n, used))
                o += n
                used += n
                if used == cap:
                    flush(pieces)
                    pieces, used = [], 0
        if pieces:
            flush(pieces)
        s.synchronize()
        self._pin.pop("export_ids", None)         # a checkpoint-sized pinned list is not kept
        return total

    # -- look-ahead staging -------------------------------------------------------------------
    def stage(self, rec):
        """Prefetch, on the planner's stream, everything window w+1 needs from the host master
        while window w still trains: the rows of the fill list and (with ``collect_losers``) the
        rows of the ids that stay un-cached, into HBM staging buffers -- gathered zero-copy over PCIe by a
        kernel (``pcie_mode`` "sm") or by host threads + cudaMemcpyAsync ("ce").  Exact under the sequential
        schedule (DESIGN.md section 2): none of these ids is cached during window w, so their master rows cannot
        change before the boundary, and the write-back of the previous boundary precedes these reads."""
        s = self.stream
        d = self.dim
        ce = self.pcie_mode == "ce" and not self.emb_tables.emb_l[0].weight.is_cuda
        if ce:
            self.flush_writeback()
        fill_jobs, loser_jobs = [], []      # (table, offset into the device id list, rows, device address of the rows)
        with torch.cuda.stream(s):
            self._buf("evict", max(sum(rec.F), 1))      # sized now (E <= F): no cudaMalloc at the boundary
            rec.stage_begin = torch.cuda.Event(enable_timing=True)
            rec.stage_begin.record(s)
            rec.fill_soff = [0] * self.T
            for k in range(1, self.T):
                rec.fill_soff[k] = rec.fill_soff[k - 1] + rec.F[k - 1]
            rec.fill_peers = None
            if self._fill_shard is not None:
                # sharded: this rank pulls its share of every table's fill list into a peer-readable buffer (two
                # alternate: the peers read the previous one at THEIR boundary); same layout on every rank
                rank, world, _group = self._fill_shard
                self._fill_no = getattr(self, "_fill_no", 0) + 1
                rec.fill_stage = None
                rec.fill_peers = self._peer_buf("fill%d" % (self._fill_no & 1), max(sum(rec.F), 1), self._fill_shard)[1]
                row_b = 4 * d
                for k in range(self.T):
                    for r in (range(world) if _group == "local" else (rank,)):
                        lo, n = wb_share_range(rec.F[k], r, world)
                        if n:
                            fill_jobs.append((k, rec.off[k] + lo, n, rec.fill_peers[r] + (rec.fill_soff[k] + lo) * row_b))
            else:
                rec.fill_stage = self._buf("fill", max(sum(rec.F), 1))
                for k in range(self.T):
                    if rec.F[k]:
                        fill_jobs.append((k, rec.off[k], rec.F[k], rec.fill_stage[rec.fill_soff[k]:].data_ptr()))
            rec.loser_shard = rec.loser_peers = None
            if rec.L is not None and self._shard is not None:
                # sharded store: this rank pulls rows [rank * shard, (rank + 1) * shard) of every table's list
                rank, world, _group = self._shard
                self._stage_no += 1
                rec.loser_shard = [(n + world - 1) // world for n in rec.L]
                rec.loser_soff = [0] * self.T
                for k in range(1, self.T):
                    rec.loser_soff[k] = rec.loser_soff[k - 1] + rec.loser_shard[k - 1]
                ptrs = self._peer_buf("loser%d" % (self._stage_no & 1), max(sum(rec.loser_shard), 1))[1]
                row_b = 4 * d
                rec.loser_peers = [[ptrs[r] + rec.loser_soff[k] * row_b for r in range(world)] for k in range(self.T)]
                for k in range(self.T):
                    for r in (range(world) if _group == "local" else (rank,)):
                        lo = r * rec.loser_shard[k]
                        n_k = min(rec.L[k], lo + rec.loser_shard[k]) - lo
                        if n_k > 0:
                            loser_jobs.append((k, rec.loser_off[k] + lo, n_k, rec.loser_peers[k][r]))
            elif rec.L is not None:
                # two loser stores alternate: the previous window's is read by the forward until the boundary
                self._stage_no += 1
                rec.loser_soff = [0] * self.T          # rows are packed by the (possibly capped) counts
                for k in range(1, self.T):
                    rec.loser_soff[k] = rec.loser_soff[k - 1] + rec.L[k - 1]
                rec.loser_stage = self._buf("loser%d" % (self._stage_no & 1), max(sum(rec.L), 1))
                for k in range(self.T):
                    if rec.L[k]:
                        loser_jobs.append((k, rec.loser_off[k], rec.L[k], rec.loser_stage[rec.loser_soff[k]:].data_ptr()))
            if not ce:
                for ids_dev, jobs in ((rec.fill_ids, fill_jobs), (rec.loser_ids, loser_jobs)):
                    for k, o, n, dst in jobs:
                        check(lib.cdlrm_move_gather_master(self.ctx, k, _vp(ids_dev[o:].data_ptr()), n, _vp(dst), _sp(s)))
        if ce:
            # everything the write-back of this window's boundary will need, sized now (E <= F) with head-room: a
            # cudaHostAlloc / cudaMalloc in the middle of a window stalls every CUDA call of the process for 10-20 ms
            n_fill = max(sum(rec.F), 1)
            self._pinned("wb_ids", 8 * n_fill)
            self._pinned("wb_prim", n_fill)
            if self.evict_victim_cache and rec.L is not None:
                self._pinned("store_ids", 8 * max(sum(rec.L), 1))     # this store's write-back, two boundaries on
            self._ce_chunks()
            for name, ids_dev, jobs in (("fill_ids", rec.fill_ids, fill_jobs), ("loser_ids", rec.loser_ids, loser_jobs)):
                if jobs:
                    hid, offs = self._ids_to_host(name, ids_dev, [(o, n) for _k, o, n, _dst in jobs])
                    self._ce_gather([(k, hid[ho:ho + n], dst) for (k, _o, n, dst), ho in zip(jobs, offs)])
        with torch.cuda.stream(s):
            rec.staged = torch.cuda.Event(enable_timing=True)
            rec.staged.record(s)
        # host-master rows pulled over PCIe by this prefetch (bench.py: prefetch GB/s = bytes / event time)
        rec.stage_bytes = 4 * d * (sum(n for _k, _o, n, _dst in fill_jobs) + sum(n for _k, _o, n, _dst in loser_jobs))
        return rec

    def install_staged(self, rec, write_master=True, average_on_writeback=False, stream=None, wb_share=None):
        """Window boundary with staged data: on ``stream`` (default: current) the evicted rows are
        copied HBM->HBM into a write-back buffer, the fills come HBM->HBM from the staging buffer
        and the loser store is switched; the write-back to the host master then runs on the
        planner's stream beside the next window's training steps.
        ``wb_share = (r, W)``: data-parallel replicas whose caches agree at the boundary (they were just aggregated)
        and that share ONE host master: this rank writes back only the r-th of W equal shares of every table's
        eviction list -- the write-back takes 1/W of the time instead of loading rank 0 alone."""
        s = stream or torch.cuda.current_stream(self.dev)
        d = self.dim
        tm = [time.perf_counter()]               # host time of the phases (Trainer.boundary_breakdown_ms)
        r_, W_ = wb_share if wb_share is not None else (0, 1)
        rec.wb_lo, rec.wb_n = zip(*[wb_share_range(E, r_, W_) for E in rec.E]) if rec.E else ((), ())
        if rec.staged is None:
            self.stage(rec)
        s.wait_event(rec.staged)
        for t in (rec.evict_ids, rec.evict_slots, rec.evict_primary, rec.fill_ids, rec.fill_slots, rec.fill_stage,
                  rec.loser_ids, rec.loser_stage):
            if t is not None and s != self.stream:
                t.record_stream(s)
        with torch.cuda.stream(s):
            eoff = [0] * self.T
            for k in range(1, self.T):
                eoff[k] = eoff[k - 1] + rec.E[k - 1]
            # (the write-back that last read this buffer precedes rec.staged on the planner stream)
            rec.evict_stage = self._buf("evict", max(sum(rec.E), 1))
            tm.append(time.perf_counter())
            for k in range(self.T):
                if rec.E[k]:
                    ids, slots, prim = rec.evict_list(k)
                    check(lib.cdlrm_move_evict(self.ctx, k, _vp(ids.data_ptr()), _vp(slots.data_ptr()),
                                               _vp(prim.data_ptr()), rec.E[k],
                                               _vp(rec.evict_stage[eoff[k]:].data_ptr()), 0, 0, _sp(s)))
            tm.append(time.perf_counter())
            if self.evict_victim_cache and self._bound is not None:
                # the bound store is still the finished window's: ids it trained are prefetched stale in this window's
                # fill and loser rows (gathered from the master while it trained); its rows replace them
                for k in range(self.T):
                    if rec.F[k]:
                        check(lib.cdlrm_move_carry_losers(self.ctx, k, _vp(rec.fill_ids[rec.off[k]:].data_ptr()), rec.F[k],
                                                          _vp(rec.fill_stage[rec.fill_soff[k]:].data_ptr()), _sp(s)))
                    if rec.L is not None and rec.L[k]:
                        check(lib.cdlrm_move_carry_losers(self.ctx, k, _vp(rec.loser_ids[rec.loser_off[k]:].data_ptr()),
                                                          rec.L[k], _vp(rec.loser_stage[rec.loser_soff[k]:].data_ptr()),
                                                          _sp(s)))
            tm.append(time.perf_counter())
            for k in range(self.T):
                if rec.F[k] and rec.fill_peers is not None:
                    # share r of the list comes out of rank r's staging buffer (local HBM or NVLink peer memory)
                    ids, slots = rec.fill_list(k)
                    world = len(rec.fill_peers)
                    for r in range(world):
                        lo, n = wb_share_range(rec.F[k], r, world)
                        if n:
                            check(lib.cdlrm_move_fill(self.ctx, k, _vp(ids[lo:].data_ptr()), _vp(slots[lo:].data_ptr()), n,
                                                      _vp(rec.fill_peers[r] + (rec.fill_soff[k] + lo) * 4 * d), None, _sp(s)))
                elif rec.F[k]:
                    ids, slots = rec.fill_list(k)
                    check(lib.cdlrm_move_fill(self.ctx, k, _vp(ids.data_ptr()), _vp(slots.data_ptr()), rec.F[k],
                                              _vp(rec.fill_stage[rec.fill_soff[k]:].data_ptr()), None, _sp(s)))
            tm.append(time.perf_counter())
            if rec.L is not None and rec.loser_peers is not None:
                world = self._shard[1]
                check(lib.cdlrm_ctx_bind_losers_sharded(
                    self.ctx,
                    _lib.ptr_array([rec.loser_ids[rec.loser_off[k]:].data_ptr() if rec.L[k] else 0
                                    for k in range(self.T)]),
                    _lib.i64_array(rec.L), _lib.i64_array(rec.loser_shard), world,
                    _lib.ptr_array([p for k in range(self.T) for p in rec.loser_peers[k]]), _sp(s)))
            elif rec.L is not None:
                check(lib.cdlrm_ctx_bind_losers(
                    self.ctx,
                    _lib.ptr_array([rec.loser_ids[rec.loser_off[k]:].data_ptr() if rec.L[k] else 0
                                    for k in range(self.T)]),
                    _lib.ptr_array([rec.loser_stage[rec.loser_soff[k]:].data_ptr() if rec.L[k] else 0
                                    for k in range(self.T)]),
                    _lib.i64_array(rec.L), _sp(s)))
            else:
                check(lib.cdlrm_ctx_bind_losers(self.ctx, None, None, None, _sp(s)))
            moved = torch.cuda.Event()
            moved.record(s)
        tm.append(time.perf_counter())
        ws = self.stream
        ws.wait_event(moved)       # later planner-stream work (next prefetch) may reuse the staging buffers
        prev, self._bound = self._bound, (rec if rec.L is not None else None)
        if self.evict_victim_cache and prev is not None and write_master:
            # the finished window's store goes back to the master before anything of the window after next reads it:
            # ce by the next flush_writeback (the plan thread, before its plan); sm right here on the planner stream.
            # Its buffers are the ones the next stage() fills: both come after this in planner-stream order
            if self.pcie_mode == "ce" and not self.emb_tables.emb_l[0].weight.is_cuda:
                self._pending_store = prev
            else:
                self._write_store(prev, ce=False)
        if write_master and sum(rec.wb_n) and self.pcie_mode == "ce" and not self.emb_tables.emb_l[0].weight.is_cuda:
            # copy engine + host threads: done by the thread that plans the next window (flush_writeback), before
            # anything of that window reads the master; callers that read the master themselves call it first
            rec.evict_stage.record_stream(ws)
            self._pending_wb = (rec, bool(average_on_writeback))
        elif write_master and sum(rec.wb_n):
            rec.evict_stage.record_stream(ws)
            with torch.cuda.stream(ws):
                for k in range(self.T):
                    lo, n = rec.wb_lo[k], rec.wb_n[k]
                    if n:
                        ids, _slots, prim = rec.evict_list(k)
                        check(lib.cdlrm_move_scatter_master2(self.ctx, k, _vp(ids[lo:].data_ptr()), _vp(prim[lo:].data_ptr()),
                                                             n, _vp(rec.evict_stage[eoff[k] + lo:].data_ptr()),
                                                             int(average_on_writeback), _sp(ws)))
        rec.wb_done = torch.cuda.Event(enable_timing=True)
        rec.wb_done.record(self.stream)
        tm.append(time.perf_counter())
        self.last_install_ms = {n: round(1e3 * (y - x), 2) for n, x, y in
                                zip(("wait_and_buffers", "evict_launches", "carry_launches", "fill_launches", "bind_losers",
                                     "writeback_launches"),
                                    tm, tm[1:])}
        return rec

    # -- install ---------------------------------------------------------------------------
    def install(self, rec, write_master=True, average_on_writeback=False, collect_evictions=False,
                fill_rows=None, stream=None):
        """Apply a plan at the window boundary on ``stream`` (default: current stream):
        evicted rows are read BEFORE any fill writes; with ``write_master`` they go straight
        back to the pinned master (zero-copy); ``collect_evictions`` additionally returns the
        reference's ``eviction_data`` list [(ids, rows)] as device tensors.
        ``fill_rows``: optional list of (rows_k, src_index_k) device tensors -- rows provided
        by the caller (reference API: ``table_cache[map[ids]]``); default reads the master."""
        s = stream or torch.cuda.current_stream(self.dev)
        out = []
        if s != self.stream:
            # the lists were allocated on the planner's stream: tell the caching allocator that
            # `s` reads them, so that freeing the record cannot hand the memory to the next plan
            # while the install kernels are still in flight
            for t in (rec.evict_ids, rec.evict_slots, rec.evict_primary, rec.fill_ids, rec.fill_slots):
                t.record_stream(s)
        with torch.cuda.stream(s):
            for k in range(self.T):
                ids, slots, prim = rec.evict_list(k)
                rows = None
                if collect_evictions:
                    rows = torch.empty(rec.E[k], self.dim, dtype=torch.float32, device=self.dev)
                if rec.E[k]:
                    check(lib.cdlrm_move_evict(self.ctx, k, _vp(ids.data_ptr()), _vp(slots.data_ptr()),
                                               _vp(prim.data_ptr()), rec.E[k],
                                               _vp(rows.data_ptr()) if rows is not None else None,
                                               int(write_master), int(average_on_writeback), _sp(s)))
                if collect_evictions:
                    out.append((ids, rows))
            for k in range(self.T):
                ids, slots = rec.fill_list(k)
                if not rec.F[k]:
                    continue
                r, si = (None, None) if fill_rows is None else fill_rows[k]
                check(lib.cdlrm_move_fill(self.ctx, k, _vp(ids.data_ptr()), _vp(slots.data_ptr()), rec.F[k],
                                          _vp(r.data_ptr()) if r is not None else None,
                                          _vp(si.data_ptr()) if si is not None else None, _sp(s)))
        return out


# ------------------------------------------------------------------------------------
# Prefetcher -- cache_manager.py:8-115
# ------------------------------------------------------------------------------------

def _util_planner(emb_tables_cpu, device, window_len):
    """A planner-only context per (master tables, device) used by the static
    ``process_batch_slice`` (it needs the unique + master-gather kernels, no cache).  Kept
    on the master-table object so that it dies with it."""
    from .model_no_ddp import Embedding_Table_Cache_Group
    reg = emb_tables_cpu.__dict__.setdefault("_cdlrm_util", {})
    key = device.index
    ent = reg.get(key)
    if ent is None or ent[1].window_len < window_len:
        ln = np.asarray([E.weight.shape[0] for E in emb_tables_cpu.emb_l])
        dim = emb_tables_cpu.emb_l[0].weight.shape[1]
        cg = Embedding_Table_Cache_Group(dim, ln, max_cache_size=2, aux_table_size=0, num_ways=1, device=device)
        ent = (cg, WindowPlanner(cg, emb_tables_cpu, window_len))
        reg[key] = ent
    return ent


class Prefetcher(threading.Thread):
    """Look-ahead scanner.  The reference runs it as a separate process with a CPU worker
    pool (cache_manager.py:66-115); here the scan is a handful of kernels, so ``run`` is a
    light host thread that only slices the loader's batches into windows of
    ``lookahead * mini_batch_size`` samples (:75,85-110) and hands the raw window ids to the
    trainer, whose ``WindowPlanner`` does the rest on a side stream."""

    def __init__(self, args, emb_tables_cpu, batch_fifo, eviction_fifo, finish_event, cache_ld):
        super().__init__(daemon=True)
        self.args = args
        self.emb_tables_cpu = emb_tables_cpu
        self.batch_fifo = batch_fifo
        self.eviction_fifo = eviction_fifo
        self.finish_event = finish_event
        self.cache_ld = cache_ld

    @staticmethod
    def pin_pool(p, core):
        """cache_manager.py:20-25 (CPU affinity of pool worker p)."""
        try:
            os.sched_setaffinity(0, {core + 3 + p})
        except (OSError, ValueError):
            pass
        return 1

    @staticmethod
    def process_batch_slice(slice, emb_tables_cpu):
        """cache_manager.py:27-46: per table the ascending unique ids of the window, the
        dense id->position map and the unique rows of the master table.  Unique and the row
        gather run on the GPU (bitmap compaction + zero-copy gather); results come back on
        the device of ``slice`` (CPU in the reference's multi-process hand-off)."""
        if not torch.cuda.is_available():
            raise _lib.CdlrmError("process_batch_slice needs a CUDA device: no CPU fallback")
        src_dev = slice.device
        dev = slice.device if slice.is_cuda else torch.device("cuda", torch.cuda.current_device())
        ids = slice.to(dev, dtype=torch.int64).contiguous()
        cg, pl = _util_planner(emb_tables_cpu, dev, int(ids.shape[1]))
        s = torch.cuda.current_stream(dev)
        check(lib.cdlrm_plan_unique(pl.ctx, _vp(ids.data_ptr()), ids.stride(0), ids.shape[1],
                                    _vp(pl._h_counts.data_ptr()), _sp(s)))
        s.synchronize()
        cg.check_device_flags()
        U = pl._h_counts.view(-1, 4)[:, 0].tolist()
        rows_l, uniq_l, maps_l = [], [], []
        for k in range(len(emb_tables_cpu.emb_l)):
            u = pl.unique_tensor(k, U[k])
            rows = torch.empty(U[k], cg.dim, dtype=torch.float32, device=dev)
            check(lib.cdlrm_move_gather_master(pl.ctx, k, _vp(u.data_ptr()), U[k], _vp(rows.data_ptr()), _sp(s)))
            m = torch.full((int(u.max().item()) + 1 if U[k] else 1, 1), -1, dtype=torch.long, device=dev)
            if U[k]:
                m[u, 0] = torch.arange(U[k], device=dev)
            uniq_l.append(u.to(src_dev))
            rows_l.append(rows.to(src_dev))
            maps_l.append(m.to(src_dev))
        return rows_l, uniq_l, maps_l

    @staticmethod
    def apply_eviction_data(emb_tables, eviction_data, average_on_writeback=False):
        """Body of the eviction loop (cache_manager.py:58-62): ``W[idxs] = emb`` or
        ``(W[idxs] + emb) / 2`` through cdlrm_move_scatter_master (zero-copy writes into the
        pinned master)."""
        dev = torch.device("cuda", torch.cuda.current_device())
        _cg, pl = _util_planner(emb_tables, dev, 1)
        s = torch.cuda.current_stream(dev)
        for k, (idxs, embeddings) in enumerate(eviction_data):
            n = int(idxs.numel())
            if n == 0:
                continue
            if average_on_writeback:
                # duplicates carry identical rows; keep one so the average is applied once
                idxs_u, inv = torch.unique(idxs, return_inverse=True)
                rep = torch.empty(idxs_u.numel(), dtype=torch.long, device=idxs.device)
                rep[inv] = torch.arange(n, device=idxs.device)
                idxs, embeddings, n = idxs_u, embeddings[rep], int(idxs_u.numel())
            i_d = idxs.to(dev, dtype=torch.int64).contiguous()
            e_d = embeddings.to(dev, dtype=torch.float32).contiguous()
            check(lib.cdlrm_move_scatter_master(pl.ctx, k, _vp(i_d.data_ptr()), n, _vp(e_d.data_ptr()),
                                                int(bool(average_on_writeback)), _sp(s)))
        s.synchronize()

    @staticmethod
    def eviction_manager(emb_tables, eviction_fifo, average_on_writeback, core, timeout):
        """cache_manager.py:48-64: pop eviction_data and write the rows back into the master
        tables.  (With ``WindowPlanner.install(write_master=True)`` the write-back already
        happened on the GPU and nothing is queued.)"""
        try:
            os.sched_setaffinity(0, {core})
        except (OSError, ValueError):
            pass
        try:
            while True:
                eviction_data = eviction_fifo.get(timeout=timeout) if timeout > 0 else eviction_fifo.get()
                Prefetcher.apply_eviction_data(emb_tables, eviction_data, average_on_writeback)
        except Exception:
            print('Eviction queue empty longer than expected. Exiting eviction manager...')

    def windows(self):
        """Generator of raw window id tensors [T, <= lookahead*mini_batch_size] in training
        order: entry w covers steps [w*lookahead, (w+1)*lookahead) (SURVEY 3.4 invariant).  With
        ``args.load_model`` the windows before the checkpoint's resume point are skipped (the loaders are
        deterministic: the run that saved saw the same windows)."""
        per = self.args.lookahead
        skip = 0
        if getattr(self.args, "load_model", ""):
            from .checkpoint import read_meta
            skip = int(read_meta(self.args.load_model)["resume"]["window"])
        w = 0
        for _epoch in range(self.args.nepochs):
            acc = []
            for _j, batch in enumerate(self.cache_ld):
                acc.append(batch[2])
                if len(acc) == per:
                    if w >= skip:
                        yield torch.cat(acc, dim=1)
                    w += 1
                    acc = []
            if acc:
                if w >= skip:
                    yield torch.cat(acc, dim=1)
                w += 1

    @property
    def fifo_payload(self):
        """What ``run`` puts on ``batch_fifo`` per window.  "tuples" (default -- the reference's contract,
        cache_manager.py:102-104): ``process_batch_slice``'s ``(rows, uniq, maps)``, consumed by
        ``load_caches_and_broadcast`` / ``CacheEmbeddings``.  "ids": the raw window ids [T, n] -- all the
        GPU-resident ``WindowPlanner`` needs (it finds the unique ids itself and reads the master rows at
        install time), without the per-window gather of every unique row.  Chosen by ``args.fifo_payload``
        (flag ``--fifo-payload`` of this package's main); the consumers accept either."""
        return getattr(self.args, "fifo_payload", None) or "tuples"

    def markers(self):
        """``ids`` payloads of a ``cache_ld`` that provides ``window_marker`` (criteo_bin.CriteoBinDataset): one marker
        per window in training order, the windows before the ``--load-model`` resume point skipped, the short last
        window of an epoch included.  Nothing is read here: the plan thread reads each window when it scans it."""
        L = self.args.lookahead
        per_epoch = -(-len(self.cache_ld) // L)
        skip = 0
        if getattr(self.args, "load_model", ""):
            from .checkpoint import read_meta
            skip = int(read_meta(self.args.load_model)["resume"]["window"])
        for w in range(skip, self.args.nepochs * per_epoch):
            yield self.cache_ld.window_marker(w % per_epoch, L)

    def payloads(self):
        """Generator of the FIFO entries in training order (what ``run`` puts)."""
        mode = self.fifo_payload
        if mode not in ("tuples", "ids"):
            raise ValueError("fifo_payload must be 'tuples' or 'ids', got %r" % (mode,))
        if mode == "ids" and hasattr(self.cache_ld, "window_marker"):
            yield from self.markers()
            return
        for win in self.windows():
            if mode == "ids":
                yield win
            else:
                a = Prefetcher.process_batch_slice(win, self.emb_tables_cpu)
                yield (a[0], a[1], a[2])                                   # cache_manager.py:102-104

    def run(self):
        """cache_manager.py:66-115: start the eviction manager, then feed ``batch_fifo`` window by window (the
        bounded queue is the back-pressure, as in the reference), then wait for ``finish_event``."""
        ev = threading.Thread(target=Prefetcher.eviction_manager, daemon=True,
                              args=(self.emb_tables_cpu, self.eviction_fifo, self.args.average_on_writeback,
                                    self.args.main_start_core + 2, self.args.eviction_fifo_timeout))
        if self.eviction_fifo is not None:
            ev.start()
        try:
            for item in self.payloads():
                self.batch_fifo.put(item)
        except Exception as e:          # surfaced by the consumer instead of a silent hang on an empty queue
            self.batch_fifo.put(e)
            raise
        if self.finish_event is not None:
            self.finish_event.wait()
