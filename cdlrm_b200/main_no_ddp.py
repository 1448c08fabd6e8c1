"""B200-native mirror of the reference's ``main_no_ddp.py`` (lkp411/cDLRM): same function
names, argument order and CLI flags, hot path in libcdlrm_b200.so.

Kept verbatim as an interface (reference file:line): ``ProcessArgs`` (:34-145),
``CacheEmbeddings`` (:148-209), ``loss_fn_wrap`` (:212-221), ``time_wrap`` (:224-226),
``wait_wrap`` (:229-231), ``aggregate_gradients`` (:234-247), ``broadcast_and_aggregate``
(:250-292), ``share_occupancy_tables`` (:295-306), ``load_caches_and_broadcast``
(:309-321), ``Run`` (:324-502).
"""
import argparse
import collections
import ctypes
import itertools
import math
import os
import queue
import sys
import time

import numpy as np
import torch
import torch.distributed as dist
import torch.nn as nn

from . import _lib
from . import checkpoint as ckpt
from ._lib import check, lib
from .cache_manager import Prefetcher, TorchGlobalRng, VictimRng, VictimRngDevice, WindowPlanner
from .model_no_ddp import (DLRM_Net, Embedding_Table_Cache_Group, Embedding_Table_Group, EvalForward, bce_mean,
                           bce_mean_with_grad)

_vp = ctypes.c_void_p

# Trainer.evaluate: loss = mean BCE, accuracy = share of round(z) == t, auc = exact ROC AUC (NaN with one class only)
EvalResult = collections.namedtuple("EvalResult", "samples loss accuracy auc positives negatives")
_ONE_ID_PER_BAG = "evaluate needs one id per bag: lS_o must be arange(batch) for every table"

# (flag, type or "flag", default) -- spelling and defaults of main_no_ddp.py:34-145
_FLAGS = [
    ("arch-sparse-feature-size", int, 2), ("arch-embedding-size", str, "4-3-2"), ("arch-mlp-bot", str, "4-3-2"),
    ("arch-mlp-top", str, "4-2-1"), ("arch-interaction-op", str, "dot"), ("arch-interaction-itself", "flag", False),
    ("activation-function", str, "relu"), ("loss-function", str, "mse"), ("loss-weights", str, "1.0-1.0"),
    ("loss-threshold", float, 0.0), ("round-targets", bool, False),
    ("data-size", int, 1), ("num-batches", int, 0), ("data-generation", str, "random"),
    ("data-trace-file", str, "./input/dist_emb_j.log"), ("data-set", str, "kaggle"), ("raw-data-file", str, ""),
    ("processed-data-file", str, ""), ("data-randomize", str, "total"), ("data-trace-enable-padding", bool, False),
    ("max-ind-range", int, -1), ("data-sub-sample-rate", float, 0.0), ("num-indices-per-lookup", int, 10),
    ("num-indices-per-lookup-fixed", bool, False), ("num-workers", int, 0), ("memory-map", "flag", False),
    ("md-flag", "flag", False), ("md-threshold", int, 200), ("md-temperature", float, 0.3),
    ("md-round-dims", "flag", False), ("qr-flag", "flag", False), ("qr-threshold", int, 200),
    ("qr-operation", str, "mult"), ("qr-collisions", int, 4),
    ("mini-batch-size", int, 1), ("nepochs", int, 1), ("learning-rate", float, 0.1), ("lr-embeds", float, 0.3),
    ("print-precision", int, 5), ("numpy-rand-seed", int, 123), ("sync-dense-params", bool, True),
    ("lookahead", int, 2), ("cache-workers", int, 2), ("cache-size", int, 10240), ("num-ways", int, 4),
    ("average-on-writeback", "flag", False), ("evict-victim-cache", "flag", False),
    ("print-freq", int, 1), ("test-freq", int, -1), ("test-mini-batch-size", int, -1), ("test-num-workers", int, -1),
    ("print-time", "flag", False), ("debug-mode", "flag", False), ("enable-profiling", "flag", False),
    ("plot-compute-graph", "flag", False), ("save-model", str, ""), ("load-model", str, ""),
    ("mlperf-logging", "flag", False), ("mlperf-acc-threshold", float, 0.0), ("mlperf-auc-threshold", float, 0.0),
    ("mlperf-bin-loader", "flag", False), ("mlperf-bin-shuffle", "flag", False), ("large-batch", "flag", False),
    ("world-size", int, 2), ("master-port", int, 12345), ("trainer-start-core", int, 7), ("main-start-core", int, 0),
    ("dense-threshold", int, 1000), ("table-agg-op", str, "mean"), ("table-agg-freq", int, 1),
    ("batch-fifo-size", int, 8), ("eviction-fifo-size", int, 8), ("eviction-fifo-timeout", int, 300),
    ("inference-only", "flag", False), ("save-onnx", "flag", False), ("use-gpu", "flag", False),
]
# additions of this implementation (not in the reference)
_EXTRA_FLAGS = [
    # Run executes the reference's literal loop: rank-0 CacheEmbeddings + full-cache broadcast at every window
    # (load_caches_and_broadcast), explicit slot windows for broadcast_and_aggregate, torch's global CPU
    # generator as the victim stream (consumed in the reference's order, so the cache decisions are those of the
    # reference program run with the same seed), no look-ahead overlap, no CUDA graph
    ("strict-reference", "flag", False),
    # index distribution of --data-generation synthetic|random (cdlrm_b200/synthetic.py)
    ("synthetic-dist", str, "zipf"), ("synthetic-zipf-a", float, 1.05),
    # what Prefetcher.run puts on batch_fifo: "tuples" = the reference's (rows, uniq, maps); "ids" = raw window ids
    ("fifo-payload", str, ""),
    ("no-cuda-graph", "flag", False),
]


def build_parser():
    parser = argparse.ArgumentParser(description="Train Deep Learning Recommendation Model (DLRM)")
    for name, typ, default in _FLAGS + _EXTRA_FLAGS:
        if typ == "flag":
            parser.add_argument("--" + name, action="store_true", default=default)
        else:
            parser.add_argument("--" + name, type=typ, default=default)
    return parser


def ProcessArgs(argv=None):
    return build_parser().parse_args(argv)


# ------------------------------------------------------------------------------------
# window install -- main_no_ddp.py:148-209
# ------------------------------------------------------------------------------------


def _planner_of(cache_group, emb_tables, need_len):
    pl = getattr(cache_group, "_compat_planner", None)
    if pl is None or pl.window_len < need_len:
        pl = WindowPlanner(cache_group, emb_tables, max(need_len, 1), rng=TorchGlobalRng())
        cache_group._compat_planner = pl
    return pl


def CacheEmbeddings(cached_entries_per_table, lists_of_unique_idxs, unique_indices_maps, cache_group, eviction_fifo,
                    rank):
    """Window install (main_no_ddp.py:148-209).  Decisions (hit / pinned / dropped / sampled
    way / evicted / last-wins duplicates) come from cdlrm_plan_phase_a/_b and are bit-exact
    with the reference; the victim way uses the global torch CPU generator exactly as
    ``Categorical.sample()`` does (:183-185).  Evicted (id, row) pairs are put on
    ``eviction_fifo`` as CPU tensors when ``rank == 0`` (:208-209)."""
    cg = cache_group
    dev = cg.device
    need = max(int(u.numel()) for u in lists_of_unique_idxs)
    cg._ensure_ctx(None)
    pl = _planner_of(cg, None, need)
    rec = pl.plan(uniq_lists=lists_of_unique_idxs)
    fill_rows = []
    for k in range(len(cached_entries_per_table)):
        ids, _slots = rec.fill_list(k)
        rows_k, map_k = cached_entries_per_table[k], unique_indices_maps[k]
        if rec.F[k] == 0:
            fill_rows.append((None, None))
        elif rows_k.is_cuda:
            src = map_k.to(dev)[ids].flatten().contiguous()              # :205
            fill_rows.append((rows_k.contiguous(), src))
        else:
            src = map_k[ids.cpu()].flatten()
            fill_rows.append((rows_k[src].to(dev, non_blocking=False).contiguous(), None))
    ev = pl.install(rec, write_master=False, collect_evictions=True, fill_rows=fill_rows)
    cg.last_plan = rec
    if rank == 0:
        eviction_fifo.put([(i.cpu(), r.cpu()) for i, r in ev])


def loss_fn_wrap(Z, T, loss_fn, args, loss_ws=None):
    if args.loss_function == "mse" or args.loss_function == "bce":
        return loss_fn(Z, T)
    elif args.loss_function == "wbce":
        loss_ws_ = loss_ws[T.data.view(-1).long()].view_as(T)
        loss_fn_ = loss_fn(Z, T)
    loss_sc_ = loss_ws_ * loss_fn_
    return loss_sc_.mean()


def time_wrap(rank):
    torch.cuda.synchronize(rank)
    return time.time()


def wait_wrap(req_objs):
    for obj in req_objs:
        obj.wait()


def _world():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def aggregate_gradients(dlrm, include_bias=False):
    """main_no_ddp.py:234-247: average the Linear WEIGHT grads over ranks (the reference never
    reduces the biases; ``include_bias=True`` fixes that).  One flat bucket, one all-reduce."""
    W = _world()
    grads = []
    for seq in (dlrm.bot_l, dlrm.top_l):
        for layer in seq:
            if isinstance(layer, nn.modules.linear.Linear):
                grads.append(layer.weight.grad)
                if include_bias:
                    grads.append(layer.bias.grad)
    if W == 1:
        return []
    flat = torch.cat([g.reshape(-1) for g in grads])
    flat /= W
    work = dist.all_reduce(flat, async_op=True)

    class _Unflatten:
        def wait(self_inner):
            work.wait()
            o = 0
            for g in grads:
                g.copy_(flat[o:o + g.numel()].view_as(g))
                o += g.numel()

    return [_Unflatten()]


# ------------------------------------------------------------------------------------
# table aggregation -- main_no_ddp.py:250-292
# ------------------------------------------------------------------------------------


class _DistComm:
    """The two collectives of the table aggregation over torch.distributed (NCCL on the GPU box).
    Tests substitute an in-process transport with the same three members to run W > 1 replicas
    of ``broadcast_and_aggregate`` on one device (tests/test_gpu_aggregate.py)."""

    @property
    def world(self):
        return _world()

    def all_gather_into(self, out, inp):
        dist.all_gather_into_tensor(out, inp)

    def all_reduce(self, buf, op):
        dist.all_reduce(buf, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)


@torch.no_grad()
def broadcast_and_aggregate(cache_group, cache_group_idxs, rank, reduce_op="mean", comm=None):
    """Every ``table_agg_freq`` steps: union over ranks of the touched slots per table,
    ``weight[u] = sum_r weight_r[u] / W`` (mean) or sum / max.  ``cache_group_idxs`` is the
    reference's int32 ``[T, n]`` slot tensor; pass ``None`` to use the dirty bitmaps that the
    fused backward maintains.  dirty bits -> all-gather + OR -> ascending slot lists ->
    pack (pre-divided by W, :277) -> ONE all-reduce on a contiguous buffer -> unpack."""
    cg = cache_group
    ctx = cg._ensure_ctx(None)
    dev = cg.device
    s = _vp(torch.cuda.current_stream(dev).cuda_stream)
    comm = comm if comm is not None else _DistComm()
    W = comm.world
    if reduce_op not in ("mean", "sum", "max"):
        raise ValueError(reduce_op)
    if cache_group_idxs is not None:
        idx = cache_group_idxs.to(dev, dtype=torch.int32)
        if idx.stride(1) != 1:
            idx = idx.contiguous()
        check(lib.cdlrm_agg_mark(ctx, _vp(idx.data_ptr()), idx.stride(0), idx.shape[1], s))
    dirty = cg.dirty_bitmap()
    T = len(cg.emb_l)
    bufs = getattr(cg, "_agg_bufs", None)
    if bufs is None or bufs[3].shape[0] != W:
        cap = int(sum(cg._cache_rows))
        bufs = (torch.empty(cap, dtype=torch.int32, device=dev), torch.empty(T, dtype=torch.int64, device=dev),
                torch.zeros(T, dtype=torch.int64).pin_memory(),
                torch.empty(W, dirty.numel(), dtype=torch.int32, device=dev))
        cg._agg_bufs = bufs
    slot_list, d_counts, h_counts, gathered = bufs
    # optional phase timing (bench.py sets cache_group._agg_prof = []): events at the phase borders of every call
    prof = getattr(cg, "_agg_prof", None)
    marks = []

    def mark():
        if prof is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record(torch.cuda.current_stream(dev))
            marks.append(e)

    mark()
    if W > 1:
        comm.all_gather_into(gathered.view(-1), dirty)
        check(lib.cdlrm_agg_or_bitmaps(ctx, _vp(gathered.data_ptr()), W, dirty.numel(), s))
    check(lib.cdlrm_agg_collect(ctx, _vp(slot_list.data_ptr()), _vp(d_counts.data_ptr()), _vp(h_counts.data_ptr()), s))
    mark()
    torch.cuda.current_stream(dev).synchronize()
    counts = h_counts.tolist()
    total = int(sum(counts))
    carr = _lib.i64_array(counts)
    if total == 0:
        return
    rows = getattr(cg, "_agg_rows", None)          # packed row buffer: grown, never shrunk
    if rows is None or rows.shape[0] < total:
        cg._agg_rows = None
        rows = cg._agg_rows = torch.empty(int(total * 1.25) + 16, cg.dim, dtype=torch.float32, device=dev)
    buf = rows[:total]
    div = float(W) if reduce_op == "mean" else 1.0
    mark()
    check(lib.cdlrm_agg_pack(ctx, _vp(slot_list.data_ptr()), carr, div, _vp(buf.data_ptr()), s))
    mark()
    if W > 1:
        comm.all_reduce(buf, reduce_op)
    mark()
    check(lib.cdlrm_agg_unpack(ctx, _vp(slot_list.data_ptr()), carr, _vp(buf.data_ptr()), 1, s))
    mark()
    if prof is not None:
        prof.append((total, marks))


def share_occupancy_tables(cache_group, occupancy_tables_fifos, rank):
    """main_no_ddp.py:295-306 shares rank 0's CPU tag tensors through host shared memory.  Here
    every rank keeps the tags in its own HBM and evolves them with the same deterministic
    plan, so there is nothing to ship; the initial state (-1) is already identical."""
    cache_group._ensure_ctx(None)


def _fifo_get(batch_fifo):
    item = batch_fifo.get()
    if isinstance(item, Exception):          # the Prefetcher thread died: say so instead of hanging
        raise item
    return item


@torch.no_grad()
def load_caches_and_broadcast(cache_group, batch_fifo, eviction_fifo, rank):
    """main_no_ddp.py:309-321, reference semantics: rank 0 pops the next window off ``batch_fifo`` and installs
    it (``CacheEmbeddings``), then every table's full cache weight (and, here, the HBM tags, which the reference
    shares through host memory, :295-306) is broadcast from rank 0.  The FIFO entry is the reference's
    ``(rows, uniq, maps)`` tuple (cache_manager.py:102-104) or a raw window id tensor [T, n], which is put
    through ``Prefetcher.process_batch_slice`` first."""
    dist_req_objs = []
    if rank == 0:
        item = _fifo_get(batch_fifo)
        if isinstance(item, torch.Tensor):
            master = getattr(cache_group, "_emb_tables", lambda: None)()
            if master is None:
                raise _lib.CdlrmError("a raw id window needs the master tables: call cache_group(...) or "
                                      "cache_group._ensure_ctx(emb_tables) once before the first install")
            item = Prefetcher.process_batch_slice(item, master)
        cached_entries_per_table, lists_of_unique_idxs, unique_indices_maps = item
        CacheEmbeddings(cached_entries_per_table, lists_of_unique_idxs, unique_indices_maps, cache_group,
                        eviction_fifo, rank)
    if _world() > 1:
        cache_group._ensure_ctx(None)
        for E, tags in zip(cache_group.emb_l, cache_group.occupancy_tables):
            dist_req_objs.append(dist.broadcast(E.weight.data, src=0, async_op=True))
            dist_req_objs.append(dist.broadcast(tags, src=0, async_op=True))
    return dist_req_objs


# ------------------------------------------------------------------------------------
# trainer -- the body of Run (main_no_ddp.py:324-502) around the new path
# ------------------------------------------------------------------------------------


class Trainer:
    """One rank of data-parallel training against a replicated look-ahead cache.

    Per step (main_no_ddp.py:401-425): cache forward -> DLRM (stock PyTorch MLPs + the
    interaction kernel) -> loss -> backward (interaction bwd, fused de-duplicated sparse
    SGD on the cache) -> MLP grad all-reduce -> SGD.  Every ``lookahead`` steps the next
    window's plan (computed ahead on a side stream by a background thread) is installed;
    every ``table_agg_freq`` steps touched cache rows are averaged over ranks.

    Differences from the reference, on purpose: every rank runs the same deterministic plan
    on the global window (same ids, same seeded victim stream, tags replicated in HBM), so
    the 1.2 GB-per-table full-cache broadcast (:318-319) disappears; at a window boundary the
    touched rows are averaged first, so rank 0 writes back the cross-rank mean.
    """

    def __init__(self, args, m_spa, ln_emb, ln_bot, ln_top, emb_tables, rank=0, world=1, device=None,
                 strict_reference=False):
        """``strict_reference``: objects are built in the reference's order with the reference's consumption
        of the global generators (Run, main_no_ddp.py:335-376), and no look-ahead planner is created -- windows
        are installed with ``load_caches_and_broadcast`` by the caller."""
        self.args = args
        self.strict = bool(strict_reference)
        self.rank, self.world = rank, world
        self.dev = device if device is not None else torch.device("cuda", rank)
        torch.cuda.set_device(self.dev)
        np.random.seed(args.numpy_rand_seed)                       # :335-337
        torch.cuda.manual_seed(args.numpy_rand_seed)
        torch.manual_seed(args.numpy_rand_seed)
        self.local_batch = math.ceil(args.mini_batch_size / world)  # :344
        self.emb_tables = emb_tables
        self.cache_group = Embedding_Table_Cache_Group(m_spa, ln_emb, max_cache_size=args.cache_size,
                                                       aux_table_size=args.mini_batch_size,
                                                       num_ways=args.num_ways, device=self.dev,
                                                       init="reference" if self.strict else "zeros")
        self.dlrm = DLRM_Net(ln_bot, ln_top, arch_interaction_op=args.arch_interaction_op,
                             arch_interaction_itself=args.arch_interaction_itself,
                             sync_dense_params=args.sync_dense_params, sigmoid_bot=-1,
                             sigmoid_top=ln_top.size - 2, loss_threshold=args.loss_threshold).to(self.dev)
        if args.loss_function == "mse":
            self.loss_fn, self.loss_ws = torch.nn.MSELoss(reduction="mean"), None
        elif args.loss_function == "bce":
            self.loss_fn, self.loss_ws = torch.nn.BCELoss(reduction="mean"), None
        elif args.loss_function == "wbce":
            self.loss_ws = torch.tensor(np.fromstring(args.loss_weights, dtype=float, sep="-")).to(self.dev)
            self.loss_fn = torch.nn.BCELoss(reduction="none")
        else:
            sys.exit("ERROR: --loss-function=" + args.loss_function + " is not supported")
        # dense parameters and their gradients in one flat bucket each (tensor-core MLP path only)
        self.flat = self.dlrm.mlp_impl == "tcgen05" and os.environ.get("CDLRM_FLAT_MLP", "1") != "0"
        if self.flat:
            self.dlrm.flatten_parameters()
            check(lib.cdlrm_mlp_set_option(5, int(os.environ.get("CDLRM_WGRAD_SIDE", "1") != "0")))
            if os.environ.get("CDLRM_DEFER_WGRAD", "1") != "0":
                self.dlrm.defer_wgrad_join(True)     # joined in the step, right before the gradients are used
        # N > 1: the top MLP's weight gradients (80 % of the dense parameters) are all-reduced as soon as its backward
        # is enqueued, beside the interaction backward and the bottom MLP; the rest follows at the end of the backward
        self._ar_stream, self._ar_work = None, None
        if self.flat and world > 1 and os.environ.get("CDLRM_EARLY_ALLREDUCE", "1") != "0":
            self._ar_stream = _lib.new_stream(self.dev, priority=-1)
            self.dlrm._mlp_state["top"].after_backward = self._early_allreduce
        self.optimizer_mlps = torch.optim.SGD(self.dlrm.parameters(), lr=args.learning_rate)
        self.optimizer_embeds = torch.optim.SGD(self.cache_group.parameters(), lr=args.lr_embeds)   # :376
        self.cache_group._ensure_ctx(emb_tables)
        self.cache_group.assume_one_id_per_bag = True              # Criteo batches (:390)
        # streams of the library's own: a pooled torch.cuda.Stream may alias the stream a graph is captured on
        self.side = _lib.new_stream(self.dev)
        # the lookup runs on its own stream beside the bottom MLP (joined before the interaction)
        self.cache_group.forward_stream = _lib.new_stream(self.dev, priority=-1)
        self.dlrm.pre_interact = self.cache_group.join_forward
        # the sparse update runs on the lookup stream beside the bottom MLP's backward (joined by
        # optimizer_embeds.step()); CDLRM_OVERLAP_UPDATE=0: from the optimizer hook, after the whole backward
        self.overlap_update = not self.strict and os.environ.get("CDLRM_OVERLAP_UPDATE", "1") != "0"
        self.planner = None
        if not self.strict:
            self.planner = WindowPlanner(self.cache_group, emb_tables, args.lookahead * args.mini_batch_size,
                                         rng=VictimRngDevice(args.numpy_rand_seed, self.dev), stream=self.side,
                                         lookahead_tags=True)
            self.planner.collect_losers = True     # un-cached ids of a window are served from an HBM loser store
            self.planner.primary_evictions_only = True   # the write-back needs the winner of a replaced slot only
            # master <-> HBM traffic of the planner: host threads + cudaMemcpyAsync ("ce": the chunk loops are native,
            # hostio.cu; hardly slows the step that runs beside it) when this rank has host cores to spare, else
            # zero-copy gather / scatter kernels ("sm": no host threads, but every system-memory access the SMs keep
            # in flight slows the training kernels 1.2-2x while it runs).  CDLRM_PREFETCH=ce|sm and
            # CDLRM_HOST_THREADS override; see DESIGN.md section 4 for the measurements behind the rule
            try:
                cores = len(os.sched_getaffinity(0))
            except (AttributeError, OSError):
                cores = os.cpu_count() or 2
            # at most half of this rank's cores (minus one) gather, at most 4: more bring nothing at one window per 2 s,
            # and the thread that enqueues the steps must never wait for a core
            threads = max(1, min(4, cores // max(world, 1) // 2 - 1))
            mode = os.environ.get("CDLRM_PREFETCH", "auto")
            self.planner.host_threads = int(os.environ.get("CDLRM_HOST_THREADS", threads))
            auto = "ce" if (world == 1 and self.planner.host_threads >= 3) else "sm"
            self.planner.pcie_mode = mode if mode in ("ce", "sm") else auto
        self._host_group = dist.new_group(backend="gloo") if world > 1 else None   # plan-thread barrier
        # write-back of a boundary's evictions shared by the ranks (they hold identical rows right after the boundary
        # aggregation and map the same host master): 1/world of every table's list each
        # (only when the master visibly IS one shared object -- a /dev/shm mapping or shared-memory tensors; with anything
        # else rank 0 writes the whole list, as the reference's one eviction manager does)
        shared_master = bool(getattr(emb_tables, "_mapped_file", False)) or \
            all(bool(e.weight.is_shared()) for e in getattr(emb_tables, "emb_l", []))
        self.shared_master = shared_master
        self.wb_sharded = (world > 1 and self.planner is not None and shared_master
                           and os.environ.get("CDLRM_WB_SHARDED", "1") != "0")
        # un-cached ids of a window (the same on every rank): one store sharded over the node's GPUs and read over
        # NVLink instead of a full copy per rank (CDLRM_LOSER_SHARDED=0: one local store per rank)
        # un-cached ids of a window at N > 1: "own" (default) = every rank stages only the ones its own batches contain
        # (a rank-private store, as small as on one GPU); CDLRM_LOSER_SHARDED=1 = one store of ALL ranks' un-cached ids
        # sharded over the node's GPUs and read over NVLink (measured at 8 GPUs: 34 k scattered 512-byte peer reads per
        # step took 410 us, the private store's local reads 25-60 us); CDLRM_LOSER_OWN=0 = the whole list on every rank
        self.sharded_losers = (world > 1 and self.planner is not None
                               and os.environ.get("CDLRM_LOSER_SHARDED", "0") == "1")
        self.own_losers = (world > 1 and self.planner is not None and not self.sharded_losers
                           and os.environ.get("CDLRM_LOSER_OWN", "1") != "0")
        if self.sharded_losers:
            self.planner.enable_sharded_losers(rank, world, self._host_group)
        # fills are the same rows on every replica: each rank pulls 1/world of them over PCIe, the boundary reads the
        # rest from the peers' staging buffers over NVLink (CDLRM_FILL_SHARDED=0: every rank pulls all of them)
        self.sharded_fills = (world > 1 and self.planner is not None
                              and os.environ.get("CDLRM_FILL_SHARDED", "1") != "0")
        if self.sharded_fills:
            self.planner.enable_sharded_fills(rank, world, self._host_group)
        # a window handed over as a marker callable (submit_window) is scanned 1/world per rank, bitmaps OR-ed over
        # NVLink (CDLRM_SCAN_SHARDED=0: every rank scans the whole global window)
        if world > 1 and self.planner is not None and os.environ.get("CDLRM_SCAN_SHARDED", "1") != "0":
            self.planner.enable_sharded_scan(rank, world, self._host_group)
        self._installed = None
        self._plan_q = queue.Queue()
        self._plan_thread = None
        self.steps_since_agg = 0
        self.caching_overhead = []
        self.input_slots = 6             # stage_inputs: device-side input slots (host runs up to 5 steps ahead)
        self.keep_losses = False         # tests: keep every step's loss tensor (no sync) in loss_history
        self.loss_history = []
        # position in the run (checkpoints): windows installed, steps run, steps of the installed window so far and
        # in all; windows submitted and the steps each one holds; victim-stream state at the start of every plan
        self._ln_bot, self._ln_top = [int(x) for x in ln_bot], [int(x) for x in ln_top]
        self.window = self.global_step = self.steps_in_window = 0
        self._window_steps = 0
        self._n_submitted = 0
        self._submitted_steps = []
        self._rng_snaps = {}
        self._finished = False

    # -- look-ahead -------------------------------------------------------------------------
    def submit_window(self, win_ids, own_ids=None):
        """Start planning a window in the background; windows must be submitted in training order.
        ``own_ids`` (N > 1): int64 device tensor [T, m] of the ids of THIS rank's own batches of the window; derived
        from ``win_ids`` when that is the global id tensor (rank r owns samples [r lb, (r+1) lb) of every step).
        ``win_ids``: int64 [T, n] tensor of the GLOBAL batch ids of the window, or the reference's FIFO entry
        ``(rows, uniq, maps)`` (cache_manager.py:102-104), of which the ascending unique id lists are what the
        plan needs (the rows are read from the master at install time: sequential schedule, DESIGN.md 2)."""
        import threading
        uniq_lists = marker = None
        if callable(win_ids):
            # chunked scan: ``win_ids(planner)`` feeds the window to ``planner.mark_ids`` chunk by chunk (on the
            # planner's stream, from the plan thread) and returns the number of ids per table of the WHOLE window;
            # with ``planner.scan_shard == (r, W)``, W > 1, it marks only the r-th of W equal shares of the window
            # (any partition will do: the ranks' bitmaps are OR-ed afterwards)
            marker = win_ids
        elif isinstance(win_ids, (tuple, list)):
            uniq_lists = [u.to(self.dev, non_blocking=True) for u in win_ids[1]]
        else:
            win_ids = win_ids.to(self.dev, non_blocking=True)
            lb, W_ = self.local_batch, self.world
            if own_ids is None and self.own_losers and win_ids.shape[1] % (lb * W_) == 0:
                own_ids = win_ids.view(win_ids.shape[0], -1, W_, lb)[:, :, self.rank].reshape(win_ids.shape[0], -1)
        if own_ids is not None and self.own_losers:
            own_ids = own_ids.to(self.dev, non_blocking=True).contiguous()
        else:
            own_ids = None
        if isinstance(win_ids, torch.Tensor):
            self._submitted_steps.append(-(-int(win_ids.shape[1]) // (self.local_batch * self.world)))
        else:
            self._submitted_steps.append(None)
        idx = self._n_submitted
        self._n_submitted += 1
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))   # ids produced on the current stream are ready
        prev = self._plan_thread

        def work():
            if prev is not None:
                prev.join()
            torch.cuda.set_device(self.dev)
            self.side.wait_event(ev)
            try:
                # the victim-stream state this plan starts from: what a checkpoint at the boundary before it records
                self._rng_snaps[idx] = self.planner.rng.snapshot(self.side)
                # (copy-engine mode) evicted rows of the window just installed go back to the host master first
                self.planner.flush_writeback()
                if own_ids is not None:
                    self.planner.mark_own_ids(own_ids)
                if marker is not None:
                    with torch.cuda.stream(self.side):
                        n_marked = marker(self.planner)      # this rank's share (planner.scan_shard) or everything
                    self.planner.merge_marks()
                    rec = self.planner.plan(marked=n_marked)
                elif uniq_lists is not None:
                    rec = self.planner.plan(uniq_lists=uniq_lists)
                else:
                    rec = self.planner.plan(win_ids=win_ids)
                if self.world > 1:
                    # the prefetch below reads master rows: rank 0's write-back of the previous
                    # boundary (asynchronous, on its planner stream) must have landed first
                    prev_rec = self._installed
                    if (self.rank == 0 or self.wb_sharded) and prev_rec is not None and prev_rec.wb_done is not None:
                        prev_rec.wb_done.synchronize()
                    dist.barrier(group=self._host_group)
                rec = self.planner.stage(rec)
                if self.sharded_losers or self.sharded_fills:
                    # a peer's forward (install) reads this rank's shard right after (at) ITS boundary: every rank's
                    # prefetch must have landed before any rank is handed the record
                    rec.staged.synchronize()
                    dist.barrier(group=self._host_group)
                self._plan_q.put(rec)
            except Exception as e:  # surfaced by install_window
                self._plan_q.put(e)

        self._plan_thread = threading.Thread(target=work, daemon=True)
        self._plan_thread.start()

    def install_window(self, steps=None):
        """Window boundary (main_no_ddp.py:393-399): wait for the plan, average touched rows
        over ranks, evict (rank 0 writes the master back), fill.  ``steps``: the number of training steps of this
        window (default: from its ids when it was submitted as an id tensor, else ``lookahead``) -- where the next
        window boundary is, for ``save_checkpoint`` / ``sync_master``."""
        t0 = time.perf_counter()
        rec = self._plan_q.get()
        if isinstance(rec, Exception):
            raise rec
        t1 = time.perf_counter()
        if self._installed is not None:
            # conditions the reference raises on the host (IndexError: aux overflow, id outside its table,
            # model_no_ddp.py:176-179) are sticky device flags here: surface them once per window
            self.cache_group.check_device_flags()
        t2 = time.perf_counter()
        if self.world > 1:
            broadcast_and_aggregate(self.cache_group, None, self.rank, self.args.table_agg_op)
            self.steps_since_agg = 0
        t3 = time.perf_counter()
        # evict / fill are HBM->HBM against the staging buffers the plan thread filled during the
        # previous window; the host write-back runs on the planner stream beside the next steps
        # the replicas were just aggregated, so their evicted rows agree: every rank writes 1/world of them back
        # into the shared host master (CDLRM_WB_SHARDED=0: rank 0 writes all of them, as the reference does)
        self.planner.install_staged(rec, write_master=(self.rank == 0 or self.wb_sharded),
                                    average_on_writeback=self.args.average_on_writeback,
                                    wb_share=(self.rank, self.world) if self.wb_sharded else None)
        self._installed = rec            # keeps the loser store of this window alive
        expected = self._submitted_steps.pop(0) if self._submitted_steps else None
        self._window_steps = int(steps or expected or self.args.lookahead)
        self.window += 1
        self.steps_in_window = 0
        self._finished = False
        for i in [i for i in self._rng_snaps if i < self.window]:
            del self._rng_snaps[i]
        t4 = time.perf_counter()
        self.caching_overhead.append(t4 - t0)
        # host milliseconds of the boundary: waiting for the plan, draining the stream for the device flags,
        # aggregation, enqueueing evict / fill
        self.boundary_breakdown_ms = {"wait_plan": round(1e3 * (t1 - t0), 2), "flags_sync": round(1e3 * (t2 - t1), 2),
                                      "aggregate": round(1e3 * (t3 - t2), 2), "install": round(1e3 * (t4 - t3), 2),
                                      "install_phases": dict(getattr(self.planner, "last_install_ms", {}))}
        return rec

    def _early_allreduce(self):
        """Called from the top MLP's backward (autograd thread, training stream current)."""
        st = self.dlrm._mlp_state["top"]
        ars = self._ar_stream
        ars.wait_stream(torch.cuda.current_stream(self.dev))
        check(lib.cdlrm_mlp_join(st.handle, ctypes.c_void_p(ars.cuda_stream)))   # its dW are complete on `ars`
        with torch.cuda.stream(ars):
            gw = self.dlrm.flat_grads[self.dlrm.flat_top_weight_off:self.dlrm.flat_weight_elems]
            gw /= self.world
            self._ar_work = dist.all_reduce(gw, async_op=True)

    # -- one training step -------------------------------------------------------------------
    def _step_eager(self, X, lS_o, lS_i, T):
        if self.overlap_update:
            self.cache_group.overlap_update = True
            self.cache_group.fused_lr = float(self.optimizer_embeds.param_groups[0]["lr"])
        lookups, _idxs = self.cache_group(lS_o, lS_i, self.emb_tables, self.dev.index)
        Z = self.dlrm(X, lookups)
        dz = None
        if self.args.loss_function == "bce" and os.environ.get("CDLRM_FUSED_LOSS", "1") != "0":
            if (self.flat and Z.is_cuda and Z.dtype == torch.float32 and T.dtype == torch.float32
                    and Z.shape == T.shape and not (0.0 < self.dlrm.loss_threshold < 1.0)):
                E, dz = bce_mean_with_grad(Z, T)   # loss and d loss / d Z in one launch, outside autograd
            else:
                E = bce_mean(Z, T)                 # BCELoss(mean) and its derivative in one launch
        else:
            E = loss_fn_wrap(Z, T, self.loss_fn, self.args, self.loss_ws)
        if self.flat:
            # the MLP backward writes dW / db into the flat bucket; weights (not biases: the reference's
            # aggregate_gradients never reduces them, :234-247) are averaged by ONE in-place all-reduce
            if dz is not None:
                Z.backward(dz)                     # == E.backward() without the ones seed and the dz * 1 launch
            else:
                E.backward()
            work = None
            if self.world > 1:
                self.dlrm.join_mlp_grads()
                early, self._ar_work = self._ar_work, None
                lo = self.dlrm.flat_top_weight_off if early is not None else self.dlrm.flat_weight_elems
                gw = self.dlrm.flat_grads[:lo]                        # what the early all-reduce did not cover
                gw /= self.world
                work = dist.all_reduce(gw, async_op=True)
            self.optimizer_embeds.step()      # applies the fused sparse update (pre-step hook)
            if work is not None:
                if early is not None:
                    early.wait()
                work.wait()
            self.dlrm.join_mlp_grads()        # weight-gradient GEMMs ran beside everything up to here
            self.dlrm.flat_sgd_step(self.optimizer_mlps.param_groups[0]["lr"])
            return E, Z
        self.optimizer_mlps.zero_grad(set_to_none=True)
        E.backward()
        reqs = aggregate_gradients(self.dlrm)
        self.optimizer_embeds.step()          # applies the fused sparse update (pre-step hook)
        wait_wrap(reqs)
        self.optimizer_mlps.step()
        return E, Z

    def capture_graph(self, X, lS_o, lS_i, T):
        """Capture one whole training step (forward, backward, both optimizers, the MLP-grad
        all-reduce) into a CUDA graph.  The captured step is NOT executed by the capture; the
        caller replays it through ``step``.  A look-ahead plan running on the side stream is waited
        for first: its stream waits, allocations and frees may not interleave with a capture."""
        dev = self.dev
        if self._plan_thread is not None:
            self._plan_thread.join()
        self._g_in = (torch.empty_like(X, device=dev), torch.empty(tuple(lS_i.shape), dtype=torch.int64, device=dev),
                      torch.empty_like(T, device=dev))
        self._g_lso = lS_o
        self.cache_group._ensure_ctx(self.emb_tables)
        check(lib.cdlrm_ctx_reserve(self.cache_group._ctx, int(lS_i.shape[1])))
        torch.cuda.synchronize(dev)
        self._graph = torch.cuda.CUDAGraph()
        n0 = lib.cdlrm_prof_launches(0)
        with torch.cuda.graph(self._graph, capture_error_mode="thread_local"):
            self._g_out = self._step_eager(self._g_in[0], lS_o, self._g_in[1], self._g_in[2])
        self.graph_launches = int(lib.cdlrm_prof_launches(0) - n0)   # library kernels per replay
        return self._graph

    def step(self, X, lS_o, lS_i, T):
        self.steps_since_agg += 1
        self.global_step += 1
        self.steps_in_window += 1
        if getattr(self, "_graph", None) is not None and tuple(lS_i.shape) == tuple(self._g_in[1].shape):
            self._g_in[0].copy_(X, non_blocking=True)
            self._g_in[1].copy_(lS_i, non_blocking=True)
            self._g_in[2].copy_(T, non_blocking=True)
            self._graph.replay()
            return self._g_out
        return self._step_eager(X, lS_o, lS_i, T)

    # -- host inputs: copy of step i+1 beside step i --------------------------------------------
    class StagedInputs:
        __slots__ = ("X", "lS_i", "T", "ready", "slot")

    def stage_inputs(self, X, lS_i, T):
        """Start the host->device copy of ONE step's inputs (pinned host tensors: dense features, ids [T, lb],
        labels) on the trainer's copy stream and return a handle for ``step_staged``.  ``input_slots`` device-side
        slots rotate, so the copies of the next steps run beside step i instead of in front of it on the training
        stream (2.2 MB per step at the Terabyte shape: ~40 us of PCIe time per step otherwise serialised with the
        step), and the host may run ``input_slots - 1`` steps ahead of the device."""
        if getattr(self, "_in_slots", None) is None:
            self._copy_stream = _lib.new_stream(self.dev, priority=-1)   # ahead of the planner's bulk copies
            self._in_slots, self._in_no = [None] * self.input_slots, 0
        k = self._in_no % len(self._in_slots)
        self._in_no += 1
        sl = self._in_slots[k]
        shapes = (tuple(X.shape), tuple(lS_i.shape), tuple(T.shape))
        if sl is None or sl[0] != shapes:
            if sl is not None:
                torch.cuda.synchronize(self.dev)
            st = Trainer.StagedInputs()
            st.X = torch.empty(shapes[0], dtype=X.dtype, device=self.dev)
            st.lS_i = torch.empty(shapes[1], dtype=torch.int64, device=self.dev)
            st.T = torch.empty(shapes[2], dtype=T.dtype, device=self.dev)
            st.ready, st.slot = torch.cuda.Event(), k
            sl = self._in_slots[k] = (shapes, st, torch.cuda.Event())
            sl[2].record(torch.cuda.current_stream(self.dev))
        _shapes, st, free = sl
        cs = self._copy_stream
        cs.wait_event(free)                 # the step that last read this slot has taken its inputs
        with torch.cuda.stream(cs):
            st.X.copy_(X, non_blocking=True)
            st.lS_i.copy_(lS_i, non_blocking=True)
            st.T.copy_(T, non_blocking=True)
            st.ready.record(cs)
        return st

    # -- per-step scalar read-back that never makes the training stream wait for PCIe ---------------
    def push_loss(self, E):
        """Queue the device scalar ``E`` (a step's loss) for an asynchronous read-back: a device-to-device copy into a
        ring slot on the training stream (E is a CUDA-graph output buffer that the next replay overwrites), then the
        4-byte device-to-host copy on a stream of its own -- so that the next step is never queued behind a PCIe
        transfer (the copy engine serves the planner's write-back chunks in front of it)."""
        if getattr(self, "_loss_ring", None) is None:
            n = self.input_slots
            self._loss_ring = (torch.zeros(n, dtype=torch.float32, device=self.dev),
                               torch.zeros(n, dtype=torch.float32, pin_memory=True),
                               [torch.cuda.Event() for _ in range(n)], [torch.cuda.Event() for _ in range(n)],
                               _lib.new_stream(self.dev, priority=-1))
            self._loss_head = self._loss_tail = 0
        ring, pin, ev_d, ev_h, ls = self._loss_ring
        n = ring.numel()
        if self._loss_head - self._loss_tail >= n:
            raise _lib.CdlrmError("push_loss: ring full, pop_loss first")
        q = self._loss_head % n
        self._loss_head += 1
        cur = torch.cuda.current_stream(self.dev)
        ring[q].copy_(E.detach().reshape(()))
        ev_d[q].record(cur)
        ls.wait_event(ev_d[q])
        with torch.cuda.stream(ls):
            pin[q].copy_(ring[q], non_blocking=True)
            ev_h[q].record(ls)

    def pending_losses(self):
        return 0 if getattr(self, "_loss_ring", None) is None else self._loss_head - self._loss_tail

    def pop_loss(self):
        """The oldest queued loss as a Python float (waits for its copy)."""
        _ring, pin, _ev_d, ev_h, _ls = self._loss_ring
        q = self._loss_tail % pin.numel()
        self._loss_tail += 1
        ev_h[q].synchronize()
        return float(pin[q])

    def step_staged(self, st, lS_o):
        """``step`` on inputs staged by ``stage_inputs``."""
        cur = torch.cuda.current_stream(self.dev)
        cur.wait_event(st.ready)
        out = self.step(st.X, lS_o, st.lS_i, st.T)
        # graph path: the replay begins with device-to-device copies into the captured input buffers, but the
        # slot is only known to be free once the whole step is enqueued behind them -- record after the step
        self._in_slots[st.slot][2].record(cur)
        return out

    def step_reference(self, X, lS_o, lS_i, T):
        """The reference's step, call for call (main_no_ddp.py:401-415); returns (E, Z, cache_group_idxs)."""
        self.cache_group.overlap_update, self.cache_group.fused_lr = False, None   # update at optimizer_embeds.step()
        lookups, cache_group_idxs = self.cache_group(lS_o, lS_i, self.emb_tables, self.dev.index)
        Z = self.dlrm(X, lookups)
        E = loss_fn_wrap(Z, T, self.loss_fn, self.args, self.loss_ws)
        self.optimizer_mlps.zero_grad()
        self.optimizer_embeds.zero_grad()
        E.backward()
        if self.flat:
            work = None
            self.dlrm.join_mlp_grads()
            if self.world > 1:
                early, self._ar_work = self._ar_work, None
                lo = self.dlrm.flat_top_weight_off if early is not None else self.dlrm.flat_weight_elems
                gw = self.dlrm.flat_grads[:lo]
                gw /= self.world
                work = dist.all_reduce(gw, async_op=True)
            self.optimizer_embeds.step()
            if work is not None:
                if early is not None:
                    early.wait()
                work.wait()
            self.dlrm.flat_sgd_step(self.optimizer_mlps.param_groups[0]["lr"])
        else:
            reqs = aggregate_gradients(self.dlrm)
            self.optimizer_embeds.step()
            wait_wrap(reqs)
            self.optimizer_mlps.step()
        return E, Z, cache_group_idxs

    def finish(self):
        """Wait for the look-ahead thread and the last asynchronous write-back; raise pending device flags."""
        if self._plan_thread is not None:
            self._plan_thread.join()
        if self.planner is not None:
            self.planner.flush_writeback()
        if self._installed is not None and self._installed.wb_done is not None:
            self._installed.wb_done.synchronize()
        torch.cuda.synchronize(self.dev)
        self.cache_group.check_device_flags()
        self._finished = True

    def maybe_aggregate(self, j):
        if self.world > 1 and j > 0 and j % self.args.table_agg_freq == 0:     # :418-420
            broadcast_and_aggregate(self.cache_group, None, self.rank, self.args.table_agg_op)
            self.steps_since_agg = 0

    # -- export, checkpoint, resume --------------------------------------------------------------
    # A checkpoint describes the boundary before window w: every step of the windows < w has run, window w is neither
    # installed nor counted as planned.  A plan(w) already in flight or staged is left alone (the run that saves goes
    # on with it); the victim-stream state recorded is the one plan(w) started from, and a resumed Trainer plans w
    # from the restored live tags and that state, as the uninterrupted run did.

    def at_boundary(self):
        """Every step of the installed window has run (or no window is installed yet)."""
        return self.steps_in_window == (self._window_steps if self._installed is not None else 0)

    def _need_planner(self, what):
        if self.planner is None:
            raise _lib.CdlrmError(f"{what} needs the look-ahead planner (not available under --strict-reference)")

    def _quiesce(self):
        """Wait for the plan thread and complete the pending eviction write-back: the master then holds every row
        evicted so far, and nothing but the caller touches the cache or the master."""
        if self._plan_thread is not None:
            self._plan_thread.join()
        self.planner.flush_writeback()
        if self._installed is not None and self._installed.wb_done is not None:
            self._installed.wb_done.synchronize()
        torch.cuda.synchronize(self.dev)
        self.cache_group.check_device_flags()

    def quiesce_ranks(self):
        """Collective over the ranks (call it on every rank at the same point): each rank completes its own plan and
        its share of the pending eviction write-back, then a host barrier.  Afterwards the master holds every row
        evicted by any rank, and no rank writes it again before the next window boundary, which waits for every rank."""
        self._need_planner("quiesce_ranks")
        self._quiesce()
        if self.world > 1:
            dist.barrier(group=self._host_group)

    def _aggregate_replicas(self):
        if self.world > 1:
            broadcast_and_aggregate(self.cache_group, None, self.rank, self.args.table_agg_op)
            self.steps_since_agg = 0
            torch.cuda.synchronize(self.dev)

    def sync_master(self):
        """Write every valid cache line into the host master: afterwards ``emb_tables.emb_l[k].weight`` is the
        trained table k.  Legal at a window boundary or after ``finish()``; under ``--average-on-writeback`` only
        after ``finish()`` (the master's stale row of a cached id is part of its later eviction average).  In the
        other modes it changes no later decision or value: the master row of a cached id is read by nobody before
        the eviction of that id overwrites it (fills and the loser store read un-cached ids only).  At N > 1 the
        replicas are aggregated first; each rank writes its share of the sets when the master is one shared object
        (``wb_sharded``), else rank 0 writes everything.  Returns the number of rows this rank wrote."""
        self._need_planner("sync_master")
        if self.args.average_on_writeback and not self._finished:
            raise _lib.CdlrmError("sync_master under --average-on-writeback needs finish() first: the master's rows of "
                                  "cached ids are part of their later eviction averages")
        if not self._finished and not self.at_boundary():
            raise _lib.CdlrmError(f"sync_master: not at a window boundary ({self.steps_in_window} of "
                                  f"{self._window_steps} steps of window {self.window - 1} have run)")
        self._quiesce()
        self._aggregate_replicas()
        n = 0
        if self.rank == 0 or self.wb_sharded:
            n = self.planner.write_cached_to_master((self.rank, self.world) if self.wb_sharded else (0, 1))
        if self.world > 1:
            dist.barrier(group=self._host_group)
        return n

    def _dense_tensors(self):
        if self.flat:
            return [self.dlrm.flat_params]
        return [p.data for p in self.dlrm.parameters()]

    def checkpoint_fields(self):
        """The meta data a checkpoint must share with this Trainer to be loaded into it (checkpoint.check_meta)."""
        a, cg = self.args, self.cache_group
        return {
            "format": ckpt.FORMAT,
            "shapes": {"ln_emb": [int(n) for n in cg.ln_emb], "dim": int(cg.dim), "ways": int(cg.num_ways),
                       "num_sets": [int(S) for S in cg.cache_sizes], "aux_rows": int(cg.aux_table_size),
                       "ln_bot": self._ln_bot, "ln_top": self._ln_top},
            "args": {"seed": int(a.numpy_rand_seed), "cache_size": int(a.cache_size), "ways": int(a.num_ways),
                     "lookahead": int(a.lookahead), "global_batch": int(a.mini_batch_size), "world_size": int(self.world),
                     "table_agg_op": a.table_agg_op, "average_on_writeback": bool(a.average_on_writeback),
                     "learning_rate": float(a.learning_rate), "lr_embeds": float(a.lr_embeds)},
        }

    def save_checkpoint(self, path, epoch=0):
        """Write the state at the current window boundary into the directory ``path`` (checkpoint.py: written as
        ``path.tmp``, then renamed into place).  Changes no training state: the cache rows are NOT written into the
        master.  At N > 1 the replicas are aggregated first (the install of the next window then finds nothing dirty),
        and rank 0 writes, with host barriers around the write.  ``epoch``: the epoch the resume point lies in.
        ``last_checkpoint_s``: seconds of device-to-host copies and of file I/O."""
        self._need_planner("save_checkpoint")
        if not self.at_boundary():
            raise _lib.CdlrmError(f"save_checkpoint: not at a window boundary ({self.steps_in_window} of "
                                  f"{self._window_steps} steps of window {self.window - 1} have run)")
        w = self.window
        self._quiesce()
        snap = self._rng_snaps.get(w)
        if snap is None:                          # plan(w) not submitted: the stream stands where plan(w) will start
            snap = self.planner.rng.snapshot(self.side)
        state, draws, ev = snap
        ev.synchronize()
        self._aggregate_replicas()
        meta = dict(self.checkpoint_fields(),
                    resume={"epoch": int(epoch), "window": int(w), "global_step": int(self.global_step)},
                    rng={"state": [int(x) for x in state.numpy().view(np.uint32)], "draws": int(draws)})
        if self.world > 1:
            dist.barrier(group=self._host_group)  # every rank's share of the write-back is in the shared master
        d2h = 0.0
        if self.rank == 0:
            wr = ckpt.Writer(path)
            t0 = time.perf_counter()
            dense = torch.cat([t.reshape(-1) for t in self._dense_tensors()]).cpu()
            d2h += time.perf_counter() - t0
            wr.put("dense.bin", dense.numpy())
            cg = self.cache_group
            for k in range(len(cg.emb_l)):
                t0 = time.perf_counter()
                tags = cg.occupancy_tables[k].cpu()
                rows = cg.emb_l[k].weight.data[:cg.num_ways * cg.cache_sizes[k]].cpu()
                d2h += time.perf_counter() - t0
                wr.put(f"tags_{k}.bin", tags.numpy())
                wr.put(f"cache_{k}.bin", rows.numpy())
                del tags, rows
                M = self.emb_tables.emb_l[k].weight.data
                wr.put(f"master_{k}.bin", (M.cpu() if M.is_cuda else M).numpy())    # straight from host storage
            wr.commit(meta)
            self.last_checkpoint_s = {"device_to_host": round(d2h, 4), "file_io": round(wr.io_s, 4)}
        if self.world > 1:
            dist.barrier(group=self._host_group)
        return meta

    def load_checkpoint(self, path):
        """Restore a checkpoint into this freshly built Trainer (same arguments and shapes; a mismatch raises
        ``checkpoint.CheckpointMismatch`` naming the field) and return the window w to submit next.  Restores the
        live and the planner's tags, the cache rows, the master (at N > 1 rank 0 writes a shared master, the others
        wait), the dense parameters and the victim-stream state as of the start of plan(w).  The CUDA graph is
        captured afterwards, as usual."""
        self._need_planner("load_checkpoint")
        if self._installed is not None or self.global_step or self._n_submitted:
            raise _lib.CdlrmError("load_checkpoint needs a freshly built Trainer")
        meta = ckpt.read_meta(path)
        ckpt.check_meta(meta, self.checkpoint_fields())
        rd = ckpt.Reader(path, meta)
        dev, cg = self.dev, self.cache_group
        h2d = 0.0
        for k in range(len(cg.emb_l)):
            S, ways = cg.cache_sizes[k], cg.num_ways
            tags = rd.read_into(f"tags_{k}.bin", np.empty((S, ways), np.int64))
            rows = rd.read_into(f"cache_{k}.bin", np.empty((ways * S, cg.dim), np.float32))
            t0 = time.perf_counter()
            cg.occupancy_tables[k].copy_(torch.from_numpy(tags))
            self.planner.plan_tags[k].copy_(cg.occupancy_tables[k])
            cg.emb_l[k].weight.data[:ways * S].copy_(torch.from_numpy(rows))
            h2d += time.perf_counter() - t0
        if self.rank == 0 or not self.shared_master:
            for k, E in enumerate(self.emb_tables.emb_l):
                M = E.weight.data
                if M.is_cuda:
                    M.copy_(torch.from_numpy(rd.read_into(f"master_{k}.bin", np.empty(tuple(M.shape), np.float32))))
                else:
                    rd.read_into(f"master_{k}.bin", M.numpy())
        dense_t = self._dense_tensors()
        dense = rd.read_into("dense.bin", np.empty(sum(t.numel() for t in dense_t), np.float32))
        t0 = time.perf_counter()
        o = 0
        with torch.no_grad():
            for t in dense_t:
                t.copy_(torch.from_numpy(dense[o:o + t.numel()]).view_as(t))
                o += t.numel()
        self.dlrm.invalidate_weight_splits()        # the hi / lo operand copies belong to the old weights
        self.planner.rng.set_state(np.asarray(meta["rng"]["state"], dtype=np.uint32), meta["rng"]["draws"], self.side)
        torch.cuda.synchronize(dev)
        h2d += time.perf_counter() - t0
        r = meta["resume"]
        self.window = self._n_submitted = int(r["window"])
        self.global_step = int(r["global_step"])
        self.resume_epoch = int(r["epoch"])
        self.last_checkpoint_s = {"host_to_device": round(h2d, 4), "file_io": round(rd.io_s, 4)}
        if self.world > 1:
            dist.barrier(group=self._host_group)
        return self.window

    # -- evaluation -------------------------------------------------------------------------------
    class _EvalState:
        """What ``evaluate`` keeps across calls: the forward (its own MLP handles), the metrics object, the CUDA graph
        of one evaluation step with its static inputs, and the rotating device slots of host batches."""

        def __init__(self, tr):
            self.fwd = EvalForward(tr.cache_group, tr.dlrm)
            self.handle, self.cap = None, 0
            self.graph = self.graph_key = self.static = None
            self.warm = set()           # batch shapes that ran eagerly once (a capture follows on the next batch)
            self.slots, self.slot_no = {}, 0
            self.copy_stream = None
            self.offsets_ok = None      # the last host lS_o found to be arange(batch) (loaders reuse one tensor)

        def drop_graph(self):
            if self.graph is not None:
                torch.cuda.synchronize()
            self.graph = self.graph_key = self.static = None
            self.warm.clear()

        def __del__(self):
            try:
                if self.handle is not None:
                    lib.cdlrm_eval_destroy(self.handle)
            except Exception:
                pass

    def _eval_inputs(self, ev, X, lS_i, T):
        """Device tensors of one test batch.  Host batches are copied on a copy stream of the evaluator's own into two
        rotating device slots per shape (never the training input slots of ``stage_inputs``)."""
        dev = self.dev
        if X.is_cuda and lS_i.is_cuda and T.is_cuda:
            return (X.to(dev, dtype=torch.float32), lS_i.to(dev, dtype=torch.int64), T.to(dev, dtype=torch.float32)), None
        if ev.copy_stream is None:
            ev.copy_stream = _lib.new_stream(dev, priority=-1)
        key = (tuple(X.shape), tuple(lS_i.shape), tuple(T.shape))
        pair = ev.slots.get(key)
        if pair is None:
            pair = ev.slots[key] = [(torch.empty(key[0], dtype=torch.float32, device=dev),
                                     torch.empty(key[1], dtype=torch.int64, device=dev),
                                     torch.empty(key[2], dtype=torch.float32, device=dev),
                                     torch.cuda.Event(), torch.cuda.Event()) for _ in range(2)]
        ev.slot_no += 1
        Xd, Id, Td, ready, free = pair[ev.slot_no % 2]
        cs, cur = ev.copy_stream, torch.cuda.current_stream(dev)
        cs.wait_event(free)                 # the evaluation step that last read this slot is enqueued before it
        with torch.cuda.stream(cs):
            Xd.copy_(X, non_blocking=True)
            Id.copy_(lS_i, non_blocking=True)
            Td.copy_(T, non_blocking=True)
            ready.record(cs)
        cur.wait_event(ready)
        return (Xd, Id, Td), free

    def _eval_step(self, ev, X, ids, T):
        """Predictions of one batch, accumulated into the metrics on the current stream: a replay of the captured
        step for the graph's shape, else eagerly with the same kernels.  The first shape that runs twice is captured."""
        dev = self.dev
        cur = torch.cuda.current_stream(dev)
        B = int(T.shape[0])
        key = (tuple(X.shape), tuple(ids.shape), tuple(T.shape))
        if ev.fwd.reserve(B, dev):
            ev.drop_graph()             # a captured step holds the old MLP handles
        use_graph = not getattr(self.args, "no_cuda_graph", False)
        if use_graph and ev.graph is None and key in ev.warm:
            torch.cuda.synchronize(dev)
            ev.static = (torch.empty_like(X), torch.empty_like(ids), torch.empty_like(T))
            ev.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(ev.graph, capture_error_mode="thread_local"):
                sx, si, st = ev.static
                p = ev.fwd(sx, si)
                check(lib.cdlrm_eval_accumulate(ev.handle, _vp(p.data_ptr()), p.stride(0), _vp(st.data_ptr()),
                                                st.stride(0), B, _vp(torch.cuda.current_stream(dev).cuda_stream)))
            ev.graph_key = key
        if ev.graph is not None and ev.graph_key == key:
            sx, si, st = ev.static
            sx.copy_(X)
            si.copy_(ids)
            st.copy_(T)
            ev.graph.replay()
            return
        p = ev.fwd(X, ids)
        check(lib.cdlrm_eval_accumulate(ev.handle, _vp(p.data_ptr()), p.stride(0), _vp(T.data_ptr()), T.stride(0), B,
                                        _vp(cur.cuda_stream)))
        ev.warm.add(key)

    def evaluate(self, loader, max_samples=None):
        """Forward-only pass over ``loader`` (``(X, lS_o, lS_i, T)`` batches, one id per bag, CPU or CUDA tensors) on the
        trained model, returning ``EvalResult``: samples, mean BCE loss, accuracy (round(z) == t), exact ROC AUC,
        positives and negatives.  The model read is the cached rows plus the host master: ``_quiesce`` first joins the
        plan thread and completes this rank's pending eviction write-back (``last_quiesce_s``: seconds it took).  At
        N > 1 with a shared master every rank writes back a share of the evicted rows: call ``quiesce_ranks()`` on
        every rank first (``Run`` does), so that the other ranks' shares have landed too.  Nothing the training step
        reads or writes is touched, so training goes on as if no evaluation had happened.  One host sync at the end.
        ``max_samples``: capacity of the metrics (default ``len(loader)`` times the first batch size).  Raises
        ``ValueError`` for a prediction outside [0, 1] or a label outside {0, 1}, ``CdlrmError`` for offsets that are
        not one id per bag."""
        self._need_planner("evaluate")
        t0 = time.perf_counter()
        self._quiesce()
        self.last_quiesce_s = time.perf_counter() - t0
        dev = self.dev
        ev = getattr(self, "_ev", None)
        if ev is None:
            ev = self._ev = Trainer._EvalState(self)
        it = iter(loader)
        first = next(it, None)
        if first is None:
            return EvalResult(0, float("nan"), float("nan"), float("nan"), 0, 0)
        cap = int(max_samples) if max_samples is not None else len(loader) * int(first[3].shape[0])
        if cap > ev.cap:
            ev.drop_graph()             # the captured step accumulates into the old metrics object
            if ev.handle is not None:
                check(lib.cdlrm_eval_destroy(ev.handle))
                ev.handle, ev.cap = None, 0
            h = _vp()
            check(lib.cdlrm_eval_create(ctypes.byref(h), dev.index, cap))
            ev.handle, ev.cap = h, cap
        cur = torch.cuda.current_stream(dev)
        ev.fwd.begin()
        check(lib.cdlrm_eval_reset(ev.handle, _vp(cur.cuda_stream)))
        seen = 0
        off_bad = torch.zeros((), dtype=torch.bool, device=dev)
        for X, lS_o, lS_i, T in itertools.chain([first], it):
            B = int(T.shape[0])
            if int(lS_i.shape[1]) != B or int(lS_o.shape[1]) != B or X.shape[0] != B:
                raise _lib.CdlrmError("evaluate needs one id per bag (lS_i and lS_o of shape [tables, batch])")
            if lS_o is not ev.offsets_ok:
                if not lS_o.is_cuda:
                    if not bool((lS_o == torch.arange(B, dtype=lS_o.dtype)).all()):
                        raise _lib.CdlrmError(_ONE_ID_PER_BAG)
                    ev.offsets_ok = lS_o
                else:                       # checked on the device, read at the one sync below
                    torch.logical_or(off_bad, (lS_o != torch.arange(B, dtype=lS_o.dtype, device=lS_o.device)).any().to(dev),
                                     out=off_bad)
            seen += B
            if seen > ev.cap:
                raise _lib.CdlrmError(f"evaluate: more than {ev.cap} samples (pass max_samples)")
            (Xd, Id, Td), free = self._eval_inputs(ev, X, lS_i, T)
            self._eval_step(ev, Xd, Id, Td)
            if free is not None:
                free.record(cur)
        st = _lib.EvalStats()
        check(lib.cdlrm_eval_result(ev.handle, _vp(ctypes.addressof(st)), _vp(cur.cuda_stream)))
        self.cache_group.check_device_flags()
        if bool(off_bad):
            raise _lib.CdlrmError(_ONE_ID_PER_BAG)
        if st.flags & 4:
            raise _lib.CdlrmError(f"evaluate: more than {ev.cap} samples")
        if st.flags & 1:
            raise ValueError("evaluate: a prediction outside [0, 1] or NaN")
        if st.flags & 2:
            raise ValueError("evaluate: a label outside {0, 1}")
        n, P, N = int(st.samples), int(st.positives), int(st.negatives)
        auc = float(st.auc_2u) / (2.0 * P * N) if P > 0 and N > 0 else float("nan")
        return EvalResult(n, st.loss_sum / n if n else float("nan"), int(st.correct) / n if n else float("nan"), auc,
                          P, N)


def _bcast_fifo_entry(item, rank, dev):
    """One shared ``batch_fifo`` read by rank 0 only (the reference's wiring, main_no_ddp.py:624,638-643): rank 0
    ships the window to the other ranks, which need it to run the same deterministic plan.  Raw id windows go as
    one int64 [T, n] tensor, ``(rows, uniq, maps)`` tuples as their unique-id lists (padded to one tensor)."""
    hdr = [None]
    if rank == 0:
        if isinstance(item, torch.Tensor):
            hdr[0] = ("ids", tuple(item.shape))
        else:
            hdr[0] = ("uniq", [int(u.numel()) for u in item[1]])
    dist.broadcast_object_list(hdr, src=0)
    kind, meta = hdr[0]
    if kind == "ids":
        t = item.to(dev) if rank == 0 else torch.empty(meta, dtype=torch.int64, device=dev)
        dist.broadcast(t, src=0)
        return t
    ld = max(max(meta), 1)
    buf = torch.zeros(len(meta), ld, dtype=torch.int64, device=dev)
    if rank == 0:
        for k, u in enumerate(item[1]):
            buf[k, :meta[k]].copy_(u)
    dist.broadcast(buf, src=0)
    return (None, [buf[k, :meta[k]] for k in range(len(meta))], None)


def slice_batch(rank, local_batch_size, X, lS_o, lS_i, T):
    """main_no_ddp.py:388-391: rank r trains on samples [r*lb, (r+1)*lb) of the global batch every rank loads;
    the offsets are cut to the first lb columns, which assumes one id per bag (P = 1, Criteo)."""
    lo, hi = rank * local_batch_size, (rank + 1) * local_batch_size
    return X[lo:hi, :], lS_o[:, :local_batch_size], lS_i[:, lo:hi], T[lo:hi, :]


def _print_eval(r):
    print('Test accuracy = {}%'.format(100 * r.accuracy))
    print('Test loss = {}, AUC = {}'.format(r.loss, r.auc))


def Run(rank, m_spa, ln_emb, ln_bot, ln_top, train_ld, test_ld, batch_fifo, eviction_fifo, occupancy_tables_fifos,
        emb_tables, args):
    """main_no_ddp.py:324-502.  ``batch_fifo`` carries one entry per window in training order: the reference's
    ``(rows, uniq, maps)`` tuples or raw window id tensors [T, n] (``Prefetcher.fifo_payload``).

    Default: every rank plans the window itself one window ahead on a side stream (``Trainer``), the step is a
    CUDA graph, metrics are read every ``print_freq`` steps only.  With one ``batch_fifo`` shared by the ranks
    (the reference's wiring) rank 0 reads it and ships the window to the others; ``args.fifo_per_rank`` (set by
    this package's ``__main__``, where every rank runs its own Prefetcher on the deterministic loader) makes
    every rank read its own.

    ``--strict-reference``: the reference's literal loop (:393-425) on the same-named functions --
    ``load_caches_and_broadcast`` + ``wait_wrap`` at every window, ``cache_group(...)``, ``dlrm(...)``,
    ``aggregate_gradients``, both optimizers, ``broadcast_and_aggregate`` on explicit slot windows.

    ``--save-model PATH``: a checkpoint (Trainer.save_checkpoint) at the end of every epoch, replacing the previous
    one, and ``sync_master()`` after the last step, so that ``emb_tables`` holds the trained tables when Run returns.
    ``--load-model PATH``: resume at the checkpoint's window; the steps before it are skipped (``batch_fifo`` must
    start at that window: ``Prefetcher`` skips the windows before it).  Neither works with ``--strict-reference``.

    The test pass (``--test-freq`` and the end of the epoch, rank 0) is ``Trainer.evaluate``: accuracy, loss and AUC
    on the GPU; ``--strict-reference`` keeps the reference's eager loop.  ``--inference-only``: build the Trainer, load
    ``--load-model`` if given, evaluate ``test_ld`` once and return (one GPU, not with ``--strict-reference``)."""
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", str(args.master_port))
    if args.world_size > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", rank=rank, world_size=args.world_size)
    strict = bool(getattr(args, "strict_reference", False))
    if strict and (args.save_model or args.load_model):
        raise _lib.CdlrmError("--save-model / --load-model need the look-ahead trainer (not --strict-reference)")
    if args.inference_only and (strict or args.world_size > 1):
        raise _lib.CdlrmError("--inference-only evaluates on one GPU with the look-ahead trainer "
                              "(--world-size 1, not --strict-reference)")
    tr = Trainer(args, m_spa, ln_emb, ln_bot, ln_top, emb_tables, rank=rank, world=args.world_size,
                 strict_reference=strict)
    if args.inference_only:          # the model of --load-model, else the freshly initialised one; nothing is trained
        if args.load_model:
            tr.load_checkpoint(args.load_model)
        if test_ld is not None:
            _print_eval(tr.evaluate(test_ld))
        return tr
    dev, lb, L = tr.dev, tr.local_batch, args.lookahead
    # training on a high-priority stream: the look-ahead planner (side stream, default priority) only
    # takes the SM slots the training step leaves free
    torch.cuda.set_stream(torch.cuda.Stream(dev, priority=-1))
    share_occupancy_tables(tr.cache_group, occupancy_tables_fifos, rank)
    shared_fifo = args.world_size > 1 and not getattr(args, "fifo_per_rank", False)
    per_epoch = math.ceil(len(train_ld) / L)
    n_windows = args.nepochs * per_epoch
    start_w = tr.load_checkpoint(args.load_model) if args.load_model else 0
    popped = start_w

    def next_entry():
        nonlocal popped
        if popped >= n_windows:
            return None
        popped += 1
        item = _fifo_get(batch_fifo) if (rank == 0 or not shared_fifo) else None
        return _bcast_fifo_entry(item, rank, dev) if shared_fifo else item

    use_graph = not strict and not getattr(args, "no_cuda_graph", False)
    total_time = total_loss = total_accu = 0.0
    total_iter = total_samp = 0
    idxs_window = []
    if not strict and popped < n_windows:
        tr.submit_window(next_entry())
    step_no = 0
    for epoch in range(args.nepochs):
        for j, (X, lS_o, lS_i, T) in enumerate(train_ld):
            if epoch * per_epoch + j // L < start_w:                                 # before the resume point
                continue
            X, lS_o, lS_i, T = slice_batch(rank, lb, X, lS_o, lS_i, T)               # :388-391
            X, lS_i, T = (t.to(dev, non_blocking=True) for t in (X, lS_i, T))
            if j % L == 0:                                                           # :393-399
                t0 = time.perf_counter()
                if strict:
                    popped += 1
                    wait_wrap(load_caches_and_broadcast(tr.cache_group, batch_fifo, eviction_fifo, rank))
                    tr.caching_overhead.append(time.perf_counter() - t0)
                else:
                    tr.install_window(steps=min(L, len(train_ld) - j))
                    nxt = next_entry()
                    if nxt is not None:
                        tr.submit_window(nxt)
            if use_graph and step_no == 2 and tuple(lS_i.shape) == (len(ln_emb), lb):
                tr.capture_graph(X, lS_o, lS_i, T)           # after two eager steps (lazy initialisation)
            t1 = time.perf_counter()
            if strict:
                E, Z, idxs = tr.step_reference(X, lS_o, lS_i, T)
                if args.world_size > 1:
                    if j > 0 and j % args.table_agg_freq == 0:                       # :418-423
                        broadcast_and_aggregate(tr.cache_group, torch.cat(idxs_window + [torch.stack(idxs)], dim=1),
                                                rank, args.table_agg_op)
                        idxs_window = []
                    else:
                        idxs_window.append(torch.stack(idxs))
            else:
                E, Z = tr.step(X, lS_o, lS_i, T)
                tr.maybe_aggregate(j)
            step_no += 1
            if tr.keep_losses:
                tr.loss_history.append(E.detach().clone())
            if rank == 0 and j > 0 and j % args.print_freq == 0:
                torch.cuda.synchronize(dev)
                tr.cache_group.check_device_flags()
                total_time += time.perf_counter() - t1
                L_ = E.item()
                A = float(((Z.detach().round() == T).sum()).item())
                mbs = T.shape[0]
                total_iter += 1
                gT = 1000.0 * total_time / max(total_iter, 1)
                ovh = 1000 * (np.mean(tr.caching_overhead) / L) if tr.caching_overhead else 0.0
                tr.caching_overhead = []
                print('Epoch {}: Finished {}/{} in {} ms/it. Caching overhead = {}. Loss = {}, Train Acc = {}'.format(
                    epoch, j, len(train_ld), gT, ovh, L_, A / mbs))
                total_time, total_iter = 0.0, 0
            test_point = (args.test_freq > 0 and j > 0 and j % args.test_freq == 0) or j == len(train_ld) - 1
            if test_point and not strict and args.world_size > 1:
                tr.quiesce_ranks()          # every rank's share of the write-back lands before rank 0 reads the master
            if rank == 0 and test_ld is not None and test_point:
                print('Testing at {}/{}....'.format(j, len(train_ld)))
                if not strict:
                    _print_eval(tr.evaluate(test_ld))
                    continue
                test_samp = total_test_acc = 0
                with torch.no_grad():
                    for _i, (Xt, lS_ot, lS_it, Tt) in enumerate(test_ld):
                        lookups, _ = tr.cache_group(lS_ot, lS_it.to(dev), emb_tables, rank)
                        Zt = tr.dlrm(Xt.to(dev), lookups)
                        total_test_acc += int((Zt.round().cpu() == Tt).sum())
                        test_samp += Tt.shape[0]
                # a test batch larger than the aux region raises IndexError in the reference (:176-179)
                tr.cache_group.check_device_flags()
                print('Test accuracy = {}%'.format(100 * (total_test_acc / max(test_samp, 1))))
        if args.save_model and (epoch + 1) * per_epoch > start_w:
            tr.save_checkpoint(args.save_model, epoch=epoch + 1)
    torch.cuda.synchronize(dev)
    tr.finish()
    if args.save_model:
        tr.sync_master()
    return tr


# ------------------------------------------------------------------------------------
# __main__ -- main_no_ddp.py:505-646
# ------------------------------------------------------------------------------------


def _derive_topology(args):
    """:525-616: table sizes, MLP shapes and the reference's sanity checks (same messages)."""
    ln_bot = np.fromstring(args.arch_mlp_bot, dtype=int, sep="-")
    if args.data_generation == "dataset":
        sys.exit("ERROR: --data-generation=dataset needs the Criteo loaders (dlrm_data_pytorch.py), which are outside "
                 "the cache hot path this package implements; use --data-generation=synthetic")
    ln_emb = np.fromstring(args.arch_embedding_size, dtype=int, sep="-")
    m_den = ln_bot[0]
    m_spa = args.arch_sparse_feature_size
    num_fea = ln_emb.size + 1
    m_den_out = ln_bot[ln_bot.size - 1]
    if args.arch_interaction_op == "dot":
        if args.arch_interaction_itself:
            num_int = (num_fea * (num_fea + 1)) // 2 + m_den_out
        else:
            num_int = (num_fea * (num_fea - 1)) // 2 + m_den_out
    elif args.arch_interaction_op == "cat":
        num_int = num_fea * m_den_out
    else:
        sys.exit("ERROR: --arch-interaction-op=" + args.arch_interaction_op + " is not supported")
    ln_top = np.fromstring(str(num_int) + "-" + args.arch_mlp_top, dtype=int, sep="-")
    if m_spa != m_den_out:
        sys.exit("ERROR: arch-sparse-feature-size " + str(m_spa) + " does not match last dim of bottom mlp "
                 + str(m_den_out))
    if num_int != ln_top[0]:
        sys.exit("ERROR: # of feature interactions " + str(num_int) + " does not match first dimension of top mlp "
                 + str(ln_top[0]))
    if args.qr_flag or args.md_flag:
        sys.exit("ERROR: QR / mixed-dimension embeddings are outside the cache hot path (unreachable from the "
                 "reference's own Run as well)")
    return ln_emb, ln_bot, ln_top, m_spa, m_den


def _rank_main(rank, args, shm_prefix=None):
    """One trainer process: its own loaders, Prefetcher thread and FIFOs over the deterministic synthetic
    stream (every rank sees the same windows), master tables shared through /dev/shm when world_size > 1."""
    import threading
    from .synthetic import make_synthetic_data_and_loaders
    ln_emb, ln_bot, ln_top, m_spa, m_den = _derive_topology(args)
    np.random.seed(args.numpy_rand_seed)
    torch.manual_seed(args.numpy_rand_seed)
    train_ld, test_ld, cache_ld = make_synthetic_data_and_loaders(args, ln_emb, m_den)
    torch.cuda.set_device(rank)
    if args.world_size > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", str(args.master_port))
        dist.init_process_group("nccl", rank=rank, world_size=args.world_size, device_id=torch.device("cuda", rank))
        if rank == 0:
            emb_tables = Embedding_Table_Group(m_spa, ln_emb, init=f"shm:{shm_prefix}:create")
        dist.barrier()
        if rank != 0:
            emb_tables = Embedding_Table_Group(m_spa, ln_emb, init=f"shm:{shm_prefix}:attach")
    else:
        big = int(np.sum(ln_emb)) * int(m_spa) > (1 << 28)
        emb_tables = Embedding_Table_Group(m_spa, ln_emb, init="device" if big else "reference")    # :621
    batch_fifo = queue.Queue(maxsize=args.batch_fifo_size)                                           # :624-626
    eviction_fifo = queue.Queue(maxsize=args.eviction_fifo_size)
    finish_event = threading.Event()
    args.fifo_per_rank = True
    if not args.fifo_payload:
        args.fifo_payload = "tuples" if args.strict_reference else "ids"
    cm = None
    if not args.inference_only:
        cm = Prefetcher(args, emb_tables, batch_fifo, eviction_fifo, finish_event, cache_ld)         # :630
        cm.start()
    try:
        tr = Run(rank, m_spa, ln_emb, ln_bot, ln_top, train_ld, test_ld, batch_fifo, eviction_fifo, [], emb_tables,
                 args)
    finally:
        finish_event.set()
        if args.world_size > 1:
            dist.barrier()
            if rank == 0:
                for k in range(len(ln_emb)):
                    try:
                        os.unlink(f"{shm_prefix}_{k}.bin")
                    except OSError:
                        pass
    if cm is not None:
        cm.join(timeout=5)
    return tr


def main(argv=None):
    """python -m cdlrm_b200.main_no_ddp [the reference's flags] -- README.md:7 of the reference, with
    ``--data-generation synthetic`` (Criteo-shaped synthetic batches, cdlrm_b200/synthetic.py)."""
    args = ProcessArgs(argv)
    np.set_printoptions(precision=args.print_precision)
    torch.set_printoptions(precision=args.print_precision)
    if args.test_mini_batch_size < 0:                    # :517-522
        args.test_mini_batch_size = args.mini_batch_size
    if args.test_num_workers < 0:
        args.test_num_workers = args.num_workers
    _derive_topology(args)                               # argument errors before any process is spawned
    if args.inference_only and (args.world_size > 1 or args.strict_reference):
        sys.exit("ERROR: --inference-only evaluates on one GPU with the look-ahead trainer: use --world-size 1 and "
                 "no --strict-reference")
    if args.world_size <= 1:
        args.world_size = 1
        return _rank_main(0, args)
    import torch.multiprocessing as mp
    prefix = f"/dev/shm/cdlrm_master_{os.getpid()}"
    mp.spawn(_rank_main, args=(args, prefix), nprocs=args.world_size, join=True)    # :638-643
    return None


if __name__ == "__main__":
    main()
