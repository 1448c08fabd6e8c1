"""B200-native mirror of the reference's ``model_no_ddp.py`` (lkp411/cDLRM).

Same class names, constructor arguments, attribute names and error behaviour as the
reference so that ``main_no_ddp.py`` can import it unchanged; the cache hot path runs in
hand-written sm_100a CUDA kernels behind the C ABI of ``libcdlrm_b200.so``
(``include/cdlrm_b200.h``).  There is no CPU / eager-PyTorch fallback: using the cache
group or the dot interaction without a CUDA device raises.

Reference citations are ``file:line`` in the reference tree.
"""
import ctypes
import os
import sys
import weakref

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from ._lib import check, lib

_vp = ctypes.c_void_p


def _stream_ptr(device):
    return _vp(torch.cuda.current_stream(device).cuda_stream)


def isPrime(n):
    """model_no_ddp.py:319-331 (quirky on purpose: see cdlrm_is_prime_ref)."""
    return bool(lib.cdlrm_is_prime_ref(int(n)))


# ------------------------------------------------------------------------------------
# master tables (host) -- model_no_ddp.py:21-98
# ------------------------------------------------------------------------------------


class Embedding_Table_Group(nn.Module):
    """CPU master embedding tables (model_no_ddp.py:21-98).  ``emb_l[k].weight`` is an
    ``nn.EmbeddingBag`` weight initialised U(+-sqrt(1/n)) from the numpy global RNG
    exactly as the reference does (:66-74).  ``device_pointers(device)`` pins the tables
    (cudaHostRegister, mapped) and returns the device-visible addresses the kernels read
    (zero-copy) and write back to."""

    def __init__(self, m_spa=None, ln_emb=None, qr_flag=False, qr_operation="mult", qr_collisions=0,
                 qr_threshold=200, md_flag=False, md_threshold=200, init="reference"):
        super().__init__()
        self._registered = {}
        if (m_spa is not None) and (ln_emb is not None):
            if qr_flag or md_flag:
                # unreachable in the reference as well (main_no_ddp.py:621 never passes them)
                raise NotImplementedError("QR / mixed-dimension embeddings are outside the cache hot path")
            self.qr_flag = qr_flag
            self.md_flag = md_flag
            self._mapped_file = isinstance(init, str) and init.startswith("shm:")
            self.emb_l = self.create_emb(m_spa, np.asarray(ln_emb), init)

    def create_emb(self, m, ln, init="reference"):
        emb_l = nn.ModuleList()
        for i in range(0, ln.size):
            n = int(ln[i])
            if init == "reference":
                W = np.random.uniform(low=-np.sqrt(1 / n), high=np.sqrt(1 / n), size=(n, m)).astype(np.float32)
                wt = torch.from_numpy(W)
            elif init == "device" or (isinstance(init, str) and init.startswith("shm:")):
                # same distribution, generated on the GPU and copied into page-locked host
                # memory (or into a /dev/shm file shared by all ranks: "shm:<prefix>")
                bound = float(np.sqrt(1 / n))
                if init == "device":
                    wt = torch.empty(n, m, dtype=torch.float32, pin_memory=True)
                    fill = True
                else:
                    prefix, role = init[4:].rsplit(":", 1)          # role: "create" | "attach"
                    wt = torch.from_file(f"{prefix}_{i}.bin", shared=True, size=n * m,
                                         dtype=torch.float32).view(n, m)
                    fill = role == "create"
                if fill:
                    g = torch.Generator(device="cuda").manual_seed(1000 + i)
                    step = 1 << 22
                    for lo in range(0, n, step):
                        hi = min(n, lo + step)
                        wt[lo:hi].copy_(torch.empty(hi - lo, m, device="cuda").uniform_(-bound, bound, generator=g))
            else:  # "fast": same distribution, chunked float32 generation on the host
                wt = torch.empty(n, m, dtype=torch.float32)
                bound = float(np.sqrt(1 / n))
                g = torch.Generator().manual_seed(1000 + i)
                step = 1 << 20
                for lo in range(0, n, step):
                    wt[lo:lo + step].uniform_(-bound, bound, generator=g)
            EE = nn.EmbeddingBag(n, m, mode="sum", sparse=True, _weight=wt)
            EE.weight.requires_grad = False
            emb_l.append(EE)
        return emb_l

    def fetch_unique_idx_slices(self, lists_of_unique_indices):
        """model_no_ddp.py:80-87.  CUDA id lists are gathered by the zero-copy kernel
        (cdlrm_move_gather_master) by callers that own a context; host id lists index
        the host table directly (pure addressing, no arithmetic)."""
        return [self.emb_l[k].weight.data[u.to(self.emb_l[k].weight.device)]
                for k, u in enumerate(lists_of_unique_indices)]

    def forward(self, lS_o, lS_i):
        return [self.emb_l[k](lS_i[k], lS_o[k]) for k in range(len(lS_i))]

    # -- pinning ---------------------------------------------------------------------
    def device_pointers(self, device):
        """Device-visible addresses of every table for ``device`` (int)."""
        ptrs = []
        for k, E in enumerate(self.emb_l):
            w = E.weight.data
            if w.is_cuda:                       # master kept in HBM (optional mode)
                ptrs.append(w.data_ptr())
                continue
            if not w.is_pinned() and not w.is_shared() and not getattr(self, "_mapped_file", False):
                # ordinary heap memory shares pages with its neighbours; registering it would
                # leave those neighbours "partially pinned" and break their later copies.
                # Re-home the table in page-locked memory of its own (one copy, at bind time).
                E.weight.data = w.pin_memory()
                w = E.weight.data
            key = (w.data_ptr(), device)
            if key not in self._registered:
                if w.is_pinned():
                    # torch-pinned memory is mapped and portable; under UVA the device
                    # address equals the host address
                    self._registered[key] = w.data_ptr()
                else:
                    dev = _vp()
                    check(lib.cdlrm_host_register(int(device), _vp(w.data_ptr()), w.numel() * 4,
                                                  ctypes.byref(dev)))
                    self._registered[key] = dev.value
            ptrs.append(self._registered[key])
        return ptrs

    def __del__(self):
        try:
            self.unpin()
        except Exception:
            pass

    def unpin(self):
        pinned = {E.weight.data_ptr() for E in self.emb_l if E.weight.data.is_pinned()}
        for (hptr, _), _dev in list(self._registered.items()):
            if hptr not in pinned:
                lib.cdlrm_host_unregister(_vp(hptr))
        self._registered.clear()


# ------------------------------------------------------------------------------------
# cache group -- model_no_ddp.py:101-212
# ------------------------------------------------------------------------------------

_GROUPS = weakref.WeakSet()      # cache groups with a pending fused update (optimizer hook)
_GRAD_READY = {}                 # data_ptr of the interaction backward's gradient planes -> event recorded behind it


class _LookupFn(torch.autograd.Function):
    """Autograd bridge: forward = cdlrm_embed_fwd, backward = de-duplicated sparse SGD
    (cdlrm_embed_bwd_plan + cdlrm_embed_bwd_sgd).  The update is applied when
    ``optimizer_embeds.step()`` runs (see ``_install_optimizer_hook``), or immediately
    when ``group.fused_lr`` is set."""

    @staticmethod
    def forward(ctx, anchor, group, ids, offsets, n_idx, n_bags, tb):
        out, slots, bag_ids = group._launch_forward(ids, offsets, n_idx, n_bags, tb)
        ctx.group = group
        ctx.tb = tb
        ctx.slots = slots
        ctx.bag_ids = bag_ids
        ctx.n_idx = n_idx
        # the backward's de-duplication plan only needs the slots: build it now on a side
        # stream so that it overlaps the MLP forward instead of sitting on the critical path
        ctx.plan = group._early_plan(tb, slots, n_idx) if group.early_plan else None
        ctx.mark_non_differentiable(slots)
        ctx.set_materialize_grads(False)      # no zero tensor for the (integer) slots output on every backward
        return (slots,) + tuple(out.unbind(0))

    @staticmethod
    def backward(ctx, _gslots, *grads):
        group = ctx.group
        T = len(grads)
        g0 = next((g for g in grads if g is not None), None)
        if g0 is None:
            return (None,) * 7
        d = group.dim
        # fast path: the T grads are planes of one buffer (what the interaction backward makes)
        uniform = all(g is not None and g.stride(1) == 1 for g in grads)
        if uniform:
            rs = grads[0].stride(0)
            ld = (grads[1].data_ptr() - grads[0].data_ptr()) // 4 if T > 1 else 0
            uniform = all(g.stride(0) == rs and g.data_ptr() - grads[0].data_ptr() == 4 * ld * k
                          for k, g in enumerate(grads)) and (T == 1 or ld > 0)
        if uniform:
            base, keep = grads[0], grads
        else:
            zero = torch.zeros_like(g0)
            keep = torch.stack([g if g is not None else zero for g in grads]).contiguous()
            base, rs, ld = keep, d, keep.stride(0)
        group._queue_update(ctx.tb, ctx.slots, ctx.bag_ids, ctx.n_idx, base, ld, rs, keep, ctx.plan)
        return (None,) * 7


class Embedding_Table_Cache_Group(nn.Module):
    """Set-associative GPU cache of embedding rows (model_no_ddp.py:101-212).

    Attributes kept from the reference: ``ln_emb, num_ways, max_cache_size, emb_l``
    (``nn.EmbeddingBag(num_ways*num_sets + aux, dim)`` per table), ``cache_sizes``,
    ``occupancy_tables`` (int64 ``[num_sets, num_ways]``, -1 = empty; moved to the GPU
    with the module), ``victim_cache_entries``.
    """

    def __init__(self, m_spa, ln_emb, max_cache_size, aux_table_size, num_ways, device=None, init="zeros"):
        """``init="reference"``: build every ``nn.EmbeddingBag`` exactly as model_no_ddp.py:138 does (N(0,1)
        rows drawn from torch's global CPU generator, then moved to ``device``).  The rows are never read before
        a fill, but the draws advance the generator that ``Categorical.sample()`` later consumes for the victim
        ways (main_no_ddp.py:183-185): ``--strict-reference`` needs the same offset to reproduce the reference
        program's cache decisions.  Default "zeros": no draws, rows zeroed on the device."""
        super().__init__()
        self._init_mode = init
        self.ln_emb = np.asarray(ln_emb)
        self.dim = int(m_spa)
        self.num_ways = int(num_ways)
        self.aux_table_size = int(aux_table_size)
        self.raw_cache_size = int(max_cache_size)
        self.max_cache_size = self.find_next_prime(int(max_cache_size))
        self.emb_l, self.cache_sizes = self.create_emb(m_spa, self.ln_emb, self.max_cache_size, num_ways,
                                                       aux_table_size, device)
        self.occupancy_tables = self.create_occupancy_tables(self.cache_sizes, num_ways, device)
        self.victim_cache_entries = [None] * len(self.emb_l)
        self.record_victims = False        # True: fill victim_cache_entries (costs a device sync)
        self.assume_one_id_per_bag = None  # None: check lS_o on the host when it is a CPU tensor
        self.fused_lr = None               # set to apply the SGD update inside backward
        self.early_plan = True             # build the backward plan during forward, on a side stream
        self.forward_stream = None         # set: lookup kernels run on this stream; consumers call join_forward()
        # with fused_lr and forward_stream set: the sparse update is launched from backward on forward_stream, behind
        # the event that marks the lookups' gradients ready, beside the rest of the backward (the bottom MLP);
        # optimizer_embeds.step() (pre-step hook) joins it
        self.overlap_update = False
        self._upd_done = None
        self._fwd_done = None
        self._plan_stream = None
        self.last_n_miss = None
        self._ctx = None
        self._bound_key = None
        self._pending = []
        self._plan_buf = None
        self._dirty = None
        _install_optimizer_hook()

    # -- geometry (model_no_ddp.py:122-147) -----------------------------------------------
    def find_next_prime(self, max_cache_size):
        r = lib.cdlrm_find_next_prime(int(max_cache_size))
        return None if r < 0 else int(r)

    def compute_set_indices(self, table_idx, lookup_idxs):
        return torch.remainder(lookup_idxs, self.cache_sizes[table_idx])

    def create_emb(self, m, ln, max_cache_size, num_ways, aux_table_size, device=None):
        emb_l = nn.ModuleList()
        cache_sizes = []
        for i in range(0, ln.size):
            n = int(ln[i])
            num_rows = n if n < max_cache_size else max_cache_size
            cache_sizes.append(num_rows)
            if getattr(self, "_init_mode", "zeros") == "reference":
                EE = nn.EmbeddingBag(num_ways * num_rows + aux_table_size, m, mode="sum", sparse=True)   # :138
                emb_l.append(EE.to(device) if device is not None else EE)
                continue
            # rows are only ever read after a fill: skip the N(0,1) init of nn.EmbeddingBag
            w = torch.zeros(num_ways * num_rows + aux_table_size, m, dtype=torch.float32, device=device)
            emb_l.append(nn.EmbeddingBag(num_ways * num_rows + aux_table_size, m, mode="sum", sparse=True,
                                         _weight=w))
        return emb_l, cache_sizes

    def create_occupancy_tables(self, cache_sizes, num_ways, device=None):
        return [torch.full((cache_sizes[i], num_ways), -1, dtype=torch.int64, device=device)
                for i in range(len(cache_sizes))]

    def _apply(self, fn, *a, **kw):
        super()._apply(fn, *a, **kw)
        self.occupancy_tables = [fn(t) for t in self.occupancy_tables]
        self._bound_key = None
        return self

    # -- context / binding -------------------------------------------------------------------
    @property
    def device(self):
        return self.emb_l[0].weight.device

    def _ensure_ctx(self, emb_tables=None):
        dev = self.device
        if dev.type != "cuda":
            raise _lib.CdlrmError("Embedding_Table_Cache_Group needs a CUDA device: the cache hot path has no "
                                  "CPU fallback (move the module with .to(rank) first)")
        if self._ctx is None:
            h = _vp()
            n_rows = _lib.i64_array([int(n) for n in self.ln_emb])
            check(lib.cdlrm_ctx_create(ctypes.byref(h), dev.index, len(self.emb_l), self.dim, self.num_ways,
                                       self.aux_table_size, n_rows, self.raw_cache_size))
            self._ctx = h
            T = len(self.emb_l)
            sets = (ctypes.c_int64 * T)()
            rows = (ctypes.c_int64 * T)()
            check(lib.cdlrm_ctx_geometry(self._ctx, sets, rows))
            assert list(sets) == [int(s) for s in self.cache_sizes]
            self._cache_rows = list(rows)
        self.occupancy_tables = [t if t.device == dev else t.to(dev) for t in self.occupancy_tables]
        key = tuple(e.weight.data_ptr() for e in self.emb_l) + tuple(t.data_ptr() for t in self.occupancy_tables)
        if key != self._bound_key:
            check(lib.cdlrm_ctx_bind_cache(self._ctx, _lib.ptr_array([e.weight.data_ptr() for e in self.emb_l]),
                                           _lib.ptr_array([t.data_ptr() for t in self.occupancy_tables])))
            # a planner running ahead of the live tags owns a separate copy (WindowPlanner.enable_lookahead_tags):
            # a re-bind (module moved, state dict assigned) must not point the planner back at the live tags
            ptags = getattr(self, "_plan_tags", None)
            if ptags is not None:
                ptags[:] = [t if t.device == dev else t.to(dev) for t in ptags]
            check(lib.cdlrm_ctx_bind_plan_tags(self._ctx, _lib.ptr_array(
                [t.data_ptr() for t in (ptags if ptags is not None else self.occupancy_tables)])))
            words = [(r + 31) // 32 for r in self._cache_rows]
            if self._dirty is None or self._dirty.numel() != sum(words):
                self._dirty = torch.zeros(sum(words), dtype=torch.int32, device=dev)
            elif self._dirty.device != dev:      # pending dirty bits survive the move (rows touched since the last aggregation)
                self._dirty = self._dirty.to(dev)
            offs = np.concatenate([[0], np.cumsum(words)[:-1]])
            check(lib.cdlrm_ctx_bind_dirty(self._ctx, _lib.ptr_array(
                [self._dirty.data_ptr() + 4 * int(o) for o in offs])))
            self._bound_key = key
        if emb_tables is not None:
            mkey = (id(emb_tables), tuple(E.weight.data_ptr() for E in emb_tables.emb_l))
            if getattr(self, "_master_key", None) != mkey:
                check(lib.cdlrm_ctx_bind_master(self._ctx, _lib.ptr_array(emb_tables.device_pointers(dev.index))))
                self._master_key = mkey
                self._emb_tables = weakref.ref(emb_tables)
        return self._ctx

    def __del__(self):
        try:
            if self._ctx is not None:
                lib.cdlrm_ctx_destroy(self._ctx)
        except Exception:
            pass

    # -- forward (model_no_ddp.py:149-212) --------------------------------------------------------
    def _launch_forward(self, ids, offsets, n_idx, n_bags, tb=0):
        dev = self.device
        T = ids.shape[0]
        out = torch.empty(T, n_bags, self.dim, dtype=torch.float32, device=dev)
        slots = torch.empty(T, max(n_idx, 1), dtype=torch.int32, device=dev)
        n_miss = torch.empty(T, dtype=torch.int32, device=dev)
        bag_ids = None
        if offsets is not None:
            bag_ids = torch.empty(T, max(n_idx, 1), dtype=torch.int32, device=dev)
        fs = self.forward_stream
        if fs is not None:
            # fork: the lookup (HBM gather + zero-copy PCIe miss fetch) overlaps whatever the caller
            # enqueues next on the current stream (the bottom MLP); join_forward() is the join
            fs.wait_stream(torch.cuda.current_stream(dev))
            sptr = _vp(fs.cuda_stream)
            ids.record_stream(fs)              # inputs may be temporaries of the caller's stream
            if offsets is not None:
                offsets.record_stream(fs)
        else:
            sptr = _stream_ptr(dev)
        check(lib.cdlrm_embed_fwd(
            self._ctx, tb, T, _vp(ids.data_ptr()), ids.stride(0),
            _vp(offsets.data_ptr()) if offsets is not None else None,
            offsets.stride(0) if offsets is not None else 0,
            n_idx, n_bags, _vp(out.data_ptr()), out.stride(0), _vp(slots.data_ptr()), slots.stride(0),
            _vp(n_miss.data_ptr()), _vp(bag_ids.data_ptr()) if bag_ids is not None else None,
            bag_ids.stride(0) if bag_ids is not None else 0, sptr))
        if fs is not None:
            self._fwd_done = torch.cuda.Event()
            self._fwd_done.record(fs)
        if tb == 0 and T == len(self.emb_l):
            self.last_n_miss = n_miss
        else:
            if self.last_n_miss is None or self.last_n_miss.numel() != len(self.emb_l):
                self.last_n_miss = torch.zeros(len(self.emb_l), dtype=torch.int32, device=dev)
            self.last_n_miss[tb:tb + T] = n_miss
        return out, slots, bag_ids

    def join_forward(self):
        """Make the current stream wait for the lookup kernels launched on ``forward_stream``."""
        if self._fwd_done is not None:
            torch.cuda.current_stream(self.device).wait_event(self._fwd_done)
            self._fwd_done = None

    def _one_id_per_bag(self, lS_o, n_idx, n_bags):
        if n_idx != n_bags:
            return False
        if self.assume_one_id_per_bag is not None:
            return bool(self.assume_one_id_per_bag)
        if isinstance(lS_o, torch.Tensor) and not lS_o.is_cuda:
            ar = torch.arange(n_bags, dtype=lS_o.dtype)
            return bool((lS_o == ar).all()) if lS_o.dim() == 2 else bool(torch.equal(lS_o, ar))
        return False   # device offsets: cannot be inspected without a sync -> general pooling path

    def forward(self, lS_o, lS_i, emb_tables, rank):
        if (len(self.emb_l) != len(lS_o)) or (len(self.emb_l) != len(lS_i)):
            sys.exit("ERROR: corrupted model input detected in parallel_forward call")
        self._ensure_ctx(emb_tables)
        dev = self.device
        if isinstance(rank, int) and rank != dev.index:
            raise _lib.CdlrmError(f"cache group lives on {dev}, forward called with rank={rank}")
        uniform = isinstance(lS_i, torch.Tensor) and lS_i.dim() == 2 and isinstance(lS_o, torch.Tensor) \
            and lS_o.dim() == 2
        if not uniform:   # ragged lists: one table per call
            lens_i = {int(t.numel()) for t in lS_i}
            lens_o = {int(t.numel()) for t in lS_o}
            if len(lens_i) == 1 and len(lens_o) == 1:
                lS_i, lS_o, uniform = torch.stack(list(lS_i)), torch.stack(list(lS_o)), True
        if uniform:
            outs, slots = self._forward_uniform(lS_o, lS_i)
            slots = [slots[k] for k in range(slots.shape[0])]
        else:             # ragged: tables with different numbers of ids / bags, one launch set per table
            outs, slots = [], []
            for k in range(len(self.emb_l)):
                o, s_ = self._forward_uniform(lS_o[k].reshape(1, -1), lS_i[k].reshape(1, -1), tb=k)
                outs.append(o[0])
                slots.append(s_[0])
        if len(self.emb_l) != len(outs):
            sys.exit("ERROR: corrupted intermediate result in parallel_forward call")
        if self.record_victims:
            self.join_forward()
            nm = self.last_n_miss.tolist()
            for k in range(len(self.emb_l)):
                base = self.cache_sizes[k] * self.num_ways
                aux = torch.arange(base, base + nm[k], device=dev)
                sl = slots[k].long()
                miss_pos = (sl >= base).nonzero().flatten()
                self.victim_cache_entries[k] = (aux, lS_i[k].to(dev)[miss_pos])
        return list(outs), slots

    def _forward_uniform(self, lS_o, lS_i, tb=0):
        dev = self.device
        n_idx, n_bags = int(lS_i.shape[1]), int(lS_o.shape[1])
        p1 = self._one_id_per_bag(lS_o, n_idx, n_bags)
        ids = lS_i.to(dev, dtype=torch.int64, non_blocking=True)
        if ids.stride(1) != 1:
            ids = ids.contiguous()
        offsets = None
        if not p1:
            offsets = lS_o.to(dev, dtype=torch.int64, non_blocking=True).contiguous()
        # (overflow of the aux region is detected on the device: check_device_flags)
        if torch.is_grad_enabled():
            # A fresh zero-size leaf per call: autograd needs one differentiable input to call backward at all.  A
            # long-lived leaf would do, except that its AccumulateGrad node is pinned to the stream of the step
            # that created it for as long as ANY earlier graph is alive (a caller still holding last step's loss):
            # the engine then syncs that stream at the end of every backward -- inside a CUDA-graph capture that is
            # "dependency created on uncaptured work in another stream" and the capture dies.
            anchor = torch.empty(0, device=dev, requires_grad=True)
            res = _LookupFn.apply(anchor, self, ids, offsets, n_idx, n_bags, tb)
            slots, outs = res[0], res[1:]
        else:
            out, slots, _ = self._launch_forward(ids, offsets, n_idx, n_bags, tb)
            outs = out.unbind(0)
        return outs, slots[:, :n_idx]

    def check_device_flags(self):
        """Raise what the reference would have raised on the host (IndexError) for
        conditions detected on the device.  Synchronises."""
        f = ctypes.c_uint32(0)
        check(lib.cdlrm_ctx_check(self._ctx, _stream_ptr(self.device), ctypes.byref(f)))
        if f.value & 1:
            raise IndexError("aux (victim) region overflow: more misses than aux_table_size "
                             "(model_no_ddp.py:177-179)")
        if f.value & 2:
            raise IndexError("sparse index outside its embedding table")
        return f.value

    # -- backward + SGD (main_no_ddp.py:376,409,413) ----------------------------------------------
    def _early_plan(self, tb, slots, n_idx):
        if n_idx == 0:
            return None
        dev = self.device
        cur = torch.cuda.current_stream(dev)
        if self.forward_stream is not None:
            ps = self.forward_stream           # stream order after the lookup that produced the slots
        else:
            if self._plan_stream is None:
                self._plan_stream = _lib.new_stream(dev)
            ps = self._plan_stream
            ps.wait_stream(cur)
        T = slots.shape[0]
        nbytes = lib.cdlrm_embed_bwd_plan_bytes(T, n_idx)
        with torch.cuda.stream(ps):
            buf = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
            base = (buf.data_ptr() + 255) // 256 * 256
            check(lib.cdlrm_embed_bwd_plan(self._ctx, tb, T, _vp(slots.data_ptr()), slots.stride(0), n_idx,
                                           _vp(base), _vp(ps.cuda_stream)))
            done = torch.cuda.Event()
            done.record(ps)
        slots.record_stream(ps)
        return (buf, base, done)

    def _queue_update(self, tb, slots, bag_ids, n_idx, dbase, ld, rs, keep, plan=None):
        item = (tb, slots, bag_ids, n_idx, dbase, ld, rs, keep, plan)
        if self.fused_lr is not None:
            self._apply_update(item, float(self.fused_lr))
            if self._upd_done is not None:
                _GROUPS.add(self)
        else:
            self._pending.append(item)
            _GROUPS.add(self)

    def _apply_update(self, item, lr):
        tb, slots, bag_ids, n_idx, dbase, ld, rs, _keep, plan = item
        if n_idx == 0:
            return
        dev = self.device
        T = slots.shape[0]
        cur = torch.cuda.current_stream(dev)
        us = self.forward_stream if (self.overlap_update and self.forward_stream is not None) else None
        if us is not None:
            # not wait_stream(cur): autograd has usually enqueued the bottom MLP's backward on `cur` already, and
            # the point is to run beside it -- wait for the producer of the gradients only
            ready = _GRAD_READY.pop(dbase.data_ptr(), None)
            if ready is not None:
                us.wait_event(ready)
            else:
                us.wait_stream(cur)
            for t in (dbase, slots, bag_ids):
                if t is not None:
                    t.record_stream(us)
            cur = us
        s = _vp(cur.cuda_stream)
        if plan is not None:
            buf, base, done = plan
            cur.wait_event(done)
            buf.record_stream(cur)
        else:
            nbytes = lib.cdlrm_embed_bwd_plan_bytes(T, n_idx)
            if self._plan_buf is None or self._plan_buf.numel() < nbytes + 256:
                self._plan_buf = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
            base = (self._plan_buf.data_ptr() + 255) // 256 * 256
            check(lib.cdlrm_embed_bwd_plan(self._ctx, tb, T, _vp(slots.data_ptr()), slots.stride(0), n_idx,
                                           _vp(base), s))
        check(lib.cdlrm_embed_bwd_sgd(self._ctx, tb, T, _vp(base), n_idx,
                                      _vp(bag_ids.data_ptr()) if bag_ids is not None else None,
                                      bag_ids.stride(0) if bag_ids is not None else 0,
                                      _vp(dbase.data_ptr()), ld, rs, lr, s))
        if us is not None:
            self._upd_done = torch.cuda.Event()
            self._upd_done.record(us)

    def join_update(self):
        """Make the current stream wait for a sparse update launched on ``forward_stream`` (``overlap_update``)."""
        if self._upd_done is not None:
            torch.cuda.current_stream(self.device).wait_event(self._upd_done)
            self._upd_done = None

    def apply_pending_updates(self, lr):
        """Apply the sparse SGD updates queued by backward (called by the optimizer hook
        with the learning rate of the param group that holds this module's weights)."""
        pend, self._pending = self._pending, []
        for item in pend:
            self._apply_update(item, lr)

    def dirty_bitmap(self):
        return self._dirty


def _optimizer_pre_step(optimizer, args, kwargs):
    if not _GROUPS:
        return
    for group in list(_GROUPS):
        if not group._pending and group._upd_done is None:
            continue
        mine = {id(e.weight) for e in group.emb_l}
        for pg in optimizer.param_groups:
            if any(id(p) in mine for p in pg["params"]):
                if group._pending:
                    group.apply_pending_updates(float(pg["lr"]))
                group.join_update()      # an update launched from backward on the lookup stream is complete here
                break


_HOOK = []


def _install_optimizer_hook():
    """``torch.optim.SGD(cache_group.parameters(), lr=args.lr_embeds)`` (main_no_ddp.py:376)
    keeps working unmodified: the weights never get a ``.grad`` (so the stock step is a
    no-op for them) and this global pre-step hook applies the fused update with the
    optimizer's own learning rate at the moment ``optimizer_embeds.step()`` is called."""
    if not _HOOK:
        from torch.optim.optimizer import register_optimizer_step_pre_hook
        _HOOK.append(register_optimizer_step_pre_hook(_optimizer_pre_step))


# ------------------------------------------------------------------------------------
# DLRM_Net -- model_no_ddp.py:215-316
# ------------------------------------------------------------------------------------


class _InteractFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, itself, x, *ly):
        feats = (x,) + ly
        B, d = x.shape
        dev = x.device
        rs = feats[0].stride(0)
        ok = all(f.is_cuda and f.dtype == torch.float32 and f.shape == x.shape and f.stride(1) == 1 and
                 f.stride(0) == rs for f in feats)
        if not ok:
            feats = tuple(f.contiguous().float() for f in feats)
            rs = d
        nf = len(feats)
        npair = nf * (nf + 1) // 2 if itself else nf * (nf - 1) // 2
        out = torch.empty(B, d + npair, dtype=torch.float32, device=dev)
        check(lib.cdlrm_interact_fwd(dev.index, _lib.ptr_array([f.data_ptr() for f in feats]), nf, rs, B, d,
                                     int(itself), _vp(out.data_ptr()), out.stride(0), _stream_ptr(dev)))
        ctx.feats = feats
        ctx.itself = itself
        ctx.rs = rs
        return out

    @staticmethod
    def backward(ctx, dR):
        feats = ctx.feats
        B, d = feats[0].shape
        dev = dR.device
        if dR.stride(1) != 1:
            dR = dR.contiguous()
        nf = len(feats)
        dfeat = torch.empty(nf, B, d, dtype=torch.float32, device=dev)
        check(lib.cdlrm_interact_bwd(dev.index, _lib.ptr_array([f.data_ptr() for f in feats]), nf, ctx.rs, B, d,
                                     int(ctx.itself), _vp(dR.data_ptr()), dR.stride(0), _vp(dfeat.data_ptr()),
                                     dfeat.stride(0), _stream_ptr(dev)))
        if nf > 1:
            # the lookups' gradients (planes 1..) are ready here: a cache group that overlaps its sparse update with
            # the rest of the backward waits for this event instead of the whole stream (Embedding_Table_Cache_Group)
            _GRAD_READY.clear()
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(dev))
            _GRAD_READY[dfeat[1].data_ptr()] = ev
        return (None,) + tuple(dfeat.unbind(0))


class _BceMeanFn(torch.autograd.Function):
    """torch.nn.BCELoss(reduction="mean")(Z, T) (main_no_ddp.py:355-369,403-405) with its derivative computed
    in the same launch (cdlrm_bce_mean): two launches per step instead of PyTorch's five."""

    @staticmethod
    def forward(ctx, Z, T):
        dev = Z.device
        n = Z.numel()
        Zc = Z if (Z.dim() == 2 and Z.shape[1] == 1) or Z.is_contiguous() else Z.contiguous()
        Tc = T if (T.dim() == 2 and T.shape[1] == 1) or T.is_contiguous() else T.contiguous()
        ldz = Zc.stride(0) if Zc.dim() == 2 and Zc.shape[1] == 1 else 1
        ldt = Tc.stride(0) if Tc.dim() == 2 and Tc.shape[1] == 1 else 1
        loss = torch.empty((), dtype=torch.float32, device=dev)
        dz = torch.empty(Z.shape, dtype=torch.float32, device=dev)
        check(lib.cdlrm_bce_mean(dev.index, _vp(Zc.data_ptr()), ldz, _vp(Tc.data_ptr()), ldt, n, _vp(loss.data_ptr()),
                                 _vp(dz.data_ptr()), _stream_ptr(dev)))
        ctx.save_for_backward(dz)
        return loss

    @staticmethod
    def backward(ctx, g):
        (dz,) = ctx.saved_tensors
        return dz * g, None


def bce_mean_with_grad(Z, T):
    """(loss, d loss / d Z) of BCELoss(mean) in one launch, outside autograd: a training loop that calls
    ``Z.backward(dz)`` instead of ``loss.backward()`` saves the two launches autograd spends on seeding the scalar
    loss with ones and scaling dz by it."""
    dev = Z.device
    Zc, Tc = Z.detach(), T
    n = Zc.numel()
    ldz = Zc.stride(0) if Zc.dim() == 2 and Zc.shape[1] == 1 else 1
    ldt = Tc.stride(0) if Tc.dim() == 2 and Tc.shape[1] == 1 else 1
    if ldz == 1 and not Zc.is_contiguous():
        Zc = Zc.contiguous()
    if ldt == 1 and not Tc.is_contiguous():
        Tc = Tc.contiguous()
    loss = torch.empty((), dtype=torch.float32, device=dev)
    dz = torch.empty(Z.shape, dtype=torch.float32, device=dev)
    check(lib.cdlrm_bce_mean(dev.index, _vp(Zc.data_ptr()), ldz, _vp(Tc.data_ptr()), ldt, n, _vp(loss.data_ptr()),
                             _vp(dz.data_ptr()), _stream_ptr(dev)))
    return loss, dz


def bce_mean(Z, T):
    """Fused BCELoss(mean) + derivative for float32 CUDA tensors; anything else goes to torch."""
    if Z.is_cuda and Z.dtype == torch.float32 and T.dtype == torch.float32 and Z.shape == T.shape and Z.numel() > 0:
        return _BceMeanFn.apply(Z, T)
    return torch.nn.functional.binary_cross_entropy(Z, T)


# ------------------------------------------------------------------------------------
# dense MLPs on the tensor cores (cdlrm_mlp_*: 3xTF32 split GEMMs, FP32 accuracy)
# ------------------------------------------------------------------------------------


class _MlpState:
    """One cdlrm_mlp object (C ABI) + its workspace for an nn.Sequential built by
    DLRM_Net.create_mlp (model_no_ddp.py:244-270): the layer list, the batch capacity and the
    activations the last forward left behind for the backward."""

    def __init__(self, seq, sigmoid_layer):
        self.linears = [m for m in seq if isinstance(m, nn.Linear)]
        self.dims = [self.linears[0].in_features] + [m.out_features for m in self.linears]
        self.sigmoid_layer = int(sigmoid_layer)
        self.handle = None
        self.cap = 0
        self.ws = None
        self.fwd_id = 0
        self.flat_grads = None     # ([dW views], [db views]) into DLRM_Net's flat gradient bucket, or None
        self.defer_join = False    # cdlrm_mlp_set_defer_join: dW / db complete only after DLRM_Net.join_mlp_grads()
        self.after_backward = None  # optional callable run right after this MLP's backward was enqueued (Trainer:
                                    # starts the all-reduce of the top MLP's weight gradients beside the rest)

    def ensure(self, batch, dev):
        if self.handle is not None and batch <= self.cap and self.ws.device == dev:
            return
        self.close()
        L = len(self.linears)
        dims = (ctypes.c_int32 * (L + 1))(*self.dims)
        need = lib.cdlrm_mlp_workspace_bytes(L, dims, batch)
        if need <= 0:
            raise _lib.CdlrmError("cdlrm_mlp_workspace_bytes failed")
        self.ws = torch.empty(need + 256, dtype=torch.uint8, device=dev)
        base = (self.ws.data_ptr() + 255) & ~255
        h = ctypes.c_void_p()
        check(lib.cdlrm_mlp_create(ctypes.byref(h), dev.index, L, dims, batch, self.sigmoid_layer, _vp(base), need))
        self.handle, self.cap = h, batch
        if self.defer_join:
            check(lib.cdlrm_mlp_set_defer_join(self.handle, 1))

    def set_defer_join(self, on):
        self.defer_join = bool(on)
        if self.handle is not None:
            check(lib.cdlrm_mlp_set_defer_join(self.handle, int(self.defer_join)))

    def close(self):
        if self.handle is not None:
            lib.cdlrm_mlp_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _MlpFn(torch.autograd.Function):
    """y = seq(x) for a create_mlp Sequential; params = W_0, b_0, W_1, b_1, ... as autograd inputs, or none of
    them in flat-bucket mode (the backward writes dW / db straight into the bucket: the parameters then stay out
    of the graph -- see the note on long-lived leaves in Embedding_Table_Cache_Group._forward_uniform -- and a
    fresh zero-size ``anchor`` leaf makes autograd call the backward)."""

    @staticmethod
    def forward(ctx, state, x, anchor, *params):
        dev = x.device
        if not params:
            params = [p for m in state.linears for p in (m.weight, m.bias)]
        if x.dtype != torch.float32 or x.stride(1) != 1:
            x = x.contiguous().float()
        B = x.shape[0]
        state.ensure(B, dev)
        Ws = [p if p.is_contiguous() else p.contiguous() for p in params[0::2]]
        bs = [p if p.is_contiguous() else p.contiguous() for p in params[1::2]]
        y = torch.empty(B, state.dims[-1], dtype=torch.float32, device=dev)
        check(lib.cdlrm_mlp_forward(state.handle, _vp(x.data_ptr()), x.stride(0), B,
                                    _lib.ptr_array([w.data_ptr() for w in Ws]),
                                    _lib.ptr_array([b.data_ptr() for b in bs]),
                                    _vp(y.data_ptr()), y.stride(0), _stream_ptr(dev)))
        state.fwd_id += 1
        ctx.state, ctx.fwd_id, ctx.batch = state, state.fwd_id, B
        ctx.need_dx = ctx.needs_input_grad[1]
        ctx.n_params = len(ctx.needs_input_grad) - 3
        return y

    @staticmethod
    def backward(ctx, dy):
        st = ctx.state
        if ctx.fwd_id != st.fwd_id:
            raise _lib.CdlrmError("MLP backward after another forward of the same MLP: its saved activations are gone")
        dev = dy.device
        if dy.stride(1) != 1 or dy.dtype != torch.float32:
            dy = dy.contiguous().float()
        B = ctx.batch
        if st.flat_grads is not None:      # DLRM_Net.flatten_parameters: dW / db land in the flat gradient bucket
            dWs, dbs = st.flat_grads
        else:
            dWs = [torch.empty(st.dims[i + 1], st.dims[i], dtype=torch.float32, device=dev) for i in range(len(st.linears))]
            dbs = [torch.empty(st.dims[i + 1], dtype=torch.float32, device=dev) for i in range(len(st.linears))]
        dx = None
        dx_ptr, lddx = None, 0
        if ctx.need_dx:
            ld = (st.dims[0] + 3) & ~3
            dx = torch.empty(B, ld, dtype=torch.float32, device=dev)[:, :st.dims[0]]
            dx_ptr, lddx = dx.data_ptr(), ld
        check(lib.cdlrm_mlp_backward(st.handle, _vp(dy.data_ptr()), dy.stride(0), _vp(dx_ptr), lddx,
                                     _lib.ptr_array([t.data_ptr() for t in dWs]),
                                     _lib.ptr_array([t.data_ptr() for t in dbs]), _stream_ptr(dev)))
        if st.after_backward is not None:
            st.after_backward()
        if st.flat_grads is not None:      # the bucket already holds them (p.grad is a view of it): nothing for autograd
            return (None, dx, None) + (None,) * ctx.n_params
        grads = []
        for w, b in zip(dWs, dbs):
            grads += [w, b]
        return (None, dx, None) + tuple(grads)


class EvalForward:
    """Forward-only pass of a trained ``Embedding_Table_Cache_Group`` + ``DLRM_Net`` for evaluation, one id per bag:
    read-only lookup (cdlrm_embed_fwd_eval: cache row, else the installed window's loser store, else the master),
    bottom MLP, interaction, top MLP.  The MLPs run on cdlrm_mlp handles of its own, sized for the evaluation batch:
    the training handles, their workspaces and the context's miss bitmap are never resized or written, so a training
    step captured in a CUDA graph keeps every pointer it holds.  Every launch goes to the current stream."""

    def __init__(self, cache_group, dlrm):
        self.cg, self.dlrm = cache_group, dlrm
        sig = getattr(dlrm, "_sigmoid", {})
        self.mlp = {"bot": _MlpState(dlrm.bot_l, sig.get("bot", -1)), "top": _MlpState(dlrm.top_l, sig.get("top", -1))}

    def begin(self):
        """Start of an evaluation: the next forward of each MLP splits the current weights into its hi / lo operands."""
        for st in self.mlp.values():
            if st.handle is not None:
                check(lib.cdlrm_mlp_invalidate_split(st.handle))

    def reserve(self, batch, dev):
        """Size both MLP handles for ``batch``; True when a handle was (re)allocated (graphs holding it are void)."""
        old = [st.handle for st in self.mlp.values()]
        for st in self.mlp.values():
            st.ensure(batch, dev)
        return [st.handle for st in self.mlp.values()] != old

    def _mlp(self, which, x):
        st = self.mlp[which]
        if self.dlrm.mlp_impl != "tcgen05":
            return (self.dlrm.bot_l if which == "bot" else self.dlrm.top_l)(x)
        dev, B = x.device, x.shape[0]
        if x.dtype != torch.float32 or x.stride(1) != 1:
            x = x.contiguous().float()
        if st.handle is None or B > st.cap:
            raise _lib.CdlrmError(f"EvalForward: batch {B} above the reserved capacity (reserve() first)")
        y = torch.empty(B, st.dims[-1], dtype=torch.float32, device=dev)
        Ws = [m.weight if m.weight.is_contiguous() else m.weight.contiguous() for m in st.linears]
        bs = [m.bias if m.bias.is_contiguous() else m.bias.contiguous() for m in st.linears]
        check(lib.cdlrm_mlp_forward(st.handle, _vp(x.data_ptr()), x.stride(0), B,
                                    _lib.ptr_array([w.data_ptr() for w in Ws]), _lib.ptr_array([b.data_ptr() for b in bs]),
                                    _vp(y.data_ptr()), y.stride(0), _stream_ptr(dev)))
        return y

    @torch.no_grad()
    def __call__(self, X, ids):
        """X: float32 [B, m_den], ids: int64 [T, B], both on the device; returns the predictions [B, 1]."""
        cg, net = self.cg, self.dlrm
        dev = X.device
        T, B = int(ids.shape[0]), int(ids.shape[1])
        if T != len(cg.emb_l):
            raise _lib.CdlrmError(f"EvalForward: {T} id rows for {len(cg.emb_l)} tables")
        if ids.stride(1) != 1:
            ids = ids.contiguous()
        ly = torch.empty(T, B, cg.dim, dtype=torch.float32, device=dev)
        check(lib.cdlrm_embed_fwd_eval(cg._ctx, 0, T, _vp(ids.data_ptr()), ids.stride(0), B, _vp(ly.data_ptr()),
                                       ly.stride(0), _stream_ptr(dev)))
        x = self._mlp("bot", X)
        if net.arch_interaction_op == "dot":
            feats = [x] + list(ly.unbind(0))
            if x.stride(0) != cg.dim or x.shape[1] != cg.dim:
                raise _lib.CdlrmError("EvalForward: the bottom MLP must end in the embedding dimension")
            itself = bool(net.arch_interaction_itself)
            nf = T + 1
            npair = nf * (nf + 1) // 2 if itself else nf * (nf - 1) // 2
            R = torch.empty(B, cg.dim + npair, dtype=torch.float32, device=dev)
            check(lib.cdlrm_interact_fwd(dev.index, _lib.ptr_array([f.data_ptr() for f in feats]), nf, cg.dim, B, cg.dim,
                                         int(itself), _vp(R.data_ptr()), R.stride(0), _stream_ptr(dev)))
        else:
            R = net.interact_features(x, list(ly.unbind(0)))
        p = self._mlp("top", R)
        if 0.0 < net.loss_threshold < 1.0:
            p = torch.clamp(p, min=net.loss_threshold, max=(1.0 - net.loss_threshold))
        return p


class DLRM_Net(nn.Module):
    """model_no_ddp.py:215-316.  bot_l / top_l are the reference's nn.Sequential stacks (same parameters, same
    numpy-RNG initialisation); on CUDA they execute through cdlrm_mlp_* (TMA + tcgen05 3xTF32 GEMMs, FP32
    accuracy; ``mlp_impl = "torch"`` / CDLRM_MLP=torch runs the stock modules).  The pairwise-dot
    interaction (:272-293) runs in cdlrm_interact_fwd/_bwd."""

    def __init__(self, ln_bot=None, ln_top=None, arch_interaction_op=None, arch_interaction_itself=False,
                 sync_dense_params=True, sigmoid_bot=-1, sigmoid_top=-1, loss_threshold=0.0):
        super().__init__()
        if (ln_bot is not None) and (ln_top is not None) and (arch_interaction_op is not None):
            self.output_d = 0
            self.parallel_model_batch_size = -1
            self.parallel_model_is_not_prepared = True
            self.arch_interaction_op = arch_interaction_op
            self.arch_interaction_itself = arch_interaction_itself
            self.sync_dense_params = sync_dense_params
            self.loss_threshold = loss_threshold
            self.cpu = torch.device("cpu")
            self.bot_l = self.create_mlp(ln_bot, sigmoid_bot)
            self.top_l = self.create_mlp(ln_top, sigmoid_top)
            self._sigmoid = {"bot": int(sigmoid_bot), "top": int(sigmoid_top)}
        self.pre_interact = None   # optional callable run between the bottom MLP and the interaction
        # "tcgen05": cdlrm_mlp_* (3xTF32 tensor-core GEMMs with fused epilogues, FP32 accuracy);
        # "torch": the stock nn.Sequential (cuBLAS SIMT sgemm)
        self.mlp_impl = os.environ.get("CDLRM_MLP", "tcgen05")
        self.fused_sgd_split = os.environ.get("CDLRM_SGD_SPLIT", "1") != "0"
        self._mlp_state = {}

    def create_mlp(self, ln, sigmoid_layer):
        """:244-270 -- numpy-RNG initialisation in the reference's draw order."""
        layers = nn.ModuleList()
        for i in range(0, ln.size - 1):
            n, m = int(ln[i]), int(ln[i + 1])
            LL = nn.Linear(n, m, bias=True)
            W = np.random.normal(0.0, np.sqrt(2 / (m + n)), size=(m, n)).astype(np.float32)
            bt = np.random.normal(0.0, np.sqrt(1 / m), size=m).astype(np.float32)
            LL.weight.data = torch.tensor(W, requires_grad=True)
            LL.bias.data = torch.tensor(bt, requires_grad=True)
            layers.append(LL)
            layers.append(nn.Sigmoid() if i == sigmoid_layer else nn.ReLU())
        return torch.nn.Sequential(*layers)

    def interact_features(self, x, ly):
        if self.arch_interaction_op == "dot":
            if not x.is_cuda:
                raise _lib.CdlrmError("interact_features('dot') needs CUDA tensors: no CPU fallback")
            return _InteractFn.apply(bool(self.arch_interaction_itself), x, *ly)
        elif self.arch_interaction_op == "cat":
            return torch.cat([x] + list(ly), dim=1)
        else:
            sys.exit("ERROR: --arch-interaction-op=" + self.arch_interaction_op + " is not supported")

    def flatten_parameters(self):
        """Flat-bucket mode for the dense parameters (SURVEY 8f.2; the reference all-reduces the Linear
        weight gradients one tensor at a time, main_no_ddp.py:234-247, and steps a per-tensor SGD, :413).
        Every nn.Linear parameter of bot_l / top_l is re-pointed at one flat FP32 buffer -- all weights first,
        then all biases, each 16-byte aligned -- and a gradient bucket of the same layout is allocated.  The
        tensor-core MLP backward then writes dW / db straight into the bucket (no autograd accumulation), the
        weight part is ONE all-reduce operand with no flatten / unflatten copies, and SGD is ONE axpy over
        the bucket (``flat_sgd_step``).  ``p.grad`` of every parameter is a view of the bucket."""
        lin = [m for seq in (self.bot_l, self.top_l) for m in seq if isinstance(m, nn.Linear)]
        params = [m.weight for m in lin] + [m.bias for m in lin]
        dev = params[0].device
        offs, o = [], 0
        n_bot = sum(1 for m in self.bot_l if isinstance(m, nn.Linear))
        for q in params:
            if q is lin[n_bot].weight:
                self.flat_top_weight_off = o      # [0, off): bottom MLP weights, [off, flat_weight_elems): top MLP weights
            offs.append(o)
            o += (q.numel() + 3) & ~3
            if q is lin[-1].weight:
                n_w = o
        flat_p = torch.zeros(o, dtype=torch.float32, device=dev)
        flat_g = torch.zeros(o, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for q, off in zip(params, offs):
                v = flat_p[off:off + q.numel()].view_as(q)
                v.copy_(q.data)
                q.data = v
                q.grad = flat_g[off:off + q.numel()].view_as(q)
        self.flat_params, self.flat_grads, self.flat_weight_elems = flat_p, flat_g, n_w
        for which, seq in (("bot", self.bot_l), ("top", self.top_l)):
            st = self._mlp_state.get(which)
            if st is None:
                st = self._mlp_state[which] = _MlpState(seq, getattr(self, "_sigmoid", {}).get(which, -1))
            st.flat_grads = ([m.weight.grad for m in st.linears], [m.bias.grad for m in st.linears])
        self.flat_mode = True
        return flat_p, flat_g

    def defer_wgrad_join(self, on=True):
        """Flat-bucket mode only: let the weight-gradient GEMMs of an MLP backward (side stream, csrc/mlp.cu) keep
        running after ``cdlrm_mlp_backward`` returns -- beside the interaction backward and the bottom MLP -- and
        make the caller responsible for ``join_mlp_grads()`` before it reads the gradient bucket."""
        if not getattr(self, "flat_mode", False):
            raise _lib.CdlrmError("defer_wgrad_join needs flatten_parameters(): autograd consumes dW / db otherwise")
        for st in self._mlp_state.values():
            st.set_defer_join(on)

    def join_mlp_grads(self):
        """Make the dW / db written by the last MLP backwards visible to the current stream."""
        for st in self._mlp_state.values():
            if st.handle is not None:
                check(lib.cdlrm_mlp_join(st.handle, _stream_ptr(self.flat_params.device)))

    @torch.no_grad()
    def flat_sgd_step(self, lr):
        """p -= lr * g over the whole flat bucket: one launch for all dense parameters.  On the tensor-core path the
        same launch also leaves the hi / lo operand copies of the UPDATED weights behind (cdlrm_mlp_sgd_split), so
        that the next forward of either MLP starts with its first GEMM instead of a split launch.  Dense parameters
        changed by anything else afterwards (``.data.copy_``) need ``invalidate_weight_splits()``;
        ``load_state_dict`` and ``.to()`` do it themselves."""
        sts = [self._mlp_state.get("bot"), self._mlp_state.get("top")]
        if (self.mlp_impl == "tcgen05" and self.fused_sgd_split
                and all(st is not None and st.handle is not None for st in sts)):
            lin = [m for st in sts for m in st.linears]
            n_w = self.flat_weight_elems
            check(lib.cdlrm_mlp_sgd_split(
                2, _lib.ptr_array([st.handle.value for st in sts]),
                _lib.ptr_array([m.weight.data_ptr() for m in lin]),
                _lib.ptr_array([g.data_ptr() for st in sts for g in st.flat_grads[0]]), float(lr),   # views of the bucket
                _vp(self.flat_params.data_ptr() + 4 * n_w), _vp(self.flat_grads.data_ptr() + 4 * n_w),
                self.flat_params.numel() - n_w, _stream_ptr(self.flat_params.device)))
            return
        self.flat_params.add_(self.flat_grads, alpha=-float(lr))

    def invalidate_weight_splits(self):
        for st in self._mlp_state.values():
            if st.handle is not None:
                check(lib.cdlrm_mlp_invalidate_split(st.handle))

    def load_state_dict(self, *a, **kw):
        r = super().load_state_dict(*a, **kw)
        self.invalidate_weight_splits()
        return r

    def _apply(self, fn, *a, **kw):
        r = super()._apply(fn, *a, **kw)
        if hasattr(self, "_mlp_state"):
            self.invalidate_weight_splits()
        return r

    def apply_mlp(self, which, x):
        """bot_l / top_l (:306-309).  On CUDA with mlp_impl == "tcgen05" the whole Sequential runs
        in cdlrm_mlp_forward/_backward; the nn.Linear parameters stay the trainable state."""
        seq = self.bot_l if which == "bot" else self.top_l
        if self.mlp_impl != "tcgen05" or not x.is_cuda:
            return seq(x)
        st = self._mlp_state.get(which)
        if st is None:
            st = self._mlp_state[which] = _MlpState(seq, getattr(self, "_sigmoid", {}).get(which, -1))
        if st.flat_grads is not None and torch.is_grad_enabled():
            return _MlpFn.apply(st, x, torch.empty(0, device=x.device, requires_grad=True))
        params = []
        for m in st.linears:
            params += [m.weight, m.bias]
        return _MlpFn.apply(st, x, None, *params)

    def forward(self, dense_x, ly):
        x = self.apply_mlp("bot", dense_x)
        if self.pre_interact is not None:
            self.pre_interact()    # e.g. cache_group.join_forward: lookups ran beside the bottom MLP
        z = self.interact_features(x, ly)
        p = self.apply_mlp("top", z)
        if 0.0 < self.loss_threshold < 1.0:
            return torch.clamp(p, min=self.loss_threshold, max=(1.0 - self.loss_threshold))
        return p
