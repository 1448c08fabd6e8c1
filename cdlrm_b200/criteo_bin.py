"""Criteo datasets in the MLPerf binary format (``--mlperf-bin-loader``): the data path of data_loader_terabyte.py
(facebookresearch/dlrm, SURVEY section 2 rows 12-13) with the per-step decode on the GPU.

Format: a data file is little-endian int32 records of 40 fields ``[label, 13 dense, 26 categorical]`` (160 bytes),
concatenated; batch j is the records ``[j B, (j + 1) B)``, the last one may be short.  A batch decodes to
(``_transform_features``, :68-87)::

    X    = torch.log(x_int.float() + 1)                                   [B, 13]
    lS_o = arange(B) repeated over the 26 tables                          [26, B]
    lS_i = (x_cat % max_ind_range if max_ind_range > 0 else x_cat).long().t()   [26, B]
    T    = y.float().view(-1, 1)                                          [B, 1]

``CriteoBinDataset`` decodes on the host with exactly those torch expressions (the reference semantics:
``--strict-reference``, the ``tuples`` FIFO payload, the tests' oracle).  ``device_batches`` streams a file to the
GPU and decodes there (``cdlrm_criteo_decode``); ``window_marker`` feeds one look-ahead window to the planner's
chunked scan without ever building the window's ids as one tensor.  DESIGN.md section 12.
"""
import math
import os
import queue
import threading

import numpy as np
import torch

from . import _lib
from ._lib import check, lib

RECORD_FIELDS = 40                 # label, 13 dense, 26 categorical
DENSE, SPARSE = 13, 26
RECORD_BYTES = 4 * RECORD_FIELDS
CHUNK_BYTES = 64 << 20             # host reads and host-to-device copies move this much at a time

_vp = _lib.vp
_STOP = object()


def _lso(n, device=None):
    return torch.arange(n, device=device).reshape(1, -1).repeat(SPARSE, 1)


def _transform_features(x_int, x_cat, y, max_ind_range):
    """data_loader_terabyte.py:68-87 with flag_input_torch_tensor=True."""
    if max_ind_range > 0:
        x_cat = x_cat % max_ind_range
    X = torch.log(x_int.float() + 1)
    return X, _lso(x_cat.shape[0]), x_cat.long().t(), y.float().view(-1, 1)


class CriteoBinDataset(torch.utils.data.Dataset):
    """data_loader_terabyte.py:195-235: batch ``idx`` of ``batch_size`` records of ``data_file``, decoded on the host.
    ``counts``: the 26 table sizes of ``counts_file`` (``np.load(counts_file)["counts"]``)."""

    def __init__(self, data_file, counts_file, batch_size=1, max_ind_range=-1, bytes_per_feature=4):
        if bytes_per_feature != 4:
            raise ValueError(f"{data_file}: only 4-byte (int32) features are supported, got {bytes_per_feature}")
        self.tar_fea, self.den_fea, self.spa_fea = 1, DENSE, SPARSE
        self.tad_fea = self.tar_fea + self.den_fea
        self.tot_fea = self.tad_fea + self.spa_fea
        self.m_den = DENSE
        self.batch_size = int(batch_size)
        self.max_ind_range = int(max_ind_range)
        self.bytes_per_feature = bytes_per_feature
        self.bytes_per_entry = bytes_per_feature * self.tot_fea * self.batch_size
        self.data_file, self.counts_file = data_file, counts_file
        size = os.path.getsize(data_file)
        if size % RECORD_BYTES:
            raise ValueError(f"{data_file}: {size} bytes is not a whole number of {RECORD_BYTES}-byte records")
        self.num_samples = size // RECORD_BYTES
        self.num_entries = math.ceil(size / self.bytes_per_entry)
        with np.load(counts_file) as z:
            counts = np.asarray(z["counts"]) if "counts" in z.files else None
        if counts is None or counts.ndim != 1 or counts.size != SPARSE:
            raise ValueError(f"{counts_file}: needs 'counts' with {SPARSE} table sizes, "
                             f"got {None if counts is None else tuple(counts.shape)}")
        self.counts = counts
        self._fd = os.open(data_file, os.O_RDONLY)
        self._scan = {}                # device index -> buffers of the window scan (window_marker)

    def __len__(self):
        return self.num_entries

    def records(self, j):
        """(first record, number of records) of batch j."""
        lo = j * self.batch_size
        return lo, min(self.batch_size, self.num_samples - lo)

    def __getitem__(self, idx):
        if not 0 <= idx < self.num_entries:
            raise IndexError(idx)
        lo, n = self.records(idx)
        raw = _pread(self._fd, n * RECORD_BYTES, lo * RECORD_BYTES, self.data_file)
        t = torch.from_numpy(np.frombuffer(raw, dtype="<i4").copy()).view(-1, self.tot_fea)
        return _transform_features(t[:, self.tar_fea:self.tad_fea], t[:, self.tad_fea:], t[:, 0], self.max_ind_range)

    def __iter__(self):
        for j in range(self.num_entries):
            yield self[j]

    def __del__(self):
        fd = getattr(self, "_fd", None)
        if fd is not None:
            os.close(fd)
            self._fd = None

    # -- GPU paths ---------------------------------------------------------------------------------
    def device_batches(self, device, start=0):
        """The batches ``[start, len)`` as CUDA tensors, read and decoded ahead of the consumer (``DeviceBatches``)."""
        return DeviceBatches(self, device, start)

    def window_marker(self, w, lookahead):
        """The marker callable of ``Trainer.submit_window`` for window ``w`` (batches ``[w L, (w + 1) L)``): on the plan
        thread it reads the window's records chunk by chunk, decodes their ids on ``planner.stream`` and marks them
        (``planner.mark_ids``); returns the window's number of ids per table."""
        lo = min(w * lookahead * self.batch_size, self.num_samples)
        hi = min((w + 1) * lookahead * self.batch_size, self.num_samples)
        return lambda planner: self._scan_window(planner, lo, hi)

    def _scan_window(self, planner, lo, hi):
        r, W = planner.scan_shard
        n = hi - lo
        a, b = lo + n * r // W, lo + n * (r + 1) // W
        dev = planner.dev
        s = planner.stream
        bufs = self._scan.get(dev.index)
        if bufs is None:
            m = CHUNK_BYTES // RECORD_BYTES
            with torch.cuda.stream(s):
                bufs = dict(m=m, pin=[torch.empty(m * RECORD_BYTES, dtype=torch.uint8, pin_memory=True) for _ in range(2)],
                            ev=[None, None], raw=torch.empty(m * RECORD_FIELDS, dtype=torch.int32, device=dev),
                            ids=torch.empty(SPARSE * m, dtype=torch.int64, device=dev))
            self._scan[dev.index] = bufs
        m, pin, ev = bufs["m"], bufs["pin"], bufs["ev"]
        raw, ids = bufs["raw"], bufs["ids"]
        i = 0
        for c0 in range(a, b, m):
            k = min(m, b - c0)
            q = i % 2
            if ev[q] is not None:
                ev[q].synchronize()        # the copy that read this pinned buffer has completed
            nbytes = k * RECORD_BYTES
            _preadv_into(self._fd, pin[q], nbytes, c0 * RECORD_BYTES, self.data_file)
            self.scan_bytes_read = getattr(self, "scan_bytes_read", 0) + nbytes
            with torch.cuda.stream(s):
                raw.view(torch.uint8)[:nbytes].copy_(pin[q][:nbytes], non_blocking=True)
                ev[q] = torch.cuda.Event()
                ev[q].record(s)
                out = ids[:SPARSE * k].view(SPARSE, k)
                check(lib.cdlrm_criteo_decode(dev.index, _vp(raw.data_ptr()), k, DENSE, SPARSE, self.max_ind_range,
                                              None, 0, _vp(out.data_ptr()), k, None, _vp(s.cuda_stream)))
                planner.mark_ids(out)
            i += 1
        return n


def _pread(fd, nbytes, offset, name):
    buf = bytearray(nbytes)
    got = os.preadv(fd, [buf], offset)
    if got != nbytes:
        raise IOError(f"{name}: short read at byte {offset}: {got} of {nbytes} bytes")
    return bytes(buf)


def _preadv_into(fd, pinned, nbytes, offset, name):
    """One positional read of ``nbytes`` into the pinned uint8 tensor (drops the interpreter lock while it reads)."""
    mv = memoryview(pinned.numpy())[:nbytes]
    got = os.preadv(fd, [mv], offset)
    if got != nbytes:
        raise IOError(f"{name}: short read at byte {offset}: {got} of {nbytes} bytes")


class DeviceBatches:
    """Iterable of the batches ``[start, len(dataset))`` as CUDA ``(X, lS_o, lS_i, T)`` tuples, the form ``Run`` and
    ``Trainer.evaluate`` take.  Every iteration runs its own pipeline (``_DeviceBatchIter``); ``iter_from(j)`` starts
    one at batch j without reading anything before it.  ``bytes_read``: file bytes read by all its iterations."""

    def __init__(self, dataset, device, start=0):
        self.ds, self.dev, self.start = dataset, torch.device(device), int(start)
        self.bytes_read = 0
        self._lso = None
        self._streams = None           # (copy, decode): library streams, created once and shared by the iterations

    def __len__(self):
        return max(0, self.ds.num_entries - self.start)

    def __iter__(self):
        return _DeviceBatchIter(self, self.start)

    def iter_from(self, j):
        return _DeviceBatchIter(self, self.start + int(j))


def _reader(fd, name, free_q, filled_q, stop, chunk_recs, first_rec, end_rec, pins):
    """Reader thread: fill pinned chunk c (records from first_rec on, chunk_recs each) once the copy that last read
    its buffer has completed; hand (c, records, bytes) over.  Errors go to the consumer."""
    try:
        c = 0
        for lo in range(first_rec, end_rec, chunk_recs):
            ev = free_q.get()
            if ev is _STOP or stop.is_set():
                return
            if ev is not None:
                ev.synchronize()
            k = min(chunk_recs, end_rec - lo)
            _preadv_into(fd, pins[c % 2], k * RECORD_BYTES, lo * RECORD_BYTES, name)
            filled_q.put((c, k))
            c += 1
    except BaseException as e:      # raised in the consumer
        filled_q.put(e)


class _DeviceBatchIter:
    """reader thread -> two pinned chunks (one ``os.preadv`` each) -> one ``cudaMemcpyAsync`` per chunk on a copy
    stream -> one ``cdlrm_criteo_decode`` per batch on a decode stream into a ring of device slots.  The consumer's
    current stream waits for its batch's ready event; a slot is decoded into again only after the event recorded on the
    consumer's stream when the batch after it was requested.  The copy of chunk c + 1 is issued when chunk c's first
    batch is taken, so it runs beside the decodes of chunk c."""

    SLOTS = 4

    def __init__(self, owner, j0):
        ds = owner.ds
        self.owner, self.ds, self.dev = owner, ds, owner.dev
        self.B = ds.batch_size
        self.j = j0
        self.end = ds.num_entries
        self.bytes_read = 0
        self.thread = None
        if self.j >= self.end:
            return
        dev = self.dev
        self.cb = max(1, CHUNK_BYTES // (RECORD_BYTES * self.B))          # batches per chunk
        self.chunk_recs = self.cb * self.B
        self.first_rec = self.j * self.B
        chunk_bytes = self.chunk_recs * RECORD_BYTES
        self.pins = [torch.empty(chunk_bytes, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
        self.raw = [torch.empty(self.chunk_recs * RECORD_FIELDS, dtype=torch.int32, device=dev) for _ in range(2)]
        if owner._streams is None:
            owner._streams = (_lib.new_stream(dev, priority=-1), _lib.new_stream(dev, priority=-1))
        self.h2d, self.dec = owner._streams
        self.copied = [torch.cuda.Event(), torch.cuda.Event()]      # chunk c on the device (c % 2)
        self.decoded = [None, None]                                 # last decode from raw[c % 2]
        B = self.B
        self.slots = [(torch.empty(B, DENSE, dtype=torch.float32, device=dev),
                       torch.empty(SPARSE * B, dtype=torch.int64, device=dev),
                       torch.empty(B, dtype=torch.float32, device=dev)) for _ in range(self.SLOTS)]
        self.ready = [torch.cuda.Event() for _ in range(self.SLOTS)]
        self.free = [None] * self.SLOTS
        if owner._lso is None:
            owner._lso = _lso(B, dev)
        self.lso_short = None
        self.n_out = 0
        self.prev_slot = None
        self.issued = -1                    # chunks whose copy has been enqueued
        self.chunk_recs_of = {}
        self.free_q, self.filled_q, self.stop = queue.Queue(), queue.Queue(), threading.Event()
        self.free_q.put(None)
        self.free_q.put(None)
        self.thread = threading.Thread(
            target=_reader, name="criteo-bin-reader", daemon=True,
            args=(ds._fd, ds.data_file, self.free_q, self.filled_q, self.stop, self.chunk_recs, self.first_rec,
                  ds.num_samples, self.pins))
        self.thread.start()

    def __iter__(self):
        return self

    def _issue(self, c):
        """Enqueue the host-to-device copy of chunk c (waits for the reader)."""
        item = self.filled_q.get()
        if isinstance(item, BaseException):
            self.close()
            raise item
        cc, k = item
        assert cc == c
        q = c % 2
        nbytes = k * RECORD_BYTES
        if self.decoded[q] is not None:
            self.h2d.wait_event(self.decoded[q])           # every decode of chunk c - 2 has read raw[q]
        with torch.cuda.stream(self.h2d):
            self.raw[q].view(torch.uint8)[:nbytes].copy_(self.pins[q][:nbytes], non_blocking=True)
            self.copied[q].record(self.h2d)
        ev = torch.cuda.Event()
        ev.record(self.h2d)
        self.free_q.put(ev)                                 # the reader may refill pins[q] once the copy has completed
        self.chunk_recs_of[c] = k
        self.bytes_read += nbytes
        self.owner.bytes_read += nbytes
        self.issued = c

    def __next__(self):
        if self.thread is None or self.j >= self.end:
            self.close()
            raise StopIteration
        cur = torch.cuda.current_stream(self.dev)
        if self.prev_slot is not None:                      # the consumer has enqueued its use of the previous batch
            ev = self.free[self.prev_slot] = torch.cuda.Event()
            ev.record(cur)
        rel = self.j * self.B - self.first_rec
        c, r0 = rel // self.chunk_recs, rel % self.chunk_recs
        while self.issued < c:
            self._issue(self.issued + 1)
        n_chunks = -(-(self.ds.num_samples - self.first_rec) // self.chunk_recs)
        if r0 == 0 and c + 1 < n_chunks and self.issued < c + 1:
            self._issue(c + 1)                              # copy ahead: beside the decodes of chunk c
        q = c % 2
        _lo, n = self.ds.records(self.j)
        s = self.n_out % self.SLOTS
        X, I, T = self.slots[s]
        dec = self.dec
        dec.wait_event(self.copied[q])
        if self.free[s] is not None:
            dec.wait_event(self.free[s])
        ids = I[:SPARSE * n].view(SPARSE, n)
        check(lib.cdlrm_criteo_decode(self.dev.index, _vp(self.raw[q].data_ptr() + r0 * RECORD_BYTES), n, DENSE, SPARSE,
                                      self.ds.max_ind_range, _vp(X.data_ptr()), DENSE, _vp(ids.data_ptr()), n,
                                      _vp(T.data_ptr()), _vp(dec.cuda_stream)))
        self.ready[s].record(dec)
        last_of_chunk = r0 + n >= self.chunk_recs_of[c] or self.j + 1 >= self.end
        if last_of_chunk:
            self.decoded[q] = torch.cuda.Event()
            self.decoded[q].record(dec)
        cur.wait_event(self.ready[s])
        self.prev_slot = s
        self.n_out += 1
        self.j += 1
        if n == self.B:
            lso = self.owner._lso
        else:
            if self.lso_short is None or self.lso_short.shape[1] != n:
                self.lso_short = _lso(n, self.dev)
            lso = self.lso_short
        return X[:n], lso, ids, T[:n].view(n, 1)

    def close(self):
        """Stop and join the reader thread; wait for this iterator's copies and decodes."""
        th, self.thread = self.thread, None
        if th is None:
            return
        self.stop.set()
        self.free_q.put(_STOP)
        th.join()
        self.h2d.synchronize()
        self.dec.synchronize()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def numpy_to_binary(input_files, output_file_path, split="train"):
    """data_loader_terabyte.py:238-275: the npz files' ``y``, ``X_int``, ``X_cat`` as int32 records.  ``train``:
    every file, concatenated; ``test`` / ``val``: the first ceil(n / 2) / the remaining rows of one file."""
    def rows(f):
        with np.load(f) as d:
            return np.concatenate([d["y"].reshape(-1, 1), d["X_int"], d["X_cat"]], axis=1).astype(np.int32)

    with open(output_file_path, "wb") as out:
        if split == "train":
            for f in input_files:
                out.write(rows(f).astype("<i4").tobytes())
            return
        if len(input_files) != 1:
            raise ValueError(f"split {split!r} takes one input file, got {len(input_files)}")
        a = rows(input_files[0])
        mid = int(np.ceil(a.shape[0] / 2.0))
        if split == "test":
            a = a[:mid]
        elif split == "val":
            a = a[mid:]
        else:
            raise ValueError(f"unknown split {split!r}")
        out.write(a.astype("<i4").tobytes())


def bin_paths(args):
    """(train file, test file, counts file) of upstream's make_criteo_data_and_loaders, mlperf-bin branch."""
    lstr = args.processed_data_file.split("/")
    d_path = "/".join(lstr[0:-1]) + "/" + lstr[-1].split(".")[0]
    return d_path + "_train.bin", d_path + "_test.bin", args.raw_data_file + "_fea_count.npz"


def table_sizes(args):
    """ln_emb: the counts file's 26 table sizes, each clamped to --max-ind-range when that is > 0."""
    _tr, _te, counts_file = bin_paths(args)
    with np.load(counts_file) as z:
        if "counts" not in z.files or np.asarray(z["counts"]).shape != (SPARSE,):
            raise ValueError(f"{counts_file}: needs 'counts' with {SPARSE} table sizes")
        ln = np.asarray(z["counts"]).astype(np.int64)
    if args.max_ind_range > 0:
        ln = np.minimum(ln, args.max_ind_range)
    return ln


def make_criteo_bin_loaders(args, device):
    """(train_ld, test_ld, cache_ld, ln_emb).  Default: device streams for training and test, and the train dataset as
    cache_ld (its window markers feed the planner).  ``--strict-reference``: host datasets all three."""
    train_file, test_file, counts_file = bin_paths(args)
    tb = args.test_mini_batch_size if getattr(args, "test_mini_batch_size", -1) > 0 else args.mini_batch_size
    train = CriteoBinDataset(train_file, counts_file, args.mini_batch_size, args.max_ind_range)
    test = CriteoBinDataset(test_file, counts_file, tb, args.max_ind_range)
    ln_emb = table_sizes(args)
    if getattr(args, "strict_reference", False):
        cache = CriteoBinDataset(train_file, counts_file, args.mini_batch_size, args.max_ind_range)
        return train, test, cache, ln_emb
    return train.device_batches(device), test.device_batches(device), train, ln_emb
