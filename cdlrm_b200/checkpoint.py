"""On-disk layout of a training checkpoint (``Trainer.save_checkpoint`` / ``load_checkpoint``, ``--save-model`` /
``--load-model``).  No reference counterpart: the reference parses those flags and ignores them.

A checkpoint is a directory::

    meta.json            format, shapes, the arguments that decide the plan and the values, the resume point
                         (epoch, window w, global step), the victim-stream state as of the start of plan(w), and the
                         dtype / shape of every file below
    dense.bin            float32: the flat dense parameter buffer
    tags_<k>.bin         int64 [num_sets_k, ways]: live tags of table k
    cache_<k>.bin        float32 [ways * num_sets_k, dim]: cache rows of table k (the aux rows are scratch)
    master_<k>.bin       float32 [n_k, dim]: master table k

The files are raw little-endian arrays.  They are written into ``<path>.tmp`` and the directory is renamed into
place, so a crash never leaves half a checkpoint behind ``<path>``; a crash between the two renames of a replacement
leaves the previous checkpoint as ``<path>.old``, which ``resolve`` falls back to."""
import json
import os
import shutil
import time

import numpy as np

FORMAT = 1
META = "meta.json"
_CHUNK = 1 << 30          # bytes per read / write call


class CheckpointMismatch(ValueError):
    """A checkpoint that does not fit the Trainer it is loaded into; the message names the field."""


def resolve(path):
    """The directory to read for ``path``: ``path`` itself, or ``path.old`` when a replacement was interrupted."""
    if not os.path.isdir(path) and os.path.isdir(path + ".old"):
        return path + ".old"
    return path


def read_meta(path):
    with open(os.path.join(resolve(path), META)) as f:
        return json.load(f)


def check_meta(saved, expected):
    """Raise ``CheckpointMismatch`` naming the first field of ``expected`` ("format", "shapes.*", "args.*") that the
    saved meta data does not hold with the same value."""
    if saved.get("format") != expected["format"]:
        raise CheckpointMismatch("checkpoint field format: saved %r, this trainer reads %r"
                                 % (saved.get("format"), expected["format"]))
    ws, we = saved.get("args", {}).get("world_size"), expected["args"]["world_size"]
    if ws != we:
        raise CheckpointMismatch("checkpoint field args.world_size: saved at world size %r, loading at %r "
                                 "(resuming at a different world size is not supported)" % (ws, we))
    for sec in ("shapes", "args"):
        for key, want in expected[sec].items():
            got = saved.get(sec, {}).get(key, "<missing>")
            if got != want:
                raise CheckpointMismatch("checkpoint field %s.%s: saved %r, this trainer has %r" % (sec, key, got, want))


def _bytes(arr):
    a = np.asarray(arr)
    if not a.flags.c_contiguous:
        raise ValueError("checkpoint arrays must be contiguous")
    return memoryview(a.reshape(-1).view(np.uint8))


class Writer:
    """Files of one checkpoint, written into ``<path>.tmp``; ``commit`` adds meta.json and renames the directory
    into place.  ``io_s``: seconds spent in file I/O (writes and fsyncs)."""

    def __init__(self, path):
        self.path = os.path.abspath(path)
        self.tmp = self.path + ".tmp"
        if os.path.isdir(self.tmp):
            shutil.rmtree(self.tmp)
        os.makedirs(self.tmp)
        self.files = {}
        self.io_s = 0.0

    def put(self, name, arr):
        t0 = time.perf_counter()
        a = np.asarray(arr)
        mv = _bytes(a)
        with open(os.path.join(self.tmp, name), "wb") as f:
            for o in range(0, len(mv), _CHUNK):
                f.write(mv[o:o + _CHUNK])
            f.flush()
            os.fsync(f.fileno())
        self.files[name] = {"dtype": a.dtype.str, "shape": list(a.shape)}
        self.io_s += time.perf_counter() - t0

    def commit(self, meta):
        t0 = time.perf_counter()
        meta = dict(meta, files=self.files)
        with open(os.path.join(self.tmp, META), "w") as f:
            json.dump(meta, f, indent=1)
            f.flush()
            os.fsync(f.fileno())
        old = self.path + ".old"
        if os.path.isdir(old):
            shutil.rmtree(old)
        if os.path.isdir(self.path):
            os.rename(self.path, old)
        os.rename(self.tmp, self.path)
        parent = os.open(os.path.dirname(self.path), os.O_RDONLY)
        try:
            os.fsync(parent)
        finally:
            os.close(parent)
        shutil.rmtree(old, ignore_errors=True)
        self.io_s += time.perf_counter() - t0


class Reader:
    """Reads the files of a checkpoint straight into caller-owned arrays.  ``io_s``: seconds of file I/O."""

    def __init__(self, path, meta=None):
        self.path = resolve(path)
        self.meta = meta if meta is not None else read_meta(path)
        self.io_s = 0.0

    def read_into(self, name, out):
        ent = self.meta["files"].get(name)
        if ent is None:
            raise CheckpointMismatch("checkpoint file %s is missing" % name)
        out = np.asarray(out)
        if np.dtype(ent["dtype"]) != out.dtype or list(ent["shape"]) != list(out.shape):
            raise CheckpointMismatch("checkpoint file %s: saved %s %s, this trainer has %s %s"
                                     % (name, ent["dtype"], ent["shape"], out.dtype.str, list(out.shape)))
        t0 = time.perf_counter()
        mv = _bytes(out)
        with open(os.path.join(self.path, name), "rb") as f:
            o = 0
            while o < len(mv):
                n = f.readinto(mv[o:o + _CHUNK])
                if not n:
                    raise CheckpointMismatch("checkpoint file %s is truncated" % name)
                o += n
        self.io_s += time.perf_counter() - t0
        return out
