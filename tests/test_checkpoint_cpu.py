"""CPU checks of the checkpoint support: the meta-data check names the mismatched field, the on-disk layout round
trips and is replaced atomically, and the new entry points fail without a CUDA device."""
import ctypes
import json
import os

import numpy as np
import pytest

import util  # noqa: F401  (puts the repository on sys.path)


def _fields():
    return {"format": 1,
            "shapes": {"ln_emb": [3000, 37], "dim": 16, "ways": 4, "num_sets": [53, 37], "aux_rows": 64,
                       "ln_bot": [13, 32, 16], "ln_top": [19, 32, 1]},
            "args": {"seed": 123, "cache_size": 50, "ways": 4, "lookahead": 6, "global_batch": 64, "world_size": 1,
                     "table_agg_op": "mean", "average_on_writeback": False, "learning_rate": 0.1, "lr_embeds": 0.3}}


@pytest.mark.parametrize("sec,key,value", [("args", "seed", 7), ("args", "cache_size", 60), ("args", "ways", 8),
                                           ("shapes", "dim", 32), ("shapes", "num_sets", [53, 36]),
                                           ("args", "average_on_writeback", True), ("args", "lr_embeds", 0.2)])
def test_meta_mismatch_names_the_field(sec, key, value):
    from cdlrm_b200.checkpoint import CheckpointMismatch, check_meta
    want = _fields()
    check_meta(json.loads(json.dumps(want)), want)        # survives a JSON round trip unchanged
    saved = json.loads(json.dumps(want))
    saved[sec][key] = value
    with pytest.raises(CheckpointMismatch, match=rf"{sec}\.{key}"):
        check_meta(saved, want)


def test_meta_refuses_another_world_size_and_format():
    from cdlrm_b200.checkpoint import CheckpointMismatch, check_meta
    want = _fields()
    saved = json.loads(json.dumps(want))
    saved["args"]["world_size"] = 2
    with pytest.raises(CheckpointMismatch, match=r"args\.world_size.*different world size"):
        check_meta(saved, want)
    saved = dict(_fields(), format=99)
    with pytest.raises(CheckpointMismatch, match="format"):
        check_meta(saved, want)
    saved = _fields()
    del saved["shapes"]["aux_rows"]
    with pytest.raises(CheckpointMismatch, match=r"shapes\.aux_rows"):
        check_meta(saved, want)


def test_files_round_trip_and_replace_atomically(tmp_path):
    from cdlrm_b200.checkpoint import CheckpointMismatch, Reader, Writer, read_meta
    path = str(tmp_path / "ck")
    rng = np.random.default_rng(0)
    a = rng.standard_normal((37, 16)).astype(np.float32)
    t = rng.integers(-1, 3000, (53, 4)).astype(np.int64)
    for gen in (1, 2):
        wr = Writer(path)
        wr.put("a.bin", a * gen)
        wr.put("t.bin", t)
        wr.commit({"format": 1, "gen": gen})
        assert sorted(os.listdir(tmp_path)) == ["ck"]          # no .tmp / .old left behind
    meta = read_meta(path)
    assert meta["gen"] == 2 and meta["files"]["a.bin"] == {"dtype": "<f4", "shape": [37, 16]}
    rd = Reader(path)
    assert np.array_equal(rd.read_into("a.bin", np.empty((37, 16), np.float32)), 2 * a)
    assert np.array_equal(rd.read_into("t.bin", np.empty((53, 4), np.int64)), t)
    with pytest.raises(CheckpointMismatch, match="t.bin"):
        rd.read_into("t.bin", np.empty((53, 4), np.int32))
    with pytest.raises(CheckpointMismatch, match="missing"):
        rd.read_into("b.bin", np.empty(1, np.float32))
    # a replacement interrupted between its two renames leaves the previous checkpoint as <path>.old
    os.rename(path, path + ".old")
    assert read_meta(path)["gen"] == 2


def test_checkpoint_entry_points_fail_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from cdlrm_b200 import _lib
    lib, vp = _lib.lib, ctypes.c_void_p
    h = vp()
    assert lib.cdlrm_rngdev_create(ctypes.byref(h), 0, 123) != 0
    state = np.zeros(625, np.uint32)
    draws = ctypes.c_uint64()
    assert lib.cdlrm_rngdev_get_state(None, vp(state.ctypes.data), ctypes.byref(draws), None) != 0
    assert lib.cdlrm_rngdev_set_state(None, vp(state.ctypes.data), 0, None) != 0
    slots = np.zeros(8, np.int32)
    ids = np.zeros(8, np.int64)
    counts = np.zeros(2, np.int64)
    assert lib.cdlrm_cache_collect_valid(None, 0, 1, vp(slots.ctypes.data), vp(ids.ctypes.data), _lib.i64_array([0, 4]),
                                         vp(counts.ctypes.data), None) != 0
    assert lib.cdlrm_last_error()
    c = vp()
    assert lib.cdlrm_ctx_create(ctypes.byref(c), 0, 2, 8, 2, 4, _lib.i64_array([100, 20]), 16) != 0
