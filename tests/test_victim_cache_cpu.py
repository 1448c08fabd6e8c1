"""``--evict-victim-cache`` without a GPU: the command-line refusals, the checkpoint field, and the new entry points
(cdlrm_embed_victim_update[_dlr], cdlrm_move_carry_losers) rejecting bad arguments."""
import ctypes

import pytest

import util  # noqa: F401  (puts the repository on sys.path)

BASE = ["--data-generation", "random", "--arch-sparse-feature-size", "16", "--arch-mlp-bot", "13-16",
        "--arch-mlp-top", "8-1", "--arch-embedding-size", "100-20", "--evict-victim-cache"]


@pytest.mark.parametrize("extra", [["--world-size", "2"], ["--world-size", "1", "--strict-reference"]])
def test_cli_refuses_the_flag_outside_the_look_ahead_trainer(extra, capsys):
    from cdlrm_b200 import main_no_ddp as R
    with pytest.raises(SystemExit) as e:
        R.main(BASE + extra)
    assert str(e.value).startswith("ERROR: --evict-victim-cache") and "world-size 1" in str(e.value)


def test_inference_only_ignores_the_flag():
    from cdlrm_b200 import main_no_ddp as R
    args = R.ProcessArgs(BASE + ["--world-size", "1", "--strict-reference", "--inference-only"])
    R._derive_topology(args)          # no refusal for the flag (main refuses --inference-only with the reference path)


def test_checkpoint_field_defaults_to_off():
    from cdlrm_b200 import checkpoint as ck
    expected = {"format": ck.FORMAT, "shapes": {"dim": 16},
                "args": {"world_size": 1, "lr_num_warmup_steps": 0, "evict_victim_cache": False}}
    old = {"format": ck.FORMAT, "shapes": {"dim": 16}, "args": {"world_size": 1}}
    ck.check_meta(old, expected)                                  # written before the field existed: trained without it
    on = dict(expected, args=dict(expected["args"], evict_victim_cache=True))
    with pytest.raises(ck.CheckpointMismatch, match=r"args\.evict_victim_cache"):
        ck.check_meta(old, on)
    with pytest.raises(ck.CheckpointMismatch, match=r"args\.evict_victim_cache"):
        ck.check_meta(on, expected)


def test_entry_points_reject_bad_arguments():
    from cdlrm_b200._lib import lib
    vp = ctypes.c_void_p
    buf = (ctypes.c_int64 * 64)()
    p = vp(ctypes.addressof(buf))
    # no context (none can be created without a device): an error before anything is touched
    assert lib.cdlrm_embed_victim_update(None, 0, 1, p, 8, p, 8, 8, None, 0, p, 8, 8, 0.1, None) != 0
    assert lib.cdlrm_embed_victim_update_dlr(None, 0, 1, p, 8, p, 8, 8, None, 0, p, 8, 8, p, None) != 0
    assert lib.cdlrm_move_carry_losers(None, 0, p, 8, p, None) != 0
    assert b"bad argument" in lib.cdlrm_last_error()
    assert not any(buf)


def test_no_context_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from cdlrm_b200 import _lib
    h = ctypes.c_void_p()
    assert _lib.lib.cdlrm_ctx_create(ctypes.byref(h), 0, 2, 8, 2, 4, _lib.i64_array([100, 20]), 16) != 0
