"""CPU-only checks of the evaluation entry points: they fail without a device, and ``--inference-only`` refuses the
configurations it does not support before anything is spawned."""
import ctypes

import pytest


def test_eval_entry_points_fail_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from cdlrm_b200 import _lib
    from cdlrm_b200._lib import lib
    h = ctypes.c_void_p()
    assert lib.cdlrm_eval_create(ctypes.byref(h), 0, 1000) != 0 and lib.cdlrm_last_error() != b""
    assert not h.value
    assert lib.cdlrm_embed_fwd_eval(None, 0, 1, None, 0, 4, None, 0, None) != 0
    assert lib.cdlrm_eval_accumulate(None, None, 1, None, 1, 4, None) != 0
    assert lib.cdlrm_eval_result(None, ctypes.addressof(_lib.EvalStats()), None) != 0


def test_eval_create_rejects_bad_capacity():
    from cdlrm_b200._lib import lib
    h = ctypes.c_void_p()
    assert lib.cdlrm_eval_create(ctypes.byref(h), 0, 0) != 0
    assert lib.cdlrm_eval_create(ctypes.byref(h), 0, (1 << 30) + 1) != 0
    assert not h.value


@pytest.mark.parametrize("extra", [["--world-size", "2"], ["--world-size", "1", "--strict-reference"]])
def test_inference_only_refuses_multi_rank_and_strict(extra):
    from cdlrm_b200 import main_no_ddp as R
    with pytest.raises(SystemExit) as e:
        R.main(["--inference-only"] + extra)
    assert "inference-only" in str(e.value)
