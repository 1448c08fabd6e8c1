"""CPU checks of the learning-rate schedule (--lr-num-warmup-steps, --lr-decay-start-step, --lr-num-decay-steps):
``lr_policy`` against an upstream-style stateful scheduler, the flags and their refusal, the checkpoint meta data of
runs from before the schedule existed, and the argument checks of the new C entry points."""
import ctypes
import json
import math
import warnings

import numpy as np
import pytest
import torch

import util  # noqa: F401  (puts the repository on sys.path)

CONFIGS = [(0, 0, 0), (0, 0, 5), (1, 3, 4), (4, 4, 3), (5, 9, 0), (5, 9, 6), (100, 300, 1000)]


class _UpstreamPolicy(torch.optim.lr_scheduler.LRScheduler):
    """Upstream DLRM's LRPolicyScheduler (dlrm_s_pytorch.py), restated: stateful, keeps ``last_lr``, stepped after
    every ``optimizer.step()``.  Where upstream reads a ``last_lr`` it never set (it raises there), this returns NaN."""

    def __init__(self, optimizer, num_warmup_steps, decay_start_step, num_decay_steps):
        self.num_warmup_steps = num_warmup_steps
        self.decay_start_step = decay_start_step
        self.decay_end_step = decay_start_step + num_decay_steps
        self.num_decay_steps = num_decay_steps
        super().__init__(optimizer)

    def get_lr(self):
        step_count = self._step_count
        if step_count < self.num_warmup_steps:
            scale = 1.0 - (self.num_warmup_steps - step_count) / self.num_warmup_steps
            lr = [base_lr * scale for base_lr in self.base_lrs]
            self.last_lr = lr
        elif self.decay_start_step <= step_count and step_count < self.decay_end_step:
            decayed_steps = step_count - self.decay_start_step
            scale = ((self.num_decay_steps - decayed_steps) / self.num_decay_steps) ** 2
            min_lr = 0.0000001
            lr = [max(min_lr, base_lr * scale) for base_lr in self.base_lrs]
            self.last_lr = lr
        else:
            if self.num_decay_steps > 0:
                lr = getattr(self, "last_lr", [math.nan] * len(self.base_lrs))
            else:
                lr = self.base_lrs
        return lr


def _upstream_lrs(bases, W, D, N, steps):
    """The learning rate of every param group during steps c = 1..steps, as upstream's training loop sees them."""
    p = [torch.nn.Parameter(torch.zeros(1)) for _ in bases]
    opt = torch.optim.SGD([{"params": [q], "lr": b} for q, b in zip(p, bases)])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sch = _UpstreamPolicy(opt, W, D, N)
        out = []
        for _c in range(1, steps + 1):
            out.append([g["lr"] for g in opt.param_groups])
            opt.step()
            sch.step()
    return np.asarray(out, dtype=np.float64)


@pytest.mark.parametrize("W,D,N", CONFIGS)
def test_lr_policy_equals_upstream_scheduler(W, D, N):
    from cdlrm_b200.main_no_ddp import lr_policy
    bases = [0.1, 0.3, 1.0, 7.0]
    steps = D + N + 50
    want = _upstream_lrs(bases, W, D, N, steps)
    deviations = 0
    for c in range(1, steps + 1):
        for g, b in enumerate(bases):
            got = lr_policy(b, c, W, D, N)
            assert got == float(np.float32(got)), "lr_policy returns fp32 values"
            if math.isnan(want[c - 1, g]):
                # upstream has no value to hold: between warmup and decay with fewer than two warmup steps
                assert W < 2 and W <= c < D and N > 0, (c, W, D, N)
                assert got == float(np.float32(b))
                deviations += 1
                continue
            assert got == float(np.float32(want[c - 1, g])), (b, c, W, D, N, got, want[c - 1, g])
    assert deviations == (len(bases) * (D - max(W, 1)) if (W < 2 and N > 0 and D > 1) else 0)


def test_lr_policy_regions():
    from cdlrm_b200.main_no_ddp import lr_policy
    W, D, N, b = 4, 6, 4, 1.0
    got = [lr_policy(b, c, W, D, N) for c in range(1, 13)]
    f = lambda v: float(np.float32(v))   # noqa: E731
    assert got[:3] == [f(0.25), f(0.5), f(0.75)]                       # warmup c = 1..3
    assert got[3:5] == [f(0.75)] * 2                                    # held at step W - 1 until the decay
    assert got[5:9] == [f(1.0), f(0.5625), f(0.25), f(0.0625)]          # decay c = 6..9
    assert got[9:] == [f(0.0625)] * 3                                   # held at step D + N - 1
    assert lr_policy(1e-9, 7, W, D, N) == f(1e-7)                       # the floor of the decay
    assert lr_policy(0.5, 10 ** 6, 0, 0, 0) == f(0.5)


def test_flags_default_to_zero_and_refuse_decay_before_warmup_end(capsys):
    from cdlrm_b200.main_no_ddp import ProcessArgs, main
    a = ProcessArgs([])
    assert (a.lr_num_warmup_steps, a.lr_decay_start_step, a.lr_num_decay_steps) == (0, 0, 0)
    a = ProcessArgs("--lr-num-warmup-steps 10 --lr-decay-start-step 20 --lr-num-decay-steps 30".split())
    assert (a.lr_num_warmup_steps, a.lr_decay_start_step, a.lr_num_decay_steps) == (10, 20, 30)
    with pytest.raises(SystemExit, match="Learning rate warmup must finish before the decay starts"):
        main("--lr-num-warmup-steps 10 --lr-decay-start-step 9".split())
    with pytest.raises(SystemExit, match="must not be negative"):
        main("--lr-num-decay-steps -1".split())


def _fields(W=0, D=0, N=0):
    return {"format": 1,
            "shapes": {"ln_emb": [3000, 37], "dim": 16, "ways": 4, "num_sets": [53, 37], "aux_rows": 64,
                       "ln_bot": [13, 32, 16], "ln_top": [19, 32, 1]},
            "args": {"seed": 123, "cache_size": 50, "ways": 4, "lookahead": 6, "global_batch": 64, "world_size": 1,
                     "table_agg_op": "mean", "average_on_writeback": False, "learning_rate": 0.1, "lr_embeds": 0.3,
                     "lr_num_warmup_steps": W, "lr_decay_start_step": D, "lr_num_decay_steps": N}}


def test_checkpoint_meta_without_schedule_loads_as_no_schedule():
    from cdlrm_b200.checkpoint import CheckpointMismatch, check_meta
    old = _fields()
    for key in ("lr_num_warmup_steps", "lr_decay_start_step", "lr_num_decay_steps"):
        del old["args"][key]
    old = json.loads(json.dumps(old))
    check_meta(old, _fields())
    with pytest.raises(CheckpointMismatch, match=r"args\.lr_decay_start_step"):
        check_meta(old, _fields(0, 5, 0))
    saved = json.loads(json.dumps(_fields(2, 5, 7)))
    check_meta(saved, _fields(2, 5, 7))
    for i, key in enumerate(("lr_num_warmup_steps", "lr_decay_start_step", "lr_num_decay_steps")):
        want = _fields(*[v + (i == j) for j, v in enumerate((2, 5, 7))])
        with pytest.raises(CheckpointMismatch, match=rf"args\.{key}"):
            check_meta(saved, want)
    other = _fields()
    del other["args"]["lr_embeds"]             # the default covers the schedule fields only
    with pytest.raises(CheckpointMismatch, match=r"args\.lr_embeds"):
        check_meta(other, _fields())


def test_lr_entry_points_refuse_bad_arguments_and_a_missing_device():
    from cdlrm_b200 import _lib
    lib, vp = _lib.lib, ctypes.c_void_p
    fake = vp(4096)
    bad = [(None, 0, 0, 0, 0), (fake, -1, 0, 0, 0), (fake, 0, -1, 0, 0), (fake, 0, 0, -1, 0), (fake, 5, 4, 3, 0),
           (fake, 0, 0, 0, -1), (fake, 0, 2 ** 62, 2 ** 62, 0)]
    for st, W, D, N, c in bad:
        assert lib.cdlrm_lr_set(0, st, 0.1, 0.3, W, D, N, c, None) == -1, (W, D, N, c)
        assert b"bad argument" in lib.cdlrm_last_error()
    assert lib.cdlrm_lr_advance(0, None, None) == -1
    assert lib.cdlrm_embed_bwd_sgd_dlr(None, 0, 1, fake, 4, None, 0, fake, 0, 16, None, None) == -1
    assert lib.cdlrm_mlp_sgd_split_dlr(1, None, None, None, None, None, None, 0, None) == -1
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert lib.cdlrm_lr_set(0, fake, 0.1, 0.3, 2, 5, 7, 0, None) == -2
    assert lib.cdlrm_lr_advance(0, fake, None) == -2
