"""The learning-rate schedule on the GPU (--lr-num-warmup-steps / --lr-decay-start-step / --lr-num-decay-steps, and
host-side changes of ``param_groups[0]["lr"]``):

* ``cdlrm_lr_advance`` writes the fp32 values of ``lr_policy`` bit for bit, with step counts past 2^31 and 2^32;
* the device-pointer update variants equal the float ones bit for bit (sparse update with hot duplicate rows on
  dyadic values, so that the order of the atomic adds cannot change a bit; fused dense SGD + hi/lo split);
* a scheduled run replayed from the CUDA graph equals the eager run, and equals a run without schedule flags whose
  param groups are set from ``lr_policy`` before every step; a graph run whose learning rate changes mid-window
  equals the eager run with the same change; save / load inside warmup and inside decay equals the uninterrupted
  run.  Decisions are compared exactly, values at the graph-vs-eager bars of test_gpu_trainer.py (the sparse
  update adds the rows of hot ids with atomics, in no fixed order);
* the switches that bypass the fused updates refuse a schedule and a learning rate changed after the capture;
* ``main`` with the flags trains differently, ``--strict-reference`` steps the optimizers' lr by ``lr_policy``."""
import ctypes
import queue
import threading

import numpy as np
import pytest
import torch

import util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CONFIGS = [(0, 0, 0), (0, 0, 5), (1, 3, 4), (4, 4, 3), (5, 9, 0), (5, 9, 6), (100, 300, 1000)]
# 6 windows of 4 steps: warmup c = 1..5, held c = 6..8, decay c = 9..16, held after the decay c = 17..24
SCHED = (6, 9, 8)


def _vp(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


# ---- kernels -------------------------------------------------------------------------------------------------------

def test_lr_advance_equals_lr_policy():
    from cdlrm_b200 import _lib
    from cdlrm_b200.main_no_ddp import lr_policy
    lib, check = _lib.lib, _lib.check
    st = torch.zeros(ctypes.sizeof(_lib.LrState) // 8, dtype=torch.int64, device=DEV)
    lrs = st.view(torch.float32)[:2]
    bases = (0.1, 0.3)
    runs = [((W, D, N), 0, D + N + 50) for W, D, N in CONFIGS]
    runs += [((2 ** 31, 2 ** 31, 2 ** 32), 2 ** 31 - 4, 8), ((2 ** 31, 2 ** 31, 2 ** 32), 2 ** 32 - 4, 8),
             ((2 ** 31, 2 ** 31, 2 ** 32), 2 ** 31 + 2 ** 32 - 4, 8), ((0, 2 ** 32, 3), 2 ** 32 - 2, 8)]
    for (W, D, N), c0, n in runs:
        check(lib.cdlrm_lr_set(0, _vp(st), bases[0], bases[1], W, D, N, c0, _stream()))
        out = torch.empty(n + 1, 2, dtype=torch.float32, device=DEV)
        out[0].copy_(lrs)
        for i in range(n):
            check(lib.cdlrm_lr_advance(0, _vp(st), _stream()))
            out[i + 1].copy_(lrs)
        got = out.cpu().numpy()
        assert int(st[6]) == c0 + n, "step count"
        for i in range(n + 1):
            want = [lr_policy(b, c0 + i, W, D, N) for b in bases]
            assert [float(x) for x in got[i]] == want, ((W, D, N), c0 + i, got[i], want)


@pytest.mark.parametrize("dim", [128, 16, 6])
def test_sparse_update_device_lr_equals_float_lr(dim):
    """cdlrm_embed_bwd_sgd_dlr == cdlrm_embed_bwd_sgd on a cache with hot duplicate rows (runs that cross the
    warps' ranges take the atomic path).  Rows, gradients and lr are dyadic with few bits, so every sum is exact and
    both equal numpy."""
    from cdlrm_b200 import cache_manager as C
    from cdlrm_b200 import model_no_ddp as M
    ln, B, ways, lr = [5000, 40, 900], 1024, 4, 0.375
    rng = np.random.default_rng(dim)
    ids = np.stack([(rng.zipf(1.2, size=B) * 7919 + k) % n for k, n in enumerate(ln)]).astype(np.int64)
    ids[:, rng.random(B) < 0.3] = 11                   # one very hot id per table
    np.random.seed(1)
    master = M.Embedding_Table_Group(dim, np.asarray(ln))
    for e in master.emb_l:                             # misses are served from master rows
        e.weight.data.copy_(torch.from_numpy(rng.integers(-64, 64, tuple(e.weight.shape)).astype(np.float32) / 64))
    cg = M.Embedding_Table_Cache_Group(dim, np.asarray(ln), 200, B, ways).to(DEV)
    cg._ensure_ctx(master)
    planner = C.WindowPlanner(cg, master, B, rng=C.VictimRng(7), lookahead_tags=True)
    planner.install(planner.plan(win_ids=torch.from_numpy(ids).to(DEV)), write_master=False)
    lS_o = torch.arange(B).reshape(1, -1).repeat(len(ln), 1)
    g = torch.Generator(device=DEV).manual_seed(dim)
    w0 = [torch.randint(-64, 64, tuple(e.weight.shape), device=DEV, generator=g).float() / 64 for e in cg.emb_l]
    G = [torch.randint(-8, 8, (B, dim), device=DEV, generator=g).float() / 64 for _ in ln]
    d_lr = torch.tensor([lr], dtype=torch.float32, device=DEV)
    out = {}
    for name, fused in (("float", lr), ("device", d_lr)):
        with torch.no_grad():
            for e, w in zip(cg.emb_l, w0):
                e.weight.data.copy_(w)
        cg.fused_lr = fused
        ly, slots = cg(lS_o, torch.from_numpy(ids), master, 0)
        torch.cuda.synchronize()
        pre = [e.weight.data.cpu().numpy().copy() for e in cg.emb_l]      # with the misses' rows in the aux region
        sum((y * gk).sum() for y, gk in zip(ly, G)).backward()
        torch.cuda.synchronize()
        out[name] = [e.weight.data.cpu().numpy().copy() for e in cg.emb_l]
    cg.fused_lr = None
    for k in range(len(ln)):
        assert np.array_equal(out["device"][k], out["float"][k]), f"table {k}"
        want = pre[k].copy()
        np.add.at(want, slots[k].cpu().numpy(), -lr * G[k].cpu().numpy())
        assert np.array_equal(out["float"][k], want), f"table {k} against numpy"
    cg.check_device_flags()


def test_dense_update_device_lr_equals_float_lr():
    """cdlrm_mlp_sgd_split_dlr == cdlrm_mlp_sgd_split: weights, biases and the hi / lo operand splits (the MLP
    workspaces, which hold them) bit for bit."""
    from cdlrm_b200 import model_no_ddp as M
    np.random.seed(17)
    net = M.DLRM_Net(np.asarray([13, 512, 256, 128]), np.asarray([479, 512, 256, 1]), arch_interaction_op="dot",
                     sigmoid_bot=-1, sigmoid_top=2).to(DEV)
    net.flatten_parameters()
    g = torch.Generator(device=DEV).manual_seed(3)
    B = 2048
    X = torch.randn(B, 13, device=DEV, generator=g)
    ly = [torch.randn(B, 128, device=DEV, generator=g) * 0.05 for _ in range(26)]
    Y = (torch.rand(B, 1, device=DEV, generator=g) < 0.25).float()
    torch.nn.functional.binary_cross_entropy(net(X, ly), Y).backward()
    net.join_mlp_grads()
    torch.cuda.synchronize()
    p0 = net.flat_params.clone()
    sts = [net._mlp_state["bot"], net._mlp_state["top"]]
    out = {}
    for name, lr in (("float", 0.0625 * 1.7), ("device", torch.tensor([0.0625 * 1.7], device=DEV))):
        with torch.no_grad():
            net.flat_params.copy_(p0)
        net.flat_sgd_step(lr)
        torch.cuda.synchronize()
        out[name] = [net.flat_params.cpu().numpy().copy()] + [st.ws.cpu().numpy().copy() for st in sts]
    assert not np.array_equal(out["float"][0], p0.cpu().numpy())
    for what, a, b in zip(("parameters", "bottom workspace", "top workspace"), out["device"], out["float"]):
        assert np.array_equal(a, b), what


# ---- the trainer ---------------------------------------------------------------------------------------------------

def _setup():
    cfg = dict(ln_emb=[3000, 37, 800, 5, 12000], dim=16, cache_size=20, num_ways=2, batch=64, lookahead=4,
               n_windows=6, lr_embeds=0.3, lr_mlp=0.1, seed=5, data_seed=41, dist="zipf", zipf_a=1.05)
    rng = np.random.default_rng(7)
    n = cfg["n_windows"] * cfg["lookahead"]
    X = rng.standard_normal((n, cfg["batch"], 13)).astype(np.float32)
    Y = (rng.random((n, cfg["batch"], 1)) < 0.3).astype(np.float32)
    return dict(cfg=cfg, ids=util.make_ids(cfg), X=X, Y=Y, ln_bot=np.asarray([13, 32, 16]),
                ln_top=np.asarray([31, 32, 1]))


def _args(cfg, sched=(0, 0, 0), extra=()):
    from cdlrm_b200 import main_no_ddp as R
    W, D, N = sched
    return R.ProcessArgs(["--arch-sparse-feature-size", str(cfg["dim"]), "--loss-function", "bce", "--learning-rate",
                          str(cfg["lr_mlp"]), "--lr-embeds", str(cfg["lr_embeds"]), "--mini-batch-size",
                          str(cfg["batch"]), "--lookahead", str(cfg["lookahead"]), "--cache-size",
                          str(cfg["cache_size"]), "--num-ways", str(cfg["num_ways"]), "--numpy-rand-seed",
                          str(cfg["seed"]), "--world-size", "1", "--lr-num-warmup-steps", str(W),
                          "--lr-decay-start-step", str(D), "--lr-num-decay-steps", str(N)] + list(extra))


def _build(s, sched=(0, 0, 0)):
    from cdlrm_b200 import main_no_ddp as R
    from cdlrm_b200 import model_no_ddp as M
    cfg = s["cfg"]
    np.random.seed(cfg["seed"])
    torch.manual_seed(cfg["seed"])
    master = M.Embedding_Table_Group(cfg["dim"], np.asarray(cfg["ln_emb"]))
    tr = R.Trainer(_args(cfg, sched), cfg["dim"], np.asarray(cfg["ln_emb"]), s["ln_bot"], s["ln_top"], master, rank=0,
                   world=1, device=torch.device(DEV))
    return tr, master


def _train(s, use_graph, sched=(0, 0, 0), before_step=None, w_end=None, load=None, save_at=None, path=None):
    """Windows [w0, w_end) as test_gpu_checkpoint.py drives them; ``before_step(tr, c)`` runs before step c (1-based).
    Returns decisions, per-step losses and learning rates, and the final state."""
    cfg = s["cfg"]
    B, L, nw, T = cfg["batch"], cfg["lookahead"], cfg["n_windows"], len(cfg["ln_emb"])
    w_end = nw if w_end is None else w_end
    tr, master = _build(s, sched)
    w0 = tr.load_checkpoint(load) if load else 0
    lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
    X, Y = torch.from_numpy(s["X"]).to(DEV), torch.from_numpy(s["Y"]).to(DEV)
    win = lambda w: torch.from_numpy(s["ids"][:, w * L * B:(w + 1) * L * B]).to(DEV)   # noqa: E731
    out = dict(w0=w0, tags=[], E=[], F=[], losses=[], lrs=[])
    tr.submit_window(win(w0))
    local = 0
    for w in range(w0, w_end):
        if save_at == w:
            tr.save_checkpoint(path)
        rec = tr.install_window()
        if w + 1 < nw:
            tr.submit_window(win(w + 1))
        torch.cuda.synchronize()
        out["tags"].append(np.concatenate([t.cpu().numpy().ravel() for t in tr.cache_group.occupancy_tables]))
        out["E"].append(list(rec.E))
        out["F"].append(list(rec.F))
        cur = win(w)
        for b in range(L):
            step = w * L + b
            if use_graph and getattr(tr, "_graph", None) is None and local == 1:
                tr.capture_graph(X[step], lS_o, cur[:, b * B:(b + 1) * B], Y[step])
            if before_step is not None:
                before_step(tr, step + 1)
            E, _Z = tr.step(X[step], lS_o, cur[:, b * B:(b + 1) * B], Y[step])
            out["losses"].append(E.detach().clone())
            out["lrs"].append(tr.current_lr())
            local += 1
    if save_at == w_end:
        tr.save_checkpoint(path)
    torch.cuda.synchronize()
    tr.finish()
    out["losses"] = np.asarray([float(x) for x in out["losses"]], dtype=np.float64)
    out["dense"] = torch.cat([p.detach().reshape(-1) for p in tr.dlrm.parameters()]).cpu().numpy()
    out["weights"] = [e.weight.data[:cfg["num_ways"] * S].cpu().numpy() for e, S in
                      zip(tr.cache_group.emb_l, tr.cache_group.cache_sizes)]
    out["master"] = [e.weight.data.numpy().copy() for e in master.emb_l]
    if tr._lr_state is not None:
        out["device_lr"] = tuple(float(x) for x in tr._lr_state.view(torch.float32)[:2].cpu())
    out["tr"] = tr
    return out


def _assert_same_run(a, b, tag):
    assert len(a["tags"]) == len(b["tags"])
    for w, (ta, tb) in enumerate(zip(a["tags"], b["tags"])):
        assert np.array_equal(ta, tb), f"{tag}: tags after window {w} differ"
    assert a["E"] == b["E"] and a["F"] == b["F"], f"{tag}: eviction / fill list lengths differ"
    assert a["lrs"] == b["lrs"], f"{tag}: learning rates differ"
    np.testing.assert_allclose(a["losses"], b["losses"], rtol=1e-6, err_msg=f"{tag}: losses")
    np.testing.assert_allclose(a["dense"], b["dense"], rtol=0, atol=1e-6, err_msg=f"{tag}: dense parameters")
    for name in ("weights", "master"):
        for x, y in zip(a[name], b[name]):
            np.testing.assert_allclose(x, y, rtol=0, atol=1e-6, err_msg=f"{tag}: {name}")


def _policy_lrs(s, sched, steps):
    from cdlrm_b200.main_no_ddp import lr_policy
    cfg = s["cfg"]
    return [(lr_policy(cfg["lr_mlp"], c, *sched), lr_policy(cfg["lr_embeds"], c, *sched)) for c in range(1, steps + 1)]


def test_scheduled_graph_run_equals_eager_and_host_driven_runs():
    s = _setup()
    n = s["cfg"]["n_windows"] * s["cfg"]["lookahead"]
    g = _train(s, True, SCHED)
    e = _train(s, False, SCHED)
    want = _policy_lrs(s, SCHED, n)
    assert g["lrs"] == want and g["device_lr"] == want[-1]
    _assert_same_run(g, e, "schedule: graph vs eager")

    def host(tr, c):       # no schedule flags: the bases follow lr_policy, written by cdlrm_lr_set before the replay
        tr.optimizer_mlps.param_groups[0]["lr"], tr.optimizer_embeds.param_groups[0]["lr"] = want[c - 1]
    h = _train(s, True, before_step=host)
    assert h["lrs"] == want and h["device_lr"] == want[-1]
    _assert_same_run(g, h, "schedule vs host-set learning rates")
    plain = _train(s, True)
    assert np.abs(plain["losses"] - g["losses"]).max() > 1e-3, "the schedule changed nothing"


@pytest.mark.parametrize("sched", [(0, 0, 0), SCHED])
def test_learning_rate_changed_mid_window_takes_effect_in_the_graph(sched):
    s = _setup()

    def change(tr, c):
        if c in (6, 15):        # inside windows 1 and 3
            for opt in (tr.optimizer_mlps, tr.optimizer_embeds):
                opt.param_groups[0]["lr"] *= 0.25 if c == 6 else 3.0
    g = _train(s, True, sched, before_step=change)
    e = _train(s, False, sched, before_step=change)
    _assert_same_run(g, e, f"lr changed at steps 6 and 15, schedule {sched}")
    plain = _train(s, True, sched)
    assert np.abs(plain["losses"][6:] - g["losses"][6:]).max() > 1e-3, "the change was ignored"
    if sched == (0, 0, 0):
        assert g["lrs"][5] == (np.float32(0.1 * 0.25), np.float32(0.3 * 0.25))


@pytest.mark.parametrize("save_at", [1, 3])      # the boundary after step 4 (warmup) / after step 12 (decay)
def test_resume_inside_the_schedule_equals_uninterrupted_run(save_at, tmp_path):
    s = _setup()
    path = str(tmp_path / "ck")
    a = _train(s, True, SCHED)
    b1 = _train(s, True, SCHED, w_end=save_at, save_at=save_at, path=path)
    b2 = _train(s, True, SCHED, load=path)
    L = s["cfg"]["lookahead"]
    assert b2["w0"] == save_at and b2["tr"].global_step == s["cfg"]["n_windows"] * L
    joined = dict(b2)
    for key in ("tags", "E", "F", "lrs"):
        joined[key] = b1[key] + b2[key]
    joined["losses"] = np.concatenate([b1["losses"], b2["losses"]])
    _assert_same_run(a, joined, f"resume at window {save_at}")
    from cdlrm_b200.checkpoint import CheckpointMismatch
    tr, _m = _build(s)
    with pytest.raises(CheckpointMismatch, match=r"args\.lr_num_warmup_steps"):
        tr.load_checkpoint(path)
    tr.finish()


@pytest.mark.parametrize("switch", [("CDLRM_MLP", "torch"), ("CDLRM_FLAT_MLP", "0"), ("CDLRM_SGD_SPLIT", "0"),
                                    ("CDLRM_OVERLAP_UPDATE", "0")])
def test_bypass_switches_refuse_what_they_cannot_follow(switch, monkeypatch):
    from cdlrm_b200._lib import CdlrmError
    monkeypatch.setenv(*switch)
    s = _setup()
    with pytest.raises(CdlrmError, match="lr-num-warmup-steps"):
        _build(s, SCHED)

    def change(tr, c):
        if c == 5:
            tr.optimizer_mlps.param_groups[0]["lr"] = 0.05
    e = _train(s, False, before_step=change)     # eager steps read the host floats: a change takes effect
    assert e["lrs"][3][0] == np.float32(0.1) and e["lrs"][4][0] == np.float32(0.05)
    cfg = s["cfg"]
    B, L, T = cfg["batch"], cfg["lookahead"], len(cfg["ln_emb"])
    tr, _m = _build(s)
    ids = torch.from_numpy(s["ids"][:, :L * B]).to(DEV)
    X, Y = torch.from_numpy(s["X"]).to(DEV), torch.from_numpy(s["Y"]).to(DEV)
    lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
    tr.submit_window(ids)
    tr.install_window()
    tr.step(X[0], lS_o, ids[:, :B], Y[0])
    tr.capture_graph(X[1], lS_o, ids[:, B:2 * B], Y[1])
    tr.step(X[1], lS_o, ids[:, B:2 * B], Y[1])
    tr.optimizer_embeds.param_groups[0]["lr"] = 0.5
    with pytest.raises(CdlrmError, match="captured"):
        tr.step(X[2], lS_o, ids[:, 2 * B:3 * B], Y[2])
    tr.finish()


# ---- main / Run ----------------------------------------------------------------------------------------------------

def _losses(out):
    return [float(line.split("Loss = ")[1].split(",")[0]) for line in out.splitlines() if "Loss = " in line]


def test_main_with_schedule_trains_differently(capsys):
    from cdlrm_b200 import main_no_ddp as R
    base = ["--data-generation", "synthetic", "--arch-embedding-size", "3000-37-800-5-12000",
            "--arch-sparse-feature-size", "16", "--arch-mlp-bot", "13-32-16", "--arch-mlp-top", "32-1",
            "--loss-function", "bce", "--mini-batch-size", "64", "--num-batches", "20", "--lookahead", "6",
            "--cache-size", "50", "--num-ways", "4", "--world-size", "1", "--print-freq", "5", "--nepochs", "2",
            "--learning-rate", "0.1", "--lr-embeds", "0.3", "--test-mini-batch-size", "32",
            "--eviction-fifo-timeout", "2"]
    R.main(base)
    plain = _losses(capsys.readouterr().out)
    tr = R.main(base + ["--lr-num-warmup-steps", "8", "--lr-decay-start-step", "20", "--lr-num-decay-steps", "15"])
    sched = _losses(capsys.readouterr().out)
    assert len(plain) == len(sched) == 6
    assert tr.global_step == 40 and tr.current_lr() == (R.lr_policy(0.1, 40, 8, 20, 15), R.lr_policy(0.3, 40, 8, 20, 15))
    assert max(abs(a - b) for a, b in zip(plain, sched)) > 1e-4, (plain, sched)


def test_strict_reference_steps_the_optimizers_by_lr_policy():
    from cdlrm_b200 import cache_manager as C
    from cdlrm_b200 import main_no_ddp as R
    from cdlrm_b200 import model_no_ddp as M
    g = util.load_golden("run_strict.npz")
    cfg = util.golden_cfg(g)
    sched = (3, 5, 6)
    args = R.ProcessArgs(["--arch-sparse-feature-size", str(cfg["dim"]), "--loss-function", "bce", "--learning-rate",
                          str(cfg["lr_mlp"]), "--lr-embeds", str(cfg["lr_embeds"]), "--mini-batch-size",
                          str(cfg["batch"]), "--lookahead", str(cfg["lookahead"]), "--cache-size",
                          str(cfg["cache_size"]), "--num-ways", str(cfg["num_ways"]), "--numpy-rand-seed",
                          str(cfg["seed"]), "--world-size", "1", "--nepochs", "1", "--print-freq", "7",
                          "--eviction-fifo-timeout", "2", "--strict-reference", "--lr-num-warmup-steps", "3",
                          "--lr-decay-start-step", "5", "--lr-num-decay-steps", "6"])
    np.random.seed(cfg["seed"])
    torch.manual_seed(cfg["seed"])
    master = M.Embedding_Table_Group(cfg["dim"], np.asarray(cfg["ln_emb"]))
    ids = util.make_ids(cfg)
    B, T = cfg["batch"], len(cfg["ln_emb"])
    lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
    n = cfg["n_windows"] * cfg["lookahead"]
    loader = [(torch.from_numpy(g["X"][i]), lS_o, torch.from_numpy(ids[:, i * B:(i + 1) * B]),
               torch.from_numpy(g["Y"][i])) for i in range(n)]
    seen = []
    orig = R.Trainer.step_reference

    def spy(self, *a):
        seen.append((self.optimizer_mlps.param_groups[0]["lr"], self.optimizer_embeds.param_groups[0]["lr"]))
        return orig(self, *a)
    batch_fifo, evq, fin = queue.Queue(maxsize=args.batch_fifo_size), queue.Queue(), threading.Event()
    cm = C.Prefetcher(args, master, batch_fifo, evq, fin, loader)
    cm.start()
    R.Trainer.step_reference = spy
    try:
        tr = R.Run(0, cfg["dim"], np.asarray(cfg["ln_emb"]), g["ln_bot"], g["ln_top"], loader, None, batch_fifo, evq,
                   [], master, args)
    finally:
        R.Trainer.step_reference = orig
        fin.set()
    cm.join(timeout=10)
    assert len(seen) == n
    assert seen == [(R.lr_policy(cfg["lr_mlp"], c, *sched), R.lr_policy(cfg["lr_embeds"], c, *sched))
                    for c in range(1, n + 1)]
    for e in tr.cache_group.emb_l:
        assert torch.isfinite(e.weight.data).all()
