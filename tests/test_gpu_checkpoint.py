"""Export, checkpoint and resume of the look-ahead ``Trainer`` on the GPU.

* ``sync_master`` after ``finish`` writes every cached row into the master: against tests/golden/dlrm_trainer.npz
  (the reference's final master with its final cache rows written at the ids of its last tags), in both PCIe modes;
* a run that saves at a window boundary, is rebuilt from scratch (new Trainer, new master object) and loads, equals
  the uninterrupted run: decisions bit for bit, values to the graph-vs-eager bars of test_gpu_trainer.py;
* saving and ``sync_master`` mid-run change nothing that follows;
* cdlrm_cache_collect_valid against numpy, the victim-stream state round trip, the refusals, and ``Run`` with
  ``--save-model`` / ``--load-model``."""
import json
import os
import queue
import shutil
import subprocess
import sys
import threading

import numpy as np
import pytest
import torch

import util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _setup(kind):
    """Configuration, ids and dense inputs: the trainer golden, or an undersized cache with many evictions."""
    if kind == "golden":
        g = util.load_golden("dlrm_trainer.npz")
        cfg = util.golden_cfg(g)
        return dict(cfg=cfg, ids=util.make_ids(cfg), X=g["X"], Y=g["Y"], ln_bot=g["ln_bot"], ln_top=g["ln_top"],
                    extra=[], golden=g)
    cfg = dict(ln_emb=[3000, 37, 800, 5, 12000], dim=16, cache_size=20, num_ways=2, batch=64, lookahead=4,
               n_windows=6, lr_embeds=0.3, lr_mlp=0.1, seed=5, data_seed=41, dist="zipf", zipf_a=1.05)
    rng = np.random.default_rng(7)
    n = cfg["n_windows"] * cfg["lookahead"]
    X = rng.standard_normal((n, cfg["batch"], 13)).astype(np.float32)
    Y = (rng.random((n, cfg["batch"], 1)) < 0.3).astype(np.float32)
    return dict(cfg=cfg, ids=util.make_ids(cfg), X=X, Y=Y, ln_bot=np.asarray([13, 32, 16]),
                ln_top=np.asarray([31, 32, 1]), extra=["--average-on-writeback"] if kind == "avgwb" else [])


def _args(cfg, extra=()):
    from cdlrm_b200 import main_no_ddp as R
    return R.ProcessArgs(["--arch-sparse-feature-size", str(cfg["dim"]), "--loss-function", "bce", "--learning-rate",
                          str(cfg["lr_mlp"]), "--lr-embeds", str(cfg["lr_embeds"]), "--mini-batch-size",
                          str(cfg["batch"]), "--lookahead", str(cfg["lookahead"]), "--cache-size",
                          str(cfg["cache_size"]), "--num-ways", str(cfg["num_ways"]), "--numpy-rand-seed",
                          str(cfg["seed"]), "--world-size", "1"] + list(extra))


def _build(s, extra=()):
    from cdlrm_b200 import main_no_ddp as R
    from cdlrm_b200 import model_no_ddp as M
    cfg = s["cfg"]
    np.random.seed(cfg["seed"])
    torch.manual_seed(cfg["seed"])
    master = M.Embedding_Table_Group(cfg["dim"], np.asarray(cfg["ln_emb"]))
    tr = R.Trainer(_args(cfg, list(s["extra"]) + list(extra)), cfg["dim"], np.asarray(cfg["ln_emb"]), s["ln_bot"],
                   s["ln_top"], master, rank=0, world=1, device=torch.device(DEV))
    return tr, master


def _train(s, use_graph, w_end=None, load=None, save_at=None, path=None, sync_at=None):
    """Windows [w0, w_end) through the Trainer as test_gpu_trainer.py drives it.  ``load``: resume from that
    checkpoint first (w0 = its window).  ``save_at`` / ``sync_at``: save to ``path`` / sync_master at the boundary
    before that window.  Returns per-window decisions, per-step values and the final state."""
    cfg = s["cfg"]
    B, L, nw, T = cfg["batch"], cfg["lookahead"], cfg["n_windows"], len(cfg["ln_emb"])
    w_end = nw if w_end is None else w_end
    tr, master = _build(s)
    w0 = tr.load_checkpoint(load) if load else 0
    lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
    X, Y = torch.from_numpy(s["X"]).to(DEV), torch.from_numpy(s["Y"]).to(DEV)
    win = lambda w: torch.from_numpy(s["ids"][:, w * L * B:(w + 1) * L * B]).to(DEV)   # noqa: E731
    out = dict(w0=w0, tags=[], E=[], F=[], losses=[], n_miss=[])
    tr.submit_window(win(w0))
    local = 0
    for w in range(w0, w_end):
        if save_at == w:
            tr.save_checkpoint(path)
        if sync_at == w:
            tr.sync_master()
        rec = tr.install_window()
        if w + 1 < nw:
            tr.submit_window(win(w + 1))       # left in flight when the caller stops at w_end
        torch.cuda.synchronize()
        out["tags"].append(np.concatenate([t.cpu().numpy().ravel() for t in tr.cache_group.occupancy_tables]))
        out["E"].append(list(rec.E))
        out["F"].append(list(rec.F))
        cur = win(w)
        for b in range(L):
            step = w * L + b
            if use_graph and getattr(tr, "_graph", None) is None and local == 1:
                tr.capture_graph(X[step], lS_o, cur[:, b * B:(b + 1) * B], Y[step])
            E, _Z = tr.step(X[step], lS_o, cur[:, b * B:(b + 1) * B], Y[step])
            out["losses"].append(E.detach().clone())
            out["n_miss"].append(tr.cache_group.last_n_miss.clone())
            local += 1
    if save_at == w_end:
        tr.save_checkpoint(path)
    torch.cuda.synchronize()
    tr.finish()
    out["losses"] = np.asarray([float(x) for x in out["losses"]], dtype=np.float64)
    out["n_miss"] = torch.stack(out["n_miss"]).cpu().numpy() if out["n_miss"] else np.zeros((0, T), np.int32)
    out["params"] = [p.detach().cpu().numpy().copy() for p in tr.dlrm.parameters()]
    out["weights"] = [e.weight.data[:cfg["num_ways"] * S].cpu().numpy() for e, S in
                      zip(tr.cache_group.emb_l, tr.cache_group.cache_sizes)]
    out["master"] = [e.weight.data.numpy().copy() for e in master.emb_l]
    out["draws"] = tr.planner.rng.draws
    out["rng_state"] = tr.planner.rng.get_state()[0]
    out["tr"], out["emb"] = tr, master
    return out


def _assert_same_run(a, b, tag):
    assert len(a["tags"]) == len(b["tags"])
    for w, (ta, tb) in enumerate(zip(a["tags"], b["tags"])):
        assert np.array_equal(ta, tb), f"{tag}: tags after window {w} differ"
    assert a["E"] == b["E"] and a["F"] == b["F"], f"{tag}: eviction / fill list lengths differ"
    assert np.array_equal(a["n_miss"], b["n_miss"]), f"{tag}: miss counts differ"
    assert a["draws"] == b["draws"] and np.array_equal(a["rng_state"], b["rng_state"]), f"{tag}: victim stream differs"
    np.testing.assert_allclose(a["losses"], b["losses"], rtol=1e-6, err_msg=f"{tag}: losses")
    for name in ("params", "weights", "master"):
        for x, y in zip(a[name], b[name]):
            np.testing.assert_allclose(x, y, rtol=0, atol=1e-6, err_msg=f"{tag}: {name}")


def _join(p1, p2):
    """Run B = its first part (windows < k) followed by the resumed part."""
    out = dict(p2)
    for key in ("tags", "E", "F"):
        out[key] = p1[key] + p2[key]
    out["losses"] = np.concatenate([p1["losses"], p2["losses"]])
    out["n_miss"] = np.concatenate([p1["n_miss"], p2["n_miss"]])
    return out


@pytest.mark.parametrize("mode", ["sm", "ce"])
def test_sync_master_exports_trained_tables(mode):
    s = _setup("golden")
    g, cfg = s["golden"], s["cfg"]
    a = _train(s, use_graph=True)
    tr, master = a["tr"], a["emb"]
    before = [m.copy() for m in a["master"]]
    tr.planner.pcie_mode = mode
    n = tr.sync_master()
    last = g[f"w{cfg['n_windows'] - 1}_tags"]
    o = 0
    total = 0
    for k, nk in enumerate(cfg["ln_emb"]):
        S = tr.cache_group.cache_sizes[k]
        ways = cfg["num_ways"]
        tags = last[o:o + S * ways].reshape(S, ways)
        o += S * ways
        want = g[f"final_master_{k}"].copy()
        sets, wys = np.nonzero(tags >= 0)
        want[tags[sets, wys]] = g[f"final_weight_{k}"][wys * S + sets]
        total += len(sets)
        got = master.emb_l[k].weight.data.numpy()
        util.assert_close_fp32(got, want, err_msg=f"exported table {k}")
        uncached = np.setdiff1d(np.arange(nk), tags[sets, wys])
        assert np.array_equal(got[uncached], before[k][uncached]), f"table {k}: un-cached rows changed"
    assert n == total


@pytest.mark.parametrize("use_graph", [True, False])
@pytest.mark.parametrize("kind", ["golden", "evict", "avgwb"])
def test_resume_equals_uninterrupted_run(kind, use_graph, tmp_path):
    s = _setup(kind)
    k = s["cfg"]["n_windows"] // 2
    path = str(tmp_path / "ck")
    a = _train(s, use_graph)
    if kind != "golden":
        assert sum(sum(e) for e in a["E"]) > 0, "the undersized cache must evict"
    b1 = _train(s, use_graph, w_end=k, save_at=k, path=path)
    del b1["tr"]
    b2 = _train(s, use_graph, load=path)
    assert b2["w0"] == k and b2["tr"].global_step == s["cfg"]["n_windows"] * s["cfg"]["lookahead"]
    _assert_same_run(a, _join(b1, b2), f"{kind} graph={use_graph}")


def test_save_and_sync_do_not_perturb(tmp_path):
    s = _setup("evict")
    a = _train(s, True)
    c = _train(s, True, save_at=2, sync_at=4, path=str(tmp_path / "ck"))
    # the master rows of ids still cached at the end differ by design (the mid-run sync wrote them): compare the
    # exported tables, which is what the master is read for
    for r in (a, c):
        r["tr"].sync_master()
        r["master"] = [e.weight.data.numpy().copy() for e in r["emb"].emb_l]
    _assert_same_run(a, c, "save at 2, sync_master at 4")


def test_collect_valid_matches_numpy():
    from cdlrm_b200 import cache_manager as C
    from cdlrm_b200 import model_no_ddp as M
    rng = np.random.default_rng(3)
    for ln, csz, ways in (([5000, 37, 800], 50, 4), ([10_000_000], 150000, 16)):
        cg = M.Embedding_Table_Cache_Group(4, np.asarray(ln), csz, 8, ways).to(DEV)
        cg._ensure_ctx(None)
        pl = C.WindowPlanner(cg, None, 16)
        tags = []
        for k, t in enumerate(cg.occupancy_tables):
            v = rng.integers(0, ln[k], t.shape)
            v[rng.random(t.shape) < 0.3] = -1
            t.copy_(torch.from_numpy(v))
            tags.append(v)
        if len(ln) == 1:
            assert cg.cache_sizes == [150001]
        for W in (1, 2, 3):
            seen = [[] for _ in ln]
            for r in range(W):
                slots, ids, off, cnt = pl.collect_valid((r, W))
                for k, v in enumerate(tags):
                    S = v.shape[0]
                    sl = slots[off[k]:off[k] + cnt[k]].cpu().numpy()
                    got_ids = ids[off[k]:off[k] + cnt[k]].cpu().numpy()
                    lo, hi = S * r // W, S * (r + 1) // W
                    way, st = np.nonzero(v.T >= 0)              # way-major: ascending slot = S * way + set
                    keep = (st >= lo) & (st < hi)
                    want = (way * S + st)[keep]
                    assert np.array_equal(sl, want), f"W={W} r={r} table {k}: slots"
                    assert np.array_equal(got_ids, v[st[keep], way[keep]]), f"W={W} r={r} table {k}: ids"
                    seen[k].append(sl)
            for k, v in enumerate(tags):
                allv = np.concatenate(seen[k])
                assert len(allv) == int((v >= 0).sum()) and len(np.unique(allv)) == len(allv), "shares overlap or miss"


def test_victim_stream_state_round_trip():
    from cdlrm_b200.cache_manager import VictimRngDevice
    r = VictimRngDevice(123, DEV)
    r.exponential(1001)
    state, draws = r.get_state()
    assert draws == 1001 and state.shape == (625,)
    for m in (5, 7_000_000):
        x = r.exponential(m).cpu().numpy()
        r.set_state(state, draws)
        assert np.array_equal(r.exponential(m).cpu().numpy(), x)
        fresh = VictimRngDevice(9, DEV)
        fresh.set_state(state, draws)
        assert np.array_equal(fresh.exponential(m).cpu().numpy(), x) and fresh.draws == draws + m
        r.set_state(state, draws)
    from cdlrm_b200._lib import CdlrmError
    with pytest.raises(CdlrmError, match="position"):
        r.set_state(state, draws + 1)


def test_refusals(tmp_path):
    from cdlrm_b200._lib import CdlrmError
    from cdlrm_b200.checkpoint import CheckpointMismatch
    s = _setup("golden")
    path = str(tmp_path / "ck")
    _train(s, False, w_end=1, save_at=1, path=path)
    meta = json.load(open(os.path.join(path, "meta.json")))
    for sec, key, val in (("args", "seed", 1), ("args", "cache_size", 99), ("args", "ways", 8), ("shapes", "dim", 8),
                          ("args", "world_size", 2)):
        bad = str(tmp_path / f"bad_{key}")
        shutil.copytree(path, bad)
        m = json.loads(json.dumps(meta))
        m[sec][key] = val
        json.dump(m, open(os.path.join(bad, "meta.json"), "w"))
        tr, _m = _build(s)
        with pytest.raises(CheckpointMismatch, match=rf"{sec}\.{key}"):
            tr.load_checkpoint(bad)
        tr.finish()
    # off a window boundary
    tr, _m = _build(s)
    cfg = s["cfg"]
    B, L, T = cfg["batch"], cfg["lookahead"], len(cfg["ln_emb"])
    ids = torch.from_numpy(s["ids"][:, :L * B]).to(DEV)
    tr.submit_window(ids)
    tr.install_window()
    lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
    tr.step(torch.from_numpy(s["X"][0]).to(DEV), lS_o, ids[:, :B], torch.from_numpy(s["Y"][0]).to(DEV))
    with pytest.raises(CdlrmError, match="window boundary"):
        tr.save_checkpoint(str(tmp_path / "off"))
    with pytest.raises(CdlrmError, match="window boundary"):
        tr.sync_master()
    assert not os.path.exists(str(tmp_path / "off")) and not os.path.exists(str(tmp_path / "off.tmp"))
    tr.finish()
    # --average-on-writeback: only after finish()
    sa = _setup("avgwb")
    tr, _m = _build(sa)
    with pytest.raises(CdlrmError, match="finish"):
        tr.sync_master()
    tr.finish()
    tr.sync_master()


def test_run_save_then_load_equals_two_epochs(tmp_path):
    from cdlrm_b200 import cache_manager as C
    from cdlrm_b200 import main_no_ddp as R
    g = util.load_golden("dlrm_trainer.npz")
    cfg = util.golden_cfg(g)
    ids = util.make_ids(cfg)
    B, T = cfg["batch"], len(cfg["ln_emb"])
    lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
    n = cfg["n_windows"] * cfg["lookahead"]
    loader = lambda: [(torch.from_numpy(g["X"][i]), lS_o, torch.from_numpy(ids[:, i * B:(i + 1) * B]),   # noqa: E731
                       torch.from_numpy(g["Y"][i])) for i in range(n)]
    path = str(tmp_path / "ck")

    def run(epochs, extra):
        args = _args(cfg, ["--nepochs", str(epochs), "--print-freq", "100", "--eviction-fifo-timeout", "2",
                           "--fifo-payload", "ids"] + extra)
        np.random.seed(cfg["seed"])
        torch.manual_seed(cfg["seed"])
        from cdlrm_b200 import model_no_ddp as M
        master = M.Embedding_Table_Group(cfg["dim"], np.asarray(cfg["ln_emb"]))
        fifo, evq, fin = queue.Queue(maxsize=2), queue.Queue(), threading.Event()
        cm = C.Prefetcher(args, master, fifo, evq, fin, loader())
        cm.start()
        orig = R.Trainer.__init__

        def _init(self, *a, **kw):
            orig(self, *a, **kw)
            self.keep_losses = True
        R.Trainer.__init__ = _init
        try:
            tr = R.Run(0, cfg["dim"], np.asarray(cfg["ln_emb"]), g["ln_bot"], g["ln_top"], loader(), None, fifo, evq,
                       [], master, args)
        finally:
            R.Trainer.__init__ = orig
            fin.set()
        cm.join(timeout=10)
        assert not cm.is_alive() and fifo.empty()
        return tr, master

    a, ma = run(2, [])
    b1, _mb1 = run(1, ["--save-model", path])
    assert json.load(open(os.path.join(path, "meta.json")))["resume"] == {"epoch": 1, "window": 4, "global_step": n}
    b2, mb2 = run(2, ["--load-model", path])
    la = np.asarray([float(x) for x in a.loss_history])
    lb1 = np.asarray([float(x) for x in b1.loss_history])
    lb2 = np.asarray([float(x) for x in b2.loss_history])
    assert len(la) == 2 * n and len(lb1) == n and len(lb2) == n
    np.testing.assert_allclose(lb1, la[:n], rtol=1e-6)
    np.testing.assert_allclose(lb2, la[n:], rtol=1e-6)
    for ta, tb in zip(a.cache_group.occupancy_tables, b2.cache_group.occupancy_tables):
        assert torch.equal(ta, tb)
    for x, y in zip(ma.emb_l, mb2.emb_l):
        np.testing.assert_allclose(x.weight.data.numpy(), y.weight.data.numpy(), rtol=0, atol=1e-6)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_checkpoint_resume(tmp_path):
    env = dict(os.environ, CKPT_DIR=str(tmp_path))

    def torchrun(phase, port):
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
               "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "mgpu_ckpt_check.py"), phase]
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
        assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
        return res.stdout

    torchrun("full", 29831)
    torchrun("save", 29832)
    out = torchrun("resume", 29833)
    assert "mgpu_ckpt_check OK" in out
