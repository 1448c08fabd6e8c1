"""``--evict-victim-cache`` on the GPU: the update of cache misses into the loser store (cdlrm_embed_victim_update),
the boundary carry (cdlrm_move_carry_losers), and the trainer-level contract: with the flag, an undersized cache
trains the same model as a cache that holds every id.

* the update kernel against a sequential numpy sum per store row (ids repeated 1, 2, 31, 33 and 200 times, the
  first and last ids of the store), deterministic, graph = eager, ``_dlr`` = float;
* the carry kernel against numpy (empty store, no ids, ids absent from the store);
* an undersized cache (the one of test_gpu_checkpoint.py: drops, contested claims, evictions, losers that recur)
  against the all-cached run: losses, dense parameters, the exported master and ``evaluate``, in both PCIe modes,
  graph and eager -- held to the bars two identically fed runs meet; without the flag the missed rows differ;
* checkpoint, resume, refusals, launch count and the CLI."""
import json
import os
import queue
import re
import shutil
import threading

import numpy as np
import pytest
import torch

import util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
# the bars of two identically fed runs (test_gpu_checkpoint.py): losses relative, parameters / tables absolute
LOSS_RTOL, VAL_ATOL = 1e-6, 1e-6
# exact AUC: swapping two near-tied predictions moves it by 1 / (positives * negatives)
AUC_ATOL = 1e-4


def _vp(t):
    import ctypes
    return ctypes.c_void_p(t.data_ptr() if isinstance(t, torch.Tensor) else t)


def _sp():
    import ctypes
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _bind_store(cg, store_ids, store_rows):
    from cdlrm_b200 import _lib
    from cdlrm_b200._lib import check, lib
    check(lib.cdlrm_ctx_bind_losers(cg._ctx, _lib.ptr_array([i.data_ptr() for i in store_ids]),
                                    _lib.ptr_array([r.data_ptr() for r in store_rows]),
                                    _lib.i64_array([i.numel() for i in store_ids]), _sp()))


def victim_update_numpy(store, store_ids, miss_ids, miss_pos, G, lr):
    """store[i] = fma(-lr, sum of G[p] over the misses on store id i in ascending p, store[i]) (fp32 sum, fp64 fma)."""
    out = store.copy()
    order = np.lexsort((miss_pos, miss_ids))
    ids_s, pos_s = miss_ids[order], miss_pos[order]
    lr32 = np.float32(lr)
    for u in np.unique(ids_s):
        i = int(np.searchsorted(store_ids, u))
        acc = np.zeros(store.shape[1], np.float32)
        for p in pos_s[ids_s == u]:
            acc = (acc + G[p]).astype(np.float32)
        out[i] = (-np.float64(lr32) * acc.astype(np.float64) + store[i].astype(np.float64)).astype(np.float32)
    return out


def _update_case(dim=16, seed=0):
    from cdlrm_b200 import model_no_ddp as M
    rng = np.random.default_rng(seed)
    ln, n_idx, ways, csz = [50_000, 9_000], 4096, 2, 31
    cg = M.Embedding_Table_Cache_Group(dim, np.asarray(ln), csz, n_idx, ways).to(DEV)
    cg._ensure_ctx(None)
    case = dict(cg=cg, n_idx=n_idx, tabs=[])
    for k, n in enumerate(ln):
        sid = np.sort(rng.choice(n, 1500, replace=False)).astype(np.int64)
        rows = rng.standard_normal((sid.size, dim)).astype(np.float32)
        # misses: ids repeated 1, 2, 31, 33 and 200 times, the first and last ids of the store, a spread of others
        reps = [(sid[0], 1), (sid[-1], 2), (sid[7], 31), (sid[500], 33), (sid[1000], 200)]
        reps += [(x, 1 + int(rng.integers(0, 3))) for x in rng.choice(sid[1:-1], 400, replace=False) if x not in
                 (sid[7], sid[500], sid[1000])]
        miss = np.concatenate([np.full(r, x, np.int64) for x, r in reps])
        pos = rng.choice(n_idx, miss.size, replace=False)
        ids = rng.integers(0, n, n_idx).astype(np.int64)
        S = cg.cache_sizes[k]
        aux_base = S * ways
        slots = rng.integers(0, aux_base, n_idx).astype(np.int32)          # hits: not touched by the update
        slots[rng.random(n_idx) < 0.02] = -1                                # unresolved positions: skipped
        ids[pos] = miss
        order = np.argsort(pos)                                             # aux slots in batch order, as the forward
        slots[pos[order]] = aux_base + np.arange(pos.size, dtype=np.int32)
        case["tabs"].append(dict(sid=sid, rows=rows, ids=ids, slots=slots, miss=miss, pos=pos))
    case["G"] = rng.standard_normal((len(ln), n_idx, dim)).astype(np.float32)
    return case


def _run_update(case, lr, dlr=False, graph=False):
    from cdlrm_b200._lib import check, lib
    cg, n_idx = case["cg"], case["n_idx"]
    T = len(case["tabs"])
    sid = [torch.from_numpy(t["sid"]).to(DEV) for t in case["tabs"]]
    rows = [torch.from_numpy(t["rows"]).to(DEV) for t in case["tabs"]]
    _bind_store(cg, sid, rows)
    ids = torch.from_numpy(np.stack([t["ids"] for t in case["tabs"]])).to(DEV)
    slots = torch.from_numpy(np.stack([t["slots"] for t in case["tabs"]])).to(DEV)
    G = torch.from_numpy(case["G"]).to(DEV)
    d = G.shape[2]
    lr_t = torch.tensor([lr], dtype=torch.float32, device=DEV)

    def launch():
        a = (cg._ctx, 0, T, _vp(slots), slots.stride(0), _vp(ids), ids.stride(0), n_idx, None, 0, _vp(G), n_idx * d, d)
        if dlr:
            check(lib.cdlrm_embed_victim_update_dlr(*a, _vp(lr_t), _sp()))
        else:
            check(lib.cdlrm_embed_victim_update(*a, float(lr), _sp()))
    if graph:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            launch()
        g.replay()
    else:
        launch()
    torch.cuda.synchronize()
    cg.check_device_flags()
    return [r.cpu().numpy() for r in rows]


@pytest.mark.parametrize("dim", [16, 128])
def test_update_kernel_matches_numpy(dim):
    case = _update_case(dim)
    lr = 0.37
    got = _run_update(case, lr)
    for k, t in enumerate(case["tabs"]):
        want = victim_update_numpy(t["rows"], t["sid"], t["miss"], t["pos"], case["G"][k], lr)
        np.testing.assert_array_max_ulp(got[k], want, maxulp=1)
        untouched = np.setdiff1d(np.arange(t["sid"].size), np.searchsorted(t["sid"], np.unique(t["miss"])))
        assert untouched.size > 0 and np.array_equal(got[k][untouched], t["rows"][untouched])
    again = _run_update(case, lr)
    graph = _run_update(case, lr, graph=True)
    dlr = _run_update(case, lr, dlr=True)
    for k in range(len(got)):
        assert np.array_equal(got[k], again[k]), "two launches differ"
        assert np.array_equal(got[k], graph[k]), "graph replay differs from the eager launch"
        assert np.array_equal(got[k], dlr[k]), "_dlr differs from the float variant"


def test_update_of_an_id_outside_the_store_raises():
    from cdlrm_b200._lib import CdlrmError
    case = _update_case(16, seed=1)
    t = case["tabs"][0]
    absent = np.setdiff1d(np.arange(1, 50_000), t["sid"])[0]
    t["ids"][t["pos"][0]] = absent
    with pytest.raises(CdlrmError, match="not in the loser store"):
        _run_update(case, 0.1)
    case["cg"].check_device_flags()                  # the flag is cleared once reported


def test_carry_kernel_matches_numpy():
    from cdlrm_b200 import model_no_ddp as M
    from cdlrm_b200._lib import check, lib
    rng = np.random.default_rng(3)
    d = 16
    cg = M.Embedding_Table_Cache_Group(d, np.asarray([100_000, 500]), 31, 64, 2).to(DEV)
    cg._ensure_ctx(None)
    q = torch.from_numpy(rng.integers(0, 500, 300).astype(np.int64)).to(DEV)
    r0 = torch.from_numpy(rng.standard_normal((300, d)).astype(np.float32)).to(DEV)
    r = r0.clone()
    check(lib.cdlrm_move_carry_losers(cg._ctx, 1, _vp(q), 300, _vp(r), _sp()))     # no store was ever bound
    torch.cuda.synchronize()
    assert torch.equal(r, r0)
    for n_store in (0, 40, 300):          # empty, the plain search, the bucket index (>= 64 ids)
        sid = [np.sort(rng.choice(n, n_store, replace=False)).astype(np.int64) for n in (100_000, 500)]
        rows = [rng.standard_normal((s.size, d)).astype(np.float32) for s in sid]
        bound = ([torch.from_numpy(s).to(DEV) for s in sid], [torch.from_numpy(x).to(DEV) for x in rows])
        _bind_store(cg, *bound)               # (the store's tensors must outlive its use)
        for k, n in enumerate((100_000, 500)):
            present = sid[k][rng.integers(0, sid[k].size, 200)] if sid[k].size else np.zeros(0, np.int64)
            q_np = np.concatenate([present, rng.integers(0, n, 300)]).astype(np.int64)
            rng.shuffle(q_np)
            base = rng.standard_normal((q_np.size, d)).astype(np.float32)
            got = torch.from_numpy(base).to(DEV)
            check(lib.cdlrm_move_carry_losers(cg._ctx, k, _vp(torch.from_numpy(q_np).to(DEV)), q_np.size, _vp(got), _sp()))
            check(lib.cdlrm_move_carry_losers(cg._ctx, k, None, 0, None, _sp()))           # n = 0: nothing to do
            want = base.copy()
            hit = np.isin(q_np, sid[k])
            want[hit] = rows[k][np.searchsorted(sid[k], q_np[hit])]
            assert np.array_equal(got.cpu().numpy(), want), f"store of {n_store}, table {k}"


# ---- trainer level ----------------------------------------------------------------------------------------------

def _setup(n_windows=6):
    cfg = dict(ln_emb=[3000, 37, 800, 5, 12000], dim=16, cache_size=20, num_ways=2, batch=64, lookahead=4,
               n_windows=n_windows, lr_embeds=0.3, lr_mlp=0.1, seed=5, data_seed=41, dist="zipf", zipf_a=1.05)
    rng = np.random.default_rng(7)
    n = cfg["n_windows"] * cfg["lookahead"]
    X = rng.standard_normal((n, cfg["batch"], 13)).astype(np.float32)
    Y = (rng.random((n, cfg["batch"], 1)) < 0.3).astype(np.float32)
    return dict(cfg=cfg, ids=util.make_ids(cfg), X=X, Y=Y, ln_bot=np.asarray([13, 32, 16]),
                ln_top=np.asarray([31, 32, 1]))


ALL_CACHED = 12000          # >= every table: each id has a set of its own, nothing ever misses


def _argv(cfg, cache_size, extra=()):
    return ["--arch-sparse-feature-size", str(cfg["dim"]), "--loss-function", "bce", "--learning-rate",
            str(cfg["lr_mlp"]), "--lr-embeds", str(cfg["lr_embeds"]), "--mini-batch-size", str(cfg["batch"]),
            "--lookahead", str(cfg["lookahead"]), "--cache-size", str(cache_size), "--num-ways",
            str(cfg["num_ways"]), "--numpy-rand-seed", str(cfg["seed"]), "--world-size", "1"] + list(extra)


def _build(s, cache_size, flag, mode=None):
    from cdlrm_b200 import main_no_ddp as R
    from cdlrm_b200 import model_no_ddp as M
    cfg = s["cfg"]
    np.random.seed(cfg["seed"])
    torch.manual_seed(cfg["seed"])
    master = M.Embedding_Table_Group(cfg["dim"], np.asarray(cfg["ln_emb"]))
    args = R.ProcessArgs(_argv(cfg, cache_size, ["--evict-victim-cache"] if flag else []))
    tr = R.Trainer(args, cfg["dim"], np.asarray(cfg["ln_emb"]), s["ln_bot"], s["ln_top"], master, rank=0, world=1,
                   device=torch.device(DEV))
    if mode is not None:
        tr.planner.pcie_mode = mode
    return tr, master


def _test_loader(s, nb=4):
    cfg = s["cfg"]
    rng = np.random.default_rng(11)
    B, T = cfg["batch"], len(cfg["ln_emb"])
    lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
    ids = s["ids"]
    out = []
    for b in range(nb):
        cols = rng.integers(0, ids.shape[1], B)
        out.append((torch.from_numpy(rng.standard_normal((B, 13)).astype(np.float32)), lS_o,
                    torch.from_numpy(ids[:, cols].copy()), torch.from_numpy((rng.random((B, 1)) < 0.3).astype(np.float32))))
    return out


def _train(s, cache_size, flag, use_graph=True, mode=None, w_end=None, load=None, save_at=None, sync_at=None,
           path=None, evaluate=True):
    cfg = s["cfg"]
    B, L, nw, T = cfg["batch"], cfg["lookahead"], cfg["n_windows"], len(cfg["ln_emb"])
    w_end = nw if w_end is None else w_end
    tr, master = _build(s, cache_size, flag, mode)
    w0 = tr.load_checkpoint(load) if load else 0
    lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
    X, Y = torch.from_numpy(s["X"]).to(DEV), torch.from_numpy(s["Y"]).to(DEV)
    win = lambda w: torch.from_numpy(s["ids"][:, w * L * B:(w + 1) * L * B]).to(DEV)   # noqa: E731
    out = dict(losses=[], losers=[set() for _ in range(T)], E=0)
    tr.submit_window(win(w0))
    local = 0
    for w in range(w0, w_end):
        if save_at == w:
            tr.save_checkpoint(path)
        if sync_at == w:
            tr.sync_master()
        rec = tr.install_window()
        if w + 1 < nw:
            tr.submit_window(win(w + 1))
        out["E"] += sum(rec.E)
        for k in range(T):
            out["losers"][k].update(rec.loser_list(k).cpu().tolist())
        cur = win(w)
        for b in range(L):
            step = w * L + b
            if use_graph and getattr(tr, "_graph", None) is None and local == 1:
                tr.capture_graph(X[step], lS_o, cur[:, b * B:(b + 1) * B], Y[step])
            E, _Z = tr.step(X[step], lS_o, cur[:, b * B:(b + 1) * B], Y[step])
            out["losses"].append(E.detach().clone())
            local += 1
    if save_at == w_end:
        tr.save_checkpoint(path)
    torch.cuda.synchronize()
    tr.finish()
    out["losses"] = np.asarray([float(x) for x in out["losses"]], dtype=np.float64)
    out["params"] = [p.detach().cpu().numpy().copy() for p in tr.dlrm.parameters()]
    if evaluate:
        out["eval"] = tr.evaluate(_test_loader(s))
    tr.sync_master()
    out["master"] = [e.weight.data.numpy().copy() for e in master.emb_l]
    out["tr"] = tr
    return out


def _diffs(a, b):
    return dict(loss=float(np.max(np.abs(a["losses"] - b["losses"]) / np.abs(b["losses"]))),
                params=max(float(np.max(np.abs(x - y))) for x, y in zip(a["params"], b["params"])),
                master=max(float(np.max(np.abs(x - y))) for x, y in zip(a["master"], b["master"])))


def _assert_within_bars(a, b, tag):
    d = _diffs(a, b)
    print(tag, d)
    assert d["loss"] <= LOSS_RTOL and d["params"] <= VAL_ATOL and d["master"] <= VAL_ATOL, (tag, d)
    if "eval" in a and "eval" in b:
        assert abs(a["eval"].loss - b["eval"].loss) <= LOSS_RTOL * abs(b["eval"].loss), (tag, a["eval"], b["eval"])
        assert abs(a["eval"].auc - b["eval"].auc) <= AUC_ATOL, (tag, a["eval"], b["eval"])


@pytest.fixture(scope="module")
def reference_runs():
    """The all-cached run twice (the spread of two identically fed runs) and the undersized run without the flag."""
    s = _setup()
    full = _train(s, ALL_CACHED, flag=False)
    full2 = _train(s, ALL_CACHED, flag=False)
    plain = _train(s, s["cfg"]["cache_size"], flag=False)
    return s, full, full2, plain


def test_two_identical_runs_meet_the_bars(reference_runs):
    _s, full, full2, _plain = reference_runs
    assert sum(len(x) for x in full["losers"]) == 0 and full["E"] == 0, "the large cache must hold every id"
    _assert_within_bars(full2, full, "all-cached twice")


@pytest.mark.parametrize("use_graph", [True, False])
@pytest.mark.parametrize("mode", ["sm", "ce"])
def test_undersized_cache_trains_the_all_cached_model(reference_runs, mode, use_graph):
    s, full, _full2, plain = reference_runs
    v = _train(s, s["cfg"]["cache_size"], flag=True, use_graph=use_graph, mode=mode)
    assert v["E"] > 0 and sum(len(x) for x in v["losers"]) > 0, "the undersized cache must evict and miss"
    _assert_within_bars(v, full, f"flag mode={mode} graph={use_graph}")
    # negative control: without the flag the rows of the ids that missed lose their updates
    worst = max(float(np.max(np.abs(plain["master"][k][sorted(ids)] - full["master"][k][sorted(ids)])))
                for k, ids in enumerate(plain["losers"]) if ids)
    assert worst > 1000 * VAL_ATOL, worst


def test_resume_equals_uninterrupted_run(tmp_path):
    s = _setup()
    k = s["cfg"]["n_windows"] // 2
    path = str(tmp_path / "ck")
    a = _train(s, s["cfg"]["cache_size"], True, evaluate=False)
    b1 = _train(s, s["cfg"]["cache_size"], True, w_end=k, save_at=k, path=path, evaluate=False)
    b2 = _train(s, s["cfg"]["cache_size"], True, load=path, evaluate=False)
    b = dict(b2, losses=np.concatenate([b1["losses"], b2["losses"]]))
    _assert_within_bars(b, a, "resume")


def test_save_and_sync_do_not_perturb(tmp_path):
    s = _setup()
    a = _train(s, s["cfg"]["cache_size"], True, evaluate=False)
    c = _train(s, s["cfg"]["cache_size"], True, save_at=2, sync_at=4, path=str(tmp_path / "ck"), evaluate=False)
    _assert_within_bars(c, a, "save at 2, sync_master at 4")


def test_checkpoint_field(tmp_path):
    from cdlrm_b200.checkpoint import CheckpointMismatch
    s = _setup(2)
    path = str(tmp_path / "ck")
    _train(s, s["cfg"]["cache_size"], True, w_end=1, save_at=1, path=path, evaluate=False)
    assert json.load(open(os.path.join(path, "meta.json")))["args"]["evict_victim_cache"] is True
    tr, _m = _build(s, s["cfg"]["cache_size"], flag=False)
    with pytest.raises(CheckpointMismatch, match=r"args\.evict_victim_cache"):
        tr.load_checkpoint(path)
    tr.finish()
    old = str(tmp_path / "old")                # written before the field existed: trained without the flag
    shutil.copytree(path, old)
    m = json.load(open(os.path.join(old, "meta.json")))
    del m["args"]["evict_victim_cache"]
    json.dump(m, open(os.path.join(old, "meta.json"), "w"))
    tr, _m = _build(s, s["cfg"]["cache_size"], flag=False)
    assert tr.load_checkpoint(old) == 1
    tr.finish()
    tr, _m = _build(s, s["cfg"]["cache_size"], flag=True)
    with pytest.raises(CheckpointMismatch, match=r"args\.evict_victim_cache"):
        tr.load_checkpoint(old)
    tr.finish()


def test_capped_store_is_refused(monkeypatch):
    from cdlrm_b200._lib import CdlrmError
    monkeypatch.setenv("CDLRM_LOSER_STORE_GB", "0.000001")          # 15 rows of 16 floats
    s = _setup(2)
    tr, _m = _build(s, s["cfg"]["cache_size"], flag=True)
    tr.submit_window(torch.from_numpy(s["ids"][:, :s["cfg"]["lookahead"] * s["cfg"]["batch"]]).to(DEV))
    with pytest.raises(CdlrmError, match="CDLRM_LOSER_STORE_GB"):
        tr.install_window()


def test_batch_outside_its_window_raises():
    from cdlrm_b200._lib import CdlrmError
    s = _setup()
    cfg = s["cfg"]
    B, L, T = cfg["batch"], cfg["lookahead"], len(cfg["ln_emb"])
    tr, _m = _build(s, cfg["cache_size"], flag=True)
    tr.submit_window(torch.from_numpy(s["ids"][:, :L * B]).to(DEV))
    tr.install_window()
    lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
    far = torch.from_numpy(s["ids"][:, 5 * L * B:5 * L * B + B].copy()).to(DEV)      # a batch of window 5
    tr.step(torch.from_numpy(s["X"][0]).to(DEV), lS_o, far, torch.from_numpy(s["Y"][0]).to(DEV))
    torch.cuda.synchronize()
    with pytest.raises(CdlrmError, match="not in the loser store"):
        tr.cache_group.check_device_flags()
    tr.finish()


def test_one_more_launch_per_step():
    s = _setup(1)
    cfg = s["cfg"]
    B, L, T = cfg["batch"], cfg["lookahead"], len(cfg["ln_emb"])
    counts = {}
    for flag in (False, True):
        tr, _m = _build(s, cfg["cache_size"], flag)
        win = torch.from_numpy(s["ids"][:, :L * B]).to(DEV)
        tr.submit_window(win)
        tr.install_window()
        lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
        X, Y = torch.from_numpy(s["X"][0]).to(DEV), torch.from_numpy(s["Y"][0]).to(DEV)
        tr.step(X, lS_o, win[:, :B], Y)
        tr.capture_graph(X, lS_o, win[:, B:2 * B], Y)
        counts[flag] = tr.graph_launches
        tr.finish()
    assert counts[True] == counts[False] + 1, counts


def _run_cli(s, cache_size, extra, capsys):
    from cdlrm_b200 import cache_manager as C
    from cdlrm_b200 import main_no_ddp as R
    from cdlrm_b200 import model_no_ddp as M
    cfg = s["cfg"]
    B, T = cfg["batch"], len(cfg["ln_emb"])
    lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
    n = cfg["n_windows"] * cfg["lookahead"]
    loader = lambda: [(torch.from_numpy(s["X"][i]), lS_o, torch.from_numpy(s["ids"][:, i * B:(i + 1) * B]),   # noqa: E731
                       torch.from_numpy(s["Y"][i])) for i in range(n)]
    args = R.ProcessArgs(_argv(cfg, cache_size, ["--print-freq", "100", "--eviction-fifo-timeout", "2",
                                                 "--fifo-payload", "ids"] + list(extra)))
    np.random.seed(cfg["seed"])
    torch.manual_seed(cfg["seed"])
    master = M.Embedding_Table_Group(cfg["dim"], np.asarray(cfg["ln_emb"]))
    fifo, evq, fin = queue.Queue(maxsize=2), queue.Queue(), threading.Event()
    cm = C.Prefetcher(args, master, fifo, evq, fin, loader())
    cm.start()
    capsys.readouterr()
    try:
        R.Run(0, cfg["dim"], np.asarray(cfg["ln_emb"]), s["ln_bot"], s["ln_top"], loader(), _test_loader(s), fifo, evq,
              [], master, args)
    finally:
        fin.set()
    cm.join(timeout=10)
    text = capsys.readouterr().out
    res = [tuple(float(x) for x in m) for m in re.findall(r"Test loss = ([-0-9.e]+), AUC = ([-0-9.e]+)", text)]
    return res, [e.weight.data.numpy().copy() for e in master.emb_l]


def test_cli_with_the_flag(tmp_path, capsys):
    s = _setup(4)
    full, _ = _run_cli(s, ALL_CACHED, [], capsys)
    vic, _ = _run_cli(s, s["cfg"]["cache_size"], ["--evict-victim-cache"], capsys)
    assert len(vic) == len(full) >= 1
    for (lv, av), (lf, af) in zip(vic, full):
        assert abs(lv - lf) <= LOSS_RTOL * abs(lf) and abs(av - af) <= AUC_ATOL, (vic, full)
    # --save-model after epoch 1 of 2, --load-model: the second epoch equals the uninterrupted run's
    path = str(tmp_path / "ck")
    a, ma = _run_cli(s, s["cfg"]["cache_size"], ["--evict-victim-cache", "--nepochs", "2"], capsys)
    _run_cli(s, s["cfg"]["cache_size"], ["--evict-victim-cache", "--nepochs", "1", "--save-model", path], capsys)
    assert json.load(open(os.path.join(path, "meta.json")))["args"]["evict_victim_cache"] is True
    b, mb = _run_cli(s, s["cfg"]["cache_size"], ["--evict-victim-cache", "--nepochs", "2", "--load-model", path],
                     capsys)
    for x, y in zip(ma, mb):
        np.testing.assert_allclose(x, y, rtol=0, atol=VAL_ATOL)
    assert abs(a[-1][0] - b[-1][0]) <= LOSS_RTOL * abs(a[-1][0]) and abs(a[-1][1] - b[-1][1]) <= AUC_ATOL, (a, b)
