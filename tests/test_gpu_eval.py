"""Forward-only evaluation on the GPU: ``cdlrm_embed_fwd_eval``, the metrics object (``cdlrm_eval_*``) and
``Trainer.evaluate``.

* the read-only lookup equals a numpy gather from the live tags, the cache rows and the master, bit for bit, on an
  undersized cache after several windows (loser-store ids, ids outside the window, more misses than aux rows);
* counts and 2U are exact against numpy integer arithmetic, the loss matches numpy fp64, on ties, degenerate inputs
  and sizes up to 10^7;
* ``evaluate`` agrees with an eager forward through the training path, and graph replay with eager evaluation;
* an evaluation (test batch 4x the training batch) changes nothing in the training run that follows, with the graph,
  mid-window and at a boundary, in both PCIe modes; right after a boundary it reads no stale master row;
* ``Run`` prints accuracy, loss and AUC, and ``--inference-only`` evaluates a saved checkpoint without changing it."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
_vp = ctypes.c_void_p


def _setup():
    """The undersized-cache configuration of test_gpu_checkpoint.py: batch 64 = aux rows, many evictions."""
    cfg = dict(ln_emb=[3000, 37, 800, 5, 12000], dim=16, cache_size=20, num_ways=2, batch=64, lookahead=4,
               n_windows=6, lr_embeds=0.3, lr_mlp=0.1, seed=5, data_seed=41, dist="zipf", zipf_a=1.05)
    rng = np.random.default_rng(7)
    n = cfg["n_windows"] * cfg["lookahead"]
    X = rng.standard_normal((n, cfg["batch"], 13)).astype(np.float32)
    Y = (rng.random((n, cfg["batch"], 1)) < 0.3).astype(np.float32)
    return dict(cfg=cfg, ids=util.make_ids(cfg), X=X, Y=Y, ln_bot=np.asarray([13, 32, 16]),
                ln_top=np.asarray([31, 32, 1]))


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
    tr = R.Trainer(_args(cfg, extra), cfg["dim"], np.asarray(cfg["ln_emb"]), s["ln_bot"], s["ln_top"], master, rank=0,
                   world=1, device=torch.device(DEV))
    return tr, master


def _test_loader(s, batch, n_batches, seed=3, labels=None):
    """CPU batches of test ids drawn over the whole id space of every table (most of them outside any window)."""
    cfg = s["cfg"]
    rng = np.random.default_rng(seed)
    T = len(cfg["ln_emb"])
    lS_o = torch.arange(batch).reshape(1, -1).repeat(T, 1)
    out = []
    for _ in range(n_batches):
        ids = np.stack([rng.integers(0, n, batch) for n in cfg["ln_emb"]]).astype(np.int64)
        X = rng.standard_normal((batch, 13)).astype(np.float32)
        Y = (rng.random((batch, 1)) < 0.3).astype(np.float32) if labels is None else np.full((batch, 1), labels,
                                                                                                np.float32)
        out.append((torch.from_numpy(X), lS_o, torch.from_numpy(ids), torch.from_numpy(Y)))
    return out


def _train(s, use_graph=True, mode=None, w_end=None, hook=None):
    """Windows [0, w_end) as test_gpu_checkpoint.py drives them.  ``hook(tr, w, b)`` runs before step b of window w
    (b == 0: right after the install of w; b == -1: at the boundary before that install)."""
    cfg = s["cfg"]
    B, L, nw, T = cfg["batch"], cfg["lookahead"], cfg["n_windows"], len(cfg["ln_emb"])
    w_end = nw if w_end is None else w_end
    tr, master = _build(s)
    if mode is not None:
        tr.planner.pcie_mode = mode
    lS_o = torch.arange(B).reshape(1, -1).repeat(T, 1)
    X, Y = torch.from_numpy(s["X"]).to(DEV), torch.from_numpy(s["Y"]).to(DEV)
    win = lambda w: torch.from_numpy(s["ids"][:, w * L * B:(w + 1) * L * B]).to(DEV)   # noqa: E731
    out = dict(tags=[], E=[], F=[], losses=[], n_miss=[])
    tr.submit_window(win(0))
    local = 0
    for w in range(w_end):
        if hook is not None:
            hook(tr, w, -1)
        rec = tr.install_window()
        if w + 1 < nw:
            tr.submit_window(win(w + 1))
        torch.cuda.synchronize()
        out["tags"].append(np.concatenate([t.cpu().numpy().ravel() for t in tr.cache_group.occupancy_tables]))
        out["E"].append(list(rec.E))
        out["F"].append(list(rec.F))
        cur = win(w)
        for b in range(L):
            if hook is not None:
                hook(tr, w, b)
            step = w * L + b
            if use_graph and getattr(tr, "_graph", None) is None and local == 1:
                tr.capture_graph(X[step], lS_o, cur[:, b * B:(b + 1) * B], Y[step])
            E, _Z = tr.step(X[step], lS_o, cur[:, b * B:(b + 1) * B], Y[step])
            out["losses"].append(E.detach().clone())
            out["n_miss"].append(tr.cache_group.last_n_miss.clone())
            local += 1
    torch.cuda.synchronize()
    tr.finish()
    out["losses"] = np.asarray([float(x) for x in out["losses"]], dtype=np.float64)
    out["n_miss"] = torch.stack(out["n_miss"]).cpu().numpy()
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


# ---------------------------------------------------------------------------------------------------------------------
# 1. the read-only lookup
# ---------------------------------------------------------------------------------------------------------------------

def _lookup(tr, ids):
    from cdlrm_b200._lib import check, lib
    cg = tr.cache_group
    ids = ids.to(DEV).contiguous()
    T, n = ids.shape
    out = torch.full((T, n, cg.dim), float("nan"), dtype=torch.float32, device=DEV)
    check(lib.cdlrm_embed_fwd_eval(cg._ctx, 0, T, _vp(ids.data_ptr()), ids.stride(0), n, _vp(out.data_ptr()),
                                   out.stride(0), _vp(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _gather(tr, master, ids):
    """Expected rows: the cache row when the id is in its set's tag line, else master[id]."""
    cg = tr.cache_group
    want = []
    for k, idk in enumerate(ids):
        tags = cg.occupancy_tables[k].cpu().numpy()
        W = cg.emb_l[k].weight.data.cpu().numpy()
        M = master.emb_l[k].weight.data.numpy()
        S = cg.cache_sizes[k]
        rows = M[idk].copy()
        s = idk % S
        for way in range(cg.num_ways - 1, -1, -1):
            hit = tags[s, way] == idk
            rows[hit] = W[S * way + s[hit]]
        want.append(rows)
    return np.stack(want)


def test_lookup_matches_cache_and_master_gather():
    s = _setup()
    cfg = s["cfg"]
    B, L = cfg["batch"], cfg["lookahead"]
    stop = {}

    def hook(tr, w, b):
        if w == 3 and b == 2 and not stop:       # mid-window 3: a loser store is installed
            stop["tr"] = tr
            tr._quiesce()
            win = s["ids"][:, 3 * L * B:4 * L * B]
            rng = np.random.default_rng(11)
            outside = np.stack([rng.integers(0, n, 700) for n in cfg["ln_emb"]]).astype(np.int64)
            for ids in (win, outside, np.concatenate([win, outside], axis=1)):   # up to 956 ids per table >> 64 aux
                got = _lookup(tr, torch.from_numpy(ids))
                want = _gather(tr, tr.emb_tables, ids)
                assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
            # the uncached ids of the window are served and are many more than the aux rows
            tags = [t.cpu().numpy() for t in tr.cache_group.occupancy_tables]
            miss = sum(int((~(tags[k][win[k] % tr.cache_group.cache_sizes[k]] == win[k][:, None]).any(1)).sum())
                       for k in range(len(tags)))
            assert miss > cfg["batch"]
            bad = torch.from_numpy(outside[:, :64].copy())
            bad[2, 5] = cfg["ln_emb"][2]
            got = _lookup(tr, bad)
            assert not got[2, 5].any()
            with pytest.raises(IndexError):
                tr.cache_group.check_device_flags()

    _train(s, use_graph=True, w_end=4, hook=hook)
    assert "tr" in stop


# ---------------------------------------------------------------------------------------------------------------------
# 2. the metrics object against numpy
# ---------------------------------------------------------------------------------------------------------------------

class _Metrics:
    def __init__(self, cap):
        from cdlrm_b200._lib import check, lib
        self.check, self.lib = check, lib
        self.h = _vp()
        check(lib.cdlrm_eval_create(ctypes.byref(self.h), 0, cap))

    def run(self, z, t, splits=(0.37, 0.81)):
        from cdlrm_b200._lib import EvalStats
        s = _vp(torch.cuda.current_stream().cuda_stream)
        zd, td = torch.from_numpy(z).to(DEV).reshape(-1, 1), torch.from_numpy(t).to(DEV).reshape(-1, 1)
        self.check(self.lib.cdlrm_eval_reset(self.h, s))
        cuts = [0] + [int(f * z.size) for f in splits] + [z.size]
        for a, b in zip(cuts[:-1], cuts[1:]):       # batches that do not line up with the loss chunks
            self.check(self.lib.cdlrm_eval_accumulate(self.h, _vp(zd[a:].data_ptr()), 1, _vp(td[a:].data_ptr()), 1,
                                                      b - a, s))
        st = EvalStats()
        self.check(self.lib.cdlrm_eval_result(self.h, _vp(ctypes.addressof(st)), s))
        return st

    def close(self):
        self.lib.cdlrm_eval_destroy(self.h)


def _numpy_metrics(z, t):
    keys, inv = np.unique(z.astype(np.float64), return_inverse=True)
    pos = np.bincount(inv, weights=(t == 1), minlength=keys.size).astype(np.int64)
    neg = np.bincount(inv, weights=(t == 0), minlength=keys.size).astype(np.int64)
    below = np.concatenate([[0], np.cumsum(neg)[:-1]])
    two_u = int(np.sum(pos * (2 * below + neg)))
    z64, t64 = z.astype(np.float64), t.astype(np.float64)
    with np.errstate(divide="ignore"):
        loss = -np.sum(t64 * np.maximum(np.log(z64), -100.0) + (1 - t64) * np.maximum(np.log(1 - z64), -100.0))
    return dict(samples=z.size, positives=int((t == 1).sum()), negatives=int((t == 0).sum()),
                correct=int((np.rint(z) == t).sum()), two_u=two_u, loss=float(loss))


def _cases():
    rng = np.random.default_rng(0)
    lab = lambda n, p=0.3: (rng.random(n) < p).astype(np.float32)   # noqa: E731
    yield "random", rng.random(100_000).astype(np.float32), lab(100_000)
    yield "q3", (rng.integers(0, 3, 50_000) / 2).astype(np.float32), lab(50_000)
    yield "q1000", (rng.integers(0, 1000, 200_000) / 999).astype(np.float32), lab(200_000)
    yield "all_equal", np.full(70_000, 0.3, np.float32), lab(70_000)
    base = np.float32(0.2).view(np.uint32) & ~np.uint32(0x3FFF)
    yield "one_2^14_ulp_range", (base + rng.integers(0, 1 << 14, 150_000).astype(np.uint32)).view(np.float32), \
        lab(150_000)
    yield "zero_one", rng.integers(0, 2, 40_000).astype(np.float32), lab(40_000)
    yield "one_class", rng.random(5000).astype(np.float32), np.ones(5000, np.float32)
    yield "half", np.full(999, 0.5, np.float32), lab(999)
    for n in (1, 31, 4097):
        yield f"size_{n}", rng.random(n).astype(np.float32), lab(n)
    z = rng.random(10_000_000).astype(np.float32)
    z[::7] = np.float32(0.0625)                       # one big tie group: a bucket split over many CTAs
    yield "size_1e7", z, lab(10_000_000)


def test_metrics_match_numpy():
    from scipy.stats import mannwhitneyu
    m = _Metrics(10_000_000)
    try:
        for name, z, t in _cases():
            st = m.run(z, t)
            want = _numpy_metrics(z, t)
            assert st.flags == 0, name
            got = dict(samples=st.samples, positives=st.positives, negatives=st.negatives, correct=st.correct,
                       two_u=int(st.auc_2u))
            assert got == {k: want[k] for k in got}, name
            np.testing.assert_allclose(st.loss_sum, want["loss"], rtol=1e-12, err_msg=name)
            P, N = st.positives, st.negatives
            if name in ("random", "q3", "q1000", "half"):
                u = mannwhitneyu(z[t == 1].astype(np.float64), z[t == 0].astype(np.float64)).statistic
                assert abs(u / (P * N) - st.auc_2u / (2.0 * P * N)) < 1e-12, name
            st2 = m.run(z, t)                         # the same batches again: the same result, bit for bit
            assert (st2.auc_2u, st2.correct, st2.loss_sum) == (st.auc_2u, st.correct, st.loss_sum), name
            st3 = m.run(z, t, splits=(0.5,))          # another split: counts exact, the loss summed in another order
            assert (st3.auc_2u, st3.correct) == (st.auc_2u, st.correct), name
            np.testing.assert_allclose(st3.loss_sum, st.loss_sum, rtol=1e-13, err_msg=name)
        z = np.asarray([0.2, 1.5, 0.3], np.float32)
        assert m.run(z, np.zeros(3, np.float32)).flags & 1
        assert m.run(np.asarray([0.2, np.nan], np.float32), np.zeros(2, np.float32)).flags & 1
        assert m.run(np.asarray([0.2, 0.4], np.float32), np.asarray([0, 2], np.float32)).flags & 2
    finally:
        m.close()


def test_bad_labels_raise_value_error():
    s = _setup()
    tr, _m = _build(s)
    tr.submit_window(torch.from_numpy(s["ids"][:, :s["cfg"]["lookahead"] * s["cfg"]["batch"]]).to(DEV))
    tr.install_window()
    with pytest.raises(ValueError):
        tr.evaluate(_test_loader(s, 64, 2, labels=2.0))
    r = tr.evaluate(_test_loader(s, 64, 2, labels=1.0))          # one class: AUC is NaN
    assert r.samples == 128 and r.negatives == 0 and np.isnan(r.auc)
    from cdlrm_b200._lib import CdlrmError
    ld = _test_loader(s, 64, 2)
    bad = ld[1][1].clone()
    bad[3, 10] = 11                                              # two ids in bag 11 of table 3, none in bag 10
    with pytest.raises(CdlrmError):
        tr.evaluate([ld[0], (ld[1][0], bad, ld[1][2], ld[1][3])])            # host offsets
    with pytest.raises(CdlrmError):
        tr.evaluate([(X.to(DEV), o.to(DEV), i.to(DEV), t.to(DEV)) for X, o, i, t in ld[:1]] +
                    [(ld[1][0].to(DEV), bad.to(DEV), ld[1][2].to(DEV), ld[1][3].to(DEV))])   # device offsets


# ---------------------------------------------------------------------------------------------------------------------
# 3. evaluate against an eager forward through the training path
# ---------------------------------------------------------------------------------------------------------------------

def test_evaluate_matches_eager_reference():
    s = _setup()
    res = {}

    def hook(tr, w, b):
        if w == 3 and b == 1 and not res:
            loader = _test_loader(s, 64, 5)
            r1 = tr.evaluate(loader)       # batch 1 eager, batch 2 captured, the rest replayed
            r2 = tr.evaluate(loader)       # all replayed
            tr.args.no_cuda_graph = True
            r3 = tr.evaluate(loader)       # all eager
            tr.args.no_cuda_graph = False
            assert r1 == r2 == r3
            ev = tr._ev
            Zs, Ze, Ts = [], [], []
            with torch.no_grad():
                for X, lS_o, lS_i, T in loader:
                    Zs.append(ev.fwd(X.to(DEV), lS_i.to(DEV)).cpu().numpy())
                    lookups, _ = tr.cache_group(lS_o, lS_i.to(DEV), tr.emb_tables, 0)
                    Ze.append(tr.dlrm(X.to(DEV), lookups).cpu().numpy())
                    Ts.append(T.numpy())
            tr.cache_group.check_device_flags()
            zs, ze, t = (np.concatenate(a).ravel() for a in (Zs, Ze, Ts))
            np.testing.assert_allclose(zs, ze, rtol=1e-5)
            want = _numpy_metrics(ze, t)
            n = want["samples"]
            assert r1.samples == n and r1.positives == want["positives"] and r1.negatives == want["negatives"]
            assert r1.accuracy == want["correct"] / n
            assert abs(r1.auc - want["two_u"] / (2.0 * want["positives"] * want["negatives"])) < 1e-6
            np.testing.assert_allclose(r1.loss, want["loss"] / n, rtol=1e-6)
            res["ok"] = True

    _train(s, use_graph=True, w_end=4, hook=hook)
    assert res


# ---------------------------------------------------------------------------------------------------------------------
# 4. / 5. training is untouched; no stale master row
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", ["ce", "sm"])
@pytest.mark.parametrize("where", ["mid_window", "after_boundary"])
def test_evaluation_does_not_perturb_training(mode, where):
    s = _setup()
    at = (2, 2) if where == "mid_window" else (3, 0)
    loader = _test_loader(s, 4 * s["cfg"]["batch"], 3)          # test batch 4x the training batch
    seen = []

    def hook(tr, w, b):
        if (w, b) == at:
            seen.append(tr.evaluate(loader))

    a = _train(s, use_graph=True, mode=mode, hook=hook)
    b = _train(s, use_graph=True, mode=mode)
    assert len(seen) == 1 and seen[0].samples == 3 * 4 * s["cfg"]["batch"]
    _assert_same_run(a, b, f"{mode}/{where}")


@pytest.mark.parametrize("mode", ["ce", "sm"])
def test_no_stale_rows_after_boundary(mode):
    s = _setup()
    loader = _test_loader(s, 256, 4)
    got = []

    def hook(tr, w, b):
        if w == 4 and b == -1:            # boundary before window 4: the write-back of window 3's evictions pending
            r1 = tr.evaluate(loader)
            tr.sync_master()
            got.append((r1, tr.evaluate(loader)))

    a = _train(s, use_graph=True, mode=mode, hook=hook)
    assert sum(a["E"][3]) > 0
    r1, r2 = got[0]
    assert r1 == r2


@pytest.mark.parametrize("mode", ["ce", "sm"])
def test_evaluate_right_after_install_waits_for_the_write_back(mode):
    """Right after the install of a window with evictions (their write-back and the next plan still running),
    evaluate must first complete both: the lookups then read the master as it is after an explicit quiesce."""
    s = _setup()
    loader = _test_loader(s, 256, 4)
    got, state = [], []

    def hook(tr, w, b):
        if w == 3 and b == 0:
            orig = tr._quiesce

            def spy():
                orig()
                wb = tr._installed.wb_done
                state.append((tr._plan_thread is None or not tr._plan_thread.is_alive(), wb is None or wb.query()))
            tr._quiesce = spy
            r1 = tr.evaluate(loader)
            tr._quiesce = orig
            tr._quiesce()
            got.append((r1, tr.evaluate(loader)))

    a = _train(s, use_graph=True, mode=mode, hook=hook)
    assert sum(a["E"][3]) > 0
    assert state == [(True, True)]
    r1, r2 = got[0]
    assert r1 == r2


_MGPU = """
import sys
sys.path.insert(0, {root!r})
from cdlrm_b200.main_no_ddp import main
main({argv!r})
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_run_test_pass_after_a_boundary_is_deterministic():
    """N = 2, one shared master: every rank writes back half of a boundary's evictions.  The test pass right after
    each install (--test-freq = --lookahead) must see both halves: two identical runs print identical metrics."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = []
    for port in (29871, 29872):
        argv = [a for a in _RUN] + ["--test-freq", "4", "--master-port", str(port)]
        argv[argv.index("--world-size") + 1] = "2"
        argv[argv.index("--mini-batch-size") + 1] = "128"
        res = subprocess.run([sys.executable, "-c", _MGPU.format(root=root, argv=argv)], capture_output=True,
                             text=True, timeout=600, cwd=root)
        assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
        outs.append(re.findall(r"^Test (?:accuracy|loss) = .*$", res.stdout, re.M))
    assert len(outs[0]) == 2 * 4 and outs[0] == outs[1]


# ---------------------------------------------------------------------------------------------------------------------
# 6. Run and --inference-only
# ---------------------------------------------------------------------------------------------------------------------

_RUN = ["--data-generation", "synthetic", "--arch-embedding-size", "3000-40-900", "--arch-sparse-feature-size", "16",
        "--arch-mlp-bot", "13-32-16", "--arch-mlp-top", "32-1", "--loss-function", "bce", "--mini-batch-size", "64",
        "--num-batches", "16", "--lookahead", "4", "--cache-size", "50", "--num-ways", "2", "--world-size", "1",
        "--print-freq", "100", "--eviction-fifo-timeout", "2", "--numpy-rand-seed", "9"]


def _old_test_accuracy(tr, test_ld):
    acc = samp = 0
    with torch.no_grad():
        for Xt, lS_ot, lS_it, Tt in test_ld:
            lookups, _ = tr.cache_group(lS_ot, lS_it.to(DEV), tr.emb_tables, 0)
            Zt = tr.dlrm(Xt.to(DEV), lookups)
            acc += int((Zt.round().cpu() == Tt).sum())
            samp += Tt.shape[0]
    tr.cache_group.check_device_flags()
    return 100 * (acc / max(samp, 1))


def _test_ld(argv):
    from cdlrm_b200 import main_no_ddp as R
    from cdlrm_b200.synthetic import make_synthetic_data_and_loaders
    args = R.ProcessArgs(argv)
    ln_emb, _b, _t, _m, m_den = R._derive_topology(args)
    return make_synthetic_data_and_loaders(args, ln_emb, m_den)[1]


def test_run_prints_accuracy_loss_and_auc(capsys):
    from cdlrm_b200 import main_no_ddp as R
    argv = _RUN + ["--test-freq", "8"]
    tr = R.main(argv)
    out = capsys.readouterr().out
    acc = re.findall(r"^Test accuracy = (.*)%$", out, re.M)
    la = re.findall(r"^Test loss = (.*), AUC = (.*)$", out, re.M)
    assert len(acc) == 2 and len(la) == 2
    assert 0.0 < float(la[-1][0]) and 0.0 <= float(la[-1][1]) <= 1.0
    assert acc[-1] == str(_old_test_accuracy(tr, _test_ld(argv)))


def test_inference_only_evaluates_a_checkpoint(tmp_path, capsys):
    from cdlrm_b200 import main_no_ddp as R
    path = str(tmp_path / "ck")
    R.main(_RUN + ["--save-model", path])
    capsys.readouterr()
    files = {f: open(os.path.join(path, f), "rb").read() for f in sorted(os.listdir(path))}
    tr = R.main(_RUN + ["--inference-only", "--load-model", path])
    out = capsys.readouterr().out
    la = re.findall(r"^Test loss = (.*), AUC = (.*)$", out, re.M)
    assert len(re.findall(r"^Test accuracy = .*%$", out, re.M)) == 1 and len(la) == 1
    assert tr.global_step == 16 and tr._n_submitted == tr.window    # nothing trained, no window submitted
    assert {f: open(os.path.join(path, f), "rb").read() for f in sorted(os.listdir(path))} == files
    for k, E in enumerate(tr.emb_tables.emb_l):
        assert E.weight.data.numpy().tobytes() == files[f"master_{k}.bin"]
    test_ld = _test_ld(_RUN)
    r = tr.evaluate(test_ld)
    assert repr(r.auc) == la[0][1] or str(r.auc) == la[0][1]
    tr2 = R.Trainer(tr.args, 16, np.asarray([3000, 40, 900]), np.asarray([13, 32, 16]), np.asarray([22, 32, 1]),
                    tr.emb_tables, rank=0, world=1, device=torch.device(DEV))
    tr2.load_checkpoint(path)
    assert tr2.evaluate(test_ld).auc == r.auc
