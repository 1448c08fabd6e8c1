"""The MLPerf binary Criteo loader on the GPU (cdlrm_b200/criteo_bin.py, csrc/criteo.cu):

(a) cdlrm_criteo_decode against the host decode (ids, offsets, labels exact; X bit for bit equal to torch's CUDA log
    and within 1 ulp of its CPU log), padded leading dimensions, NULL outputs;
(b) the device batch stream against the host batches, its resume point, its errors and its reader thread;
(c) the window scan through markers against planning the concatenated window ids;
(d) a Trainer fed by the device stream and markers against the same batches fed as tensors (decisions bit for bit);
(e) main(--data-generation dataset --mlperf-bin-loader): training lifts the AUC, save + load resume equals the
    uninterrupted run, --inference-only evaluates the test file.
Files are written under tmp_path (a few MB)."""
import re
import threading

import numpy as np
import pytest
import torch

import util  # noqa: F401

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rand_records(n, seed, neg=True, hi=1 << 20):
    rng = np.random.default_rng(seed)
    rec = np.empty((n, 40), np.int32)
    rec[:, 0] = rng.integers(0, 2, n)
    rec[:, 1:14] = rng.integers(-2 if neg else 0, 1 << 16, (n, 13))
    rec[:, 14:] = rng.integers(-hi if neg else 0, hi, (n, 26))
    return rec


def _write(path, rec):
    rec.astype("<i4").tofile(str(path))
    return str(path)


def _counts(path, counts):
    np.savez(str(path), counts=np.asarray(counts))
    return str(path)


def _decode(rec_d, n, mir, ld_x=13, ld_ids=None, want=(True, True, True)):
    from cdlrm_b200._lib import check, lib, vp
    ld_ids = n if ld_ids is None else ld_ids
    X = torch.full((max(n, 1), ld_x), 7.0, device=DEV)
    ids = torch.full((26, max(ld_ids, 1)), -7, dtype=torch.int64, device=DEV)
    T = torch.full((max(n, 1),), 7.0, device=DEV)
    s = torch.cuda.current_stream()
    check(lib.cdlrm_criteo_decode(0, vp(rec_d.data_ptr()), n, 13, 26, mir, vp(X.data_ptr()) if want[0] else None,
                                  ld_x, vp(ids.data_ptr()) if want[1] else None, ld_ids,
                                  vp(T.data_ptr()) if want[2] else None, vp(s.cuda_stream)))
    torch.cuda.synchronize()
    return X, ids, T


def _host(rec, mir):
    from cdlrm_b200.criteo_bin import _transform_features
    t = torch.from_numpy(rec)
    return _transform_features(t[:, 1:14], t[:, 14:], t[:, 0], mir)


def _ulp_le1(a, b):
    a, b = a.cpu().numpy(), b.cpu().numpy()
    assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.isinf(a), np.isinf(b))
    f = np.isfinite(b)
    assert np.array_equal(a[~f & ~np.isnan(a)], b[~f & ~np.isnan(b)])
    np.testing.assert_array_max_ulp(a[f], b[f], maxulp=1)


@pytest.mark.parametrize("n", [1, 127, 128, 8192, 8193, 1000003])
@pytest.mark.parametrize("mir", [-1, 1000])
def test_decode_matches_host(n, mir):
    rec = _rand_records(n, seed=n)
    rec_d = torch.from_numpy(rec).to(DEV)
    hX, hO, hI, hT = _host(rec, mir)
    X, ids, T = _decode(rec_d, n, mir)
    assert torch.equal(ids.cpu(), hI) and torch.equal(T.view(-1, 1).cpu(), hT)
    assert torch.equal(hO, torch.arange(n).reshape(1, -1).repeat(26, 1))
    ref = torch.log(rec_d[:, 1:14].float() + 1)
    assert torch.equal(torch.nan_to_num(X, nan=1e30), torch.nan_to_num(ref, nan=1e30))
    assert torch.equal(X.isnan(), ref.isnan())
    _ulp_le1(X, hX)
    # padded leading dimensions: the padding is left alone
    X2, ids2, _T2 = _decode(rec_d, n, mir, ld_x=16, ld_ids=n + 5)
    assert torch.equal(torch.nan_to_num(X2[:, :13], nan=1e30), torch.nan_to_num(X, nan=1e30))
    assert bool((X2[:, 13:] == 7.0).all()) and torch.equal(ids2[:, :n], ids) and bool((ids2[:, n:] == -7).all())
    # NULL outputs are not written (the window scan asks for ids only)
    X3, ids3, T3 = _decode(rec_d, n, mir, want=(False, True, False))
    assert torch.equal(ids3, ids) and bool((X3 == 7.0).all()) and bool((T3 == 7.0).all())


def test_dense_log_within_one_ulp_of_host_for_every_integer():
    vals = np.arange(-1, (1 << 24) + 1, dtype=np.int64)
    n = -(-vals.size // 13)
    rec = np.zeros((n, 40), np.int32)
    flat = np.full(n * 13, 5, np.int64)
    flat[:vals.size] = vals
    rec[:, 1:14] = flat.reshape(n, 13)
    rec_d = torch.from_numpy(rec).to(DEV)
    X, _ids, _T = _decode(rec_d, n, -1, want=(True, False, False))
    assert torch.equal(X, torch.log(rec_d[:, 1:14].float() + 1))
    _ulp_le1(X, torch.log(torch.from_numpy(rec[:, 1:14]).float() + 1))


def _dataset(tmp_path, n=3000, B=256, seed=1, mir=-1, name="d_train.bin"):
    from cdlrm_b200.criteo_bin import CriteoBinDataset
    rec = _rand_records(n, seed, hi=5000)
    f = _write(tmp_path / name, rec)
    return CriteoBinDataset(f, _counts(tmp_path / "c.npz", [5000] * 26), batch_size=B, max_ind_range=mir), rec


def _same_batch(got, want):
    X, lS_o, lS_i, T = got
    hX, hO, hI, hT = want
    assert X.is_cuda and lS_o.is_cuda and lS_i.is_cuda and T.is_cuda
    assert torch.equal(lS_o.cpu(), hO) and torch.equal(lS_i.cpu(), hI) and torch.equal(T.cpu(), hT)
    assert lS_i.is_contiguous() and X.shape == hX.shape
    _ulp_le1(X, hX)


@pytest.mark.parametrize("mir", [-1, 777])
def test_device_stream_equals_host_batches(tmp_path, monkeypatch, mir):
    from cdlrm_b200 import criteo_bin as CB
    monkeypatch.setattr(CB, "CHUNK_BYTES", 3 * 256 * 160)       # 3 batches per chunk: many chunk turns
    ds, _rec = _dataset(tmp_path, mir=mir)
    assert len(ds) == 12                                          # 11 full batches and 184 records
    stream = ds.device_batches(DEV)
    lsos = set()
    for j, b in enumerate(stream):
        _same_batch(b, ds[j])
        if j < 11:
            lsos.add(id(b[1]))
    assert j == 11 and len(lsos) == 1 and stream.bytes_read == 3000 * 160
    # resume at a batch: nothing before it is read
    st = ds.device_batches(DEV, start=5)
    assert len(st) == 7
    it = iter(st)
    for j, b in enumerate(it, 5):
        _same_batch(b, ds[j])
    assert it.bytes_read == (3000 - 5 * 256) * 160 and it.thread is None
    # an iterator dropped part-way, or closed, joins its reader
    it = iter(ds.device_batches(DEV))
    next(it)
    th = it.thread
    it.close()
    assert not th.is_alive()
    it = iter(ds.device_batches(DEV))
    next(it)
    th = it.thread
    del it
    assert not th.is_alive()
    assert not any(t.name == "criteo-bin-reader" for t in threading.enumerate())


def test_device_stream_raises_a_short_read_in_the_consumer(tmp_path, monkeypatch):
    from cdlrm_b200 import criteo_bin as CB
    monkeypatch.setattr(CB, "CHUNK_BYTES", 2 * 256 * 160)
    ds, _rec = _dataset(tmp_path)
    with open(ds.data_file, "r+b") as f:
        f.truncate(5 * 256 * 160)                                 # the file shrinks after the dataset was opened
    it = iter(ds.device_batches(DEV))
    with pytest.raises(IOError, match="short read"):
        for _ in it:
            pass
    assert it.thread is None


# ---- planner and trainer ------------------------------------------------------------------------------------------

LN = [8] + [int(x) for x in np.random.default_rng(4).integers(20, 500, 25)]


def _trainer_args(B, L, extra=()):
    from cdlrm_b200 import main_no_ddp as R
    return R.ProcessArgs(["--arch-sparse-feature-size", "16", "--loss-function", "bce", "--learning-rate", "0.1",
                          "--lr-embeds", "0.3", "--mini-batch-size", str(B), "--lookahead", str(L), "--cache-size",
                          "16", "--num-ways", "4", "--numpy-rand-seed", "3", "--world-size", "1"] + list(extra))


def _trainer(B, L):
    from cdlrm_b200 import main_no_ddp as R
    from cdlrm_b200 import model_no_ddp as M
    np.random.seed(3)
    torch.manual_seed(3)
    master = M.Embedding_Table_Group(16, np.asarray(LN))
    tr = R.Trainer(_trainer_args(B, L), 16, np.asarray(LN), np.asarray([13, 32, 16]),
                   np.asarray([27 * 26 // 2 + 16, 32, 1]), master, rank=0, world=1, device=torch.device(DEV))
    return tr, master


def _ds_small(tmp_path, n, B, seed=2):
    from cdlrm_b200.criteo_bin import CriteoBinDataset
    rng = np.random.default_rng(seed)
    rec = np.empty((n, 40), np.int32)
    rec[:, 1:14] = rng.integers(0, 101, (n, 13))
    for k, m in enumerate(LN):
        rec[:, 14 + k] = rng.integers(0, m, n)
    rec[:, 0] = rec[:, 14] < 4
    f = _write(tmp_path / "s_train.bin", rec)
    return CriteoBinDataset(f, _counts(tmp_path / "s_fea_count.npz", LN), batch_size=B), rec


def _decisions(tr, rec):
    torch.cuda.synchronize()
    out = [np.concatenate([t.cpu().numpy().ravel() for t in tr.cache_group.occupancy_tables])]
    for k in range(len(LN)):
        out += [x.cpu().numpy().copy() for x in rec.fill_list(k)]
        out += [x.cpu().numpy().copy() for x in rec.evict_list(k)]
        out.append(rec.loser_list(k).cpu().numpy().copy())
    return out


def test_window_scan_equals_concatenated_window_ids(tmp_path, monkeypatch):
    from cdlrm_b200 import criteo_bin as CB
    monkeypatch.setattr(CB, "CHUNK_BYTES", 1000 * 160)            # several chunks per window, one chunk across windows
    B, L = 128, 5
    ds, _rec = _ds_small(tmp_path, 128 * 5 * 3 + 300, B)          # 3 full windows, a short one of 3 batches
    nw = -(-len(ds) // L)
    assert nw == 4
    a, _ma = _trainer(B, L)
    b, _mb = _trainer(B, L)
    for w in range(nw):
        a.submit_window(ds.window_marker(w, L))
        b.submit_window(torch.cat([ds[j][2] for j in range(w * L, min((w + 1) * L, len(ds)))], dim=1).to(DEV))
        ra, rb = a.install_window(), b.install_window()
        da, db = _decisions(a, ra), _decisions(b, rb)
        assert list(ra.E) == list(rb.E) and list(ra.F) == list(rb.F) and list(ra.L) == list(rb.L), w
        for x, y in zip(da, db):
            assert np.array_equal(x, y), f"window {w}"
    a.finish()
    b.finish()


def _run(tr, windows, batches, L, n_steps):
    """Windows submitted one ahead, a boundary every L steps, the step captured after one eager step."""
    losses, tags = [], []
    tr.submit_window(windows(0))
    nw = -(-n_steps // L)
    for w in range(nw):
        tr.install_window()
        if w + 1 < nw:
            tr.submit_window(windows(w + 1))
        tags.append(np.concatenate([t.cpu().numpy().ravel() for t in tr.cache_group.occupancy_tables]))
        for _ in range(w * L, min((w + 1) * L, n_steps)):
            X, lS_o, lS_i, T = next(batches)
            if getattr(tr, "_graph", None) is None and len(losses) == 1:
                tr.capture_graph(X, lS_o, lS_i, T)
            E, _Z = tr.step(X, lS_o, lS_i, T)
            losses.append(E.detach().clone())
    tr.finish()
    return np.asarray([float(x) for x in losses]), tags


def test_trainer_fed_from_the_file_equals_tensor_fed(tmp_path):
    B, L = 128, 4
    ds, _rec = _ds_small(tmp_path, B * L * 3, B)
    n = len(ds)
    assert n == 12
    same = [tuple(t.clone() for t in b) for b in ds.device_batches(DEV)]     # the stream's own decoded batches
    a, ma = _trainer(B, L)
    it = iter(ds.device_batches(DEV))
    la, ta = _run(a, lambda w: ds.window_marker(w, L), it, L, n)
    b, mb = _trainer(B, L)
    lb, tb = _run(b, lambda w: torch.cat([same[j][2] for j in range(w * L, (w + 1) * L)], dim=1), iter(same), L, n)
    assert a._graph is not None and b._graph is not None
    # cache decisions bit for bit; values to the bars test_gpu_checkpoint.py uses for two runs: two Trainers fed the same
    # tensors differ in the last bit of some losses and parameters, so the file-fed run is held to that bar too
    for x, y in zip(ta, tb):
        assert np.array_equal(x, y)
    assert np.all(np.isfinite(la))
    np.testing.assert_allclose(la, lb, rtol=1e-6)
    for e, f in zip(a.cache_group.emb_l, b.cache_group.emb_l):
        torch.testing.assert_close(e.weight.data, f.weight.data, rtol=0, atol=1e-6)
    for e, f in zip(ma.emb_l, mb.emb_l):
        torch.testing.assert_close(e.weight.data, f.weight.data, rtol=0, atol=1e-6)
    for p, q in zip(a.dlrm.parameters(), b.dlrm.parameters()):
        torch.testing.assert_close(p.data, q.data, rtol=0, atol=1e-6)


# ---- CLI ----------------------------------------------------------------------------------------------------------

def _cli_files(tmp_path):
    rng = np.random.default_rng(11)

    def rec(n):
        r = np.empty((n, 40), np.int32)
        r[:, 1:14] = rng.integers(0, 101, (n, 13))
        for k, m in enumerate(LN):
            r[:, 14 + k] = rng.integers(0, m, n)
        r[:, 0] = r[:, 14] < 4                   # the label is a function of the id of table 0 (8 rows)
        return r

    _write(tmp_path / "tb_train.bin", rec(128 * 16 + 64))       # 17 batches of 128: 5 windows of 4, the last short
    _write(tmp_path / "tb_test.bin", rec(1000))
    _counts(tmp_path / "day_fea_count.npz", LN)
    return ["--data-generation", "dataset", "--mlperf-bin-loader", "--processed-data-file",
            str(tmp_path / "tb.npz"), "--raw-data-file", str(tmp_path / "day"), "--world-size", "1",
            "--arch-sparse-feature-size", "16", "--arch-mlp-bot", "13-32-16", "--arch-mlp-top", "32-1",
            "--loss-function", "bce", "--learning-rate", "0.1", "--lr-embeds", "0.3", "--mini-batch-size", "128",
            "--test-mini-batch-size", "256", "--lookahead", "4", "--cache-size", "16", "--num-ways", "4",
            "--print-freq", "8", "--eviction-fifo-timeout", "2"]


def _auc(out):
    la = re.findall(r"^Test loss = (.*), AUC = (.*)$", out, re.M)
    assert la, out
    return [float(a) for _l, a in la]


def _main_keep(argv):
    from cdlrm_b200 import main_no_ddp as R
    orig = R.Trainer.__init__

    def _init(self, *a, **kw):
        orig(self, *a, **kw)
        self.keep_losses = True
    R.Trainer.__init__ = _init
    try:
        return R.main(argv)
    finally:
        R.Trainer.__init__ = orig


def test_main_trains_on_a_binary_dataset_and_resumes(tmp_path, capsys):
    from cdlrm_b200 import main_no_ddp as R
    base = _cli_files(tmp_path)
    R.main(base + ["--inference-only"])                          # the freshly initialised model
    fresh = _auc(capsys.readouterr().out)
    assert len(fresh) == 1
    a = _main_keep(base + ["--nepochs", "2"])
    out = capsys.readouterr().out
    auc = _auc(out)
    assert out.count("Finished") == 4 and len(auc) == 2 and a._graph is not None
    assert auc[-1] > 0.75 and auc[-1] > fresh[0], (fresh, auc)
    path = str(tmp_path / "ck")
    b1 = _main_keep(base + ["--nepochs", "1", "--save-model", path])
    auc1 = _auc(capsys.readouterr().out)[-1]
    b2 = _main_keep(base + ["--nepochs", "2", "--load-model", path])
    out = capsys.readouterr().out
    la = np.asarray([float(x) for x in a.loss_history])
    lb = np.asarray([float(x) for x in b1.loss_history + b2.loss_history])
    assert len(la) == 34 and len(lb) == 34
    np.testing.assert_allclose(lb, la, rtol=1e-6)
    for x, y in zip(a.cache_group.occupancy_tables, b2.cache_group.occupancy_tables):
        assert torch.equal(x, y)
    for x, y in zip(a.emb_tables.emb_l, b2.emb_tables.emb_l):
        np.testing.assert_allclose(x.weight.data.numpy(), y.weight.data.numpy(), rtol=0, atol=1e-6)
    np.testing.assert_allclose(_auc(out)[-1], auc[-1], rtol=0, atol=1e-4)    # (last-bit value differences may swap a tie)
    tr = R.main(base + ["--inference-only", "--load-model", path])
    ev = _auc(capsys.readouterr().out)
    assert len(ev) == 1 and tr.global_step == 17
    np.testing.assert_allclose(ev[0], auc1, rtol=0, atol=1e-6)
