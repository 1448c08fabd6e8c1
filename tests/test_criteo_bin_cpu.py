"""The MLPerf binary Criteo loader on the host (cdlrm_b200/criteo_bin.py): ``CriteoBinDataset`` against a numpy
restatement of the format, ``numpy_to_binary``, the upstream path rules, ``ln_emb`` / ``ln_bot[0]`` from the counts
file, the refusals, and ``cdlrm_criteo_decode``'s argument checks and its failure without a device."""
import ctypes
import os

import numpy as np
import pytest
import torch

import util  # noqa: F401  (puts the repository on sys.path)


def _records(n, seed=0, neg=False, hi=1000):
    rng = np.random.default_rng(seed)
    y = rng.integers(0, 2, n)
    X_int = rng.integers(-3 if neg else 0, 101, (n, 13))
    X_cat = rng.integers(-hi if neg else 0, hi, (n, 26))
    return y, X_int, X_cat


def _npz(path, y, X_int, X_cat):
    np.savez(path, y=y, X_int=X_int, X_cat=X_cat)
    return str(path)


def _counts(path, counts):
    np.savez(path, counts=np.asarray(counts))
    return str(path)


def _expect(y, X_int, X_cat, B, j, mir):
    """numpy restatement of batch j: X = log(x + 1) in float32, ids = x_cat floor-mod mir (sign of the divisor),
    table-major; offsets arange(b) per table; labels [b, 1]."""
    lo, hi = j * B, min((j + 1) * B, len(y))
    c = X_cat[lo:hi].astype(np.int64)
    if mir > 0:
        c = np.mod(c, mir)
    with np.errstate(divide="ignore", invalid="ignore"):
        X = np.log(X_int[lo:hi].astype(np.float32) + np.float32(1))
    return X, np.tile(np.arange(hi - lo), (26, 1)), c.T, y[lo:hi].astype(np.float32).reshape(-1, 1)


@pytest.mark.parametrize("mir", [-1, 0, 97])
@pytest.mark.parametrize("neg", [False, True])
def test_dataset_matches_numpy_restatement(tmp_path, mir, neg):
    from cdlrm_b200.criteo_bin import CriteoBinDataset, numpy_to_binary
    y, X_int, X_cat = _records(1000, seed=3, neg=neg)
    data = str(tmp_path / "d_train.bin")
    numpy_to_binary([_npz(tmp_path / "a.npz", y, X_int, X_cat)], data)
    cnt = _counts(tmp_path / "c.npz", [1000] * 26)
    B = 64
    ds = CriteoBinDataset(data, cnt, batch_size=B, max_ind_range=mir)
    assert len(ds) == 16 and ds.num_samples == 1000 and ds.m_den == 13     # ceil(1000 / 64), the last batch is short
    assert list(ds.counts) == [1000] * 26
    for j in range(len(ds)):
        X, lS_o, lS_i, T = ds[j]
        eX, eo, ei, eT = _expect(y, X_int, X_cat, B, j, mir)
        b = 1000 - 15 * B if j == 15 else B
        assert X.shape == (b, 13) and X.dtype == torch.float32
        assert lS_i.shape == (26, b) and lS_i.dtype == torch.int64 and T.shape == (b, 1) and T.dtype == torch.float32
        assert np.array_equal(lS_o.numpy(), eo) and np.array_equal(lS_i.numpy(), ei) and np.array_equal(T.numpy(), eT)
        got = X.numpy()
        assert np.array_equal(np.isnan(got), np.isnan(eX)) and np.array_equal(np.isinf(got), np.isinf(eX))
        fin = np.isfinite(eX)
        np.testing.assert_array_max_ulp(got[fin], eX[fin], maxulp=1)
    with pytest.raises(IndexError):
        ds[len(ds)]
    assert sum(1 for _ in ds) == len(ds)


def test_numpy_to_binary_round_trip_and_halves(tmp_path):
    from cdlrm_b200.criteo_bin import numpy_to_binary
    parts = [_records(n, seed=n) for n in (7, 12)]
    files = [_npz(tmp_path / f"day_{i}.npz", *p) for i, p in enumerate(parts)]
    numpy_to_binary(files, str(tmp_path / "train.bin"), split="train")
    got = np.fromfile(str(tmp_path / "train.bin"), dtype="<i4").reshape(-1, 40)
    want = np.concatenate([np.concatenate([p[0].reshape(-1, 1), p[1], p[2]], axis=1) for p in parts]).astype(np.int32)
    assert np.array_equal(got, want)
    odd = _records(13, seed=5)
    f = _npz(tmp_path / "day_23.npz", *odd)
    numpy_to_binary([f], str(tmp_path / "test.bin"), split="test")
    numpy_to_binary([f], str(tmp_path / "val.bin"), split="val")
    full = np.concatenate([odd[0].reshape(-1, 1), odd[1], odd[2]], axis=1).astype(np.int32)
    assert np.array_equal(np.fromfile(str(tmp_path / "test.bin"), dtype="<i4").reshape(-1, 40), full[:7])
    assert np.array_equal(np.fromfile(str(tmp_path / "val.bin"), dtype="<i4").reshape(-1, 40), full[7:])
    with pytest.raises(ValueError):
        numpy_to_binary(files, str(tmp_path / "x.bin"), split="test")
    with pytest.raises(ValueError):
        numpy_to_binary([f], str(tmp_path / "x.bin"), split="dev")


def _args(extra):
    from cdlrm_b200.main_no_ddp import ProcessArgs
    return ProcessArgs(extra)


def test_paths_and_topology_from_the_counts_file(tmp_path):
    from cdlrm_b200.criteo_bin import bin_paths
    from cdlrm_b200.main_no_ddp import _derive_topology
    a = _args(["--processed-data-file", "/data/tb/terabyte_processed.npz", "--raw-data-file", "/data/tb/day"])
    assert bin_paths(a) == ("/data/tb/terabyte_processed_train.bin", "/data/tb/terabyte_processed_test.bin",
                            "/data/tb/day_fea_count.npz")
    counts = [5, 1000, 70, 3] + [40] * 22
    _counts(tmp_path / "day_fea_count.npz", counts)
    base = ["--data-generation", "dataset", "--mlperf-bin-loader", "--world-size", "1",
            "--processed-data-file", str(tmp_path / "t.npz"), "--raw-data-file", str(tmp_path / "day"),
            "--arch-embedding-size", "4-3-2", "--arch-mlp-bot", "4-32-16", "--arch-sparse-feature-size", "16",
            "--arch-mlp-top", "32-1"]
    ln_emb, ln_bot, ln_top, m_spa, m_den = _derive_topology(_args(base))
    assert list(ln_emb) == counts and list(ln_bot) == [13, 32, 16] and m_den == 13 and m_spa == 16
    assert list(ln_top) == [27 * 26 // 2 + 16, 32, 1]
    ln_emb, *_ = _derive_topology(_args(base + ["--max-ind-range", "50"]))
    assert list(ln_emb) == [min(c, 50) for c in counts]


def test_refusals(tmp_path):
    from cdlrm_b200.criteo_bin import CriteoBinDataset
    from cdlrm_b200.main_no_ddp import _derive_topology
    bad = tmp_path / "bad_train.bin"
    bad.write_bytes(b"\0" * 161)
    cnt = _counts(tmp_path / "c.npz", [10] * 26)
    with pytest.raises(ValueError, match="bad_train.bin"):
        CriteoBinDataset(str(bad), cnt)
    good = tmp_path / "good_train.bin"
    good.write_bytes(b"\0" * 320)
    wrong = _counts(tmp_path / "wrong_fea_count.npz", [10] * 25)
    with pytest.raises(ValueError, match="wrong_fea_count.npz"):
        CriteoBinDataset(str(good), wrong)
    _counts(tmp_path / "day_fea_count.npz", [10] * 26)
    base = ["--data-generation", "dataset", "--mlperf-bin-loader", "--processed-data-file", str(tmp_path / "t.npz"),
            "--raw-data-file", str(tmp_path / "day")]
    for extra, flag in ((["--world-size", "2"], "--world-size"),
                        (["--world-size", "1", "--mlperf-bin-shuffle"], "--mlperf-bin-shuffle")):
        with pytest.raises(SystemExit, match=flag):
            _derive_topology(_args(base + extra))
    with pytest.raises(SystemExit, match="--mlperf-bin-loader"):
        _derive_topology(_args(["--data-generation", "dataset", "--world-size", "1"]))


def test_prefetcher_puts_one_marker_per_window(tmp_path):
    from cdlrm_b200.cache_manager import Prefetcher
    from cdlrm_b200.criteo_bin import CriteoBinDataset, numpy_to_binary
    numpy_to_binary([_npz(tmp_path / "a.npz", *_records(700))], str(tmp_path / "t_train.bin"))
    ds = CriteoBinDataset(str(tmp_path / "t_train.bin"), _counts(tmp_path / "c.npz", [1000] * 26), batch_size=32)
    args = _args(["--lookahead", "4", "--nepochs", "2", "--fifo-payload", "ids"])
    got = list(Prefetcher(args, None, None, None, None, ds).payloads())
    assert len(got) == 2 * 6 and all(callable(m) for m in got)        # 22 batches: 5 full windows and a short one


def test_decode_checks_arguments_and_fails_without_a_device():
    from cdlrm_b200 import _lib
    lib, vp = _lib.lib, ctypes.c_void_p
    rec = np.zeros((8, 40), np.int32)
    X = np.zeros((8, 13), np.float32)
    ids = np.zeros((26, 8), np.int64)
    T = np.zeros(8, np.float32)
    p = lambda a, off=0: vp(a.ctypes.data + off)          # noqa: E731
    ok = (0, p(rec), 8, 13, 26, -1, p(X), 13, p(ids), 8, p(T), None)
    for i, v in ((2, -1), (3, -1), (4, -2), (7, 12), (9, 7), (1, p(rec, 2))):
        a = list(ok)
        a[i] = v
        assert lib.cdlrm_criteo_decode(*a) != 0 and b"bad argument" in lib.cdlrm_last_error()
    a = list(ok)
    a[2] = 0
    assert lib.cdlrm_criteo_decode(*a) == 0                # n == 0: nothing to launch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert lib.cdlrm_criteo_decode(*ok) != 0 and lib.cdlrm_last_error() != b""
    assert not X.any() and not ids.any() and not T.any()
    assert os.path.exists(_lib.LIB_PATH)
