#!/usr/bin/env python
"""Cost of ``Trainer.evaluate`` at the Terabyte cache shape (26 tables, 150001 sets x 16 ways, dim 128, MLPs
13-512-256-128 / 479-512-256-1):

  * evaluation throughput (samples/s) at test batch 8192 and 65536, inputs generated on the device by SyntheticStream
    (a test stream of its own seed), the evaluation step replayed from its CUDA graph;
  * the share of looked-up rows served from the cache, from the loser store of the installed window and from the
    host master (zero-copy);
  * ``cdlrm_eval_result`` (the AUC pass) at 10^7 and 9 x 10^7 accumulated samples;
  * the ``_quiesce`` wait of an evaluation that starts right after a window boundary (plan of the next window and
    write-back of the boundary's evictions still running).

The cache is trained by windows of the zipf synthetic stream (installs only: the steps would not change what is
measured).  ``--max-rows`` caps every master table so that the master fits the machine.  Writes one JSON file with
the GPU's name and power limit.  Needs a CUDA device: there is no CPU path.

  python tools/eval_time.py --json profiles/eval_time_b200.json
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def build(args, ln_emb):
    from cdlrm_b200.main_no_ddp import ProcessArgs, Trainer
    from cdlrm_b200.model_no_ddp import Embedding_Table_Group
    dev = torch.device("cuda", 0)
    pa = ProcessArgs(["--arch-sparse-feature-size", "128", "--arch-mlp-bot", "13-512-256-128", "--arch-mlp-top",
                      "512-512-256-1", "--loss-function", "bce", "--mini-batch-size", str(args.batch), "--lookahead",
                      str(args.lookahead), "--cache-size", "150000", "--num-ways", "16", "--world-size", "1"])
    master = Embedding_Table_Group(128, np.asarray(ln_emb), init="device")
    nf = len(ln_emb) + 1
    tr = Trainer(pa, 128, np.asarray(ln_emb), np.asarray([13, 512, 256, 128]),
                 np.asarray([nf * (nf - 1) // 2 + 128, 512, 256, 1]), master, rank=0, world=1, device=dev)
    return tr


def test_batches(ln_emb, batch, n, dev):
    from cdlrm_b200.synthetic import SyntheticStream
    st = SyntheticStream(ln_emb, batch, dev, seed=777)
    X, T = st.dense_and_labels(0, n)
    ids = st.ids(0, n)
    lS_o = torch.arange(batch).reshape(1, -1).repeat(len(ln_emb), 1)
    return [(X[i * batch:(i + 1) * batch], lS_o, ids[:, i * batch:(i + 1) * batch].contiguous(),
             T[i * batch:(i + 1) * batch]) for i in range(n)]


def served_from(tr, batches):
    """Rows served from the cache, the loser store and the master for the ids of ``batches``."""
    cg, rec = tr.cache_group, tr._installed
    hit = los = tot = 0
    for k in range(len(cg.emb_l)):
        tags = cg.occupancy_tables[k]
        losers = rec.loser_list(k) if rec is not None and rec.loser_ids is not None else None
        for _X, _o, ids, _T in batches:
            i = ids[k]
            h = (tags[i % cg.cache_sizes[k]] == i[:, None]).any(1)
            hit += int(h.sum())
            if losers is not None and losers.numel():
                pos = torch.searchsorted(losers, i).clamp_(max=losers.numel() - 1)
                los += int(((losers[pos] == i) & ~h).sum())
            tot += i.numel()
    return {"cache": round(hit / tot, 4), "loser_store": round(los / tot, 4), "master": round((tot - hit - los) / tot, 4)}


def result_time(n, dev, reps=3):
    from cdlrm_b200._lib import EvalStats, check, lib
    h = ctypes.c_void_p()
    check(lib.cdlrm_eval_create(ctypes.byref(h), dev.index, n))
    s = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    z = torch.rand(n, device=dev)
    t = (torch.rand(n, device=dev) < 0.25).float()
    check(lib.cdlrm_eval_reset(h, s))
    check(lib.cdlrm_eval_accumulate(h, ctypes.c_void_p(z.data_ptr()), 1, ctypes.c_void_p(t.data_ptr()), 1, n, s))
    st = EvalStats()
    times = []
    for _ in range(reps):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        check(lib.cdlrm_eval_result(h, ctypes.c_void_p(ctypes.addressof(st)), s))
        times.append(time.perf_counter() - t0)
    check(lib.cdlrm_eval_destroy(h))
    assert st.samples == n and st.flags == 0
    return {"samples": n, "ms": [round(1e3 * x, 2) for x in times], "auc": st.auc_2u / (2.0 * st.positives * st.negatives)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--json", required=True, help="result file")
    ap.add_argument("--max-rows", type=int, default=2_500_000, help="rows per master table at most")
    ap.add_argument("--batch", type=int, default=8192, help="training batch")
    ap.add_argument("--lookahead", type=int, default=1000)
    ap.add_argument("--test-samples", type=int, default=3 * 65536 * 16)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("eval_time.py needs a CUDA device")
    from cdlrm_b200.synthetic import TERABYTE_ROWS, SyntheticStream
    dev = torch.device("cuda", 0)
    ln_emb = [min(int(n), args.max_rows) for n in TERABYTE_ROWS]
    res = {"gpu": torch.cuda.get_device_name(dev), "ln_emb": ln_emb, "dim": 128, "num_ways": 16, "cache_size": 150000,
           "window": {"batch": args.batch, "lookahead": args.lookahead, "dist": "zipf"}}
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        res["power_limit"] = f"unknown ({e})"

    def dump():
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)

    tr = build(args, ln_emb)
    res["pcie_mode"] = tr.planner.pcie_mode
    sg = SyntheticStream(ln_emb, args.batch, dev, seed=3)
    tr.submit_window(sg.window_ids(0, args.lookahead))
    tr.install_window()
    tr.submit_window(sg.window_ids(1, args.lookahead))
    tr.install_window()                            # window 1 installed: evictions, write-back pending
    tr.submit_window(sg.window_ids(2, args.lookahead))
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    tr._quiesce()
    res["quiesce_after_boundary_s"] = round(time.perf_counter() - t0, 4)
    res["evictions_at_boundary"] = int(sum(tr._installed.E))
    res["valid_lines"] = int(sum(int((t >= 0).sum()) for t in tr.cache_group.occupancy_tables))
    dump()
    res["evaluate"] = {}
    for tb in (8192, 65536):
        n = max(4, args.test_samples // tb)
        batches = test_batches(ln_emb, tb, n, dev)
        tr.evaluate(batches[:3])                   # warm-up: eager batch, capture, replay
        runs = []
        for _ in range(3):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            r = tr.evaluate(batches)
            runs.append(time.perf_counter() - t0)
        res["evaluate"][str(tb)] = {"batches": n, "samples": r.samples, "s": [round(x, 4) for x in runs],
                                    "samples_per_s": round(r.samples / min(runs)), "auc": r.auc, "loss": r.loss,
                                    "served_from": served_from(tr, batches[:8])}
        del batches
        dump()
    torch.cuda.empty_cache()
    res["eval_result"] = {str(n): result_time(n, dev) for n in (10_000_000, 90_000_000)}
    dump()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
