#!/usr/bin/env python
"""Cost of ``--evict-victim-cache`` at the bench's Terabyte shape (26 tables, dim 128, bottom 13-512-256-128, top
512-512-256-1, batch 8192, 150000 sets x 16 ways; masters capped at ``--max-rows`` rows and kept in HBM, as
lr_schedule_time.py and eval_time.py keep them), for zipf and uniform ids, flag off and on alternating:

  * window 0 is installed, trained (two eager steps, then the captured step), window 1 is installed -- the boundary
    that carries window 0's trained loser rows -- and trained whole: ms/step of window 1 (CUDA events around its
    steps, which run beside the write-back of window 0's store and the prefetch of window 2);
  * the update kernel's time per launch (library event timing over eager steps) and the carry's time at the
    boundary (event timing of the boundary's launches);
  * the store write-back: rows and GB of window 1's store and the seconds ``write_store_to_master`` takes for them;
  * ``boundary_breakdown_ms["wait_plan"]`` of the boundaries.

The result is one JSON file (``--json``) with the GPU's name and power limit.  Needs a CUDA device.

  python tools/victim_cache_time.py --json profiles/victim_cache_time_b200.json
"""
import argparse
import ctypes
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def prof_ms(lib, names):
    """Summed milliseconds and calls of the named kernels since the last report (clears the records)."""
    n = lib.cdlrm_prof_num_kernels()
    ms, calls = (ctypes.c_double * n)(), (ctypes.c_int64 * n)()
    lib.cdlrm_prof_report(ms, calls, n)
    by = {lib.cdlrm_prof_kernel_name(i).decode(): (ms[i], calls[i]) for i in range(n)}
    return {k: by[k] for k in names}


def one_run(args, dist, flag, ln_emb, dev):
    from cdlrm_b200._lib import lib
    from cdlrm_b200.main_no_ddp import ProcessArgs, Trainer
    from cdlrm_b200.model_no_ddp import Embedding_Table_Group
    from cdlrm_b200.synthetic import SyntheticStream
    B, L = args.batch, args.lookahead
    pa = ProcessArgs(["--arch-sparse-feature-size", "128", "--arch-mlp-bot", "13-512-256-128", "--arch-mlp-top",
                      "512-512-256-1", "--loss-function", "bce", "--mini-batch-size", str(B), "--lookahead", str(L),
                      "--cache-size", "150000", "--num-ways", "16", "--world-size", "1", "--learning-rate", "0.1",
                      "--lr-embeds", "0.1"] + (["--evict-victim-cache"] if flag else []))
    master = Embedding_Table_Group(128, np.asarray(ln_emb), init="device")
    nf = len(ln_emb) + 1
    tr = Trainer(pa, 128, np.asarray(ln_emb), np.asarray([13, 512, 256, 128]),
                 np.asarray([nf * (nf - 1) // 2 + 128, 512, 256, 1]), master, rank=0, world=1, device=dev)
    sg = SyntheticStream(ln_emb, B, dev, dist=dist, zipf_a=1.05, seed=123)
    lS_o = torch.arange(B).reshape(1, -1).repeat(len(ln_emb), 1)
    out = {"flag": flag}
    wins = [sg.window_ids(w, L) for w in range(3)]
    X, Y = sg.dense_and_labels(0, 1)
    tr.submit_window(wins[0])
    tr.install_window()
    tr.submit_window(wins[1])
    lib.cdlrm_prof_enable(1)
    for j in range(L):
        if j == 2:
            lib.cdlrm_prof_enable(0)
            t = prof_ms(lib, ["embed_victim", "bwd_sgd"])
            out["victim_us_per_launch"] = round(1e3 * t["embed_victim"][0] / max(t["embed_victim"][1], 1), 2)
            out["bwd_sgd_us_per_launch"] = round(1e3 * t["bwd_sgd"][0] / max(t["bwd_sgd"][1], 1), 2)
            tr.capture_graph(X, lS_o, wins[0][:, j * B:(j + 1) * B].contiguous(), Y)
        tr.step(X, lS_o, wins[0][:, j * B:(j + 1) * B].contiguous(), Y)
    torch.cuda.synchronize(dev)
    out["miss_per_step"] = int(tr.cache_group.last_n_miss.sum())
    lib.cdlrm_prof_enable(1)
    rec = tr.install_window()
    torch.cuda.synchronize(dev)
    lib.cdlrm_prof_enable(0)
    t = prof_ms(lib, ["move_carry"])
    out["carry_ms"] = round(t["move_carry"][0], 3)
    out["carry_launches"] = int(t["move_carry"][1])
    out["wait_plan_ms"] = [tr.boundary_breakdown_ms["wait_plan"]]
    tr.submit_window(wins[2])
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for j in range(L):
        tr.step(X, lS_o, wins[1][:, j * B:(j + 1) * B].contiguous(), Y)
    b.record()
    b.synchronize()
    out["window_ms_per_step"] = round(a.elapsed_time(b) / L, 4)
    tr.install_window()
    out["wait_plan_ms"].append(tr.boundary_breakdown_ms["wait_plan"])
    tr.finish()
    # window 2 is installed: time the write-back of its store (what the next boundary enqueues on the planner stream)
    nrows = int(sum(tr.planner._bound.L))
    t0 = time.perf_counter()
    tr.planner.write_store_to_master()
    dt = time.perf_counter() - t0
    out["store_rows"] = nrows
    out["store_writeback_gb"] = round(nrows * 128 * 4 / 1e9, 3)
    out["store_writeback_s"] = round(dt, 4) if flag else None
    out["window1_loser_rows"] = int(sum(rec.L))
    del tr, master, sg
    gc.collect()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--json", required=True, help="result file")
    ap.add_argument("--max-rows", type=int, default=10_000_000, help="rows per master table at most")
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--lookahead", type=int, default=64, help="steps per window")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("victim_cache_time.py needs a CUDA device")
    from cdlrm_b200.synthetic import TERABYTE_ROWS
    dev = torch.device("cuda", 0)
    ln_emb = [min(int(n), args.max_rows) for n in TERABYTE_ROWS]
    res = {"gpu": torch.cuda.get_device_name(dev), "ln_emb": ln_emb, "dim": 128, "num_ways": 16, "cache_size": 150000,
           "batch": args.batch, "lookahead": args.lookahead, "master": f"in HBM, tables capped at {args.max_rows} rows"}
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        res["power_limit"] = f"unknown ({e})"
    for dist, order in (("zipf", (False, True)), ("uniform", (True, False))):
        runs = [one_run(args, dist, flag, ln_emb, dev) for flag in order]
        off = next(r for r in runs if not r["flag"])
        on = next(r for r in runs if r["flag"])
        res[dist] = {"off": off, "on": on,
                     "step_overhead_share": round(on["window_ms_per_step"] / off["window_ms_per_step"] - 1, 4)}
        print(dist, json.dumps(res[dist]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
    with open(args.json, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
