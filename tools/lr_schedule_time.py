#!/usr/bin/env python
"""Cost of the learning-rate schedule in the captured training step, at the bench's Terabyte shape (26 tables, dim 128,
bottom 13-512-256-128, top 512-512-256-1, batch 8192, 150000 sets x 16 ways; masters capped at ``--max-rows``):

  * one Trainer, one installed window (zipf synthetic ids), two CUDA graphs of the same step captured from it: without
    a schedule (the learning rates are read from the device state that cdlrm_lr_set wrote once) and with a decaying
    schedule (plus one cdlrm_lr_advance launch per step);
  * steady-state replays of the two graphs alternate in blocks of ``--steps`` on the same inputs and cache state,
    ``--rounds`` times, timed with CUDA events: ms/step of each arm (median over the blocks), the difference, and the
    block-to-block spread of each arm.

The result is one JSON file (``--json``) with the GPU's name and power limit.  Needs a CUDA device: there is no CPU
path.

  python tools/lr_schedule_time.py --json profiles/lr_schedule_time_b200.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--json", required=True, help="result file")
    ap.add_argument("--max-rows", type=int, default=10_000_000, help="rows per master table at most")
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--lookahead", type=int, default=64, help="steps of the installed window")
    ap.add_argument("--steps", type=int, default=200, help="replays per timed block")
    ap.add_argument("--rounds", type=int, default=10, help="timed blocks per arm")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("lr_schedule_time.py needs a CUDA device")
    from cdlrm_b200.main_no_ddp import ProcessArgs, Trainer
    from cdlrm_b200.model_no_ddp import Embedding_Table_Group
    from cdlrm_b200.synthetic import TERABYTE_ROWS, SyntheticStream
    dev = torch.device("cuda", 0)
    ln_emb = [min(int(n), args.max_rows) for n in TERABYTE_ROWS]
    sched = (0, 0, 10 ** 9)            # quadratic decay from the first step on, over more steps than any run here
    res = {"gpu": torch.cuda.get_device_name(dev), "ln_emb": ln_emb, "dim": 128, "num_ways": 16, "cache_size": 150000,
           "batch": args.batch, "dist": "zipf 1.05", "schedule": dict(zip(("W", "D", "N"), sched)),
           "steps_per_block": args.steps, "rounds": args.rounds}
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        res["power_limit"] = f"unknown ({e})"
    pa = ProcessArgs(["--arch-sparse-feature-size", "128", "--arch-mlp-bot", "13-512-256-128", "--arch-mlp-top",
                      "512-512-256-1", "--loss-function", "bce", "--mini-batch-size", str(args.batch), "--lookahead",
                      str(args.lookahead), "--cache-size", "150000", "--num-ways", "16", "--world-size", "1",
                      "--learning-rate", "0.1", "--lr-embeds", "0.1"])
    master = Embedding_Table_Group(128, np.asarray(ln_emb), init="device")
    nf = len(ln_emb) + 1
    tr = Trainer(pa, 128, np.asarray(ln_emb), np.asarray([13, 512, 256, 128]),
                 np.asarray([nf * (nf - 1) // 2 + 128, 512, 256, 1]), master, rank=0, world=1, device=dev)
    sg = SyntheticStream(ln_emb, args.batch, dev, dist="zipf", zipf_a=1.05, seed=123)
    win = sg.window_ids(0, args.lookahead)
    tr.submit_window(win)
    tr.install_window()
    X, Y = sg.dense_and_labels(0, 1)
    lS_i = win[:, :args.batch].contiguous()
    lS_o = torch.arange(args.batch).reshape(1, -1).repeat(len(ln_emb), 1)
    for _ in range(2):                 # lazy initialisation, as Run does before the capture
        tr.step(X, lS_o, lS_i, Y)
    graphs = {}
    for name, s in (("no_schedule", (0, 0, 0)), ("schedule", sched)):
        tr.lr_schedule = s
        tr._set_lr_state()
        tr.capture_graph(X, lS_o, lS_i, Y)
        graphs[name] = (tr._graph, tr._g_in, tr._g_out, tr.graph_launches, s)
    res["library_launches_per_step"] = {k: v[3] for k, v in graphs.items()}

    def block(name, n):
        tr._graph, tr._g_in, tr._g_out, _n, tr.lr_schedule = graphs[name]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            tr.step(X, lS_o, lS_i, Y)
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / n

    for name in graphs:                # warm-up of both graphs
        block(name, 50)
    ms = {k: [] for k in graphs}
    for r in range(args.rounds):
        order = list(graphs) if r % 2 == 0 else list(graphs)[::-1]
        for name in order:
            ms[name].append(block(name, args.steps))
    tr.finish()
    for k, v in ms.items():
        res[k] = {"ms_per_step_median": round(float(np.median(v)), 4), "min": round(min(v), 4),
                  "max": round(max(v), 4), "blocks": [round(x, 4) for x in v]}
    diff = [s - n for s, n in zip(ms["schedule"], ms["no_schedule"])]
    res["difference_ms_per_step"] = {"median": round(float(np.median(diff)), 4), "min": round(min(diff), 4),
                                     "max": round(max(diff), 4)}
    res["difference_share"] = round(float(np.median(diff)) / float(np.median(ms["no_schedule"])), 5)
    os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
    with open(args.json, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
