#!/usr/bin/env python
"""Cost of exporting and checkpointing the look-ahead cache at the Terabyte cache shape (26 tables, 150001 sets x 16
ways, dim 128: up to 62 M cached lines, 32 GB):

  * Trainer.sync_master in both PCIe modes ("sm": zero-copy evict kernel, "ce": evict kernel into HBM staging +
    cudaMemcpyAsync + host scatter): rows, GB, GB/s, against the device-to-host cudaMemcpyAsync peak of a pinned
    1 GB copy measured in the same run;
  * Trainer.save_checkpoint and load_checkpoint (into a freshly built Trainer): wall time, split into device<->host
    copies and file I/O.

The cache holds one window: a uniform synthetic window of lookahead x batch ids per table is planned and installed
(no training steps run; they do not change what is exported).  ``--max-rows`` caps every table's master so that the
master and the checkpoint fit the machine; everything is written under ``--out``, and the result is one JSON file
(``--json``) with the GPU's name and power limit.  Needs a CUDA device: there is no CPU path.

  python tools/ckpt_time.py --out /tmp/ckpt_time --json profiles/ckpt_time_b200.json
"""
import argparse
import gc
import json
import os
import shutil
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def d2h_peak_gbs(dev, nbytes=1 << 30, reps=5):
    d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    h.copy_(d, non_blocking=True)                 # warm-up
    torch.cuda.synchronize(dev)
    best = 0.0
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        h.copy_(d, non_blocking=True)             # cudaMemcpyAsync device -> pinned host
        b.record()
        b.synchronize()
        best = max(best, nbytes / (a.elapsed_time(b) * 1e-3) / 1e9)
    return best


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
    return tr, master


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True, help="directory for the checkpoint (emptied first)")
    ap.add_argument("--json", required=True, help="result file")
    ap.add_argument("--max-rows", type=int, default=2_500_000, help="rows per master table at most")
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--lookahead", type=int, default=3000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ckpt_time.py needs a CUDA device")
    from cdlrm_b200.synthetic import TERABYTE_ROWS, SyntheticStream
    dev = torch.device("cuda", 0)
    ln_emb = [min(int(n), args.max_rows) for n in TERABYTE_ROWS]
    res = {"gpu": torch.cuda.get_device_name(dev), "ln_emb": ln_emb, "dim": 128, "num_ways": 16, "cache_size": 150000,
           "window": {"batch": args.batch, "lookahead": args.lookahead, "dist": "uniform"}}
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        res["power_limit"] = f"unknown ({e})"
    res["d2h_memcpy_peak_GBps"] = round(d2h_peak_gbs(dev), 2)

    def dump():
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)

    tr, master = build(args, ln_emb)
    sg = SyntheticStream(ln_emb, args.batch, dev, dist="uniform", seed=3)
    t0 = time.perf_counter()
    tr.submit_window(sg.window_ids(0, args.lookahead))
    tr.install_window()
    torch.cuda.synchronize(dev)
    res["plan_install_s"] = round(time.perf_counter() - t0, 3)
    tr.steps_in_window = tr._window_steps          # the window's steps would not change what is exported
    res["valid_lines"] = int(sum(int((t >= 0).sum()) for t in tr.cache_group.occupancy_tables))
    res["sync_master"] = {}
    for mode in ("sm", "ce"):
        tr.planner.pcie_mode = mode
        tr.planner.host_threads = 4
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        n = tr.sync_master()
        dt = time.perf_counter() - t0
        gb = n * 128 * 4 / 1e9
        res["sync_master"][mode] = {"rows": n, "GB": round(gb, 3), "s": round(dt, 3), "GBps": round(gb / dt, 2),
                                    "share_of_d2h_peak": round(gb / dt / res["d2h_memcpy_peak_GBps"], 3)}
        dump()
    if os.path.isdir(args.out):
        shutil.rmtree(args.out)
    os.makedirs(args.out)
    path = os.path.join(args.out, "ck")
    need = sum(n * 512 for n in ln_emb) + 2 * res["valid_lines"] * 512
    free = shutil.disk_usage(args.out).free
    res["checkpoint_bytes_estimate"] = need
    if free < 1.2 * need:
        res["checkpoint"] = f"not measured: {free / 1e9:.0f} GB free under --out, about {need / 1e9:.0f} GB needed"
        dump()
        return
    t0 = time.perf_counter()
    tr.save_checkpoint(path)
    res["save_checkpoint"] = dict(s=round(time.perf_counter() - t0, 3), **tr.last_checkpoint_s)
    res["checkpoint_bytes"] = sum(os.path.getsize(os.path.join(path, f)) for f in os.listdir(path))
    dump()
    tr.finish()
    del tr, master
    gc.collect()
    torch.cuda.empty_cache()
    tr, master = build(args, ln_emb)
    t0 = time.perf_counter()
    tr.load_checkpoint(path)
    res["load_checkpoint"] = dict(s=round(time.perf_counter() - t0, 3), **tr.last_checkpoint_s)
    tr.finish()
    shutil.rmtree(args.out)
    dump()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
