#!/usr/bin/env python
"""Cost of training from an MLPerf binary Criteo file (cdlrm_b200/criteo_bin.py) against training from the device-side
synthetic stream, at the Terabyte shape (26 tables, 150001 sets x 16 ways, dim 128, MLPs 13-512-256-128 /
479-512-256-1, batch 8192, look-ahead ``--lookahead`` steps):

  * a data file of two windows (2 x lookahead x 8192 records, 7.9 GB at the default 3000) is written into a
    temporary directory (free space checked first, deleted at exit).  Its ids are those of ``SyntheticStream`` with
    the same seed and row cap, so both arms plan identical windows; dense values U{0..100}, labels Bernoulli(0.25);
  * one whole window is timed (its L steps, the plan and prefetch of the next window running beside them, the
    boundary that installs it, every loss read back), four times, the two arms in the order file, synthetic,
    synthetic, file:
      - file: batches from ``device_batches`` (reader thread, copy stream, decode per step), the next window handed
        to the planner as a ``window_marker`` (its records read again and decoded ids-only, chunk by chunk);
      - synthetic: batches staged from pinned host memory through ``Trainer.stage_inputs`` / ``step_staged`` as
        bench.py's e2e leg does, the next window as the device-generated id tensor;
  * decode time per step (CUDA events around 200 decodes of one batch), the scan's device time per window and its
    share of the planner burst (scan start to prefetch done), the wait at the boundary, and the host read rate
    (``os.preadv`` of one window's records into a pinned buffer).

The file was just written, so every read comes from the page cache: the disk's read rate is not measured.
``--rows-cap`` caps every master table (as tools/eval_time.py does) so that master and page cache fit the host.
Writes one JSON file with the GPU's name and power limit.  Needs a CUDA device.

  python tools/criteo_bin_time.py --json profiles/criteo_bin_time_b200.json
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
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
    return Trainer(pa, 128, np.asarray(ln_emb), np.asarray([13, 512, 256, 128]),
                   np.asarray([nf * (nf - 1) // 2 + 128, 512, 256, 1]), master, rank=0, world=1, device=dev)


def write_file(path, sg, n_steps, batch, dev, seed=11):
    """Records of steps [0, n_steps) of the synthetic stream: ids from ``sg``, dense U{0..100}, labels Bernoulli(0.25)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    per = max(1, (1 << 27) // (160 * batch))              # ~128 MB of records per piece
    host = torch.empty(per * batch, 40, dtype=torch.int32, pin_memory=True)
    with open(path, "wb") as f:
        for s0 in range(0, n_steps, per):
            ns = min(per, n_steps - s0)
            n = ns * batch
            rec = torch.empty(n, 40, dtype=torch.int32, device=dev)
            rec[:, 0] = (torch.rand(n, device=dev, generator=g) < 0.25).int()
            rec[:, 1:14] = torch.randint(0, 101, (n, 13), device=dev, generator=g, dtype=torch.int32)
            rec[:, 14:] = sg.ids(s0, ns).t().int()
            host[:n].copy_(rec)
            f.write(memoryview(host[:n].numpy()).cast("B"))
    return os.path.getsize(path)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--json", required=True, help="result file")
    ap.add_argument("--rows-cap", type=int, default=2_500_000, help="rows per master table at most")
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--lookahead", type=int, default=3000)
    ap.add_argument("--tmpdir", default=tempfile.gettempdir(), help="where the data file is written")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("criteo_bin_time.py needs a CUDA device")
    from cdlrm_b200 import criteo_bin as CB
    from cdlrm_b200._lib import check, lib, vp
    from cdlrm_b200.synthetic import TERABYTE_ROWS, SyntheticStream
    dev = torch.device("cuda", 0)
    B, L = args.batch, args.lookahead
    ln_emb = [min(int(n), args.rows_cap) for n in TERABYTE_ROWS]
    need = 2 * L * B * CB.RECORD_BYTES
    free = shutil.disk_usage(args.tmpdir).free
    if free < need + (2 << 30):
        sys.exit(f"criteo_bin_time.py: {need / 1e9:.1f} GB data file does not fit {args.tmpdir} "
                 f"({free / 1e9:.1f} GB free); pass --tmpdir or a smaller --lookahead")
    res = {"gpu": torch.cuda.get_device_name(dev), "ln_emb": ln_emb, "dim": 128, "num_ways": 16, "cache_size": 150000,
           "batch": B, "lookahead": L, "dist": "zipf",
           "note": "the data file was just written: reads come from the page cache, the disk's read rate is not measured"}
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        res["power_limit"] = f"unknown ({e})"

    def dump():
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)

    tmp = tempfile.mkdtemp(prefix="criteo_bin_time_", dir=args.tmpdir)
    try:
        sg = SyntheticStream(ln_emb, B, dev, seed=3)
        t0 = time.perf_counter()
        data = os.path.join(tmp, "tb_train.bin")
        res["file_bytes"] = write_file(data, sg, 2 * L, B, dev)
        res["file_write_s"] = round(time.perf_counter() - t0, 1)
        np.savez(os.path.join(tmp, "day_fea_count.npz"), counts=np.asarray(ln_emb))
        ds = CB.CriteoBinDataset(data, os.path.join(tmp, "day_fea_count.npz"), batch_size=B)
        dump()
        run(res, dump, args, ds, sg, ln_emb, dev, check, lib, vp, CB)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(res))


def run(res, dump, args, ds, sg, ln_emb, dev, check, lib, vp, CB):
    B, L, T = args.batch, args.lookahead, len(ln_emb)
    # host read rate: one window's records into a pinned buffer, 64 MB per os.preadv
    pin = torch.empty(CB.CHUNK_BYTES, dtype=torch.uint8, pin_memory=True)
    nbytes = L * B * CB.RECORD_BYTES
    t0 = time.perf_counter()
    for off in range(0, nbytes, CB.CHUNK_BYTES):
        CB._preadv_into(ds._fd, pin, min(CB.CHUNK_BYTES, nbytes - off), off, ds.data_file)
    res["host_read_gb_per_s"] = round(nbytes / (time.perf_counter() - t0) / 1e9, 2)
    del pin
    # decode of one batch (events, 200 launches)
    raw = torch.from_numpy(np.fromfile(ds.data_file, dtype=np.int32, count=B * 40)).to(dev)
    X = torch.empty(B, 13, device=dev)
    ids = torch.empty(T, B, dtype=torch.int64, device=dev)
    Y = torch.empty(B, device=dev)
    s = torch.cuda.current_stream(dev)

    def dec():
        check(lib.cdlrm_criteo_decode(0, vp(raw.data_ptr()), B, 13, 26, -1, vp(X.data_ptr()), 13, vp(ids.data_ptr()), B,
                                      vp(Y.data_ptr()), vp(s.cuda_stream)))
    for _ in range(20):
        dec()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(200):
        dec()
    e1.record()
    torch.cuda.synchronize(dev)
    res["decode_us_per_step"] = round(1e3 * e0.elapsed_time(e1) / 200, 2)
    res["decode_bytes_per_step"] = {"read": B * 160, "written": B * (13 * 4 + 26 * 8 + 4)}
    dump()

    tr = build(args, ln_emb)
    res["pcie_mode"] = tr.planner.pcie_mode
    torch.cuda.set_stream(torch.cuda.Stream(dev, priority=-1))          # as Run: training on a high-priority stream
    stream = ds.device_batches(dev)
    scans = []

    def marker(w):
        m = ds.window_marker(w, L)

        def timed(planner):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(planner.stream)
            h0 = time.perf_counter()
            n = m(planner)
            b.record(planner.stream)
            scans.append((a, b, h0, time.perf_counter()))
            return n
        return timed

    id_buf = {}

    def synth_ids(w):
        id_buf["b"] = sg.ids(w * L, L, out=id_buf.get("b"), stream=tr.side)
        return id_buf["b"]

    hI = torch.empty(L, T, B, dtype=torch.int64, pin_memory=True)
    hX = torch.empty(L, B, 13, dtype=torch.float32, pin_memory=True)
    hY = torch.empty(L, B, 1, dtype=torch.float32, pin_memory=True)

    def fill_host(w):
        for s0 in range(0, L, 100):
            ns = min(100, L - s0)
            hI[s0:s0 + ns].copy_(sg.ids(w * L + s0, ns).view(T, ns, B).permute(1, 0, 2))
        Xw, Yw = sg.dense_and_labels(w, L)
        hX.copy_(Xw.view(L, B, 13))
        hY.copy_(Yw.view(L, B, 1))
        del Xw, Yw
        torch.cuda.synchronize(dev)

    lS_o = torch.arange(B, device=dev).reshape(1, -1).repeat(T, 1)
    AHEAD = tr.input_slots - 2

    def steps(arm, w):
        loss = float("nan")
        if arm == "file":
            it = stream.iter_from(w * L)
            for _ in range(L):
                X_, o_, i_, T_ = next(it)
                E, _ = tr.step(X_, o_, i_, T_)
                tr.push_loss(E)
                if tr.pending_losses() > AHEAD:
                    loss = tr.pop_loss()
            it.close()
        else:
            staged = [tr.stage_inputs(hX[q], hI[q], hY[q]) for q in range(AHEAD)]
            for i in range(L):
                if i + AHEAD < L:
                    staged.append(tr.stage_inputs(hX[i + AHEAD], hI[i + AHEAD], hY[i + AHEAD]))
                E, _ = tr.step_staged(staged.pop(0), lS_o)
                tr.push_loss(E)
                if tr.pending_losses() > AHEAD:
                    loss = tr.pop_loss()
        while tr.pending_losses():
            loss = tr.pop_loss()
        return loss

    # window 0 installed (through a marker: the scan's buffers are allocated here), graph captured, both input paths
    # warmed (a few steps of window 0)
    tr.submit_window(marker(0))
    tr.install_window()
    it = stream.iter_from(0)
    for k in range(3):
        X_, o_, i_, T_ = next(it)
        if k == 2:
            tr.capture_graph(X_, o_, i_, T_)
        tr.step(X_, o_, i_, T_)
    it.close()
    fill_host(0)
    for q in range(8):
        tr.step_staged(tr.stage_inputs(hX[q], hI[q], hY[q]), lS_o)
    torch.cuda.synchronize(dev)
    runs = []
    for r, arm in enumerate(["file", "synthetic", "synthetic", "file"]):
        w, nxt = r % 2, (r + 1) % 2
        if arm == "synthetic":
            fill_host(w)
        torch.cuda.synchronize(dev)
        nscan = len(scans)
        t0 = time.perf_counter()
        tr.submit_window(marker(nxt) if arm == "file" else synth_ids(nxt))
        loss = steps(arm, w)
        rec = tr.install_window()
        torch.cuda.synchronize(dev)
        wall = time.perf_counter() - t0
        item = {"arm": arm, "window": w, "ms_per_step": round(1e3 * wall / L, 4), "last_loss": loss,
                "boundary_wait_plan_ms": tr.boundary_breakdown_ms["wait_plan"],
                "boundary": tr.boundary_breakdown_ms}
        if len(scans) > nscan:
            a, b, h0, h1 = scans[-1]
            scan_s = a.elapsed_time(b) / 1e3
            burst_s = a.elapsed_time(rec.staged) / 1e3 if rec.staged is not None else float("nan")
            item.update(scan_device_s=round(scan_s, 3), scan_host_s=round(h1 - h0, 3), planner_burst_s=round(burst_s, 3),
                        scan_share_of_burst=round(scan_s / burst_s, 3),
                        scan_read_gb_per_s=round(L * B * 160 / (h1 - h0) / 1e9, 2))
        runs.append(item)
        res["runs"] = runs
        dump()
    tr.finish()
    f = [x["ms_per_step"] for x in runs if x["arm"] == "file"]
    sy = [x["ms_per_step"] for x in runs if x["arm"] == "synthetic"]
    res["file_ms_per_step"], res["synthetic_ms_per_step"] = f, sy
    res["file_over_synthetic"] = round(float(np.mean(f)) / float(np.mean(sy)), 4)
    res["stream_bytes_read"] = stream.bytes_read
    dump()


if __name__ == "__main__":
    main()
