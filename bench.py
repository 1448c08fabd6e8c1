#!/usr/bin/env python
"""bench.py -- training samples/sec of the cDLRM look-ahead embedding-cache path on
Terabyte-shape synthetic data (BASELINE.json metric), one process per GPU.

  python bench.py --gpus N --steps K --warmup W            (torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py --steps K --dump-outputs DIR             (the last timed step's loss / predictions as .npy)

A step = one full training iteration over one global batch: cache forward (probe + gather +
pool), bottom/top MLPs (tcgen05 3xTF32 GEMMs, FP32 accuracy), pairwise-dot interaction fwd/bwd, BCE loss,
de-duplicated sparse SGD on the cache, dense SGD; window install every `lookahead` steps with
the next window planned concurrently on a side stream; table aggregation every
`table_agg_freq` steps when N > 1.  Prints ONE JSON line (rank 0).
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[2] (the configuration the metric is quoted on); configs[3] / [4] are this workload with
    # --cache-size / --num-ways / --dist and --batch / --table-agg-freq overridden
    "terabyte": dict(rows="terabyte", dim=128, bot="13-512-256-128", top="512-512-256-1", batch=8192,
                     cache=150000, ways=16, lookahead=3000, agg=100),
    # configs[1]
    "kaggle": dict(rows="kaggle", dim=16, bot="13-512-256-64-16", top="512-256-1", batch=2048,
                   cache=150000, ways=16, lookahead=3000, agg=100),
    # configs[0]
    "small": dict(rows=[100000] * 8, dim=16, bot="13-64-16", top="64-1", batch=128, cache=10000, ways=16,
                  lookahead=100, agg=100),
}
METRIC = "samples/sec (Terabyte-shape synthetic) at 1/2/4/8 B200; cache-op HBM GB/s"


def log(msg):
    if os.environ.get("CDLRM_BENCH_LOG", "1") != "0":
        sys.stderr.write(f"[bench {time.strftime('%H:%M:%S')} rank {os.environ.get('RANK', '0')}] {msg}\n")
        sys.stderr.flush()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)      # 0: one full window (lookahead steps)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", type=str, default="cdlrm_b200")
    ap.add_argument("--workload", type=str, default="terabyte")
    ap.add_argument("--dist", type=str, default="zipf")
    ap.add_argument("--zipf-a", type=float, default=1.05)
    ap.add_argument("--row-cap", type=int, default=40_000_000)
    ap.add_argument("--lookahead", type=int, default=0)
    ap.add_argument("--cache-size", type=int, default=0)
    ap.add_argument("--num-ways", type=int, default=0)
    ap.add_argument("--table-agg-freq", type=int, default=0)
    ap.add_argument("--batch", type=int, default=0)          # per-GPU batch
    # end-to-end leg: 0 = one whole look-ahead window starting at a window boundary (one install, the next window
    # planned and prefetched beside training, lookahead / table_agg_freq aggregations); n > 0 = n steps; -1 = skip
    ap.add_argument("--e2e-steps", type=int, default=0)
    ap.add_argument("--cpu-baseline-steps", type=int, default=4)
    ap.add_argument("--ref-window-steps", type=int, default=0)   # reference arm: steps per installed window (0: auto)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-prof", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    # measurement only: at a third of the timed region, enqueue this many GB of copy-engine host-to-device copies
    # (256 MB pinned chunks, side stream) beside the steps: what a cudaMemcpyAsync prefetch would cost the step
    ap.add_argument("--ce-probe-gb", type=float, default=0.0)
    # what the last timed step returned to its caller (Trainer.step: the loss E and the predictions Z of rank 0's
    # batch) as DIR/loss.npy and DIR/predictions.npy, float32; the inputs are seeded, so that two builds run with the
    # same arguments can be compared output for output.  Not bit for bit: sums are accumulated in a different order
    # from run to run, and two runs of the default workload (20 timed steps, one B200) differed by up to 2e-4
    # relative in the predictions
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs dumps the GPU path's outputs; the reference arm has none")
    return a


def table_rows(wl, cap):
    from cdlrm_b200.synthetic import KAGGLE_ROWS, TERABYTE_ROWS
    rows = {"terabyte": TERABYTE_ROWS, "kaggle": KAGGLE_ROWS}.get(wl["rows"], wl["rows"]) \
        if isinstance(wl["rows"], str) else wl["rows"]
    return [min(int(n), cap) for n in rows]


def workload_string(a, wl, T, world):
    return (f"{a.workload}-shape synthetic: {T} tables (row cap {a.row_cap}), dim {wl['dim']}, bot {wl['bot']}, "
            f"top {wl['top']}, batch {wl['batch']} per GPU (global {wl['batch'] * world}), cache {wl['cache']}x"
            f"{wl['ways']}-way, lookahead {wl['lookahead']}, table-agg-freq {wl['agg']}, index dist "
            f"{a.dist}(a={a.zipf_a})")


def mem_available_gb():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                return int(line.split()[1]) / 1e6
    except OSError:
        pass
    return 0.0


def model_args(wl, ln_emb, world):
    from cdlrm_b200.main_no_ddp import ProcessArgs
    argv = ["--arch-sparse-feature-size", str(wl["dim"]), "--arch-mlp-bot", wl["bot"], "--arch-mlp-top", wl["top"],
            "--loss-function", "bce", "--learning-rate", "0.8", "--lr-embeds", "0.8", "--mini-batch-size",
            str(wl["batch"]), "--lookahead", str(wl["lookahead"]), "--cache-size", str(wl["cache"]), "--num-ways",
            str(wl["ways"]), "--table-agg-freq", str(wl["agg"]), "--batch-fifo-size", "8", "--cache-workers", "4",
            "--large-batch", "--world-size", str(world)]
    args = ProcessArgs(argv)
    ln_bot = np.fromstring(wl["bot"], dtype=int, sep="-")
    nf = len(ln_emb) + 1
    num_int = nf * (nf - 1) // 2 + int(ln_bot[-1])
    ln_top = np.fromstring(str(num_int) + "-" + wl["top"], dtype=int, sep="-")
    return args, ln_bot, ln_top


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [ln.strip().split(", ") for ln in open(self.f.name) if ln.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except ValueError:
                continue
            for nm, v in zip(names, r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(nm)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle port (numpy) + stock torch CPU MLPs, on the box's host cores
# ------------------------------------------------------------------------------------------

def cpu_reference_run(wl, ln_emb, steps, warmup, budget_s, dist, zipf_a):
    """Times the reference's CPU algorithm (oracle port, kind 'port': the reference is pure
    Python and cannot travel to the GPU box) on a bounded sample of the same workload:
    same tables / dim / cache geometry / MLPs, batch scaled down to `bs` samples per step and a
    window of `look` steps so that the run fits the time budget."""
    import torch
    from oracle import oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    try:        # torchrun exports OMP_NUM_THREADS=1: give numpy's BLAS / OpenMP pools all the host cores back
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=cores)
    except Exception:
        pass
    d, T = wl["dim"], len(ln_emb)
    B = wl["batch"]
    rng = np.random.default_rng(123)

    def make_ids(n):
        out = np.empty((T, n), dtype=np.int64)
        for k, nk in enumerate(ln_emb):
            u = rng.random(n)
            if dist == "uniform" or nk == 1:
                r = np.minimum((u * nk).astype(np.int64), nk - 1)
            else:
                e = 1.0 - zipf_a
                r = np.clip((((nk + 1.0) ** e - 1.0) * u + 1.0) ** (1.0 / e) - 1, 0, nk - 1).astype(np.int64)
            out[k] = (r * 2654435761 + 40503 * k) % nk
        return out

    ln_bot = np.fromstring(wl["bot"], dtype=int, sep="-")
    nf = T + 1
    ln_top = np.fromstring(str(nf * (nf - 1) // 2 + int(ln_bot[-1])) + "-" + wl["top"], dtype=int, sep="-")

    def mlp(ln, last_sigmoid):
        layers = []
        for i in range(len(ln) - 1):
            layers.append(torch.nn.Linear(int(ln[i]), int(ln[i + 1])))
            layers.append(torch.nn.Sigmoid() if (last_sigmoid and i == len(ln) - 2) else torch.nn.ReLU())
        return torch.nn.Sequential(*layers)

    bot, top = mlp(ln_bot, False), mlp(ln_top, True)
    opt = torch.optim.SGD(list(bot.parameters()) + list(top.parameters()), lr=0.8)
    loss_fn = torch.nn.BCELoss()
    master = [np.zeros((n, d), dtype=np.float32) for n in ln_emb]   # lazily committed (calloc)
    gen = O.TorchCpuGenerator(123)

    def run(bs, look, nsteps):
        cache = O.OracleCache(d, ln_emb, wl["cache"], bs, wl["ways"])
        t_total = 0.0
        done = 0
        while done < nsteps:
            n_here = min(look, nsteps - done)
            win = make_ids(look * bs)
            Xw = np.log1p(rng.integers(0, 101, size=(look * bs, 13))).astype(np.float32)
            Yw = (rng.random((look * bs, 1)) < 0.25).astype(np.float32)
            t0 = time.perf_counter()
            O.install_window(cache, master, win, gen)
            for b in range(n_here):
                ids = win[:, b * bs:(b + 1) * bs]
                ly, slots = [], []
                for k in range(T):
                    o, s, _ = O.forward_table_fast(cache, k, ids[k], master[k])
                    ly.append(o)
                    slots.append(s)
                x = bot(torch.from_numpy(Xw[b * bs:(b + 1) * bs]))
                R, Tm = O.interact_fwd_fast(x.detach().numpy(), ly)
                Rt = torch.from_numpy(R).requires_grad_()
                loss = loss_fn(top(Rt), torch.from_numpy(Yw[b * bs:(b + 1) * bs]))
                opt.zero_grad()
                loss.backward()
                dT = O.interact_bwd_fast(Tm, Rt.grad.numpy())
                x.backward(torch.from_numpy(np.ascontiguousarray(dT[:, 0])))
                opt.step()
                for k in range(T):
                    O.backward_sgd_table_fast(cache.weight[k], slots[k], dT[:, k + 1], 0.8)
            t_total += time.perf_counter() - t0
            done += n_here
        return t_total

    # calibrate on a small sample, then size the per-step sample to the budget
    bs0 = min(B, 512)
    look0 = 2
    t_cal = run(bs0, look0, 2) / 2
    per_sample = t_cal / bs0
    total_steps = steps + warmup
    bs = int(min(B, max(64, budget_s / max(total_steps, 1) / per_sample)))
    look = max(1, min(wl["lookahead"], total_steps, 4))
    run(bs, look, warmup) if warmup else None
    t = run(bs, look, steps)
    return dict(value=steps * bs / t, ms_per_step=1000 * t / steps, cores=cores,
                sample=f"{steps} steps of {bs} samples (of the {B}-sample batch), window = {look} steps "
                       f"(of {wl['lookahead']}), all {T} tables at full cardinality, dim {d}; numpy oracle port + "
                       f"torch CPU MLPs on {cores} host threads")


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------

def pcie_peaks(torch, dev, nbytes=256 << 20, reps=5):
    """Measured cudaMemcpyAsync peaks between pinned host memory and this GPU (the denominator north_star asks
    for next to the prefetch rate): best of `reps`, CUDA events."""
    h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = {}
    for name, (dst, src) in {"h2d": (d, h), "d2h": (h, d)}.items():
        best = 1e9
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dst.copy_(src, non_blocking=True)
            e1.record()
            e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        out[name + "_GB/s"] = round(nbytes / (best * 1e-3) / 1e9, 1)
    del h, d
    return out


def gpu_run(a, wl, ln_emb):
    import torch
    import torch.distributed as dist
    from cdlrm_b200 import _lib
    from cdlrm_b200.main_no_ddp import Trainer, broadcast_and_aggregate
    from cdlrm_b200.model_no_ddp import Embedding_Table_Group
    from cdlrm_b200.synthetic import SyntheticStream

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    # training runs on a high-priority stream: the look-ahead planner's kernels (side stream, default
    # priority) then only take the SM slots the training step leaves free
    torch.cuda.set_stream(torch.cuda.Stream(dev, priority=-1))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.lib
    args, ln_bot, ln_top = model_args(wl, ln_emb, world)
    L, B, d, T = wl["lookahead"], wl["batch"], wl["dim"], len(ln_emb)
    K = a.steps if a.steps > 0 else L
    W = max(a.warmup, 3)
    lb = B                               # per-GPU batch (weak scaling); global batch = B * world
    args.mini_batch_size = B * world

    # -- master tables in page-locked host memory (one copy per box, shared by the ranks) --------
    t0 = time.time()
    log(f"start: world {world}, {T} tables, master {sum(ln_emb) * d * 4 / 1e9:.1f} GB")
    if world == 1:
        master = Embedding_Table_Group(d, np.asarray(ln_emb), init="device")
    else:
        prefix = f"/dev/shm/cdlrm_master_{os.environ.get('MASTER_PORT', '0')}"
        if rank == 0:
            master = Embedding_Table_Group(d, np.asarray(ln_emb), init=f"shm:{prefix}:create")
        dist.barrier()
        if rank != 0:
            master = Embedding_Table_Group(d, np.asarray(ln_emb), init=f"shm:{prefix}:attach")
    log(f"master tables ready ({time.time() - t0:.1f} s)")
    tr = Trainer(args, d, np.asarray(ln_emb), ln_bot, ln_top, master, rank=rank, world=world, device=dev)
    log(f"trainer ready ({time.time() - t0:.1f} s); host cores {os.cpu_count()}, planner PCIe mode "
        f"{tr.planner.pcie_mode} ({tr.planner.host_threads} host threads)")
    if world > 1:
        dist.barrier()
        if rank == 0:
            for k in range(T):
                try:
                    os.unlink(f"{prefix}_{k}.bin")      # mappings stay alive; nothing left behind
                except OSError:
                    pass
    setup_s = time.time() - t0
    pcie = pcie_peaks(torch, dev)

    Bg = lb * world                     # weak scaling: the per-GPU batch stays at the configured size
    stream_g = SyntheticStream(ln_emb, Bg, dev, dist=a.dist, zipf_a=a.zipf_a, seed=123)
    stream_l = SyntheticStream(ln_emb, lb, dev, dist=a.dist, zipf_a=a.zipf_a, seed=777 + rank)
    data = {}
    recs = {}                           # window -> PlanRecord (prefetch timing)

    mark_buf = {}
    win_bufs = []

    def prepare(w):
        """Window w on the side stream (overlaps training): this rank's slice of the ids plus its dense inputs /
        labels for the training steps, and the look-ahead plan over the GLOBAL window.  At N > 1 the global window
        ([T, L x global batch] int64: 41 GB at 8 GPUs) is never materialised: the stream is counter-based, so the
        planner's scan regenerates it chunk by chunk into one reused buffer (Trainer.submit_window(callable))."""
        # three rotating sets of persistent buffers (window w-1 may still be read when w+1 is generated): no
        # allocation beside training (a cudaMalloc of gigabytes stalls the host thread that enqueues the steps)
        if not win_bufs:
            for _ in range(3):
                win_bufs.append((torch.empty(T, L * lb, dtype=torch.int64, device=dev),
                                 torch.empty(L * lb, 13, dtype=torch.float32, device=dev),
                                 torch.empty(L * lb, 1, dtype=torch.float32, device=dev)))
        b_loc, b_X, b_Y = win_bufs[w % 3]
        # (the steps that read this set belong to window w-3: finished at least a whole window ago)
        with torch.cuda.stream(tr.side):
            loc = stream_g.ids(w * L, L, b0=rank * lb, nb=lb, out=b_loc, stream=tr.side)          # [T, L*lb]
            X, Y = stream_l.dense_and_labels(w, L, out=(b_X, b_Y))
            ready = torch.cuda.Event(enable_timing=True)
            ready.record(tr.side)
        if world == 1:
            tr.submit_window(loc)
        else:
            def mark(planner):
                cs = max(1, (1 << 22) // Bg)                 # ~4 M ids per table per chunk (0.9 GB for 26 tables)
                if "b" not in mark_buf:
                    mark_buf["b"] = torch.empty(T, cs * Bg, dtype=torch.int64, device=dev)
                r_, w_ = planner.scan_shard              # sharded scan: this rank marks steps [lo, hi) only
                per = (L + w_ - 1) // w_
                lo_s, hi_s = r_ * per, min(L, (r_ + 1) * per)
                for s0 in range(lo_s, hi_s, cs):
                    ns = min(cs, hi_s - s0)
                    planner.mark_ids(stream_g.ids(w * L + s0, ns, out=mark_buf["b"], stream=planner.stream))
                return L * Bg
            tr.submit_window(mark, own_ids=loc)
        data[w] = (loc, X, Y, ready)
        for old in [x for x in data if x < w - 1]:
            del data[old]

    def window(w):
        loc, X, Y, ready = data[w]
        torch.cuda.current_stream(dev).wait_event(ready)
        return loc, X, Y

    lS_o = torch.arange(lb).reshape(1, -1).repeat(T, 1)
    torch.cuda.synchronize(dev)
    bound_log, agg_log = [], []        # (host seconds, event pair) per boundary / aggregation of the e2e leg
    logging_on = [False]

    def timed_call(fn, sink):
        if not logging_on[0]:
            return fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0 = time.perf_counter()
        e0.record()
        r = fn()
        e1.record()
        sink.append((time.perf_counter() - h0, e0, e1))
        return r

    prep_log = []

    def boundary(j):
        recs[j // L] = timed_call(tr.install_window, bound_log)
        h0 = time.perf_counter()
        prepare(j // L + 1)
        if logging_on[0]:
            prep_log.append((round(1e3 * (time.perf_counter() - h0), 2), dict(tr.boundary_breakdown_ms)))

    def aggregate(j):
        if world > 1 and j > 0 and j % args.table_agg_freq == 0:
            timed_call(lambda: tr.maybe_aggregate(j), agg_log)

    def one_step(j, host=None):
        w, b = divmod(j, L)
        if b == 0 and j > 0:
            boundary(j)
        lo = b * lb
        if host is None:
            ids, X, Y = window(w)
            E, Z = tr.step(X[lo:lo + lb], lS_o, ids[:, lo:lo + lb], Y[lo:lo + lb])
            aggregate(j)
            return E, Z
        # end-to-end: inputs come from pinned host memory, the result goes back to the host
        hX, hI, hY = host
        E, _ = tr.step(hX[b].to(dev, non_blocking=True), lS_o, hI[b].to(dev, non_blocking=True),
                       hY[b].to(dev, non_blocking=True))
        aggregate(j)
        return E.item()

    # first window: plan + install (untimed set-up), look-ahead plan of window 1 starts
    t_w0 = time.perf_counter()
    prepare(0)
    recs[0] = tr.install_window()
    torch.cuda.synchronize(dev)
    first_install_ms = 1000 * (time.perf_counter() - t_w0)
    log(f"window 0 planned + installed in {first_install_ms:.0f} ms (not overlapped with anything)")
    j = 0
    for _ in range(3):                 # eager steps: lazy initialisation (cuBLAS handles, scratch)
        one_step(j)
        j += 1
    if not a.no_graph:                 # capture one whole step; no plan thread is running right now
        ids0, X0, Y0 = window(0)
        tr.capture_graph(X0[:lb], lS_o, ids0[:, :lb], Y0[:lb])
    log("graph captured" if not a.no_graph else "eager mode")
    prepare(1)
    if world > 1:
        # lazy initialisation of the aggregation path (NCCL connections, pinned count buffers, the packed row
        # buffer): one untimed table aggregation; measured 0.6 s when it fell into a timed region
        broadcast_and_aggregate(tr.cache_group, None, rank, args.table_agg_op)
    for _ in range(max(W - 3, 0)):
        one_step(j)
        j += 1
    # A SHORT run would otherwise sit entirely inside the planner's burst (the plan and PCIe prefetch of the next
    # window take ~0.15 s right after a boundary and slow the step 1.2-1.3x while they run, 2.5 % averaged over the
    # 2.2 s window): let the burst finish first so that the short run measures the steady state.  The end-to-end
    # leg below covers a whole window with its boundary, plan, prefetch and aggregations inside the timed region.
    plan_inside = K >= L
    if not plan_inside and tr._plan_thread is not None:
        tr._plan_thread.join()
    # the clock sampler forks nvidia-smi: start it BEFORE the barrier so that every rank enters the timed region
    # together, and keep it running through the end-to-end leg (seconds, not milliseconds, of samples)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize(dev)
    log("warm-up done, timing")
    lib.cdlrm_prof_launches(1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_boundaries = 0
    cuprof = os.environ.get("CDLRM_BENCH_CUPROF", "0") == "1"   # ncu --profile-from-start off: timed region only
    if cuprof:
        torch.cuda.profiler.start()
    seg = max(1, K // 24)                 # per-segment device times: shows what the planner / boundaries cost
    marks = []
    probe = None
    if a.ce_probe_gb > 0:
        probe = (torch.empty(256 << 20, dtype=torch.uint8, pin_memory=True),
                 torch.empty(256 << 20, dtype=torch.uint8, device=dev), _lib.new_stream(dev),
                 torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    ev0.record()
    for i in range(K):
        if j % L == 0:
            n_boundaries += 1
        if probe is not None and i == K // 3:
            with torch.cuda.stream(probe[2]):
                probe[3].record()
                for _ in range(int(a.ce_probe_gb * 4)):
                    probe[1].copy_(probe[0], non_blocking=True)
                probe[4].record()
        last = one_step(j)
        j += 1
        if (i + 1) % seg == 0 and i + 1 < K:
            m = torch.cuda.Event(enable_timing=True)
            m.record()
            marks.append((i + 1, m))
    ev1.record()
    # copied behind the timed region, before the next step (a graph replay) overwrites the output buffers
    dumped = [t.detach().clone() for t in last] if a.dump_outputs and rank == 0 else None
    torch.cuda.synchronize(dev)
    if dumped is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, t in zip(("loss", "predictions"), dumped):
            np.save(os.path.join(a.dump_outputs, name + ".npy"), t.cpu().numpy().astype(np.float32))
        log(f"last timed step's outputs written to {a.dump_outputs}")
    if cuprof:
        torch.cuda.profiler.stop()
    launches = int(lib.cdlrm_prof_launches(0))
    if getattr(tr, "_graph", None) is not None:
        launches += K * tr.graph_launches      # graph replays re-issue the captured launches
    ms = ev0.elapsed_time(ev1)
    series, prev_i, prev_e = [], 0, ev0
    for i, m in marks + [(K, ev1)]:
        series.append(round(prev_e.elapsed_time(m) / (i - prev_i), 4))
        prev_i, prev_e = i, m
    if world > 1:
        dist.barrier()
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    log(f"timed region done: {ms / K:.3f} ms/step")
    if probe is not None:
        log(f"copy-engine probe: {a.ce_probe_gb} GB host-to-device in {probe[3].elapsed_time(probe[4]):.1f} ms, started "
            f"{ev0.elapsed_time(probe[3]):.1f} ms into the timed region; per-segment ms/step: {series}")
    value = K * lb * world / (ms / 1000.0)

    # -- per-kernel durations (CUDA events around every launch of the library) ------------------
    roof = kernels = None
    if not a.no_kernel_prof:
        kernels, roof, step_bytes, j = kernel_profile(a, wl, tr, lib, _lib, torch, one_step, window, master, lS_o, j, L,
                                                      lb, T, d, dev, ln_bot, ln_top)

    # -- end to end through the public API with host buffers ---------------------------------------
    e2e = full_window = None
    if a.e2e_steps >= 0:
        whole = a.e2e_steps == 0
        n_e2e = L if whole else a.e2e_steps
        if whole:
            # run (untimed) up to the next window boundary, so that the leg is exactly one window: its install
            # first, then the plan + PCIe prefetch of the following window beside the steps, every aggregation
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n_fill = (-j) % L
            f0.record()
            for _ in range(n_fill):
                one_step(j)
                j += 1
            f1.record()
        w_e, b_e = divmod(j, L)
        if not whole:
            n_e2e = min(n_e2e, L - b_e)
        ids, X, Y = window(w_e)
        torch.cuda.synchronize(dev)
        filler_ms = f0.elapsed_time(f1) / max(n_fill, 1) if whole and n_fill else None
        # this window's inputs in pinned host memory, one contiguous block per step
        hI = torch.empty(n_e2e, T, lb, dtype=torch.int64, pin_memory=True)
        hX = torch.empty(n_e2e, lb, X.shape[1], dtype=torch.float32, pin_memory=True)
        hY = torch.empty(n_e2e, lb, 1, dtype=torch.float32, pin_memory=True)
        lo = b_e * lb
        hI.copy_(ids[:, lo:lo + n_e2e * lb].view(T, n_e2e, lb).permute(1, 0, 2))
        hX.copy_(X[lo:lo + n_e2e * lb].view(n_e2e, lb, -1))
        hY.copy_(Y[lo:lo + n_e2e * lb].view(n_e2e, lb, 1))
        hosts = (hX, hI, hY)
        del ids, X, Y
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)
        log(f"end-to-end leg: {n_e2e} steps from pinned host inputs ({(hI.nbytes + hX.nbytes + hY.nbytes) / 1e9:.1f} GB)")
        logging_on[0] = True
        tr.cache_group._agg_prof = [] if world > 1 else None      # phase events of every table aggregation of the leg
        lib.cdlrm_prof_launches(1)
        seg2 = max(1, n_e2e // 120)
        marks2 = []
        t0 = time.perf_counter()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        # Every step: its inputs come from pinned host memory (Trainer.stage_inputs: the copy of step i+1 runs on
        # the copy stream beside step i) and its loss is read back to the host (asynchronous copy into a pinned
        # ring, read one step later, so that the host can enqueue step i+1 while step i runs).
        # The host runs AHEAD steps in front of the device (a data-parallel rank that may not run ahead stalls its
        # peers in every step's all-reduce whenever its host thread hiccups): inputs of step i+AHEAD are staged while
        # step i is enqueued, the loss of step i-AHEAD is read while step i runs.
        AHEAD = tr.input_slots - 2
        loss_host = float("nan")
        e0.record()
        staged = [tr.stage_inputs(hX[q], hI[q], hY[q]) for q in range(min(AHEAD, n_e2e))]
        host_t = []                                  # host clock at the top of the first 41 iterations
        for i in range(n_e2e):
            if i <= 40:
                host_t.append(time.perf_counter())
            # (one_step indexes the host block by the step's position in its window)
            w_, b_ = divmod(j, L)
            if b_ == 0 and j > 0:
                boundary(j)
            if i + AHEAD < n_e2e:
                staged.append(tr.stage_inputs(hX[i + AHEAD], hI[i + AHEAD], hY[i + AHEAD]))
            E, _ = tr.step_staged(staged.pop(0), lS_o)
            aggregate(j)
            tr.push_loss(E)                          # device -> host read of the step's result (asynchronous)
            if tr.pending_losses() > AHEAD:
                loss_host = tr.pop_loss()            # the loss of step i - AHEAD
            j += 1
            if ((i + 1) % seg2 == 0 or i < 40) and i + 1 < n_e2e:
                m = torch.cuda.Event(enable_timing=True)
                m.record()
                marks2.append((i + 1, m))
        while tr.pending_losses():                   # the last AHEAD losses
            loss_host = tr.pop_loss()
        e1.record()
        torch.cuda.synchronize(dev)
        wall_ms = 1000 * (time.perf_counter() - t0)
        logging_on[0] = False
        e2e_launches = int(lib.cdlrm_prof_launches(0)) + (n_e2e * tr.graph_launches if getattr(tr, "_graph", None) else 0)
        ems = e0.elapsed_time(e1)
        series2, prev_i, prev_e = [], 0, e0
        for i, m in marks2 + [(n_e2e, e1)]:
            series2.append(round(prev_e.elapsed_time(m) / (i - prev_i), 4))
            prev_i, prev_e = i, m
        if world > 1:
            t = torch.tensor([ems], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t.item())
        hb = (hI[0].nbytes + hX[0].nbytes + hY[0].nbytes)
        e2e = {"value": n_e2e * lb * world / (ems / 1000.0), "unit": "samples/s", "h2d_bytes_per_step": hb * world,
               "d2h_bytes_per_step": 4 * world, "steps": n_e2e, "ms_per_step": ems / n_e2e,
               "wall_ms_per_step": wall_ms / n_e2e, "last_loss": loss_host,
               "whole_window": whole, "gpu_launches": e2e_launches}
        # what the leg contained
        rec_next = None
        if tr._plan_thread is not None:
            tr._plan_thread.join()
        try:
            rec_next = tr._plan_q.queue[0] if tr._plan_q.qsize() else None
        except Exception:
            rec_next = None
        torch.cuda.synchronize(dev)
        full_window = {
            "ms_per_step": round(ems / n_e2e, 4), "steps": n_e2e, "window_boundaries": len(bound_log),
            "boundary_ms": [round(1000 * h, 3) for h, _, _ in bound_log],
            "boundary_device_ms": [round(b0.elapsed_time(b1), 3) for _, b0, b1 in bound_log],
            "aggregations": len(agg_log),
            "agg_ms_per_call": round(float(np.mean([1000 * h for h, _, _ in agg_log])), 4) if agg_log else None,
            "agg_device_ms_per_call": round(float(np.mean([b0.elapsed_time(b1) for _, b0, b1 in agg_log])), 4) if agg_log else None,
            "agg_ms_per_step_amortised": round(float(np.sum([b0.elapsed_time(b1) for _, b0, b1 in agg_log])) / n_e2e, 5) if agg_log else 0.0,
            "ms_per_step_series": {"steps_per_segment": seg2, "first_40_steps_ms": series2[:40],
                                   # how long the HOST spent in each of those iterations (a stall here that the device
                                   # series repeats AHEAD steps later is the host thread's, not the GPU's)
                                   "first_40_host_iter_ms": [round(1e3 * (y - x), 3) for x, y in zip(host_t, host_t[1:])],
                                   "ms_per_step": series2[40:]},
            "boundary_host_breakdown_ms": [b for _, b in prep_log],
            "next_window_input_generation_host_ms": [p_ for p_, _ in prep_log],
            "steady_ms_per_step_before": round(filler_ms, 4) if filler_ms else None,
        }
        ap = getattr(tr.cache_group, "_agg_prof", None)
        tr.cache_group._agg_prof = None
        if ap:
            # [dirty-bitmap all-gather + OR + slot lists | host reads the counts | pack | all-reduce | unpack], device ms
            names = ("bitmaps_and_lists", "host_sync_gap", "pack", "all_reduce", "unpack")
            ph = np.asarray([[m[q].elapsed_time(m[q + 1]) for q in range(5)] for _t, m in ap if len(m) == 6])
            rows_ = float(np.mean([t_ for t_, _m in ap]))
            full_window["agg_phases_device_ms"] = {n_: round(float(v_), 3) for n_, v_ in zip(names, ph.mean(0))} if len(ph) else None
            full_window["agg_rows_per_call"] = int(rows_)
            full_window["agg_row_bytes_per_call"] = int(rows_ * d * 4)
            if len(ph) and ph.mean(0)[3] > 0:
                full_window["agg_all_reduce_algbw_GB/s"] = round(rows_ * d * 4 / (ph.mean(0)[3] * 1e-3) / 1e9, 1)
        if rec_next is not None and not isinstance(rec_next, Exception) and getattr(rec_next, "stage_begin", None) is not None:
            st_ms = rec_next.stage_begin.elapsed_time(rec_next.staged)
            full_window["planner_ms"] = {k: round(1000 * v, 1) for k, v in tr.planner.last_timing.items()}
            # when, after the start of the leg, each phase of the next window's look-ahead ended on the side stream
            tl = {"ids_ready": data[max(data)][3]}
            tl.update(rec_next.marks)
            tl.update(stage_begin=rec_next.stage_begin, staged=rec_next.staged)
            if tr._installed is not None and tr._installed.wb_done is not None:
                tl["writeback_done"] = tr._installed.wb_done      # the leg's own boundary: evicted rows back in the master
            full_window["planner_timeline_ms"] = {k: round(e0.elapsed_time(v), 1) for k, v in tl.items()}
            full_window["planner_ms"]["prefetch"] = round(st_ms, 1)
            pcie["prefetch_rows"] = {"fills": int(sum(rec_next.F)), "evictions": int(sum(rec_next.E)),
                                     "losers_staged": int(sum(rec_next.L)) if rec_next.L is not None else 0}
            pcie["prefetch_bytes"] = int(rec_next.stage_bytes)
            pcie["prefetch_ms"] = round(st_ms, 2)
            pcie["prefetch_GB/s"] = round(rec_next.stage_bytes / (st_ms * 1e-3) / 1e9, 2) if st_ms > 0 else None
            pcie["prefetch_frac_of_h2d_peak"] = round(pcie["prefetch_GB/s"] / pcie["h2d_GB/s"], 3) if st_ms > 0 else None
            pcie["prefetch_how"] = (("host threads (%d) gather master rows into pinned chunks, cudaMemcpyAsync on the "
                                     "planner stream (copy engine)" % tr.planner.host_threads)
                                    if tr.planner.pcie_mode == "ce" else
                                    "SM-driven zero-copy row gathers from the pinned master (32 CTAs)") + \
                                   ", beside the training steps of the end-to-end leg, all ranks at once" + \
                                   ("; fills sharded over the ranks (1/world of them per rank over PCIe, the others over NVLink "
                                    "at the boundary)" if getattr(tr, "sharded_fills", False) else "")
        del hosts, hI, hX, hY
    clocks = sampler.stop() if sampler else None

    res = None
    cache_gb = sum(int(e.weight.numel()) for e in tr.cache_group.emb_l) * 4 / 1e9
    l2_policy = (f"inputs larger than L2: every step reads a fresh {T}x{lb}-row slice of a {cache_gb:.1f} GB cache and a "
                 "new batch of the window's inputs") if cache_gb > 0.5 else \
                (f"NOT flushed: the whole {cache_gb * 1e3:.0f} MB cache fits the 126 MB L2 (a parity-test configuration of "
                 "BASELINE.json, not the bench line)")
    if rank == 0:
        peak, _src = measured_peak()
        res = {
            "metric": METRIC,
            "value": value, "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(a, wl, T, world),
                       "global_batch": Bg, "local_batch": lb, "parallelism": f"dp{world} (replicated cache)",
                       "window_boundaries_in_timed_region": n_boundaries,
                       "l2_policy": l2_policy,
                       "lookahead_plan": "planned inside the timed region" if plan_inside else
                                         "next window planned before the timed region (steps < lookahead); the e2e leg "
                                         "is a whole window with its boundary, plan, prefetch and aggregations inside",
                       "cuda_graph": getattr(tr, "_graph", None) is not None,
                       "hbm_peak_allocated_gb": round(torch.cuda.max_memory_allocated(dev) / 1e9, 1),
                       "setup_s": round(setup_s, 1), "master_host_gb": round(sum(ln_emb) * d * 4 / 1e9, 1),
                       "first_window_install_ms": round(first_install_ms, 1)},
            "e2e": e2e, "full_window": full_window, "gpu_launches": launches, "clocks": clocks, "roofline": roof,
            "pcie": pcie, "kernels": kernels,
            "caching_overhead_ms_per_window": [round(1000 * x, 2) for x in tr.caching_overhead[-3:]],
            "ms_per_step_series": {"steps_per_segment": seg, "ms_per_step": series},
        }
        if kernels is not None:
            # whole-step roofline: algorithmic bytes of the cache path + interaction per step over the step time
            res["step_roofline"] = {
                "algo_bytes_per_step": int(step_bytes), "ms_per_step": round(ms / K, 4),
                "GB/s": round(step_bytes / (ms / K * 1e-3) / 1e9, 1), "peak": peak,
                "frac": round(step_bytes / (ms / K * 1e-3) / 1e9 / peak, 3),
                "note": "HBM-bound kernels only (cache forward / miss / update, interaction fwd / bwd); the rest of the "
                        "step is the 3xTF32 MLP GEMMs (tensor-bound, kernels.mlp_gemm)"}
    if world > 1:
        dist.barrier()
    tr.finish()
    return res, rank


def kernel_profile(a, wl, tr, lib, _lib, torch, one_step, window, master, lS_o, j, L, lb, T, d, dev, ln_bot, ln_top):
    """Eager steps with every library launch bracketed by CUDA events on its own stream (every rank takes these
    steps: they contain collectives).  Returns (kernels, roofline, algorithmic bytes per step, next step index)."""
    NK = lib.cdlrm_prof_num_kernels()
    if j % L == 0:              # at a window boundary (the whole-window e2e leg ends on one): take it first
        one_step(j)
        j += 1
    if tr._plan_thread is not None:     # the look-ahead plan / prefetch of the next window must not run beside
        tr._plan_thread.join()          # the kernels being timed
    tr.side.synchronize()
    torch.cuda.synchronize(dev)
    lib.cdlrm_prof_enable(1)
    nprof = 0
    graph, tr._graph = getattr(tr, "_graph", None), None     # eager launches so that events can bracket them
    # every kernel alone on one stream (no overlap with the MLPs), so that a duration is the kernel's own
    fstream, tr.cache_group.forward_stream = tr.cache_group.forward_stream, None
    eplan, tr.cache_group.early_plan = tr.cache_group.early_plan, False
    lib.cdlrm_mlp_set_option(5, 0)      # weight-gradient GEMMs in line, not beside the data-gradient chain
    for _ in range(20):
        if j % L == 0:
            break
        # park the GPU for ~4 ms so that the host enqueues the whole step ahead of it: the event pair
        # around a launch then brackets the kernel alone, not the host's launch latency before it
        torch.cuda._sleep(8_000_000)
        one_step(j)
        for _ in range(4):          # calibration: an empty kernel through the same event pair
            lib.cdlrm_prof_null(ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        j += 1
        nprof += 1
    tr._graph = graph
    tr.cache_group.forward_stream, tr.cache_group.early_plan = fstream, eplan
    lib.cdlrm_mlp_set_option(5, int(os.environ.get("CDLRM_WGRAD_SIDE", "1") != "0"))
    msv = (ctypes.c_double * NK)()
    calls = (ctypes.c_int64 * NK)()
    _lib.check(lib.cdlrm_prof_report(msv, calls, NK))
    log(f"kernel profile over {nprof} eager steps: {lib.cdlrm_last_error().decode()}")
    lib.cdlrm_prof_enable(0)
    n_miss = int(tr.cache_group.last_n_miss.sum().item())
    w, b = divmod(j - 1, L)
    lo = b * lb
    ids = window(w)[0][:, lo:lo + lb]
    n_distinct = 0
    with torch.no_grad():
        _, sl = tr.cache_group(lS_o, ids, master, dev.index)
        tr.cache_group.join_forward()
        for s_ in sl:
            n_distinct += int(torch.unique(s_).numel())
    n = T * lb
    nfe = T + 1
    npair = nfe * (nfe - 1) // 2
    algo = {   # ALGORITHMIC bytes per launch (DESIGN.md section 4)
        # id + tag line + slot + miss-bitmap word per id; row read + out write per hit
        "embed_fwd": n * (8 + 8 * wl["ways"] + 4) + n // 8 + (n - n_miss) * 8 * d,
        # bitmap read; per miss: id + slot + row read (HBM loser store or PCIe) + aux row + out row
        "embed_miss": n // 8 + n_miss * (8 + 4 + 12 * d),
        "bwd_plan": n * (4 + 8),
        # per id: sorted (slot, position) pair + its gradient row; per distinct slot: weight row read + write
        "bwd_sgd": n * (8 + 4 * d) + n_distinct * 8 * d,
        "interact_fwd": lb * (nfe * 4 * d + (d + npair) * 4),
        "interact_bwd": lb * (2 * nfe * 4 * d + (d + npair) * 4),
    }
    peak, peak_src = measured_peak()
    kernels = {}
    names = [lib.cdlrm_prof_kernel_name(i).decode() for i in range(NK)]
    # what the event pair itself adds (an empty kernel measured the same way): reported next to the raw time
    i_null = names.index("null")
    null_us = 1000.0 * msv[i_null] / calls[i_null] if calls[i_null] else 0.0
    traffic, traffic_src = {}, None
    tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(tpath) and a.workload == "terabyte" and not (a.cache_size or a.num_ways or a.batch):
        tj = json.load(open(tpath))    # dram__bytes_read.sum + dram__bytes_write.sum per launch (one ncu pass at this configuration)
        traffic, traffic_src = tj["kernels"], tj.get("source", "profiles/r2_traffic.json")
    for i in range(NK):
        if calls[i] and i != i_null:
            nm = names[i]
            raw = 1000.0 * msv[i] / calls[i]
            us = max(raw - null_us, 0.25 * raw)
            kernels[nm] = {"us_per_launch": round(us, 2), "us_raw_event_pair": round(raw, 2),
                           "launches_per_step": calls[i] / max(nprof, 1)}
            if nm in algo:
                kernels[nm]["algo_bytes"] = int(algo[nm])
                kernels[nm]["GB/s"] = round(algo[nm] / (us * 1e-6) / 1e9, 1)
                kernels[nm]["frac_of_peak"] = round(algo[nm] / (us * 1e-6) / 1e9 / peak, 3)
                kernels[nm]["frac_of_peak_raw_event_pair"] = round(algo[nm] / (raw * 1e-6) / 1e9 / peak, 3)
            if nm in traffic:
                db = int(traffic[nm]["dram_bytes_per_launch"])
                kernels[nm]["ncu_dram_bytes_static_profile"] = db
                # the Zipf head and the tiny tables are served by L2: DRAM traffic, not algorithmic bytes, is what
                # an HBM fraction has to be quoted on when the two differ
                kernels[nm]["dram_frac_of_peak"] = round(db / (us * 1e-6) / 1e9 / peak, 3)
            if nm == "embed_miss":
                kernels[nm]["misses_per_step"] = n_miss
    # useful FP32 flops of the MLP GEMMs (forward + data gradient + weight gradient); the tcgen05 kernel
    # spends 3 TF32 products per FP32 product (3xTF32 split, DESIGN.md section 4)
    if "mlp_gemm" in kernels:
        def mlp_flops(ln):
            f = 0
            for i in range(len(ln) - 1):
                f += 2 * lb * int(ln[i]) * int(ln[i + 1]) * (3 if i > 0 else 2)    # no dgrad below layer 0 ...
            return f
        fl = mlp_flops(ln_bot) + mlp_flops(ln_top) + 2 * lb * int(ln_bot[0]) * int(ln_bot[1])  # ... except bottom dX
        g = kernels["mlp_gemm"]
        t_us = g["us_per_launch"] * g["launches_per_step"]
        g["fp32_flops_per_step"] = int(fl)
        g["us_per_step"] = round(t_us, 1)
        g["useful_TFLOP/s"] = round(fl / (t_us * 1e-6) / 1e12, 1)
        g["tf32_TFLOP/s"] = round(3 * fl / (t_us * 1e-6) / 1e12, 1)
    roof = None
    cand = [k for k in kernels if "GB/s" in kernels[k] and k != "embed_miss"]
    if cand:
        top = max(cand, key=lambda k: kernels[k]["us_per_launch"] * kernels[k]["launches_per_step"])
        roof = {"bound": "hbm", "kernel": top, "achieved": kernels[top]["GB/s"], "peak": peak, "unit": "GB/s",
                "frac": kernels[top]["frac_of_peak"],
                "traffic": kernels[top].get("ncu_dram_bytes_static_profile"),
                "traffic_source": traffic_src if kernels[top].get("ncu_dram_bytes_static_profile") else None,
                "peak_source": peak_src,
                "algo_bytes_per_launch": kernels[top]["algo_bytes"],
                "us_per_launch": kernels[top]["us_per_launch"],
                "us_raw_event_pair": kernels[top]["us_raw_event_pair"],
                "frac_raw_event_pair": kernels[top]["frac_of_peak_raw_event_pair"],
                "event_pair_overhead_us": round(null_us, 2),
                "note": "dominant HBM-bound kernel of the cache path; us_per_launch is net of the event-pair overhead "
                        "(an empty kernel through the same pair), frac_raw_event_pair is the same fraction without that "
                        "subtraction; the MLP GEMMs (tensor-bound) are under kernels.mlp_gemm"}
    step_bytes = sum(algo[k] for k in algo if k in kernels)
    return kernels, roof, step_bytes, j


def main():
    a = parse()
    # stdout carries exactly ONE JSON line: everything else a library prints there (NCCL's version banner at
    # N > 1) goes to stderr
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    try:
        _main(a, real_stdout)
    finally:
        real_stdout.flush()


def cpu_arm(a, wl, ln_emb, steps, warmup, window_steps):
    """The reference's CPU path on this box's host cores: the reference's OWN code from baseline/_ref
    (kind "reference", baseline/ref_arm.py) when the copy made by __graft_entry__.install_reference travelled with
    the snapshot, else the numpy oracle port (kind "port")."""
    sys.path.insert(0, ROOT)
    from baseline import ref_arm
    if ref_arm.available():
        r = ref_arm.run(wl, ln_emb, steps, warmup, window_steps, dist=a.dist, zipf_a=a.zipf_a, log=log)
        r["kind"] = "reference"
        return r
    log("baseline/_ref is missing: timing the numpy oracle port instead of the reference's own code")
    r = cpu_reference_run(wl, ln_emb, steps, warmup, 60.0, a.dist, a.zipf_a)
    r["kind"] = "port"
    return r


def _main(a, out):
    wl = dict(WORKLOADS[a.workload])
    for key, val in (("lookahead", a.lookahead), ("cache", a.cache_size), ("ways", a.num_ways),
                     ("agg", a.table_agg_freq), ("batch", a.batch)):
        if val:
            wl[key] = val
    ln_emb = table_rows(wl, a.row_cap)
    rank = int(os.environ.get("RANK", "0"))
    world = max(a.gpus, 1)
    if a.impl == "reference":
        if rank != 0:
            return
        K = a.steps if a.steps > 0 else 20
        W = max(a.warmup, 0)
        # a window long enough to hold the warm-up and the timed steps, at least 32 steps (bounded: the install of
        # a 3000-step window takes the reference minutes)
        Lp = a.ref_window_steps or max(32, min(wl["lookahead"], K + W))
        r = cpu_arm(a, wl, ln_emb, K, W, Lp)
        cb = {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
        for k in ("step_ms", "step_ms_median", "install_s", "window_steps", "lookahead", "batch", "installs"):
            if k in r:
                cb[k] = r[k]
        line = {"impl": "reference", "metric": METRIC,
                "value": r["value"], "unit": "samples/s", "n_gpus": a.gpus, "steps": K, "warmup": a.warmup,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_string(a, wl, len(ln_emb), world),
                           "note": "CPU arm on the box's host cores (no GPU work, nothing of cdlrm_b200 loaded): the "
                                   "reference's own functions at the full batch of ONE trainer; a CPU run does not "
                                   "scale with --gpus, the same figure stands beside every N (cpu_baseline.sample "
                                   "says what was run)"},
                "cpu_baseline": cb,
                "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        out.write(json.dumps(line) + "\n")
        return
    res, rank = gpu_run(a, wl, ln_emb)
    if rank == 0:
        if not a.no_cpu_baseline and int(os.environ.get("WORLD_SIZE", "1")) == 1:
            r = cpu_arm(a, wl, ln_emb, max(a.cpu_baseline_steps, 1), 1, 8)
            res["cpu_baseline"] = {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": r["kind"],
                                   "sample": r["sample"]}
            if "step_ms" in r:
                res["cpu_baseline"].update(step_ms=round(r["step_ms"], 2), install_s=[round(x, 2) for x in r["install_s"]])
        out.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
