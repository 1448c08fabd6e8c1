#!/usr/bin/env python
"""Two-rank checkpoint / resume check of the data-parallel Trainer (run under torchrun, one rank per GPU; used by
tests/test_gpu_checkpoint.py).  Three invocations, in this order, share $CKPT_DIR:

  full    an uninterrupted run of N_WINDOWS windows; records tags, losses and dense parameters per rank, then
          sync_master: every rank writes its share of the sets into the shared master, and the shares together
          must cover every valid cache line exactly once, with the row the cache holds
  save    the first K windows, then save_checkpoint at the boundary before window K (plan(K) in flight)
  resume  fresh processes and a fresh master: load_checkpoint, run windows K..N_WINDOWS-1, compare with "full"

  torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/mgpu_ckpt_check.py full|save|resume
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_WINDOWS, K = 4, 2


def main(phase):
    from cdlrm_b200.main_no_ddp import ProcessArgs, Trainer
    from cdlrm_b200.model_no_ddp import Embedding_Table_Group
    from cdlrm_b200.synthetic import SyntheticStream
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank)))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    out_dir = os.environ["CKPT_DIR"]
    ln_emb = [5000, 37, 90000, 1200]
    d, lb, L, ways, csz, agg = 16, 96, 5, 4, 211, 3
    Bg, T = lb * world, len(ln_emb)
    args = ProcessArgs(["--arch-sparse-feature-size", str(d), "--arch-mlp-bot", f"13-32-{d}", "--arch-mlp-top", "32-1",
                        "--loss-function", "bce", "--learning-rate", "0.1", "--lr-embeds", "0.3",
                        "--mini-batch-size", str(Bg), "--lookahead", str(L), "--cache-size", str(csz), "--num-ways",
                        str(ways), "--table-agg-freq", str(agg), "--world-size", str(world), "--numpy-rand-seed", "9"])
    nf = T + 1
    ln_bot, ln_top = np.asarray([13, 32, d]), np.asarray([nf * (nf - 1) // 2 + d, 32, 1])
    prefix = f"/dev/shm/cdlrm_ckpt_{os.environ.get('MASTER_PORT', '0')}"
    if rank == 0:
        master = Embedding_Table_Group(d, np.asarray(ln_emb), init=f"shm:{prefix}:create")
    dist.barrier()
    if rank != 0:
        master = Embedding_Table_Group(d, np.asarray(ln_emb), init=f"shm:{prefix}:attach")
    tr = Trainer(args, d, np.asarray(ln_emb), ln_bot, ln_top, master, rank=rank, world=world, device=dev)
    dist.barrier()
    if rank == 0:
        for k in range(T):
            os.unlink(f"{prefix}_{k}.bin")
    assert tr.wb_sharded, "the /dev/shm master is one shared object: the ranks share the write-back"
    sg = SyntheticStream(ln_emb, Bg, dev, dist="zipf", zipf_a=1.05, seed=11)
    rng = np.random.default_rng(5)
    X = torch.from_numpy(rng.standard_normal((N_WINDOWS * L, Bg, 13)).astype(np.float32)).to(dev)
    Y = (X[:, :, :1] > 0).float()
    lS_o = torch.arange(lb).reshape(1, -1).repeat(T, 1)
    path = os.path.join(out_dir, "ck")
    w0 = tr.load_checkpoint(path) if phase == "resume" else 0
    w_end = K if phase == "save" else N_WINDOWS
    tags, losses = [], []
    tr.submit_window(sg.window_ids(w0, L))
    for w in range(w0, w_end):
        tr.install_window()
        if w + 1 < N_WINDOWS:
            tr.submit_window(sg.window_ids(w + 1, L))
        tags.append(torch.cat([t.reshape(-1) for t in tr.cache_group.occupancy_tables]).cpu().numpy())
        g = sg.window_ids(w, L)
        for j in range(L):
            s = w * L + j
            ids = g[:, j * Bg:(j + 1) * Bg][:, rank * lb:(rank + 1) * lb].contiguous()
            E, _Z = tr.step(X[s, rank * lb:(rank + 1) * lb], lS_o, ids, Y[s, rank * lb:(rank + 1) * lb])
            tr.maybe_aggregate(j)
            losses.append(float(E))
    if phase == "save":
        tr.save_checkpoint(path)
    tr.finish()
    dense = tr.dlrm.flat_params.cpu().numpy()
    mine = os.path.join(out_dir, f"{phase}_{rank}.npz")
    if phase == "full":
        # export: each rank writes its share of the sets; together every valid line exactly once
        n = torch.tensor([tr.sync_master()], device=dev)
        dist.all_reduce(n)
        valid = sum(int((t >= 0).sum()) for t in tr.cache_group.occupancy_tables)
        assert int(n) == valid, f"the sync_master shares wrote {int(n)} rows, the caches hold {valid} valid lines"
        cg = tr.cache_group
        for k in range(T):
            t = cg.occupancy_tables[k].cpu().numpy()
            S = t.shape[0]
            sets, wys = np.nonzero(t >= 0)
            rows = cg.emb_l[k].weight.data[:ways * S].cpu().numpy()[wys * S + sets]
            assert np.array_equal(master.emb_l[k].weight.data.numpy()[t[sets, wys]], rows), f"table {k}: export"
        np.savez(mine, tags=np.stack(tags), losses=np.asarray(losses), dense=dense)
    elif phase == "resume":
        ref = np.load(os.path.join(out_dir, f"full_{rank}.npz"))
        assert np.array_equal(ref["tags"][K:], np.stack(tags)), "tags after resume differ from the uninterrupted run"
        np.testing.assert_allclose(np.asarray(losses), ref["losses"][K * L:], rtol=1e-5)
        np.testing.assert_allclose(dense, ref["dense"], rtol=0, atol=1e-5)
    dist.barrier()
    if rank == 0 and phase == "resume":
        print("mgpu_ckpt_check OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1])
