"""Window planner parity at the benchmark's table and window sizes.

bench.py plans windows of 3000 steps x 8192 ids over tables of up to 39.9 M rows.  At that size the compaction kernels
(compact.cuh, plan.cu) run code that smaller windows never reach:
  * the carry of scan_tiles_kernel from one round of 1024 tiles to the next: an id bitmap above 2^25 rows, or more
    than 2^20 unique ids, survivors, fills, evictions or losers in one table;
  * millions of survivors contesting the same (set, way) (select_kernel's atomicMax, the win flag of lists_kernel);
  * sets whose every way is pinned by a hit (drops);
  * the bucket index of a loser store over a 40 M-row table (build_loser_buckets, miss_row).
Here the production path -- Embedding_Table_Cache_Group, WindowPlanner with the device victim stream, chunked
mark_ids, plan, stage, install_staged, the forward -- runs at that size, and every decision is compared with the numpy
oracle (oracle/oracle.py, pinned to the reference's golden vectors), which plans a full-size window table by table.

The embedding dimension is 16: the planner's integer decisions do not depend on it, and it keeps the host master tables
at 5.2 GB.  No SGD step runs, so every cache row and every evicted row is a copy of its master row and the master
never changes: one master serves every configuration and both PCIe modes.
"""
import contextlib

import numpy as np
import pytest
import torch

import util
from oracle import oracle as O

DEV = "cuda:0"
ROWS = [39884406, 38532951, 2953546, 403346, 7420, 3]    # Terabyte tables: the two 40 M-row ones, mid, small, tiny
DIM, BATCH = 16, 8192
SEED_IDS, SEED_RNG = 123, 11
CHUNK_STEPS = 512            # steps per mark_ids call: 4 M ids per table, as bench.py's chunked scan
CONFIGS = {
    # the bench line: Terabyte window and cache, zipf 1.05 ids, the Trainer's eviction lists (one entry per slot)
    "A": dict(L=3000, csz=150000, ways=16, dist="zipf", primary=True, own=False),
    # BASELINE.json configs[3]: uniform ids into a 50000 x 4 cache -- dozens of claimants per line and fully pinned
    # sets; the reference's eviction lists (one entry per claimant); a rank-private loser store (first half of
    # every batch)
    "B": dict(L=1000, csz=50000, ways=4, dist="uniform", primary=False, own=True),
}


# ---------------------------------------------------------------------------------------------------------------
# reference: the oracle's pieces, assembled into what the planner returns (checked on the CPU by the last test)
# ---------------------------------------------------------------------------------------------------------------

def unique_ids(ids, n_rows):
    """Ascending distinct ids of one table's window, through a mask over the table: np.unique would sort 25 M ids,
    and the oracle's process_batch_slice builds an id -> row map of max(id) + 1 entries."""
    m = np.zeros(n_rows, dtype=bool)
    m[ids] = True
    return np.flatnonzero(m)


def claim_winners(slot):
    """win[r]: survivor r is the last claimant of its slot (the reference's single-thread index_put_)."""
    win = np.zeros(len(slot), dtype=bool)
    if len(slot):
        _, last = np.unique(slot[::-1], return_index=True)
        win[len(slot) - 1 - last] = True
    return win


def is_cached(tags, u, chunk=1 << 21):
    S = tags.shape[0]
    out = np.empty(len(u), dtype=bool)
    for i in range(0, len(u), chunk):
        x = u[i:i + chunk]
        out[i:i + chunk] = (tags[x % S] == x[:, None]).any(axis=1)
    return out


def plan_reference(tags, u, draw):
    """One table's plan for the window whose ascending unique ids are ``u`` (O.plan_table; mutates ``tags``), in the
    shape of a PlanRecord: counts, fill list, the reference's eviction list (one entry per claimant, flagged primary
    for the claimant that wins the slot) and the ascending un-cached ids."""
    before = tags.copy()
    p = O.plan_table(tags, tags.shape[0], tags.shape[1], u, draw)
    win = claim_winners(p["slot"])
    old = before[p["surv_sets"], p["way"]]
    ev = old != -1
    assert np.array_equal(old[ev], p["evict_ids"])
    return dict(uniq=len(u), hits=p["n_hit"], dropped=p["n_dropped"], rows=len(p["slot"]), F=int(win.sum()),
                fill_ids=p["surv_ids"][win], fill_slots=p["slot"][win],
                evict_ids=old[ev], evict_slots=p["slot"][ev], evict_primary=win[ev],
                losers=u[~is_cached(tags, u)], tags=tags.copy())


def primary_evictions(ref):
    """The eviction list of WindowPlanner.primary_evictions_only: the winner's entry of every replaced slot."""
    keep = ref["evict_primary"]
    return ref["evict_ids"][keep], ref["evict_slots"][keep], ref["evict_primary"][keep]


def own_mask(ids, n_rows, steps, half):
    """Ids of the first ``half`` samples of every batch of a window [steps * batch] (a data-parallel rank's own)."""
    m = np.zeros(n_rows, dtype=bool)
    m[ids.reshape(steps, -1)[:, :half]] = True
    return m


def reference_run(c, master_np, window_on_host):
    """Everything the planner must produce for two windows of configuration ``c``: per window and table the expected
    record (lists shaped as the configuration asks) and, for the first, a middle and the last step of window 2, the
    forward's slots, miss counts and pooled rows plus the missed ids that the loser store must serve."""
    T, L, ways = len(ROWS), c["L"], c["ways"]
    oc = O.OracleCache(DIM, ROWS, c["csz"], BATCH, ways)
    gen = O.TorchCpuGenerator(SEED_RNG)
    out = {"windows": [], "draws": [], "fwd": []}
    for w in range(2):
        ids = window_on_host(w)
        per = []
        for k, n in enumerate(ROWS):
            e = plan_reference(oc.tags[k], unique_ids(ids[k], n), gen.exponential_f32)
            if c["primary"]:
                e["evict_ids"], e["evict_slots"], e["evict_primary"] = primary_evictions(e)
            if c["own"]:
                e["losers"] = e["losers"][own_mask(ids[k], n, L, BATCH // 2)[e["losers"]]]
            e["E"], e["L"] = len(e["evict_ids"]), len(e["losers"])
            per.append(e)
        out["windows"].append(per)
        out["draws"].append(gen.draws)
    # window 2 is installed: with no SGD step, every live line holds its id's master row
    for k in range(T):
        S = oc.cache_sizes[k]
        sets, way = np.nonzero(oc.tags[k] >= 0)
        oc.weight[k][S * way + sets] = master_np[k][oc.tags[k][sets, way]]
    for b in (0, L // 2, L - 1):
        f = {"step": b, "rows": [], "slots": [], "n_miss": [], "store": []}
        for k in range(T):
            x = ids[k, b * BATCH:(b + 1) * BATCH]
            rows, slots, n_miss = O.forward_table_fast(oc, k, x, master_np[k])
            missed = np.unique(x[slots >= oc.cache_sizes[k] * ways])
            store = np.intersect1d(missed, out["windows"][1][k]["losers"], assume_unique=True)
            assert c["own"] or len(store) == len(missed), "a missed id of the window is not in its loser list"
            f["rows"].append(rows)
            f["slots"].append(slots)
            f["n_miss"].append(n_miss)
            f["store"].append(store)
        out["fwd"].append(f)
    return out


# ---------------------------------------------------------------------------------------------------------------
# the planner on the GPU
# ---------------------------------------------------------------------------------------------------------------

def _planner(master, ln, csz, ways, window_len, aux, primary, mode):
    from cdlrm_b200 import cache_manager as C
    from cdlrm_b200 import model_no_ddp as M
    cg = M.Embedding_Table_Cache_Group(master.emb_l[0].weight.shape[1], np.asarray(ln), csz, aux, ways).to(DEV)
    cg._ensure_ctx(master)
    rng = C.VictimRngDevice(SEED_RNG, DEV)
    pl = C.WindowPlanner(cg, master, window_len, rng=rng, lookahead_tags=True)
    pl.collect_losers = True
    pl.primary_evictions_only = primary
    pl.pcie_mode = mode
    return cg, pl, rng


def _check_plan(where, pl, rec, ref):
    """One window's plan against the reference, table by table (bit-exact).  Checked before anything consumes it."""
    torch.cuda.synchronize()
    for k, e in enumerate(ref):
        got = [rec.uniq[k], rec.hits[k], rec.dropped[k], rec.rows[k], rec.E[k], rec.F[k], rec.L[k]]
        want = [e["uniq"], e["hits"], e["dropped"], e["rows"], e["E"], e["F"], e["L"]]
        assert got == want, f"{where} table {k}: counts (uniq, hits, dropped, rows, E, F, L) {got} != {want}"
        fi, fs = (t.cpu().numpy() for t in rec.fill_list(k))
        assert np.array_equal(fi, e["fill_ids"]), f"{where} table {k}: fill ids differ"
        assert np.array_equal(fs, e["fill_slots"]), f"{where} table {k}: fill slots differ"
        ei, es, ep = (t.cpu().numpy() for t in rec.evict_list(k))
        assert np.array_equal(ei, e["evict_ids"]), f"{where} table {k}: evicted ids differ"
        assert np.array_equal(es, e["evict_slots"]), f"{where} table {k}: eviction slots differ"
        assert np.array_equal(ep.astype(bool), e["evict_primary"]), f"{where} table {k}: primary flags differ"
        assert np.array_equal(rec.loser_list(k).cpu().numpy(), e["losers"]), f"{where} table {k}: loser list differs"
        assert np.array_equal(pl.plan_tags[k].cpu().numpy(), e["tags"]), f"{where} table {k}: plan tags differ"


def _check_install(where, cg, rec, ref, master_np):
    """The cache after stage + install_staged: live tags, and the master's rows at the fill slots."""
    torch.cuda.synchronize()
    for k, e in enumerate(ref):
        assert np.array_equal(cg.occupancy_tables[k].cpu().numpy(), e["tags"]), f"{where} table {k}: live tags differ"
        if e["F"]:
            rows = cg.emb_l[k].weight.data[rec.fill_list(k)[1].long()].cpu().numpy()
            assert np.array_equal(rows, master_np[k][e["fill_ids"]]), f"{where} table {k}: filled rows differ"


@contextlib.contextmanager
def _negated(master_np, ids):
    """Master rows of ``ids[k]`` negated (exactly reversible): a missed id served from the master instead of the
    loser store then pools the wrong sign, whereas the two sources hold the same row otherwise."""
    for m, x in zip(master_np, ids):
        m[x] = -m[x]
    try:
        yield
    finally:
        for m, x in zip(master_np, ids):
            m[x] = -m[x]


@pytest.fixture(scope="module")
def master():
    from cdlrm_b200 import model_no_ddp as M
    m = M.Embedding_Table_Group(DIM, np.asarray(ROWS), init="device")
    return m, [e.weight.data.numpy() for e in m.emb_l]


@pytest.fixture(scope="module")
def reference(master):
    """reference(name): the oracle's results for configuration ``name``, computed once and shared by both PCIe modes
    (one configuration in host memory at a time)."""
    from cdlrm_b200.synthetic import SyntheticStream
    memo = {}

    def get(name):
        if name not in memo:
            memo.clear()
            c = CONFIGS[name]
            st = SyntheticStream(ROWS, BATCH, DEV, dist=c["dist"], zipf_a=1.05, seed=SEED_IDS)
            memo[name] = reference_run(c, master[1], lambda w: st.window_ids(w, c["L"]).cpu().numpy())
            torch.cuda.empty_cache()
        return memo[name]
    return get


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,mode", [("A", "sm"), ("A", "ce"), ("B", "sm"), ("B", "ce")])
def test_benchmark_size_windows_match_oracle(cfg, mode, master, reference):
    """Two windows of the benchmark's stream, planned, staged and installed, against the oracle; then the first, a
    middle and the last step of window 2 through the forward."""
    from cdlrm_b200.synthetic import SyntheticStream
    c, ref = CONFIGS[cfg], reference(cfg)
    m, master_np = master
    T, L, ways = len(ROWS), c["L"], c["ways"]
    cg, pl, rng = _planner(m, ROWS, c["csz"], ways, L * BATCH, BATCH, c["primary"], mode)
    st = SyntheticStream(ROWS, BATCH, DEV, dist=c["dist"], zipf_a=1.05, seed=SEED_IDS)
    lS_o = torch.arange(BATCH).reshape(1, -1).repeat(T, 1)
    assert max(-(-n // 32) for n in ROWS) > 1024 * 1024, "no id bitmap above 1024 tiles"
    draws = 0
    for w in range(2):
        where = f"config {cfg} ({mode}) window {w + 1}"
        if c["own"]:
            pl.mark_own_ids(st.ids(w * L, L, b0=0, nb=BATCH // 2))
        for s0 in range(0, L, CHUNK_STEPS):
            pl.mark_ids(st.ids(w * L + s0, min(CHUNK_STEPS, L - s0)))
        rec = pl.plan(marked=L * BATCH)
        draws += sum(rec.rows) * ways
        assert rng.draws == draws == ref["draws"][w], \
            f"{where}: victim draws {rng.draws}, {draws} by the counts, {ref['draws'][w]} by the oracle"
        _check_plan(where, pl, rec, ref["windows"][w])
        pl.stage(rec)
        pl.install_staged(rec)
        _check_install(where, cg, rec, ref["windows"][w], master_np)
        # what this configuration is for: carries past 1024 tiles, contested claims, a loser store with a bucket
        # index of shift > 0 (build_loser_buckets: at least 64 losers, n_rows > losers / 4 + 1)
        assert max(rec.uniq) > 1 << 20 and max(rec.rows) > 1 << 20, f"{where}: fewer than 2^20 unique ids / survivors"
        assert sum(rec.F) < sum(rec.rows), f"{where}: no contested claim"
        assert any(n > 1 << 25 and rec.L[k] >= 64 and n > rec.L[k] // 4 + 1 for k, n in enumerate(ROWS)), \
            f"{where}: no bucketed loser store over a 40 M-row table"
        if w == 1:
            assert sum(rec.E) > 0, f"{where}: no eviction"
            assert cfg != "B" or sum(rec.dropped) > 0, f"{where}: no fully pinned set"
    # the forward at scale: hits from the cache, misses through the bucket index of the loser store
    pl.flush_writeback()
    torch.cuda.synchronize()
    for f in ref["fwd"]:
        ids = st.ids(L + f["step"], 1)
        with _negated(master_np, f["store"]), torch.no_grad():
            ly, slots = cg(lS_o, ids, m, 0)
            n_miss = cg.last_n_miss.cpu().numpy()
            torch.cuda.synchronize()
        for k in range(T):
            where = f"config {cfg} ({mode}) step {L + f['step']} table {k}"
            assert np.array_equal(slots[k].cpu().numpy(), f["slots"][k]), f"{where}: slots differ"
            assert n_miss[k] == f["n_miss"][k], f"{where}: miss count {n_miss[k]} != {f['n_miss'][k]}"
            assert np.array_equal(ly[k].cpu().numpy(), f["rows"][k]), f"{where}: pooled rows differ"
    assert sum(len(x) for x in ref["fwd"][0]["store"]) > 0, "no miss was served from the loser store"
    cg.check_device_flags()


# ---------------------------------------------------------------------------------------------------------------
# the 1024-tile boundary of the id bitmap, without the stream
# ---------------------------------------------------------------------------------------------------------------

def boundary_window(n_rows, w):
    """Ids at both sides of every 1024-word tile boundary of the id bitmap, id 0 and the last id, and a dense block of
    2^20 + 1 consecutive ids (the unique, survivor, list and loser scans then span 1025 tiles).  Window 2 moves the
    block 3000 ids down: most of the cached ids (the boundary ids and the block's top) hit again and pin whole sets,
    the others miss and are evicted."""
    t = np.arange(1, 1025, dtype=np.int64) * 32768
    edges = np.concatenate([[0, 1 << 25], t - 1, t])
    block = np.arange((1 << 20) + 1, dtype=np.int64) + (3_000_000 if w == 0 else 2_997_000)
    return np.minimum(np.concatenate([edges, block]), n_rows - 1)[None, :]


@pytest.mark.gpu
@pytest.mark.parametrize("n_rows", [(1 << 25) + 1, 1 << 25])      # 1025 bitmap tiles (the last one a single word); 1024
def test_tile_boundary_windows_match_oracle(n_rows):
    from cdlrm_b200 import model_no_ddp as M
    m = M.Embedding_Table_Group(4, np.asarray([n_rows]), init="device")
    master_np = [m.emb_l[0].weight.data.numpy()]
    wins = [boundary_window(n_rows, w) for w in range(2)]
    n = wins[0].shape[1]
    cg, pl, rng = _planner(m, [n_rows], 1000, 4, n, 1024, False, "sm")
    oc = O.OracleCache(4, [n_rows], 1000, 1024, 4)
    gen = O.TorchCpuGenerator(SEED_RNG)
    for w, win in enumerate(wins):
        ref = plan_reference(oc.tags[0], unique_ids(win[0], n_rows), gen.exponential_f32)
        ref["E"], ref["L"] = len(ref["evict_ids"]), len(ref["losers"])
        x = torch.from_numpy(win).to(DEV)
        pl.mark_ids(x[:, :n // 2].contiguous())
        pl.mark_ids(x[:, n // 2:].contiguous())
        rec = pl.plan(marked=n)
        assert rng.draws == gen.draws
        _check_plan(f"{n_rows} rows, window {w + 1}", pl, rec, [ref])
        pl.stage(rec)
        pl.install_staged(rec)
        _check_install(f"{n_rows} rows, window {w + 1}", cg, rec, [ref], master_np)
        assert rec.uniq[0] > 1 << 20          # the survivor and loser scans span 1026 tiles
        if w == 0:
            assert rec.rows[0] > 1 << 20 and rec.F[0] < rec.rows[0]
        else:
            assert rec.dropped[0] > 0 and rec.hits[0] > 0 and rec.E[0] > 0 and rec.F[0] < rec.rows[0]
    cg.check_device_flags()


# ---------------------------------------------------------------------------------------------------------------
# the reference itself (CPU)
# ---------------------------------------------------------------------------------------------------------------

def test_reference_helpers_match_oracle_install_and_golden():
    """The pieces the GPU tests build their reference from, against O.install_window and the reference's own trace
    (trace_pressure.npz: an undersized cache with duplicate claims): unique ids, tags, the reference's eviction list
    (ids, and slots through the rows the oracle evicted), the fill list (through the rows the oracle's last-write-wins
    install left in the cache), the winner filter of primary evictions, and the loser list, which must hold exactly
    the ids the oracle's forward misses in the window's batches (all of them, or the first half of each)."""
    g = util.load_golden("trace_pressure.npz")
    cfg = util.golden_cfg(g)
    ln, B, L, ways = cfg["ln_emb"], cfg["batch"], cfg["lookahead"], cfg["num_ways"]
    ids, master = util.make_ids(cfg), util.master_init(cfg)
    oc = O.OracleCache(cfg["dim"], ln, cfg["cache_size"], B, ways)
    tags = [t.copy() for t in oc.tags]
    gen_o, gen_h = O.TorchCpuGenerator(cfg["seed"]), O.TorchCpuGenerator(cfg["seed"])
    contested = 0
    for w in range(cfg["n_windows"]):
        win = ids[:, w * L * B:(w + 1) * L * B]
        m0, w0 = [x.copy() for x in master], [x.copy() for x in oc.weight]
        ev, _plans, uniq = O.install_window(oc, master, win, gen_o)
        refs = []
        for k, n in enumerate(ln):
            u = unique_ids(win[k], n)
            assert np.array_equal(u, uniq[k]) and len(u) == g[f"w{w}_uniq_len"][k]
            refs.append(plan_reference(tags[k], u, gen_h.exponential_f32))
        assert gen_h.draws == gen_o.draws
        g_len = g[f"w{w}_evict_len"]
        g_off = np.concatenate([[0], np.cumsum(g_len)])
        assert np.array_equal(np.concatenate([t.ravel() for t in tags]), g[f"w{w}_tags"])
        missed, missed_half = [[] for _ in ln], [[] for _ in ln]   # ids the oracle's forward misses (first half)
        for b in range(L):
            batch = win[:, b * B:(b + 1) * B]
            _ly, slots, _nm = O.forward(oc, [np.arange(B)] * len(ln), batch, master)
            for k in range(len(ln)):
                miss = slots[k] >= oc.cache_sizes[k] * ways
                missed[k].append(batch[k][miss])
                missed_half[k].append(batch[k][:B // 2][miss[:B // 2]])
        for k, (n, e) in enumerate(zip(ln, refs)):
            assert np.array_equal(e["tags"], oc.tags[k])
            gi = g[f"w{w}_evict_ids"][g_off[k]:g_off[k + 1]]
            assert np.array_equal(e["evict_ids"], ev[k][0]) and np.array_equal(e["evict_ids"], gi)
            assert np.array_equal(ev[k][1], w0[k][e["evict_slots"]])
            assert np.array_equal(oc.weight[k][e["fill_slots"]], m0[k][e["fill_ids"]])
            assert len(np.unique(e["fill_slots"])) == e["F"] and np.isin(e["evict_slots"], e["fill_slots"]).all()
            contested += e["rows"] - e["F"]
            pi, ps, pp = primary_evictions(e)    # each evicted id once, by the claimant that took its slot
            assert np.array_equal(np.sort(pi), np.unique(gi)) and pp.all() and len(np.unique(ps)) == len(ps)
            assert np.array_equal(e["losers"], np.unique(np.concatenate(missed[k])))
            own = own_mask(win[k], n, L, B // 2)
            assert np.array_equal(e["losers"][own[e["losers"]]], np.unique(np.concatenate(missed_half[k])))
    assert contested > 50, "the undersized cache was meant to produce contested claims"
