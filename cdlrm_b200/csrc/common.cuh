// common.cuh -- shared declarations of libcdlrm_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/cdlrm_b200.h"

#define CDLRM_OK 0
#define CDLRM_ERR_ARG -1
#define CDLRM_ERR_CUDA -2
#define CDLRM_ERR_STATE -3

void cdlrm_set_error(const char* fmt, ...);

#define CU_CHECK(call)                                                                    \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            cdlrm_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return CDLRM_ERR_CUDA;                                                        \
        }                                                                                 \
    } while (0)

#define ARG_CHECK(cond)                                                                   \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            cdlrm_set_error("%s:%d bad argument: %s", __FILE__, __LINE__, #cond);         \
            return CDLRM_ERR_ARG;                                                         \
        }                                                                                 \
    } while (0)

// One per table; lives in device memory (ctx->d_tabs) and on the host (ctx->tabs).
struct TableDesc {
    float* weight;        // [cache_rows, dim]
    int64_t* tags;        // live tags [num_sets, ways]
    int64_t* plan_tags;   // planner's look-ahead copy (may alias tags)
    const float* master;  // device-visible master table [n_rows, dim]
    uint32_t* dirty;      // bitmap over cache_rows (may be null)
    int64_t num_sets;
    int64_t n_rows;
    int64_t cache_rows;
    int64_t dirty_word_off;  // offset of this table's bitmap in the concatenated bitmap
};

// Planner workspace carve-up (device pointers into the caller's buffer).
struct PlanTable {
    uint32_t* bitmap;   // n_rows bits
    uint32_t* own;      // n_rows bits: ids of THIS rank's own batches (cdlrm_plan_mark_own_ids), kept clean between windows
    int64_t* uniq;      // [umax]
    int32_t* surv;      // [umax] survivor r -> index into uniq
    uint8_t* state;     // [umax] per-unique state: hit way, 255 = miss (not cached), 254 = miss that won a slot
    int64_t umax;
};

// Loser store of one table: the window's ids that are NOT cached after the install (lost a
// contested slot, or dropped because their set was fully pinned), ascending, with a copy of
// their master rows staged in HBM; the forward serves these misses from HBM instead of PCIe.
// Sharded over the ranks of a node (shard > 0): index i of the list lives on rank i / shard, at row i % shard of
// that rank's shard (peer[r]: device address of rank r's shard of this table, readable over NVLink; peer[own
// rank] is local HBM).
struct LoserDesc {
    const int64_t* ids;
    const float* rows;
    int64_t n;
    int64_t shard;                       // 0: the whole store is local (rows)
    const float* peer[CDLRM_MAX_PEERS];
    // bucket index over the ascending ids (built by the bind call): bucket[b] = first index whose id >= b << shift, so the
    // forward's search for an id starts inside [bucket[id >> shift], bucket[(id >> shift) + 1]) -- a handful of entries
    // in one or two cache lines instead of log2(n) dependent DRAM round trips.  NULL: search the whole list.
    const int32_t* bucket;
    int32_t shift;
    int32_t nb;
};

struct cdlrm_ctx {
    int device = 0;
    int num_sms = 148;
    int T = 0, dim = 0, ways = 0;
    int64_t aux = 0;
    int64_t max_cache_size = 0;  // after find_next_prime
    std::vector<TableDesc> tabs;
    TableDesc* d_tabs = nullptr;
    bool tabs_dirty = true;
    // forward/backward scratch
    uint32_t* d_missmap = nullptr;  // [T][ceil(max_idx/32)] forward miss bitmap
    int64_t scratch_max_idx = 0;
    uint32_t* d_flags = nullptr;    // sticky error flags
    LoserDesc* d_losers = nullptr;  // [T] (device), updated in stream order by cdlrm_ctx_bind_losers
    LoserDesc* h_losers = nullptr;  // [2][T] pinned staging for the async update
    int32_t* d_lbucket = nullptr;   // bucket indices of the bound loser store (all tables, grow-only)
    int64_t lbucket_cap = 0;
    int losers_flip = 0;
    // planner
    std::vector<PlanTable> ptabs;
    PlanTable* d_ptabs = nullptr;
    int64_t plan_window_len = 0;
    bool primary_evictions = false;      // eviction lists hold only the winner of every replaced (set, way)
    bool own_marked = false;             // own-id bitmaps hold a window: cdlrm_plan_losers keeps this rank's own ids only
    char* plan_ws = nullptr;             // base of the bound planner workspace (peer copies share its carve-up)
    std::vector<unsigned long long*> pins;  // per table [num_sets] pin masks of the window being planned
    int32_t* p_blocksum2 = nullptr; // second tile-sum array
    int32_t* p_blocksum = nullptr;  // [nblk_max + 1]
    int32_t* p_claim = nullptr;     // [cache_rows_max], kept at -1 between uses
    int32_t* p_slot = nullptr;      // [umax_max] slot chosen per survivor
    int64_t* p_old = nullptr;       // [umax_max] old tag per survivor
    uint8_t* p_flag = nullptr;      // [umax_max] bit0 evict, bit1 winner
    int64_t* p_counts = nullptr;    // device counters [T*8]
    std::vector<int64_t> last_uniq; // U_k of the last phase A (host, after sync by caller)
    int64_t umax_max = 0, sets_max = 0, rows_max = 0;
};

int cdlrm_sync_tabs(cdlrm_ctx* ctx, cudaStream_t s);

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute: opt `func` in for `bytes` on the current
// device once per (function, device), thread-safe.  Returns cudaSuccess or the error of the attribute call.
cudaError_t cdlrm_smem_optin(const void* func, int bytes);

// ---- launch accounting / optional per-kernel event timing (see cdlrm_prof_* in the header) ----
enum KernelId {
    K_PROBE = 0, K_GATHER, K_POOL, K_BWD_PLAN, K_BWD_SGD, K_BWD_SGD_MULTI, K_INT_FWD, K_INT_BWD,
    K_PLAN_BITMAP_SET, K_PLAN_COMPACT, K_PLAN_PROBE, K_PLAN_SURV, K_PLAN_SELECT, K_PLAN_LISTS,
    K_MOVE_EVICT, K_MOVE_GATHER, K_MOVE_FILL, K_MOVE_SCATTER, K_AGG_MARK, K_AGG_OR, K_AGG_COLLECT,
    K_AGG_PACK, K_AGG_UNPACK, K_MISC, K_RNG_MT, K_RNG_EXP, K_MLP_GEMM, K_MLP_SPLIT, K_EMBED_EVAL, K_EVAL, K_LR, K_NULL,
    K_EMBED_VICTIM, K_MOVE_CARRY, K_COUNT
};
void cdlrm_prof_mark(int id, cudaStream_t s, int end);
// wraps one kernel launch statement
#define LAUNCH(id, stream, ...)              \
    do {                                     \
        cdlrm_prof_mark((id), (stream), 0);  \
        __VA_ARGS__;                         \
        cdlrm_prof_mark((id), (stream), 1);  \
    } while (0)

static inline int ceil_div_i(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------
// The per-step kernels are short (3-60 us) and run as one dependent chain, so the launch latency
// between two of them is a visible share of the step.  Every kernel launched through LAUNCH_PDL
// calls pdl_enter() first: it releases its dependents (they may be scheduled while this grid is still
// running -- they block in their own griddepcontrol.wait until this grid has completed and its
// writes are visible) and then waits for its own prerequisite grid.  A kernel launched WITH the
// attribute but WITHOUT pdl_enter() would race with its predecessor: only use LAUNCH_PDL with kernels
// that call it.  cdlrm_set_pdl(0) / CDLRM_PDL=0 switches the attribute off (plain stream order).
extern int g_cdlrm_pdl;

__device__ __forceinline__ void pdl_enter() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

template <typename... KArgs, typename... Args>
inline void cdlrm_launch_pdl_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                                     int cluster_x, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (g_cdlrm_pdl) {
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    if (cluster_x > 1) {     // thread-block cluster along x (grid.x must be a multiple of it)
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = (unsigned)cluster_x;
        attr[na].val.clusterDim.y = 1;
        attr[na].val.clusterDim.z = 1;
        ++na;
    }
    cfg.attrs = attr;
    cfg.numAttrs = na;
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

template <typename... KArgs, typename... Args>
inline void cdlrm_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cdlrm_launch_pdl_cluster(kernel, grid, block, smem, s, 1, static_cast<Args&&>(args)...);
}

// kern may be a parenthesised template-id: LAUNCH_PDL(id, s, (k<A, B>), grid, block, smem, args...)
#define LAUNCH_PDL(id, stream, kern, grid, block, smem, ...)                           \
    do {                                                                               \
        cdlrm_prof_mark((id), (stream), 0);                                            \
        cdlrm_launch_pdl(kern, dim3(grid), dim3(block), (smem), (stream), __VA_ARGS__); \
        cdlrm_prof_mark((id), (stream), 1);                                            \
    } while (0)

// Index of `id` in the ascending ids of a loser store (bucket index, then binary search), or -1 when the store does
// not hold it.
__device__ __forceinline__ int64_t loser_index(const LoserDesc* __restrict__ L, int64_t id) {
    const int64_t n = L->n;
    int64_t lo = 0, hi = n;                // first index with ids[idx] >= id
    if (L->bucket) {                       // bucket index: the answer lies in [bucket[b], bucket[b + 1]]
        const int64_t bk = id >> L->shift;
        lo = __ldg(L->bucket + bk);
        hi = __ldg(L->bucket + bk + 1);
    }
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(L->ids + mid) < id) lo = mid + 1; else hi = mid;
    }
    return (lo < n && __ldg(L->ids + lo) == id) ? lo : -1;
}

// Row `idx` of a loser store: local HBM, or (sharded store) the HBM of rank idx / shard over NVLink.
__device__ __forceinline__ const float* loser_row(const LoserDesc* __restrict__ L, int64_t idx, int dim) {
    if (L->shard) {
        const int64_t owner = idx / L->shard;
        return L->peer[owner] + (idx - owner * L->shard) * dim;
    }
    return L->rows + idx * dim;
}

__device__ __forceinline__ int64_t set_index(int64_t id, int64_t S) {
    // torch.remainder semantics (non-negative result for S > 0)
    if ((uint64_t)id < 0x100000000ull && (uint64_t)S < 0x100000000ull)
        return (int64_t)((uint32_t)id % (uint32_t)S);
    int64_t r = id % S;
    return r < 0 ? r + S : r;
}
