// embed.cu -- per-step cache path: probe + slot + gather + sum-pool forward
// (Embedding_Table_Cache_Group.forward, model_no_ddp.py:149-212) and the
// de-duplicated sparse-SGD backward (EmbeddingBag backward + optimizer_embeds.step(),
// main_no_ddp.py:376,409,413).  All tables of a call are covered by one launch per
// stage (grid.y = table).  HBM-bound integer/row-copy work: no tensor cores.
#include <stdlib.h>

#include "common.cuh"

namespace {


template <int VEC> struct VecT;
template <> struct VecT<4> { using type = float4; };
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<1> { using type = float; };

__device__ __forceinline__ float4 vadd(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float2 vadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float vadd(float a, float b) { return a + b; }
__device__ __forceinline__ float4 vfma(float s, float4 a, float4 b) { return make_float4(fmaf(s, a.x, b.x), fmaf(s, a.y, b.y), fmaf(s, a.z, b.z), fmaf(s, a.w, b.w)); }
__device__ __forceinline__ float2 vfma(float s, float2 a, float2 b) { return make_float2(fmaf(s, a.x, b.x), fmaf(s, a.y, b.y)); }
__device__ __forceinline__ float vfma(float s, float a, float b) { return fmaf(s, a, b); }
__device__ __forceinline__ float4 vscale(float s, float4 a) { return make_float4(s * a.x, s * a.y, s * a.z, s * a.w); }
__device__ __forceinline__ float2 vscale(float s, float2 a) { return make_float2(s * a.x, s * a.y); }
__device__ __forceinline__ float vscale(float s, float a) { return s * a; }
__device__ __forceinline__ void vzero(float4& a) { a = make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ void vzero(float2& a) { a = make_float2(0.f, 0.f); }
__device__ __forceinline__ void vzero(float& a) { a = 0.f; }

__device__ __forceinline__ void red_add(float4* p, float4 v) {
    // sm_90+ vectorised reduction: one 16-byte red per lane
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void red_add(float2* p, float2 v) {
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void red_add(float* p, float v) { atomicAdd(p, v); }

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------------------
// K1: fused probe + slot + row copy (model_no_ddp.py:166-174,200-202).
// A warp owns 32 consecutive ids of one table (= one word of the miss bitmap).
//   phase 1  lane l loads id l (one coalesced 256-byte load), set = id mod num_sets;
//   phase 2  lane l reads the whole tag line of its set (8*ways bytes: one 128-byte
//            line at 16 ways, as 16-byte loads that are all in flight together) and
//            compares in registers -> way, slot = num_sets*way + set;
//   phase 3  COPY (one id per bag, Criteo): the 32 cache rows of the warp are moved to
//            out[] by groups of G lanes, U rows (U*512 B at dim 128) in flight per
//            group; row descriptors travel by shuffle.
// Misses only set their bit in the miss bitmap (one plain store per warp, the bitmap
// is rewritten completely by every launch): the batch-order ordinal they need
// (model_no_ddp.py:177) is resolved by K2.
// ------------------------------------------------------------------------------
constexpr int FWD_NT = 128;

template <int WAYS>
__device__ __forceinline__ int probe_line(const int64_t* __restrict__ tags, int64_t s, int64_t id, int ways) {
    int way = -1;
    if constexpr (WAYS >= 2) {
        const longlong2* line = reinterpret_cast<const longlong2*>(tags + s * WAYS);
        longlong2 v[WAYS / 2];
#pragma unroll
        for (int i = 0; i < WAYS / 2; ++i) v[i] = __ldg(line + i);
#pragma unroll
        for (int i = WAYS / 2 - 1; i >= 0; --i) {   // descending: the lowest matching way wins
            if (v[i].y == id) way = 2 * i + 1;
            if (v[i].x == id) way = 2 * i;
        }
    } else {
        const int64_t* line = tags + s * ways;
        for (int w = ways - 1; w >= 0; --w)
            if (__ldg(line + w) == id) way = w;
    }
    return way;
}

// Tag probe of one id: its cache slot num_sets * way + set, or -1 when it is not cached.  An id outside its table
// raises the sticky flag 2 (IndexError in the reference, master.weight[missing], :176) and matches nothing.
template <int WAYS>
__device__ __forceinline__ int64_t probe_slot(const TableDesc& T, int64_t id, int ways, uint32_t* __restrict__ flags) {
    if ((uint64_t)id >= (uint64_t)T.n_rows) {
        atomicOr(flags, 2u);
        return -1;
    }
    const int64_t s = set_index(id, T.num_sets);
    const int way = probe_line<WAYS>(T.tags, s, id, ways);
    return way < 0 ? -1 : T.num_sets * way + s;
}

// Source row of an un-cached id: its copy in the loser store of the installed window (ascending ids: bucket index,
// then binary search; L may be null), else the master row (zero-copy PCIe).
__device__ __forceinline__ const float* miss_row(const LoserDesc* __restrict__ L, const float* __restrict__ master,
                                                 int64_t id, int dim) {
    if (L) {
        const int64_t idx = loser_index(L, id);
        if (idx >= 0) return loser_row(L, idx, dim);
    }
    return master + id * dim;
}

template <int WAYS, int G, bool COPY>
__global__ void __launch_bounds__(FWD_NT) fwd_fused_kernel(const TableDesc* __restrict__ tabs, int tb,
                                                            const int64_t* __restrict__ ids, int64_t ld_ids, int n_idx,
                                                            int32_t* __restrict__ slots, int64_t ld_slots,
                                                            uint32_t* __restrict__ missmap, int words,
                                                            float* __restrict__ out, int64_t ld_out, int dim, int ways,
                                                            uint32_t* __restrict__ flags) {
    pdl_enter();
    const int t = blockIdx.y;
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * (FWD_NT / 32) + (threadIdx.x >> 5);
    if (w >= words) return;
    const TableDesc& T = tabs[tb + t];
    const int j0 = w * 32, j = j0 + lane;
    const bool valid = j < n_idx;
    const int64_t id = valid ? __ldg(ids + (int64_t)t * ld_ids + j) : 0;
    // an id outside its table is a miss: K2 gives the position a zero row and slot -1
    const int64_t sl = probe_slot<WAYS>(T, id, ways, flags);
    const bool miss = valid && sl < 0;
    const int32_t slot = valid ? (int32_t)sl : -1;
    if (valid) slots[(int64_t)t * ld_slots + j] = slot;
    const uint32_t mm = __ballot_sync(0xffffffffu, miss);
    if (lane == 0) missmap[(int64_t)t * words + w] = mm;
    if constexpr (COPY) {
        constexpr int NGW = 32 / G;               // rows moved per warp instruction
        constexpr int ITERS = G;                  // 32 rows / NGW
        constexpr int U = ITERS < 8 ? ITERS : 8;  // row batches in flight
        const float* __restrict__ weight = T.weight;
        float* tout = out + (int64_t)t * ld_out + (int64_t)j0 * dim;
        const int cpr = dim >> 2;
        const int gl = lane % G, g = lane / G;
#pragma unroll 1
        for (int it0 = 0; it0 < ITERS; it0 += U) {
            float4 v[U];
            int32_t sl[U];
#pragma unroll
            for (int u = 0; u < U; ++u) sl[u] = __shfl_sync(0xffffffffu, slot, (it0 + u) * NGW + g);
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (sl[u] >= 0 && gl < cpr) v[u] = reinterpret_cast<const float4*>(weight + (int64_t)sl[u] * dim)[gl];
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (sl[u] >= 0 && gl < cpr)
                    reinterpret_cast<float4*>(tout + (int64_t)((it0 + u) * NGW + g) * dim)[gl] = v[u];
        }
    }
}

// ------------------------------------------------------------------------------
// K2: resolve the misses (model_no_ddp.py:176-179).  Miss i (batch order = rank of its
// bit in the table's miss bitmap) takes aux slot num_sets*ways + i, reads the master row
// (zero-copy from pinned host memory), parks it in the aux row and, when every bag
// holds one id, also writes out[j].  CTA c of table t owns a contiguous range of bitmap
// words; the ordinal base of the range is the popcount of everything before it.  With
// no misses (the common case) every CTA leaves after reading the bitmap.
// ------------------------------------------------------------------------------
constexpr int MISS_NT = 256;

template <int VEC, bool COPY>
__global__ void __launch_bounds__(MISS_NT) fwd_miss_kernel(const TableDesc* __restrict__ tabs, int tb,
                                                            const int64_t* __restrict__ ids, int64_t ld_ids, int n_idx,
                                                            int32_t* __restrict__ slots, int64_t ld_slots,
                                                            const uint32_t* __restrict__ missmap, int words, int wpc,
                                                            const LoserDesc* __restrict__ losers,
                                                            float* __restrict__ out, int64_t ld_out,
                                                            int32_t* __restrict__ n_miss, uint32_t* __restrict__ flags,
                                                            int dim, int ways, int64_t aux_rows) {
    pdl_enter();
    using V = typename VecT<VEC>::type;
    constexpr int NW = MISS_NT / 32;
    __shared__ int s_red[2][NW];
    const int t = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t* mm = missmap + (int64_t)t * words;
    const int w_lo = blockIdx.x * wpc, w_hi = min(words, w_lo + wpc);
    // popcount of the words before the range (ordinal base) and inside it
    int before = 0, inside = 0;
    for (int w = threadIdx.x; w < w_hi; w += MISS_NT) {
        const int c = __popc(mm[w]);
        if (w < w_lo) before += c; else inside += c;
    }
    before = warp_sum(before);
    inside = warp_sum(inside);
    if (lane == 0) { s_red[0][warp] = before; s_red[1][warp] = inside; }
    __syncthreads();
    before = inside = 0;
#pragma unroll
    for (int i = 0; i < NW; ++i) { before += s_red[0][i]; inside += s_red[1][i]; }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) n_miss[t] = before + inside;
    if (inside == 0) return;
    const TableDesc& T = tabs[tb + t];
    float* __restrict__ weight = T.weight;
    const float* __restrict__ master = T.master;
    const int64_t aux_base = T.num_sets * ways;
    const int cpr = dim / VEC;
    // loser store of the installed window: ascending ids + their master rows staged in HBM
    const LoserDesc* __restrict__ l_desc = losers ? losers + tb + t : nullptr;
    // warp `warp` owns words w_lo + warp, w_lo + warp + NW, ... ; its running ordinal starts at the
    // popcount of the range's words that precede each of them, recomputed per word (ranges are short)
    for (int w = w_lo + warp; w < w_hi; w += NW) {
        const uint32_t bits = mm[w];
        if (!bits) continue;
        int ord0 = 0;
        for (int x = w_lo + lane; x < w; x += 32) ord0 += __popc(mm[x]);
        ord0 = warp_sum(ord0) + before;
        const bool mine = (bits >> lane) & 1u;
        const int j = w * 32 + lane;
        const int64_t ord = ord0 + __popc(bits & ((1u << lane) - 1u));
        const float* src_l = nullptr;
        int64_t aux_l = -1;
        if (mine) {
            const int64_t id = __ldg(ids + (int64_t)t * ld_ids + j);
            const bool bad_id = (uint64_t)id >= (uint64_t)T.n_rows;       // flag 2 was raised by K1
            if (ord >= aux_rows || bad_id) {
                // IndexError in the reference.  Here: sticky flag (check_device_flags raises it on the host),
                // the position keeps slot -1 (skipped by the pooling and by the backward) and pools a zero row.
                if (!bad_id) atomicOr(flags, 1u);
                if (COPY) {
                    float* orow = out + (int64_t)t * ld_out + (int64_t)j * dim;
                    for (int c = 0; c < dim; ++c) orow[c] = 0.f;
                }
            } else {
                aux_l = aux_base + ord;
                src_l = miss_row(l_desc, master, id, dim);
                slots[(int64_t)t * ld_slots + j] = (int32_t)aux_l;
            }
        }
        const unsigned long long src_bits = (unsigned long long)src_l;
        uint32_t rem = bits;
        constexpr int U = 4;
        while (rem) {
            int b[U];
            unsigned long long sp[U];
            long long ax[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                b[u] = rem ? __ffs(rem) - 1 : -1;
                if (rem) rem &= rem - 1;
                sp[u] = __shfl_sync(0xffffffffu, src_bits, b[u] < 0 ? 0 : b[u]);
                ax[u] = __shfl_sync(0xffffffffu, (long long)aux_l, b[u] < 0 ? 0 : b[u]);
                if (b[u] < 0) sp[u] = 0;
            }
            for (int c = lane; c < cpr; c += 32) {
                V v[U];
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (sp[u]) v[u] = reinterpret_cast<const V*>(sp[u])[c];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (!sp[u]) continue;
                    reinterpret_cast<V*>(weight + ax[u] * dim)[c] = v[u];
                    if (COPY) reinterpret_cast<V*>(out + (int64_t)t * ld_out + (int64_t)(w * 32 + b[u]) * dim)[c] = v[u];
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------
// Read-only lookup for evaluation (one id per bag): a warp owns 32 consecutive ids of one table; lane l probes id l
// and resolves its source row -- the cache row on a hit, else the loser store of the installed window or the master
// (probe_slot / miss_row, as K1 / K2) -- then groups of G lanes copy the 32 rows to out[], U rows in flight per group.
// Writes out[] only: no slots, aux rows, miss bitmap, miss counts or dirty bits, so any batch size works.  An id
// outside its table raises flag 2 and gets a zero row.
// ------------------------------------------------------------------------------
template <int WAYS, int VEC>
__global__ void __launch_bounds__(FWD_NT) fwd_eval_kernel(const TableDesc* __restrict__ tabs, int tb,
                                                           const int64_t* __restrict__ ids, int64_t ld_ids, int n_idx,
                                                           const LoserDesc* __restrict__ losers,
                                                           float* __restrict__ out, int64_t ld_out, int dim, int ways,
                                                           int G, uint32_t* __restrict__ flags) {
    pdl_enter();
    using V = typename VecT<VEC>::type;
    constexpr int U = 4;
    const int t = blockIdx.y;
    const int lane = threadIdx.x & 31;
    const int j0 = (blockIdx.x * (FWD_NT / 32) + (threadIdx.x >> 5)) * 32;
    if (j0 >= n_idx) return;
    const TableDesc& T = tabs[tb + t];
    const int j = j0 + lane;
    const float* src = nullptr;
    if (j < n_idx) {
        const int64_t id = __ldg(ids + (int64_t)t * ld_ids + j);
        const int64_t sl = probe_slot<WAYS>(T, id, ways, flags);
        if (sl >= 0) src = T.weight + sl * dim;
        else if ((uint64_t)id < (uint64_t)T.n_rows) src = miss_row(losers ? losers + tb + t : nullptr, T.master, id, dim);
    }
    const unsigned long long src_bits = (unsigned long long)src;
    float* tout = out + (int64_t)t * ld_out;
    const int cpr = dim / VEC;
    const int NGW = 32 / G, gl = lane % G, g = lane / G;
    // every group runs the same number of iterations (NGW * U divides 32 or exceeds it): the shuffles stay warp-wide
    for (int r0 = g; r0 < 32; r0 += NGW * U) {
        unsigned long long sp[U];
        int row[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int r = r0 + u * NGW;
            sp[u] = __shfl_sync(0xffffffffu, src_bits, r < 32 ? r : 0);
            row[u] = (r < 32 && j0 + r < n_idx) ? j0 + r : -1;
        }
        for (int c = gl; c < cpr; c += G) {
            V v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                vzero(v[u]);
                if (row[u] >= 0 && sp[u]) v[u] = reinterpret_cast<const V*>(sp[u])[c];
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (row[u] >= 0) reinterpret_cast<V*>(tout + (int64_t)row[u] * dim)[c] = v[u];
        }
    }
}

// ------------------------------------------------------------------------------
// K3: EmbeddingBag(mode="sum") over final slots for general offsets
// (model_no_ddp.py:191,200-202).  One group of G lanes per bag.
// ------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(256) pool_kernel(const TableDesc* __restrict__ tabs, int tb,
                                                   const int32_t* __restrict__ slots, int64_t ld_slots,
                                                   const int64_t* __restrict__ offsets, int64_t ld_off,
                                                   int n_idx, int n_bags, float* __restrict__ out, int64_t ld_out,
                                                   int32_t* __restrict__ bag_ids, int64_t ld_bag, int dim, int G) {
    using V = typename VecT<VEC>::type;
    const int t = blockIdx.y;
    const int gl = threadIdx.x % G, group = threadIdx.x / G, NG = 256 / G;
    const int b = blockIdx.x * NG + group;
    if (b >= n_bags) return;
    const float* __restrict__ weight = tabs[tb + t].weight;
    const int64_t* off = offsets ? offsets + (int64_t)t * ld_off : nullptr;   // null: bag b = id b
    const int32_t* tsl = slots + (int64_t)t * ld_slots;
    int64_t lo = off ? off[b] : b, hi = off ? ((b + 1 < n_bags) ? off[b + 1] : n_idx) : b + 1;
    const int cpr = dim / VEC;
    if (bag_ids && gl == 0)
        for (int64_t j = lo; j < hi; ++j) bag_ids[(int64_t)t * ld_bag + j] = b;
    for (int c = gl; c < cpr; c += G) {
        V acc;
        vzero(acc);
        for (int64_t j = lo; j < hi; ++j)
            if (tsl[j] >= 0) acc = vadd(acc, reinterpret_cast<const V*>(weight + (int64_t)tsl[j] * dim)[c]);
        reinterpret_cast<V*>(out + (int64_t)t * ld_out + (int64_t)b * dim)[c] = acc;
    }
}

// ------------------------------------------------------------------------------
// Backward plan: one 1024-thread CTA per table radix-sorts (slot, position) pairs
// in shared memory (stable LSD, 8-bit digits, ranks from __match_any_sync), then
// cuts the sorted run into chunks of <= CH equal slots.  A chunk that covers its
// whole segment is applied with a plain read-modify-write, the (rare) others with
// vector reds.  This is the "deduplicated indices instead of atomics" step.
// ------------------------------------------------------------------------------
constexpr int PLAN_NT = 1024;
constexpr int PLAN_MAX_ROUNDS = CDLRM_SORT_MAX / 1024;  // 16 keys per thread at most

struct PlanView {
    int32_t* sorted_pos;    // [tc][n_idx] absolute position j, grouped by slot (stable: ascending j within a slot)
    uint32_t* sorted_key;   // [tc][n_idx] the slot of each sorted entry
};

__host__ __device__ inline int plan_nsub(int n_idx) { return (n_idx + CDLRM_SORT_MAX - 1) / CDLRM_SORT_MAX; }

__host__ inline PlanView plan_view(void* plan, int tc, int n_idx) {
    PlanView v;
    char* p = (char*)plan;
    size_t a = (size_t)tc * n_idx * sizeof(int32_t);
    a = (a + 255) & ~(size_t)255;
    v.sorted_pos = (int32_t*)p; p += a;
    v.sorted_key = (uint32_t*)p;
    return v;
}

__device__ __forceinline__ int block_excl_scan_1024(int v, int* s_warp, int& total) {
    // exclusive sum scan over 1024 threads; s_warp: 32 ints of shared scratch
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int n = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += n;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int n = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += n;
        }
        s_warp[lane] = winc - w;  // exclusive warp offsets
        if (lane == 31) s_warp[32] = winc;
    }
    __syncthreads();
    int res = s_warp[warp] + inc - v;
    total = s_warp[32];
    __syncthreads();
    return res;
}

__device__ __forceinline__ int block_excl_maxscan_1024(int v, int* s_warp) {
    // exclusive max scan (identity -1) over 1024 threads
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int n = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc = max(inc, n);
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int n = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc = max(winc, n);
        }
        int wex = __shfl_up_sync(0xffffffffu, winc, 1);
        s_warp[lane] = lane == 0 ? -1 : wex;
    }
    __syncthreads();
    int ex = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) ex = -1;
    int res = max(s_warp[warp], ex);
    __syncthreads();
    return res;
}

__global__ void __launch_bounds__(PLAN_NT, 1) bwd_plan_kernel(const TableDesc* __restrict__ tabs, int tb,
                                                              const int32_t* __restrict__ slots, int64_t ld_slots,
                                                              int n_idx, int j0, int n, PlanView pv) {
    pdl_enter();
    extern __shared__ __align__(16) unsigned char smem[];
    // layout: keyA[n] keyB[n] (u32) | valA[n] valB[n] (u16) | cnt[8192] (u16) | scratch[40] (int)
    const int npad = (n + 7) & ~7;
    uint32_t* keyA = reinterpret_cast<uint32_t*>(smem);
    uint32_t* keyB = keyA + npad;
    uint16_t* valA = reinterpret_cast<uint16_t*>(keyB + npad);
    uint16_t* valB = valA + npad;
    uint16_t* cnt = valB + npad;                       // [256 digits][32 warps]
    int* s_scr = reinterpret_cast<int*>(cnt + 8192);

    const int t = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int32_t* tsl = slots + (int64_t)t * ld_slots + j0;
    const int64_t rows = tabs[tb + t].cache_rows;
    for (int i = tid; i < n; i += PLAN_NT) {
        // unresolved positions (slot -1: aux overflow / id out of range, flagged by the forward) sort behind
        // every real slot under the key `rows`; the apply kernel skips them
        const uint32_t k = (uint32_t)tsl[i];
        keyA[i] = k < (uint32_t)rows ? k : (uint32_t)rows;
        valA[i] = (uint16_t)i;
    }
    const int bits = 64 - __clzll((unsigned long long)(rows > 1 ? rows : 1));   // the key `rows` must be representable
    const int passes = (bits + 7) / 8;
    const int per_warp = (((n + 31) / 32) + 31) & ~31;  // keys per warp, multiple of 32
    const int rounds = per_warp / 32;                   // <= PLAN_MAX_ROUNDS
    const uint32_t lt = (1u << lane) - 1u;
    __syncthreads();

    for (int pass = 0; pass < passes; ++pass) {
        const int shift = pass * 8;
        for (int e = tid; e < 4096; e += PLAN_NT) reinterpret_cast<uint32_t*>(cnt)[e] = 0;
        __syncthreads();
        uint16_t rk[PLAN_MAX_ROUNDS];
#pragma unroll
        for (int r = 0; r < PLAN_MAX_ROUNDS; ++r) {
            if (r < rounds) {
                int i = warp * per_warp + r * 32 + lane;
                bool valid = i < n;
                uint32_t dg = valid ? ((keyA[i] >> shift) & 255u) : 256u;
                uint32_t peers = __match_any_sync(0xffffffffu, dg);
                int leader = __ffs(peers) - 1;
                int old = 0;
                if (valid && lane == leader) {
                    old = cnt[dg * 32 + warp];
                    cnt[dg * 32 + warp] = (uint16_t)(old + __popc(peers));
                }
                old = __shfl_sync(0xffffffffu, old, leader);
                rk[r] = (uint16_t)(old + __popc(peers & lt));
                __syncwarp();
            }
        }
        __syncthreads();
        {   // exclusive scan of cnt in (digit, warp) order: 8 entries per thread
            uint4 raw = reinterpret_cast<uint4*>(cnt)[tid];
            uint16_t c[8];
            c[0] = raw.x & 0xffff; c[1] = raw.x >> 16; c[2] = raw.y & 0xffff; c[3] = raw.y >> 16;
            c[4] = raw.z & 0xffff; c[5] = raw.z >> 16; c[6] = raw.w & 0xffff; c[7] = raw.w >> 16;
            int sum = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) sum += c[q];
            int total;
            int ex = block_excl_scan_1024(sum, s_scr, total);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                int v = c[q];
                c[q] = (uint16_t)ex;
                ex += v;
            }
            raw.x = c[0] | ((uint32_t)c[1] << 16); raw.y = c[2] | ((uint32_t)c[3] << 16);
            raw.z = c[4] | ((uint32_t)c[5] << 16); raw.w = c[6] | ((uint32_t)c[7] << 16);
            reinterpret_cast<uint4*>(cnt)[tid] = raw;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < PLAN_MAX_ROUNDS; ++r) {
            if (r < rounds) {
                int i = warp * per_warp + r * 32 + lane;
                if (i < n) {
                    uint32_t k = keyA[i];
                    uint32_t dg = (k >> shift) & 255u;
                    int dst = cnt[dg * 32 + warp] + rk[r];
                    keyB[dst] = k;
                    valB[dst] = valA[i];
                }
            }
        }
        __syncthreads();
        uint32_t* tk = keyA; keyA = keyB; keyB = tk;
        uint16_t* tv = valA; valA = valB; valB = tv;
    }

    // ---- the sorted run: slot keys and the positions that carry them ----------------
    const int64_t obase = (int64_t)t * n_idx + j0;
    for (int i = tid; i < n; i += PLAN_NT) {
        pv.sorted_key[obase + i] = keyA[i];
        pv.sorted_pos[obase + i] = j0 + (int)valA[i];
    }
}

// ------------------------------------------------------------------------------
// Backward plan, cluster version: the same stable LSD radix sort, but one thread-block CLUSTER of C CTAs per
// table instead of one CTA (26 CTAs on 148 SMs, 32 us, was the slowest stage of the cache path).  CTA c owns
// positions [c*chunk, (c+1)*chunk) of the current order in its shared memory; per 8-bit pass
//   1. ranks of its keys within (digit, warp)   (__match_any_sync, as above);
//   2. per-digit totals published in shared memory;  cluster barrier;
//   3. every CTA reads the C x 256 totals over DSMEM: global digit bases + what the CTAs before it hold;
//   4. keys and positions are scattered to their destination CTA's other buffer with DSMEM stores;  cluster barrier.
// Stable by construction (lane < round < warp < CTA order = position order), so the sorted run is bit-identical
// to bwd_plan_kernel's.  Unresolved positions and the padding carry the key `rows` and sort to the end.
// ------------------------------------------------------------------------------
constexpr int CPL_NT = 512;
constexpr int CPL_NW = CPL_NT / 32;
constexpr int CPL_MAX_ROUNDS = 4;                 // keys per thread: chunk <= 4 * 512 = 2048
constexpr int CPL_MAX_CHUNK = CPL_NT * CPL_MAX_ROUNDS;

__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_nctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same shared-memory variable in CTA `rank` of the cluster (shared::cluster window)
__device__ __forceinline__ uint32_t dsmem_addr(const void* local_smem, uint32_t rank) {
    uint32_t a = (uint32_t)__cvta_generic_to_shared(local_smem), r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    return r;
}
__device__ __forceinline__ uint32_t dsmem_ld_u32(uint32_t addr) {
    uint32_t v; asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v;
}
__device__ __forceinline__ void dsmem_st_u32(uint32_t addr, uint32_t v) { asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void dsmem_st_u16(uint32_t addr, uint16_t v) { asm volatile("st.shared::cluster.u16 [%0], %1;" ::"r"(addr), "h"(v) : "memory"); }

__global__ void __launch_bounds__(CPL_NT, 1) bwd_plan_cluster_kernel(const TableDesc* __restrict__ tabs, int tb,
                                                                     const int32_t* __restrict__ slots, int64_t ld_slots,
                                                                     int n_idx, int j0, int n, int chunk, PlanView pv) {
    pdl_enter();
    extern __shared__ __align__(16) unsigned char smem[];
    // layout: keyA[chunk] keyB[chunk] (u32) | valA[chunk] valB[chunk] (u16) | cnt[256][NW] (u16) | tot[256] base[256] (u32) | scratch
    uint32_t* keyA = reinterpret_cast<uint32_t*>(smem);
    uint32_t* keyB = keyA + chunk;
    uint16_t* valA = reinterpret_cast<uint16_t*>(keyB + chunk);
    uint16_t* valB = valA + chunk;
    uint16_t* cnt = valB + chunk;
    uint32_t* tot = reinterpret_cast<uint32_t*>(cnt + 256 * CPL_NW);
    uint32_t* base = tot + 256;
    int* s_scr = reinterpret_cast<int*>(base + 256);

    const int t = blockIdx.y;
    const uint32_t crank = cluster_ctarank(), C = cluster_nctarank();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int32_t* tsl = slots + (int64_t)t * ld_slots + j0;
    const int64_t rows = tabs[tb + t].cache_rows;
    const int g0 = (int)crank * chunk;
    for (int i = tid; i < chunk; i += CPL_NT) {
        const int gp = g0 + i;
        uint32_t k = (uint32_t)rows;
        if (gp < n) {
            const uint32_t sl = (uint32_t)tsl[gp];
            if (sl < (uint32_t)rows) k = sl;
        }
        keyA[i] = k;
        valA[i] = (uint16_t)gp;
    }
    const int bits = 64 - __clzll((unsigned long long)(rows > 1 ? rows : 1));
    const int passes = (bits + 7) / 8;
    const int per_warp = chunk / CPL_NW;                // multiple of 32 (chunk is a multiple of 512)
    const int rounds = per_warp / 32;                   // <= CPL_MAX_ROUNDS
    const uint32_t lt = (1u << lane) - 1u;
    __syncthreads();

    for (int pass = 0; pass < passes; ++pass) {
        const int shift = pass * 8;
        for (int e = tid; e < 256 * CPL_NW / 2; e += CPL_NT) reinterpret_cast<uint32_t*>(cnt)[e] = 0;
        __syncthreads();
        uint16_t rk[CPL_MAX_ROUNDS];
#pragma unroll
        for (int r = 0; r < CPL_MAX_ROUNDS; ++r) {
            if (r < rounds) {
                const int i = warp * per_warp + r * 32 + lane;
                const uint32_t dg = (keyA[i] >> shift) & 255u;
                const uint32_t peers = __match_any_sync(0xffffffffu, dg);
                const int leader = __ffs(peers) - 1;
                int old = 0;
                if (lane == leader) {
                    old = cnt[dg * CPL_NW + warp];
                    cnt[dg * CPL_NW + warp] = (uint16_t)(old + __popc(peers));
                }
                old = __shfl_sync(0xffffffffu, old, leader);
                rk[r] = (uint16_t)(old + __popc(peers & lt));
                __syncwarp();
            }
        }
        __syncthreads();
        if (tid < 256) {        // digit tid: exclusive prefix over this CTA's warps, total of the CTA
            uint32_t run = 0;
#pragma unroll
            for (int w = 0; w < CPL_NW; ++w) {
                const uint32_t v = cnt[tid * CPL_NW + w];
                cnt[tid * CPL_NW + w] = (uint16_t)run;
                run += v;
            }
            tot[tid] = run;
        }
        cluster_sync_all();     // every CTA's totals are visible cluster-wide
        {
            uint32_t col = 0, mine = 0;
            if (tid < 256) {
                for (uint32_t cc = 0; cc < C; ++cc) {
                    const uint32_t v = cc == crank ? tot[tid] : dsmem_ld_u32(dsmem_addr(tot + tid, cc));
                    if (cc < crank) mine += v;
                    col += v;
                }
            }
            // exclusive scan of the digit totals over the first 256 threads (8 warps)
            uint32_t inc = col;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t nb = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += nb;
            }
            if (tid < 256 && lane == 31) s_scr[warp] = (int)inc;
            __syncthreads();
            if (tid < 256) {
                uint32_t woff = 0;
                for (int w = 0; w < warp; ++w) woff += (uint32_t)s_scr[w];
                base[tid] = woff + inc - col + mine;
            }
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < CPL_MAX_ROUNDS; ++r) {
            if (r < rounds) {
                const int i = warp * per_warp + r * 32 + lane;
                const uint32_t k = keyA[i];
                const uint32_t dg = (k >> shift) & 255u;
                const uint32_t dst = base[dg] + cnt[dg * CPL_NW + warp] + rk[r];
                const uint32_t dc = dst / (uint32_t)chunk, off = dst - dc * (uint32_t)chunk;
                if (dc == crank) {
                    keyB[off] = k;
                    valB[off] = valA[i];
                } else {
                    dsmem_st_u32(dsmem_addr(keyB + off, dc), k);
                    dsmem_st_u16(dsmem_addr(valB + off, dc), valA[i]);
                }
            }
        }
        cluster_sync_all();     // all scatters of the pass have landed; nobody reads tot / writes keyB any more
        uint32_t* tk = keyA; keyA = keyB; keyB = tk;
        uint16_t* tv = valA; valA = valB; valB = tv;
    }

    const int64_t obase = (int64_t)t * n_idx + j0;
    for (int i = tid; i < chunk; i += CPL_NT) {
        const int gp = g0 + i;
        if (gp < n) {
            pv.sorted_key[obase + gp] = keyA[i];
            pv.sorted_pos[obase + gp] = j0 + (int)valA[i];
        }
    }
}

// ------------------------------------------------------------------------------
// Backward apply over the sorted run (slot keys ascending, positions ascending within a
// slot).  A warp owns 32 consecutive sorted entries of one table: one coalesced load
// brings their (slot, position) pairs, everything after that is independent row traffic.
// Groups of G lanes own a row (G = dim/4 rounded up to a power of two; 32 at dim 128), so
// a warp works on NGW = 32/G sub-ranges of EPG = G entries side by side.  A group walks
// its entries in order, CHB at a time: the gradient rows of the batch -- and the weight
// rows of the runs that end inside it -- are all in flight together; then
//     acc += g[pos]   ...   at the end of a run:  weight[slot] = fma(-lr, acc, weight[slot])
// as a plain read-modify-write when the whole run lies inside the group's entries
// (deterministic: ascending position), or a vector red when the run continues in a
// neighbouring sub-range (the hot rows of a skewed stream, the tiny tables: one red per
// 32 rows at dim 128).  No per-table counts, no chunk records, no empty CTAs: the grid is
// ceil(n/32) warps per table.
// ------------------------------------------------------------------------------
constexpr int CHB = 8;          // entries in flight per lane group
constexpr int APPLY_NT = 256;

// the learning rate of an update: a kernel argument, or (DLR) the value a device buffer holds when the kernel runs
// (cdlrm_lr_advance / cdlrm_lr_set write it earlier in stream order; read after griddepcontrol.wait)
template <bool DLR>
__device__ __forceinline__ float load_lr(float lr, const float* d_lr) {
    if constexpr (DLR) return *d_lr;
    else return lr;
}

template <int G, bool DLR>
__global__ void __launch_bounds__(APPLY_NT, 2) bwd_sgd_apply_kernel(const TableDesc* __restrict__ tabs, int tb,
                                                                     PlanView pv, int n_idx, int j0, int n,
                                                                     const int32_t* __restrict__ bag_ids, int64_t ld_bag,
                                                                     const float* __restrict__ d_out, int64_t ld_dout,
                                                                     int64_t row_stride, float lr_arg,
                                                                     const float* __restrict__ d_lr, int dim) {
    pdl_enter();
    const float lr = load_lr<DLR>(lr_arg, d_lr);
    constexpr int NGW = 32 / G;               // lane groups per warp
    constexpr int EPG = G;                    // sorted entries per group (32 / NGW)
    constexpr int NB = EPG < CHB ? EPG : CHB; // entries per batch
    const int t = blockIdx.y;
    const int lane = threadIdx.x & 31;
    const int e0 = (blockIdx.x * (APPLY_NT / 32) + (threadIdx.x >> 5)) * 32;   // first entry of the warp
    if (e0 >= n) return;
    const TableDesc& T = tabs[tb + t];
    float* __restrict__ weight = T.weight;
    const float* gbase = d_out + (int64_t)t * ld_dout;
    const int64_t obase = (int64_t)t * n_idx + j0;
    const uint32_t* keys = pv.sorted_key + obase;
    const uint32_t nkeys = (uint32_t)T.cache_rows;       // keys >= nkeys: unresolved positions, at the end of the run
    const uint32_t key_l = e0 + lane < n ? keys[e0 + lane] : 0xffffffffu;
    const bool valid_l = key_l < nkeys;
    int pos_l = valid_l ? pv.sorted_pos[obase + e0 + lane] : 0;
    if (bag_ids && valid_l) pos_l = bag_ids[(int64_t)t * ld_bag + pos_l];
    // neighbours across the warp's range
    const uint32_t key_before = e0 > 0 ? keys[e0 - 1] : 0xffffffffu;
    const uint32_t key_after = e0 + 32 < n ? keys[e0 + 32] : 0xffffffffu;
    uint32_t kp = __shfl_up_sync(0xffffffffu, key_l, 1);
    uint32_t kn = __shfl_down_sync(0xffffffffu, key_l, 1);
    if (lane == 0) kp = key_before;
    if (lane == 31) kn = key_after;
    // run structure relative to the GROUP's sub-range [g*EPG, (g+1)*EPG)
    const int within = lane % EPG;
    const bool head_true = valid_l && key_l != kp;                    // first entry of its slot
    const bool tail_true = valid_l && key_l != kn;                    // last entry of its slot
    const bool seg_head = valid_l && (head_true || within == 0);      // the group starts accumulating here
    const bool seg_tail = valid_l && (tail_true || within == EPG - 1 || e0 + lane + 1 >= n);
    if (head_true && T.dirty) atomicOr(T.dirty + (key_l >> 5), 1u << (key_l & 31));
    // a segment is the slot's only contribution iff it starts at a true head and ends at a true tail
    const uint32_t head_mask = __ballot_sync(0xffffffffu, seg_head);
    const uint32_t headtrue_mask = __ballot_sync(0xffffffffu, head_true);
    int excl_l = 0;
    if (seg_tail) {
        const uint32_t upto = head_mask & (0xffffffffu >> (31 - lane));   // segment heads at or before this lane
        const int h = 31 - __clz(upto);                                   // this segment's head lane
        excl_l = (tail_true && ((headtrue_mask >> h) & 1u)) ? 1 : 0;
    }
    const int flags_l = (seg_tail ? 1 : 0) | (excl_l << 1);

    const int gl = lane % G, g = lane / G;
    const int cpr = dim >> 2;
    const bool act = gl < cpr;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
    for (int b0 = 0; b0 < EPG; b0 += NB) {
        uint32_t key[NB];
        int pos[NB], fl[NB];
        float4 gv[NB], wv[NB];
#pragma unroll
        for (int q = 0; q < NB; ++q) {
            const int src = g * EPG + b0 + q;
            key[q] = __shfl_sync(0xffffffffu, key_l, src);
            pos[q] = __shfl_sync(0xffffffffu, pos_l, src);
            fl[q] = __shfl_sync(0xffffffffu, flags_l, src);
            if (e0 + src >= n || key[q] >= nkeys) fl[q] = -1;         // past the end of the run / unresolved
        }
#pragma unroll
        for (int q = 0; q < NB; ++q) {
            if (fl[q] >= 0 && act) {
                gv[q] = reinterpret_cast<const float4*>(gbase + (int64_t)pos[q] * row_stride)[gl];
                if (fl[q] == 3) wv[q] = reinterpret_cast<const float4*>(weight + (int64_t)key[q] * dim)[gl];
            }
        }
#pragma unroll
        for (int q = 0; q < NB; ++q) {
            if (fl[q] >= 0 && act) {
                acc = vadd(acc, gv[q]);
                if (fl[q] & 1) {
                    float4* wp = reinterpret_cast<float4*>(weight + (int64_t)key[q] * dim) + gl;
                    if (fl[q] == 3) *wp = vfma(-lr, acc, wv[q]);
                    else red_add(wp, vscale(-lr, acc));
                    acc = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        }
    }
}

// generic fallback (any dim / alignment): one lane group per sorted entry, always atomic
template <int VEC, bool DLR>
__global__ void __launch_bounds__(256) bwd_sgd_kernel(const TableDesc* __restrict__ tabs, int tb,
                                                      PlanView pv, int n_idx, int j0, int n,
                                                      const int32_t* __restrict__ bag_ids, int64_t ld_bag,
                                                      const float* __restrict__ d_out, int64_t ld_dout,
                                                      int64_t row_stride, float lr_arg, const float* __restrict__ d_lr,
                                                      int dim, int G) {
    using V = typename VecT<VEC>::type;
    const float lr = load_lr<DLR>(lr_arg, d_lr);
    const int t = blockIdx.y;
    const int gl = threadIdx.x % G, group = threadIdx.x / G, NG = 256 / G;
    const int e = blockIdx.x * NG + group;
    if (e >= n) return;
    const int64_t obase = (int64_t)t * n_idx + j0;
    const uint32_t slot = pv.sorted_key[obase + e];
    int p0 = pv.sorted_pos[obase + e];
    if (bag_ids) p0 = bag_ids[(int64_t)t * ld_bag + p0];
    const TableDesc& T = tabs[tb + t];
    if (slot >= (uint32_t)T.cache_rows) return;          // unresolved position (see bwd_plan_kernel)
    const float* g = d_out + (int64_t)t * ld_dout + (int64_t)p0 * row_stride;
    float* wrow = T.weight + (int64_t)slot * dim;
    const int cpr = dim / VEC;
    for (int cc = gl; cc < cpr; cc += G)
        red_add(reinterpret_cast<V*>(wrow) + cc, vscale(-lr, reinterpret_cast<const V*>(g)[cc]));
    if (gl == 0 && T.dirty) atomicOr(T.dirty + (slot >> 5), 1u << (slot & 31));
}

// ------------------------------------------------------------------------------
// Update of the misses (--evict-victim-cache): a miss of the step is a position whose slot is an aux slot; its row
// came from the loser store of the installed window, and its sparse update goes into that store row, not only into
// the aux row the next forward overwrites.  Per table and store row: the gradient rows of every position that
// missed on it, summed in ascending position, then ONE weight = fma(-lr, sum, weight) -- what bwd_sgd_apply_kernel
// does for a cached slot.  Duplicate misses of an id sit in separate aux slots and are summed once.
// CTA c of a table owns the ids whose hash is c (mod gridDim.x), so every store row has one owner CTA: it keeps its
// misses as keys (store index << 32 | position) in shared memory, sorts them (bitonic: the keys are distinct), and
// its warps walk the runs of equal store index, one float4 column per lane, U runs in flight.
// A miss whose id is not in the store raises flag 4 (cdlrm_ctx_check) and is not applied.
// ------------------------------------------------------------------------------
constexpr int VICTIM_NT = 512;

template <int VEC, bool DLR>
__global__ void __launch_bounds__(VICTIM_NT) victim_update_kernel(const TableDesc* __restrict__ tabs, int tb,
                                                                  const LoserDesc* __restrict__ losers,
                                                                  const int32_t* __restrict__ slots, int64_t ld_slots,
                                                                  const int64_t* __restrict__ ids, int64_t ld_ids,
                                                                  int n_idx, const int32_t* __restrict__ bag_ids,
                                                                  int64_t ld_bag, const float* __restrict__ d_out,
                                                                  int64_t ld_dout, int64_t row_stride, float lr_arg,
                                                                  const float* __restrict__ d_lr, int dim, int ways,
                                                                  int cap, uint32_t* __restrict__ flags) {
    pdl_enter();
    using V = typename VecT<VEC>::type;
    extern __shared__ __align__(16) unsigned long long s_key[];
    __shared__ int s_n;
    const int t = blockIdx.y, C = gridDim.x;
    const TableDesc& T = tabs[tb + t];
    const LoserDesc* __restrict__ L = losers ? losers + tb + t : nullptr;
    const int64_t aux_base = T.num_sets * ways;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    const int32_t* tsl = slots + (int64_t)t * ld_slots;
    const int64_t* tid = ids + (int64_t)t * ld_ids;
    for (int j = threadIdx.x; j < n_idx; j += VICTIM_NT) {
        const int64_t sl = tsl[j];
        if (sl < aux_base || sl >= T.cache_rows) continue;       // cached, or unresolved (slot -1, flagged by the forward)
        const int64_t id = tid[j];
        if ((int)((((uint64_t)id * 0x9E3779B97F4A7C15ull) >> 32) % (uint64_t)C) != (int)blockIdx.x) continue;
        const int64_t li = (L && !L->shard) ? loser_index(L, id) : -1;
        if (li < 0) {
            atomicOr(flags, 4u);
            continue;
        }
        const int e = atomicAdd(&s_n, 1);
        if (e < cap) s_key[e] = ((unsigned long long)li << 32) | (uint32_t)j;
    }
    __syncthreads();
    const int n = min(s_n, cap);
    if (n == 0) return;
    int kp = 1;
    while (kp < n) kp <<= 1;
    for (int i = n + threadIdx.x; i < kp; i += VICTIM_NT) s_key[i] = ~0ull;
    __syncthreads();
    for (int size = 2; size <= kp; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = threadIdx.x; i < (kp >> 1); i += VICTIM_NT) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const unsigned long long a = s_key[lo], b = s_key[hi];
                if ((a > b) == ((lo & size) == 0)) { s_key[lo] = b; s_key[hi] = a; }
            }
            __syncthreads();
        }
    }
    const float lr = load_lr<DLR>(lr_arg, d_lr);
    float* __restrict__ rows = const_cast<float*>(L->rows);
    const float* __restrict__ gbase = d_out + (int64_t)t * ld_dout;
    const int32_t* __restrict__ tbag = bag_ids ? bag_ids + (int64_t)t * ld_bag : nullptr;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int cpr = dim / VEC;
    constexpr int U = 4;
    for (int base = warp * 32; base < n; base += VICTIM_NT) {
        const int e = base + lane;
        const unsigned long long k = e < n ? s_key[e] : ~0ull;
        const unsigned long long kprev = (e > 0 && e < n) ? s_key[e - 1] : ~0ull;
        uint32_t heads = __ballot_sync(0xffffffffu, e < n && (k >> 32) != (kprev >> 32));
        while (heads) {
            int h[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                h[u] = heads ? base + __ffs(heads) - 1 : -1;
                if (heads) heads &= heads - 1;
            }
            for (int c = lane; c < cpr; c += 32) {
                V acc[U], wv[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (h[u] < 0) continue;
                    const unsigned long long kh = s_key[h[u]];
                    const int p = tbag ? tbag[(uint32_t)kh] : (int)(uint32_t)kh;
                    vzero(acc[u]);
                    acc[u] = vadd(acc[u], reinterpret_cast<const V*>(gbase + (int64_t)p * row_stride)[c]);
                    wv[u] = reinterpret_cast<const V*>(rows + (int64_t)(kh >> 32) * dim)[c];
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (h[u] < 0) continue;
                    const unsigned long long li = s_key[h[u]] >> 32;
                    for (int x = h[u] + 1; x < n; ++x) {
                        const unsigned long long kx = s_key[x];
                        if ((kx >> 32) != li) break;
                        const int p = tbag ? tbag[(uint32_t)kx] : (int)(uint32_t)kx;
                        acc[u] = vadd(acc[u], reinterpret_cast<const V*>(gbase + (int64_t)p * row_stride)[c]);
                    }
                    reinterpret_cast<V*>(rows + (int64_t)li * dim)[c] = vfma(-lr, acc[u], wv[u]);
                }
            }
        }
    }
}

inline int pow2_ceil(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

inline int pick_vec(int dim, const void* a, const void* b, int64_t s1, int64_t s2) {
    auto al = [](const void* p, int n) { return p == nullptr || ((uintptr_t)p % n) == 0; };
    if (dim % 4 == 0 && al(a, 16) && al(b, 16) && s1 % 4 == 0 && s2 % 4 == 0) return 4;
    if (dim % 2 == 0 && al(a, 8) && al(b, 8) && s1 % 2 == 0 && s2 % 2 == 0) return 2;
    return 1;
}

}  // namespace

static int g_plan_cluster = -1;

extern "C" int cdlrm_embed_set_option(int key, int value) {
    if (key == 0) { g_plan_cluster = value; return CDLRM_OK; }
    cdlrm_set_error("cdlrm_embed_set_option: unknown key %d", key);
    return CDLRM_ERR_ARG;
}

static int ensure_scratch(cdlrm_ctx* c, int64_t n_idx) {
    if (n_idx <= c->scratch_max_idx && c->d_missmap) return CDLRM_OK;
    return cdlrm_ctx_reserve(c, n_idx > 8192 ? n_idx : 8192);
}

extern "C" int cdlrm_embed_fwd(cdlrm_ctx* c, int tb, int tc, const int64_t* ids, int64_t ld_ids,
                               const int64_t* offsets, int64_t ld_off, int32_t n_idx, int32_t n_bags,
                               float* out, int64_t ld_out, int32_t* slots, int64_t ld_slots, int32_t* n_miss,
                               int32_t* bag_ids, int64_t ld_bag, cdlrm_stream stream) {
    ARG_CHECK(c && ids && out && slots && n_miss);
    ARG_CHECK(tb >= 0 && tc > 0 && tb + tc <= c->T);
    ARG_CHECK(n_idx >= 0 && n_bags >= 0);
    ARG_CHECK(offsets != nullptr || n_idx == n_bags);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    for (int k = tb; k < tb + tc; ++k) {
        if (!c->tabs[k].weight || !c->tabs[k].tags || !c->tabs[k].master) {
            cdlrm_set_error("table %d: cache or master not bound", k);
            return CDLRM_ERR_STATE;
        }
    }
    int rc = cdlrm_sync_tabs(c, s);
    if (rc) return rc;
    if (n_idx == 0) {
        CU_CHECK(cudaMemsetAsync(n_miss, 0, sizeof(int32_t) * tc, s));
        if (n_bags > 0)
            for (int t = 0; t < tc; ++t)
                CU_CHECK(cudaMemsetAsync(out + (int64_t)t * ld_out, 0, sizeof(float) * (int64_t)n_bags * c->dim, s));
        return CDLRM_OK;
    }
    rc = ensure_scratch(c, n_idx);
    if (rc) return rc;
    const bool p1 = offsets == nullptr;
    bool al16 = true, al8 = true, tags16 = true;
    for (int k = tb; k < tb + tc; ++k) {
        al16 = al16 && ((uintptr_t)c->tabs[k].master % 16 == 0);
        al8 = al8 && ((uintptr_t)c->tabs[k].master % 8 == 0);
        tags16 = tags16 && ((uintptr_t)c->tabs[k].tags % 16 == 0);
    }
    int vec = pick_vec(c->dim, out, nullptr, ld_out, c->dim);
    if (vec == 4 && !al16) vec = 2;
    if (vec == 2 && !al8) vec = 1;
    const int cpr = c->dim / vec;
    const int G = pow2_ceil(cpr) > 32 ? 32 : pow2_ceil(cpr);
    // K1 copies the hit rows itself when every bag holds one id and rows are <= 32 float4 wide;
    // otherwise it only probes and K3 (pool) produces the output rows from the final slots.
    const bool copy = p1 && vec == 4 && cpr <= 32;
    const int words = (n_idx + 31) / 32;
    dim3 grid((words + FWD_NT / 32 - 1) / (FWD_NT / 32), tc);
    const int wsel = !tags16 ? 0 : (c->ways == 16 ? 16 : c->ways == 8 ? 8 : c->ways == 4 ? 4 : c->ways == 2 ? 2 : 0);
#define LAUNCH_FUSED(WW, GG, CP) LAUNCH_PDL(K_PROBE, s, (fwd_fused_kernel<WW, GG, CP>), grid, FWD_NT, 0, c->d_tabs, tb, ids, ld_ids, n_idx, slots, ld_slots, c->d_missmap, words, out, ld_out, c->dim, c->ways, c->d_flags)
#define FUSED_G(WW)                                             \
    if (!copy) { LAUNCH_FUSED(WW, 32, false); }                 \
    else switch (G) {                                           \
        case 1: LAUNCH_FUSED(WW, 1, true); break;               \
        case 2: LAUNCH_FUSED(WW, 2, true); break;               \
        case 4: LAUNCH_FUSED(WW, 4, true); break;               \
        case 8: LAUNCH_FUSED(WW, 8, true); break;               \
        case 16: LAUNCH_FUSED(WW, 16, true); break;             \
        default: LAUNCH_FUSED(WW, 32, true); break;             \
    }
    switch (wsel) {
        case 16: FUSED_G(16) break;
        case 8: FUSED_G(8) break;
        case 4: FUSED_G(4) break;
        case 2: FUSED_G(2) break;
        default: FUSED_G(0) break;
    }
#undef FUSED_G
#undef LAUNCH_FUSED
    CU_CHECK(cudaGetLastError());
    // K2: one warp per bitmap word (8 words per CTA) up to 256 CTAs per table, so that the dependent
    // chain of a miss (bitmap -> id -> loser search -> row) is paid once, by all warps at the same time
    int mctas = (words + MISS_NT / 32 - 1) / (MISS_NT / 32);
    if (mctas > 256) mctas = 256;
    const int wpc = (words + mctas - 1) / mctas;
    dim3 mgrid(mctas, tc);
#define LAUNCH_MISS(VEC, CP) LAUNCH_PDL(K_GATHER, s, (fwd_miss_kernel<VEC, CP>), mgrid, MISS_NT, 0, c->d_tabs, tb, ids, ld_ids, n_idx, slots, ld_slots, c->d_missmap, words, wpc, c->d_losers, out, ld_out, n_miss, c->d_flags, c->dim, c->ways, c->aux)
    if (copy) LAUNCH_MISS(4, true);
    else if (vec == 4) LAUNCH_MISS(4, false);
    else if (vec == 2) LAUNCH_MISS(2, false);
    else LAUNCH_MISS(1, false);
#undef LAUNCH_MISS
    CU_CHECK(cudaGetLastError());
    if (!copy && n_bags > 0) {
        const int NG = 256 / G;
        dim3 pg((n_bags + NG - 1) / NG, tc);
        if (vec == 4) LAUNCH(K_POOL, s, pool_kernel<4><<<pg, 256, 0, s>>>(c->d_tabs, tb, slots, ld_slots, offsets, ld_off, n_idx, n_bags, out, ld_out, bag_ids, ld_bag, c->dim, G));
        else if (vec == 2) LAUNCH(K_POOL, s, pool_kernel<2><<<pg, 256, 0, s>>>(c->d_tabs, tb, slots, ld_slots, offsets, ld_off, n_idx, n_bags, out, ld_out, bag_ids, ld_bag, c->dim, G));
        else LAUNCH(K_POOL, s, pool_kernel<1><<<pg, 256, 0, s>>>(c->d_tabs, tb, slots, ld_slots, offsets, ld_off, n_idx, n_bags, out, ld_out, bag_ids, ld_bag, c->dim, G));
        CU_CHECK(cudaGetLastError());
    }
    return CDLRM_OK;
}

extern "C" int cdlrm_embed_fwd_eval(cdlrm_ctx* c, int tb, int tc, const int64_t* ids, int64_t ld_ids, int32_t n_idx,
                                    float* out, int64_t ld_out, cdlrm_stream stream) {
    ARG_CHECK(c && ids && out);
    ARG_CHECK(tb >= 0 && tc > 0 && tb + tc <= c->T);
    ARG_CHECK(n_idx >= 0);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    for (int k = tb; k < tb + tc; ++k) {
        if (!c->tabs[k].weight || !c->tabs[k].tags || !c->tabs[k].master) {
            cdlrm_set_error("table %d: cache or master not bound", k);
            return CDLRM_ERR_STATE;
        }
    }
    int rc = cdlrm_sync_tabs(c, s);
    if (rc) return rc;
    if (n_idx == 0) return CDLRM_OK;
    bool al16 = true, al8 = true, tags16 = true;
    for (int k = tb; k < tb + tc; ++k) {
        al16 = al16 && ((uintptr_t)c->tabs[k].master % 16 == 0);
        al8 = al8 && ((uintptr_t)c->tabs[k].master % 8 == 0);
        tags16 = tags16 && ((uintptr_t)c->tabs[k].tags % 16 == 0);
    }
    int vec = pick_vec(c->dim, out, nullptr, ld_out, c->dim);
    if (vec == 4 && !al16) vec = 2;
    if (vec == 2 && !al8) vec = 1;
    const int cpr = c->dim / vec;
    const int G = pow2_ceil(cpr) > 32 ? 32 : pow2_ceil(cpr);
    const int words = (n_idx + 31) / 32;
    dim3 grid((words + FWD_NT / 32 - 1) / (FWD_NT / 32), tc);
    const int wsel = !tags16 ? 0 : (c->ways == 16 ? 16 : c->ways == 8 ? 8 : c->ways == 4 ? 4 : c->ways == 2 ? 2 : 0);
#define LAUNCH_EVAL(WW, VV) LAUNCH_PDL(K_EMBED_EVAL, s, (fwd_eval_kernel<WW, VV>), grid, FWD_NT, 0, c->d_tabs, tb, ids, ld_ids, n_idx, c->d_losers, out, ld_out, c->dim, c->ways, G, c->d_flags)
#define EVAL_V(WW)                                  \
    if (vec == 4) { LAUNCH_EVAL(WW, 4); }           \
    else if (vec == 2) { LAUNCH_EVAL(WW, 2); }      \
    else { LAUNCH_EVAL(WW, 1); }
    switch (wsel) {
        case 16: EVAL_V(16) break;
        case 8: EVAL_V(8) break;
        case 4: EVAL_V(4) break;
        case 2: EVAL_V(2) break;
        default: EVAL_V(0) break;
    }
#undef EVAL_V
#undef LAUNCH_EVAL
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

extern "C" int64_t cdlrm_embed_bwd_plan_bytes(int tc, int32_t n_idx) {
    if (tc <= 0 || n_idx < 0) return -1;
    size_t a = (size_t)tc * (size_t)(n_idx > 0 ? n_idx : 1) * sizeof(int32_t);
    a = (a + 255) & ~(size_t)255;
    return (int64_t)(2 * a);
}

extern "C" int cdlrm_embed_bwd_plan(cdlrm_ctx* c, int tb, int tc, const int32_t* slots, int64_t ld_slots,
                                    int32_t n_idx, void* plan, cdlrm_stream stream) {
    ARG_CHECK(c && slots && plan);
    ARG_CHECK(tb >= 0 && tc > 0 && tb + tc <= c->T && n_idx >= 0);
    ARG_CHECK(((uintptr_t)plan & 255) == 0);
    if (n_idx == 0) return CDLRM_OK;
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    int rc = cdlrm_sync_tabs(c, s);
    if (rc) return rc;
    PlanView pv = plan_view(plan, tc, n_idx);
    const int nsub = plan_nsub(n_idx);
    const int max_smem = CDLRM_SORT_MAX * 12 + 8192 * 2 + 64 * 4;
    // cluster size of the multi-CTA sort (cdlrm_embed_set_option(0, .) / CDLRM_PLAN_CLUSTER; 0 = one CTA per table)
    static const int env_cluster = [] { const char* e = getenv("CDLRM_PLAN_CLUSTER"); return e ? atoi(e) : -1; }();
    const int want = g_plan_cluster >= 0 ? g_plan_cluster : (env_cluster >= 0 ? env_cluster : 8);
    for (int sub = 0; sub < nsub; ++sub) {
        const int j0 = sub * CDLRM_SORT_MAX;
        const int n = n_idx - j0 < CDLRM_SORT_MAX ? n_idx - j0 : CDLRM_SORT_MAX;
        int C = 0;
        if (want > 0) {         // smallest power of two <= want whose chunks fit a CTA, not more CTAs than 512-key chunks
            C = 1;
            while (C < want && C < 8 && (int64_t)C * 512 < n) C <<= 1;
            if (((int64_t)n + C - 1) / C > CPL_MAX_CHUNK) C = 0;
        }
        if (C > 0) {
            const int chunk = (int)((((int64_t)n + C - 1) / C + 511) / 512 * 512);
            const int smem = chunk * 12 + 256 * CPL_NW * 2 + 512 * 4 + 64 * 4;
            cdlrm_prof_mark(K_BWD_PLAN, s, 0);
            cdlrm_launch_pdl_cluster(bwd_plan_cluster_kernel, dim3(C, tc), dim3(CPL_NT), smem, s, C, c->d_tabs, tb, slots,
                                     ld_slots, n_idx, j0, n, chunk, pv);
            cdlrm_prof_mark(K_BWD_PLAN, s, 1);
        } else {
            CU_CHECK(cdlrm_smem_optin((const void*)bwd_plan_kernel, max_smem));
            const int npad = (n + 7) & ~7;
            const int smem = npad * 12 + 8192 * 2 + 64 * 4;
            LAUNCH_PDL(K_BWD_PLAN, s, bwd_plan_kernel, tc, PLAN_NT, smem, c->d_tabs, tb, slots, ld_slots, n_idx, j0, n, pv);
        }
    }
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

template <bool DLR>
static int bwd_sgd_launch(cdlrm_ctx* c, int tb, int tc, const void* plan, int32_t n_idx, const int32_t* bag_ids,
                          int64_t ld_bag, const float* d_out, int64_t ld_dout, int64_t row_stride, float lr,
                          const float* d_lr, cdlrm_stream stream) {
    ARG_CHECK(c && plan && d_out);
    ARG_CHECK(tb >= 0 && tc > 0 && tb + tc <= c->T && n_idx >= 0);
    ARG_CHECK(!DLR || d_lr);
    if (n_idx == 0) return CDLRM_OK;
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    int rc = cdlrm_sync_tabs(c, s);
    if (rc) return rc;
    PlanView pv = plan_view(const_cast<void*>(plan), tc, n_idx);
    const int nsub = plan_nsub(n_idx);
    const int vec = pick_vec(c->dim, d_out, nullptr, ld_dout, row_stride);
    const int cpr = c->dim / vec;
    const int G = pow2_ceil(cpr) > 32 ? 32 : pow2_ceil(cpr);
    const int NG = 256 / G;
    // sub-batches (sorted separately) are applied one after the other in stream order: two
    // sub-batches may hold the same slot, and each treats its own runs as exclusive
    for (int sub = 0; sub < nsub; ++sub) {
        const int j0 = sub * CDLRM_SORT_MAX;
        const int n = n_idx - j0 < CDLRM_SORT_MAX ? n_idx - j0 : CDLRM_SORT_MAX;
        if (vec == 4 && cpr <= 32) {
            dim3 grid((n + APPLY_NT - 1) / APPLY_NT, tc);     // a warp per 32 sorted entries
#define LAUNCH_SGD(GG)                                                                                         \
    LAUNCH_PDL(K_BWD_SGD, s, (bwd_sgd_apply_kernel<GG, DLR>), grid, APPLY_NT, 0, c->d_tabs, tb, pv, n_idx, j0, n, bag_ids, ld_bag, d_out, ld_dout, row_stride, lr, d_lr, c->dim)
            switch (G) {
                case 1: LAUNCH_SGD(1); break;
                case 2: LAUNCH_SGD(2); break;
                case 4: LAUNCH_SGD(4); break;
                case 8: LAUNCH_SGD(8); break;
                case 16: LAUNCH_SGD(16); break;
                default: LAUNCH_SGD(32); break;
            }
#undef LAUNCH_SGD
        } else {
            dim3 grid((n + NG - 1) / NG, tc);
            if (vec == 4) LAUNCH(K_BWD_SGD, s, (bwd_sgd_kernel<4, DLR><<<grid, 256, 0, s>>>(c->d_tabs, tb, pv, n_idx, j0, n, bag_ids, ld_bag, d_out, ld_dout, row_stride, lr, d_lr, c->dim, G)));
            else if (vec == 2) LAUNCH(K_BWD_SGD, s, (bwd_sgd_kernel<2, DLR><<<grid, 256, 0, s>>>(c->d_tabs, tb, pv, n_idx, j0, n, bag_ids, ld_bag, d_out, ld_dout, row_stride, lr, d_lr, c->dim, G)));
            else LAUNCH(K_BWD_SGD, s, (bwd_sgd_kernel<1, DLR><<<grid, 256, 0, s>>>(c->d_tabs, tb, pv, n_idx, j0, n, bag_ids, ld_bag, d_out, ld_dout, row_stride, lr, d_lr, c->dim, G)));
        }
    }
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

extern "C" int cdlrm_embed_bwd_sgd(cdlrm_ctx* c, int tb, int tc, const void* plan, int32_t n_idx,
                                   const int32_t* bag_ids, int64_t ld_bag, const float* d_out, int64_t ld_dout,
                                   int64_t row_stride, float lr, cdlrm_stream stream) {
    return bwd_sgd_launch<false>(c, tb, tc, plan, n_idx, bag_ids, ld_bag, d_out, ld_dout, row_stride, lr, nullptr, stream);
}

extern "C" int cdlrm_embed_bwd_sgd_dlr(cdlrm_ctx* c, int tb, int tc, const void* plan, int32_t n_idx,
                                       const int32_t* bag_ids, int64_t ld_bag, const float* d_out, int64_t ld_dout,
                                       int64_t row_stride, const float* d_lr, cdlrm_stream stream) {
    return bwd_sgd_launch<true>(c, tb, tc, plan, n_idx, bag_ids, ld_bag, d_out, ld_dout, row_stride, 0.f, d_lr, stream);
}

template <bool DLR>
static int victim_launch(cdlrm_ctx* c, int tb, int tc, const int32_t* slots, int64_t ld_slots, const int64_t* ids,
                         int64_t ld_ids, int32_t n_idx, const int32_t* bag_ids, int64_t ld_bag, const float* d_out,
                         int64_t ld_dout, int64_t row_stride, float lr, const float* d_lr, cdlrm_stream stream) {
    ARG_CHECK(c && slots && ids && d_out);
    ARG_CHECK(tb >= 0 && tc > 0 && tb + tc <= c->T && n_idx >= 0);
    ARG_CHECK(!DLR || d_lr);
    // misses of a table: at most one per aux row and one per position; one CTA may have to hold all of them
    const int64_t cap = c->aux < n_idx ? c->aux : n_idx;
    if (cap == 0) return CDLRM_OK;
    if (cap > CDLRM_SORT_MAX) {
        cdlrm_set_error("cdlrm_embed_victim_update: up to %d misses per table (aux rows and ids per table), got %lld",
                        CDLRM_SORT_MAX, (long long)cap);
        return CDLRM_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    int rc = cdlrm_sync_tabs(c, s);
    if (rc) return rc;
    const int vec = pick_vec(c->dim, d_out, nullptr, ld_dout, row_stride);
    const int smem = pow2_ceil((int)cap) * (int)sizeof(unsigned long long);
    int C = n_idx / 512;                   // CTAs per table: ids are spread over them by hash
    C = C < 1 ? 1 : (C > 16 ? 16 : C);
    const dim3 grid(C, tc);
#define LAUNCH_VICTIM(VV)                                                                                            \
    do {                                                                                                             \
        CU_CHECK(cdlrm_smem_optin((const void*)victim_update_kernel<VV, DLR>, smem));                                \
        LAUNCH_PDL(K_EMBED_VICTIM, s, (victim_update_kernel<VV, DLR>), grid, VICTIM_NT, smem, c->d_tabs, tb,       \
                   c->d_losers, slots, ld_slots, ids, ld_ids, n_idx, bag_ids, ld_bag, d_out, ld_dout, row_stride, lr, \
                   d_lr, c->dim, c->ways, (int)cap, c->d_flags);                                                     \
    } while (0)
    if (vec == 4) LAUNCH_VICTIM(4);
    else if (vec == 2) LAUNCH_VICTIM(2);
    else LAUNCH_VICTIM(1);
#undef LAUNCH_VICTIM
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

extern "C" int cdlrm_embed_victim_update(cdlrm_ctx* c, int tb, int tc, const int32_t* slots, int64_t ld_slots,
                                         const int64_t* ids, int64_t ld_ids, int32_t n_idx, const int32_t* bag_ids,
                                         int64_t ld_bag, const float* d_out, int64_t ld_dout, int64_t row_stride,
                                         float lr, cdlrm_stream stream) {
    return victim_launch<false>(c, tb, tc, slots, ld_slots, ids, ld_ids, n_idx, bag_ids, ld_bag, d_out, ld_dout,
                                row_stride, lr, nullptr, stream);
}

extern "C" int cdlrm_embed_victim_update_dlr(cdlrm_ctx* c, int tb, int tc, const int32_t* slots, int64_t ld_slots,
                                             const int64_t* ids, int64_t ld_ids, int32_t n_idx, const int32_t* bag_ids,
                                             int64_t ld_bag, const float* d_out, int64_t ld_dout, int64_t row_stride,
                                             const float* d_lr, cdlrm_stream stream) {
    return victim_launch<true>(c, tb, tc, slots, ld_slots, ids, ld_ids, n_idx, bag_ids, ld_bag, d_out, ld_dout,
                               row_stride, 0.f, d_lr, stream);
}
