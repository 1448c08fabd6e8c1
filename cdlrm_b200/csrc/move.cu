// move.cu -- data movers of the window install and the table aggregation.
//   evict / fill / master gather: data part of CacheEmbeddings (main_no_ddp.py:190-199,
//   :205-206), Prefetcher.eviction_manager (cache_manager.py:48-64) and
//   Embedding_Table_Group.fetch_unique_idx_slices (model_no_ddp.py:80-87).
//   collect / pack / unpack: broadcast_and_aggregate (main_no_ddp.py:250-292) around one
//   NCCL all-reduce issued by the host side.
// The master pointers are device-visible addresses of pinned host memory: the gathers
// and the write-back are zero-copy PCIe reads/writes issued by the SMs, so scattered
// 512-byte rows move without any host-side staging or CPU work.
#include <stdlib.h>

#include "common.cuh"
#include "compact.cuh"

namespace {

template <int VEC> struct VT;
template <> struct VT<4> { using type = float4; };
template <> struct VT<2> { using type = float2; };
template <> struct VT<1> { using type = float; };

__device__ __forceinline__ float4 avg2(float4 a, float4 b) { return make_float4((a.x + b.x) / 2, (a.y + b.y) / 2, (a.z + b.z) / 2, (a.w + b.w) / 2); }
__device__ __forceinline__ float2 avg2(float2 a, float2 b) { return make_float2((a.x + b.x) / 2, (a.y + b.y) / 2); }
__device__ __forceinline__ float avg2(float a, float b) { return (a + b) / 2; }
__device__ __forceinline__ float4 vdiv(float4 a, float d) { return make_float4(a.x / d, a.y / d, a.z / d, a.w / d); }
__device__ __forceinline__ float2 vdiv(float2 a, float d) { return make_float2(a.x / d, a.y / d); }
__device__ __forceinline__ float vdiv(float a, float d) { return a / d; }

// mode 0: evict   rows_out[e] = weight[slot[e]]; master[id[e]] = row (or average)
// mode 1: gather  rows_out[i] = master[id[i]]
// mode 2: fill    weight[slot[i]] = rows ? rows[src?src[i]:i] : master[id[i]]; tags updated
// mode 3: pack    buf[i] = weight[slot[i]] / divisor
// mode 4: unpack  weight[slot[i]] = buf[i]
// mode 5: scatter master[id[i]] = rows[i] (or average)
template <int VEC, int MODE>
__global__ void __launch_bounds__(256) rows_kernel(TableDesc T, const int64_t* __restrict__ ids,
                                                   const int32_t* __restrict__ slots,
                                                   const uint8_t* __restrict__ primary, int64_t n,
                                                   float* __restrict__ rows, const int64_t* __restrict__ src_index,
                                                   int write_master, int average, float divisor, int dim, int ways,
                                                   int G) {
    using V = typename VT<VEC>::type;
    const int gl = threadIdx.x % G, group = threadIdx.x / G, NG = blockDim.x / G;
    const int cpr = dim / VEC;
    float* master = const_cast<float*>(T.master);
    constexpr int U = 4;
    for (int64_t i0 = (int64_t)blockIdx.x * NG * U + group; i0 < n; i0 += (int64_t)gridDim.x * NG * U) {
        for (int c = gl; c < cpr; c += G) {
            V v[U];
            const float* src[U];
            float* dst[U];
            float* dst2[U];
            bool valid[U], avg[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t i = i0 + (int64_t)u * NG;
                valid[u] = i < n;
                src[u] = nullptr; dst[u] = nullptr; dst2[u] = nullptr; avg[u] = false;
                if (!valid[u]) continue;
                if (MODE == 0) {
                    src[u] = T.weight + (int64_t)slots[i] * dim;
                    dst[u] = rows ? rows + i * dim : nullptr;
                    if (write_master && (!average || primary[i])) {
                        dst2[u] = master + ids[i] * dim;
                        avg[u] = average != 0;
                    }
                } else if (MODE == 1) {
                    src[u] = master + ids[i] * dim;
                    dst[u] = rows + i * dim;
                } else if (MODE == 2) {
                    src[u] = rows ? rows + (src_index ? src_index[i] : i) * dim : master + ids[i] * dim;
                    dst[u] = T.weight + (int64_t)slots[i] * dim;
                } else if (MODE == 3) {
                    src[u] = T.weight + (int64_t)slots[i] * dim;
                    dst[u] = rows + i * dim;
                } else if (MODE == 4) {
                    src[u] = rows + i * dim;
                    dst[u] = T.weight + (int64_t)slots[i] * dim;
                } else {
                    src[u] = rows + i * dim;
                    if (!primary || primary[i]) {   // duplicates carry identical rows: written once
                        dst2[u] = master + ids[i] * dim;
                        avg[u] = average != 0;
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (valid[u]) v[u] = reinterpret_cast<const V*>(src[u])[c];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (!valid[u]) continue;
                if (MODE == 3 && divisor != 1.0f) v[u] = vdiv(v[u], divisor);
                if (dst[u]) reinterpret_cast<V*>(dst[u])[c] = v[u];
                if ((MODE == 0 || MODE == 5) && dst2[u]) {
                    V* m = reinterpret_cast<V*>(dst2[u]) + c;
                    *m = avg[u] ? avg2(*m, v[u]) : v[u];
                }
            }
        }
        if (MODE == 2 && gl == 0) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t i = i0 + (int64_t)u * NG;
                if (i < n) {
                    const int64_t sl = slots[i];
                    const int64_t way = sl / T.num_sets, s = sl - way * T.num_sets;
                    T.tags[s * ways + way] = ids[i];
                }
            }
        }
    }
}

__global__ void or_bitmaps_kernel(uint32_t* __restrict__ dst, const uint32_t* __restrict__ gathered, int world,
                                  int64_t words) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < words; i += stride) {
        uint32_t v = 0;
        for (int r = 0; r < world; ++r) v |= gathered[(int64_t)r * words + i];
        dst[i] = v;
    }
}

inline int pow2_ceil(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

inline int vec_for(int dim, const void* a, const void* b) {
    auto al = [](const void* p, int n) { return p == nullptr || ((uintptr_t)p % n) == 0; };
    if (dim % 4 == 0 && al(a, 16) && al(b, 16)) return 4;
    if (dim % 2 == 0 && al(a, 8) && al(b, 8)) return 2;
    return 1;
}

constexpr int mode_kid(int mode) {
    return mode == 0 ? K_MOVE_EVICT : mode == 1 ? K_MOVE_GATHER : mode == 2 ? K_MOVE_FILL
         : mode == 3 ? K_AGG_PACK : mode == 4 ? K_AGG_UNPACK : K_MOVE_SCATTER;
}

template <int MODE>
int launch_rows(cdlrm_ctx* c, int k, const int64_t* ids, const int32_t* slots, const uint8_t* primary, int64_t n,
                float* rows, const int64_t* src_index, int write_master, int average, float divisor,
                bool uses_master, cudaStream_t s) {
    if (n <= 0) return CDLRM_OK;
    const TableDesc& T = c->tabs[k];
    const int vec = vec_for(c->dim, rows, uses_master ? T.master : nullptr);
    const int cpr = c->dim / vec;
    const int G = pow2_ceil(cpr) > 32 ? 32 : pow2_ceil(cpr);
    // HBM<->HBM movers: full grid.  Movers that touch the host master are PCIe-bound and run for ~0.1 s per
    // window on the planner stream beside the training step.  What they cost the step is set by how many
    // system-memory reads they keep in flight, not by their SM footprint (B200, Terabyte shape, 7 GB prefetch):
    //     4736 CTAs x 256 thr (full occupancy)   training stalled outright, 110 ms per window
    //      148 CTAs x  64 thr (600 KB in flight)  step 2-4x slower while it runs,  ~87 ms lost per window
    //       16 CTAs x 256 thr (260 KB in flight)  step 1.15-1.3x slower,           ~25 ms lost, same PCIe rate
    //        8 CTAs x 256 thr (130 KB in flight)  step 1.1x slower but the prefetch takes 1.5x longer
    // Default: 32 CTAs x 128 threads (260 KB in flight; 9 K registers per CTA, so the 1-CTA-per-SM tensor-core
    // GEMM with its 54 K registers still fits beside it).  CDLRM_PCIE_CTAS / CDLRM_PCIE_THREADS override.
    static const int pcie_ctas = [] { const char* e = getenv("CDLRM_PCIE_CTAS"); return e ? atoi(e) : 32; }();
    static const int pcie_threads = [] { const char* e = getenv("CDLRM_PCIE_THREADS"); return e ? atoi(e) : 128; }();
    const int nt = uses_master ? (pcie_threads >= G && pcie_threads <= 256 ? pcie_threads : 128) : 256;
    const int NG = nt / G;
    int64_t blocks = (n + NG * 4 - 1) / (NG * 4);
    const int64_t cap = uses_master ? (pcie_ctas > 0 ? pcie_ctas : 32) : (int64_t)c->num_sms * 32;
    if (blocks > cap) blocks = cap;
    if (vec == 4) LAUNCH(mode_kid(MODE), s, (rows_kernel<4, MODE><<<(int)blocks, nt, 0, s>>>(T, ids, slots, primary, n, rows, src_index, write_master, average, divisor, c->dim, c->ways, G)));
    else if (vec == 2) LAUNCH(mode_kid(MODE), s, (rows_kernel<2, MODE><<<(int)blocks, nt, 0, s>>>(T, ids, slots, primary, n, rows, src_index, write_master, average, divisor, c->dim, c->ways, G)));
    else LAUNCH(mode_kid(MODE), s, (rows_kernel<1, MODE><<<(int)blocks, nt, 0, s>>>(T, ids, slots, primary, n, rows, src_index, write_master, average, divisor, c->dim, c->ways, G)));
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

}  // namespace

extern "C" int cdlrm_move_scatter_master2(cdlrm_ctx* c, int k, const int64_t* ids, const uint8_t* primary, int64_t n,
                                          const float* rows, int average, cdlrm_stream stream);

extern "C" int cdlrm_move_evict(cdlrm_ctx* c, int k, const int64_t* evict_ids, const int32_t* evict_slots,
                                const uint8_t* evict_primary, int64_t n, float* rows_out, int write_master,
                                int average, cdlrm_stream stream) {
    ARG_CHECK(c && k >= 0 && k < c->T && n >= 0);
    if (n == 0) return CDLRM_OK;
    ARG_CHECK(evict_ids && evict_slots);
    ARG_CHECK(!(write_master && average) || evict_primary);
    ARG_CHECK(c->tabs[k].weight && (!write_master || c->tabs[k].master));
    CU_CHECK(cudaSetDevice(c->device));
    return launch_rows<0>(c, k, evict_ids, evict_slots, evict_primary, n, rows_out, nullptr, write_master, average,
                          1.0f, write_master != 0, (cudaStream_t)stream);
}

extern "C" int cdlrm_move_gather_master(cdlrm_ctx* c, int k, const int64_t* ids, int64_t n, float* rows_out,
                                        cdlrm_stream stream) {
    ARG_CHECK(c && k >= 0 && k < c->T && n >= 0);
    if (n == 0) return CDLRM_OK;
    ARG_CHECK(ids && rows_out && c->tabs[k].master);
    CU_CHECK(cudaSetDevice(c->device));
    return launch_rows<1>(c, k, ids, nullptr, nullptr, n, rows_out, nullptr, 0, 0, 1.0f, true, (cudaStream_t)stream);
}

extern "C" int cdlrm_move_fill(cdlrm_ctx* c, int k, const int64_t* fill_ids, const int32_t* fill_slots, int64_t n,
                               const float* rows, const int64_t* src_index, cdlrm_stream stream) {
    ARG_CHECK(c && k >= 0 && k < c->T && n >= 0);
    if (n == 0) return CDLRM_OK;
    ARG_CHECK(fill_ids && fill_slots && c->tabs[k].weight && c->tabs[k].tags);
    ARG_CHECK(rows || c->tabs[k].master);
    CU_CHECK(cudaSetDevice(c->device));
    return launch_rows<2>(c, k, fill_ids, fill_slots, nullptr, n, const_cast<float*>(rows), src_index, 0, 0, 1.0f,
                          rows == nullptr, (cudaStream_t)stream);
}

extern "C" int cdlrm_move_scatter_master(cdlrm_ctx* c, int k, const int64_t* ids, int64_t n, const float* rows,
                                         int average, cdlrm_stream stream) {
    return cdlrm_move_scatter_master2(c, k, ids, nullptr, n, rows, average, stream);
}

extern "C" int cdlrm_move_scatter_master2(cdlrm_ctx* c, int k, const int64_t* ids, const uint8_t* primary, int64_t n,
                                          const float* rows, int average, cdlrm_stream stream) {
    ARG_CHECK(c && k >= 0 && k < c->T && n >= 0);
    if (n == 0) return CDLRM_OK;
    ARG_CHECK(ids && rows && c->tabs[k].master);
    CU_CHECK(cudaSetDevice(c->device));
    return launch_rows<5>(c, k, ids, nullptr, primary, n, const_cast<float*>(rows), nullptr, 1, average, 1.0f, true,
                          (cudaStream_t)stream);
}

// Bucket index of a loser store (LoserDesc::bucket): thread b finds the first index whose id >= b << shift.
__global__ void __launch_bounds__(256) loser_bucket_kernel(const LoserDesc* __restrict__ losers) {
    const LoserDesc& L = losers[blockIdx.y];
    if (!L.bucket || L.n <= 0) return;
    int32_t* __restrict__ bucket = const_cast<int32_t*>(L.bucket);
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < L.nb; b += gridDim.x * blockDim.x) {
        const int64_t target = (int64_t)b << L.shift;
        int64_t lo = 0, hi = L.n;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (__ldg(L.ids + mid) < target) lo = mid + 1; else hi = mid;
        }
        bucket[b] = (int32_t)lo;
    }
}

// Carve the bucket indices of the descriptors in h[0..T) out of c->d_lbucket (grown when a window needs more; the
// stores are bound at window boundaries, where a cudaMalloc does not hurt) and launch the build behind the
// descriptor copy.  About 4 ids per bucket: n / 4 + 2 buckets per table.
static int build_loser_buckets(cdlrm_ctx* c, LoserDesc* h, cudaStream_t s) {
    int64_t total = 0;
    for (int k = 0; k < c->T; ++k) {
        h[k].bucket = nullptr;
        h[k].shift = 0;
        h[k].nb = 0;
        if (h[k].n < 64 || h[k].n >= (1ll << 31)) continue;             // short lists: the plain search is as fast
        int shift = 0;
        while (shift < 40 && ((c->tabs[k].n_rows >> shift) > h[k].n / 4 + 1)) ++shift;
        const int64_t nb = (c->tabs[k].n_rows >> shift) + 2;
        if (nb >= (1ll << 31)) continue;
        h[k].shift = shift;
        h[k].nb = (int32_t)nb;
        total += nb;
    }
    if (total == 0) return CDLRM_OK;
    if (total > c->lbucket_cap) {
        if (c->d_lbucket) CU_CHECK(cudaFree(c->d_lbucket));            // (synchronises: no forward still reads it)
        c->d_lbucket = nullptr;
        c->lbucket_cap = total + total / 2 + 1024;
        CU_CHECK(cudaMalloc(&c->d_lbucket, sizeof(int32_t) * (size_t)c->lbucket_cap));
    }
    int64_t off = 0;
    int64_t nb_max = 0;
    for (int k = 0; k < c->T; ++k) {
        if (!h[k].nb) continue;
        h[k].bucket = c->d_lbucket + off;
        off += h[k].nb;
        if (h[k].nb > nb_max) nb_max = h[k].nb;
    }
    return CDLRM_OK;
}

static int launch_loser_buckets(cdlrm_ctx* c, const LoserDesc* h, cudaStream_t s) {
    int64_t nb_max = 0;
    for (int k = 0; k < c->T; ++k)
        if (h[k].nb > nb_max) nb_max = h[k].nb;
    if (nb_max == 0) return CDLRM_OK;
    const int gx = (int)((nb_max + 255) / 256 < 592 ? (nb_max + 255) / 256 : 592);
    LAUNCH(K_MOVE_GATHER, s, loser_bucket_kernel<<<dim3(gx, c->T), 256, 0, s>>>(c->d_losers));
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

// Loser store (see LoserDesc): the descriptors reach the device in stream order, so the forward
// launched after this call on `stream` sees the new store and the ones before it the old one.
extern "C" int cdlrm_ctx_bind_losers(cdlrm_ctx* c, const int64_t* const* h_ids, const float* const* h_rows,
                                     const int64_t* h_n, cdlrm_stream stream) {
    ARG_CHECK(c);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    if (!c->d_losers) {
        CU_CHECK(cudaMalloc(&c->d_losers, sizeof(LoserDesc) * c->T));
        CU_CHECK(cudaMemset(c->d_losers, 0, sizeof(LoserDesc) * c->T));
        CU_CHECK(cudaHostAlloc(&c->h_losers, sizeof(LoserDesc) * c->T * 4, cudaHostAllocDefault));
    }
    LoserDesc* h = c->h_losers + (size_t)(c->losers_flip++ & 3) * c->T;   // 4 updates may be in flight
    for (int k = 0; k < c->T; ++k) {
        memset(&h[k], 0, sizeof(LoserDesc));
        h[k].ids = h_ids ? h_ids[k] : nullptr;
        h[k].rows = h_rows ? h_rows[k] : nullptr;
        h[k].n = (h_ids && h_rows && h_n) ? h_n[k] : 0;
        ARG_CHECK(h[k].n >= 0 && (h[k].n == 0 || (h[k].ids && h[k].rows)));
    }
    if (int rc = build_loser_buckets(c, h, s)) return rc;
    CU_CHECK(cudaMemcpyAsync(c->d_losers, h, sizeof(LoserDesc) * c->T, cudaMemcpyHostToDevice, s));
    return launch_loser_buckets(c, h, s);
}

// Boundary carry (--evict-victim-cache): rows[i] = the bound loser store's row of ids[i] when the store holds ids[i].
// The next window's fill and loser rows were prefetched from the master while this window trained its store rows.
template <int VEC>
__global__ void __launch_bounds__(256) carry_kernel(const LoserDesc* __restrict__ L, const int64_t* __restrict__ ids,
                                                    int64_t n, float* __restrict__ rows, int dim, int G) {
    using V = typename VT<VEC>::type;
    const int gl = threadIdx.x % G, group = threadIdx.x / G, NG = blockDim.x / G;
    const int cpr = dim / VEC;
    for (int64_t i = (int64_t)blockIdx.x * NG + group; i < n; i += (int64_t)gridDim.x * NG) {
        const int64_t li = loser_index(L, ids[i]);
        if (li < 0) continue;
        const V* src = reinterpret_cast<const V*>(loser_row(L, li, dim));
        V* dst = reinterpret_cast<V*>(rows + i * dim);
        for (int c = gl; c < cpr; c += G) dst[c] = src[c];
    }
}

extern "C" int cdlrm_move_carry_losers(cdlrm_ctx* c, int k, const int64_t* ids, int64_t n, float* rows_inout,
                                       cdlrm_stream stream) {
    ARG_CHECK(c && k >= 0 && k < c->T && n >= 0);
    if (n == 0 || !c->d_losers) return CDLRM_OK;         // nothing to copy, or no store was ever bound
    ARG_CHECK(ids && rows_inout);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    const int vec = vec_for(c->dim, rows_inout, nullptr);
    const int cpr = c->dim / vec;
    const int G = pow2_ceil(cpr) > 32 ? 32 : pow2_ceil(cpr);
    const int NG = 256 / G;
    int64_t blocks = (n + NG - 1) / NG;
    if (blocks > (int64_t)c->num_sms * 16) blocks = (int64_t)c->num_sms * 16;
    const LoserDesc* L = c->d_losers + k;
    if (vec == 4) LAUNCH(K_MOVE_CARRY, s, (carry_kernel<4><<<(int)blocks, 256, 0, s>>>(L, ids, n, rows_inout, c->dim, G)));
    else if (vec == 2) LAUNCH(K_MOVE_CARRY, s, (carry_kernel<2><<<(int)blocks, 256, 0, s>>>(L, ids, n, rows_inout, c->dim, G)));
    else LAUNCH(K_MOVE_CARRY, s, (carry_kernel<1><<<(int)blocks, 256, 0, s>>>(L, ids, n, rows_inout, c->dim, G)));
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

extern "C" int cdlrm_ctx_bind_losers_sharded(cdlrm_ctx* c, const int64_t* const* h_ids, const int64_t* h_n,
                                             const int64_t* h_shard, int world, const float* const* h_peer,
                                             cdlrm_stream stream) {
    ARG_CHECK(c && h_ids && h_n && h_shard && h_peer && world >= 1 && world <= CDLRM_MAX_PEERS);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    if (!c->d_losers) {
        CU_CHECK(cudaMalloc(&c->d_losers, sizeof(LoserDesc) * c->T));
        CU_CHECK(cudaMemset(c->d_losers, 0, sizeof(LoserDesc) * c->T));
        CU_CHECK(cudaHostAlloc(&c->h_losers, sizeof(LoserDesc) * c->T * 4, cudaHostAllocDefault));
    }
    LoserDesc* h = c->h_losers + (size_t)(c->losers_flip++ & 3) * c->T;
    for (int k = 0; k < c->T; ++k) {
        memset(&h[k], 0, sizeof(LoserDesc));
        h[k].n = h_n[k];
        if (h[k].n == 0) continue;
        ARG_CHECK(h[k].n > 0 && h_ids[k] && h_shard[k] > 0 && h_shard[k] * world >= h[k].n);
        h[k].ids = h_ids[k];
        h[k].shard = h_shard[k];
        for (int r = 0; r < world; ++r) {
            h[k].peer[r] = h_peer[(size_t)k * world + r];
            ARG_CHECK(h[k].peer[r] || (int64_t)r * h_shard[k] >= h[k].n);     // a rank without rows may pass NULL
        }
    }
    if (int rc = build_loser_buckets(c, h, s)) return rc;
    CU_CHECK(cudaMemcpyAsync(c->d_losers, h, sizeof(LoserDesc) * c->T, cudaMemcpyHostToDevice, s));
    return launch_loser_buckets(c, h, s);
}

extern "C" int cdlrm_host_register(int device, void* h_ptr, int64_t bytes, void** dev_ptr) {
    ARG_CHECK(h_ptr && bytes > 0 && dev_ptr);
    CU_CHECK(cudaSetDevice(device));
    CU_CHECK(cudaHostRegister(h_ptr, (size_t)bytes, cudaHostRegisterMapped | cudaHostRegisterPortable));
    CU_CHECK(cudaHostGetDevicePointer(dev_ptr, h_ptr, 0));
    return CDLRM_OK;
}

extern "C" int cdlrm_host_unregister(void* h_ptr) {
    ARG_CHECK(h_ptr);
    CU_CHECK(cudaHostUnregister(h_ptr));
    return CDLRM_OK;
}

// ---- aggregation ---------------------------------------------------------------------------------

__global__ void mark_kernel(TableDesc T, const int32_t* __restrict__ idxs, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const int32_t sl = idxs[i];
        if (sl >= 0 && sl < T.cache_rows) atomicOr(T.dirty + (sl >> 5), 1u << (sl & 31));
    }
}

extern "C" int cdlrm_agg_mark(cdlrm_ctx* c, const int32_t* idxs, int64_t ld, int64_t n, cdlrm_stream stream) {
    ARG_CHECK(c && n >= 0);
    if (n == 0) return CDLRM_OK;
    ARG_CHECK(idxs);
    CU_CHECK(cudaSetDevice(c->device));
    for (int k = 0; k < c->T; ++k) {
        ARG_CHECK(c->tabs[k].dirty);
        int64_t blocks = (n + 255) / 256;
        if (blocks > 1184) blocks = 1184;
        LAUNCH(K_AGG_MARK, (cudaStream_t)stream, mark_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(c->tabs[k], idxs + k * ld, n));
    }
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

static int dirty_is_concatenated(const cdlrm_ctx* c) {
    for (int k = 0; k < c->T; ++k)
        if (!c->tabs[k].dirty || c->tabs[k].dirty != c->tabs[0].dirty + c->tabs[k].dirty_word_off) return 0;
    return 1;
}

extern "C" int cdlrm_agg_or_bitmaps(cdlrm_ctx* c, const uint32_t* gathered, int world, int64_t words_total,
                                    cdlrm_stream stream) {
    ARG_CHECK(c && gathered && world >= 1);
    const TableDesc& last = c->tabs[c->T - 1];
    ARG_CHECK(words_total == last.dirty_word_off + (last.cache_rows + 31) / 32);
    if (!dirty_is_concatenated(c)) {
        cdlrm_set_error("dirty bitmaps must be bound as one concatenated buffer");
        return CDLRM_ERR_STATE;
    }
    CU_CHECK(cudaSetDevice(c->device));
    LAUNCH(K_AGG_OR, (cudaStream_t)stream, or_bitmaps_kernel<<<592, 256, 0, (cudaStream_t)stream>>>(c->tabs[0].dirty, gathered, world, words_total));
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

extern "C" int cdlrm_agg_collect(cdlrm_ctx* c, int32_t* slot_list, int64_t* d_counts, int64_t* h_counts,
                                 cdlrm_stream stream) {
    ARG_CHECK(c && slot_list && d_counts);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    int64_t words_max = 0;
    for (int k = 0; k < c->T; ++k) {
        ARG_CHECK(c->tabs[k].dirty);
        int64_t w = (c->tabs[k].cache_rows + 31) / 32;
        words_max = w > words_max ? w : words_max;
    }
    static thread_local int32_t* bs = nullptr;
    static thread_local int64_t bs_cap = 0;
    const int64_t need = (words_max + TILE - 1) / TILE + 1;
    if (need > bs_cap) {
        if (bs) cudaFree(bs);
        CU_CHECK(cudaMalloc(&bs, sizeof(int32_t) * need));
        bs_cap = need;
    }
    int64_t cap_off = 0;
    for (int k = 0; k < c->T; ++k) {
        const TableDesc& t = c->tabs[k];
        const int64_t nwords = (t.cache_rows + 31) / 32;
        const int nblk = (int)((nwords + TILE - 1) / TILE);
        LAUNCH(K_AGG_COLLECT, s, bitmap_count_kernel<<<nblk, 256, 0, s>>>(t.dirty, nwords, bs));
        LAUNCH(K_AGG_COLLECT, s, scan_tiles_kernel<<<1, 1024, 0, s>>>(bs, nblk, reinterpret_cast<unsigned long long*>(d_counts + k)));
        LAUNCH(K_AGG_COLLECT, s, (bitmap_emit_kernel<int32_t, false><<<nblk, 256, 0, s>>>(t.dirty, nwords, bs, slot_list + cap_off)));
        cap_off += t.cache_rows;
    }
    CU_CHECK(cudaGetLastError());
    if (h_counts) CU_CHECK(cudaMemcpyAsync(h_counts, d_counts, sizeof(int64_t) * c->T, cudaMemcpyDeviceToHost, s));
    return CDLRM_OK;
}

extern "C" int cdlrm_agg_pack(cdlrm_ctx* c, const int32_t* slot_list, const int64_t* h_counts, float divisor,
                              float* buf, cdlrm_stream stream) {
    ARG_CHECK(c && slot_list && h_counts && buf && divisor != 0.0f);
    CU_CHECK(cudaSetDevice(c->device));
    int64_t cap_off = 0, boff = 0;
    for (int k = 0; k < c->T; ++k) {
        ARG_CHECK(h_counts[k] >= 0 && h_counts[k] <= c->tabs[k].cache_rows);
        int rc = launch_rows<3>(c, k, nullptr, slot_list + cap_off, nullptr, h_counts[k], buf + boff * c->dim, nullptr,
                                0, 0, divisor, false, (cudaStream_t)stream);
        if (rc) return rc;
        cap_off += c->tabs[k].cache_rows;
        boff += h_counts[k];
    }
    return CDLRM_OK;
}

extern "C" int cdlrm_agg_unpack(cdlrm_ctx* c, const int32_t* slot_list, const int64_t* h_counts, const float* buf,
                                int clear_dirty, cdlrm_stream stream) {
    ARG_CHECK(c && slot_list && h_counts && buf);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    int64_t cap_off = 0, boff = 0;
    for (int k = 0; k < c->T; ++k) {
        ARG_CHECK(h_counts[k] >= 0 && h_counts[k] <= c->tabs[k].cache_rows);
        int rc = launch_rows<4>(c, k, nullptr, slot_list + cap_off, nullptr, h_counts[k],
                                const_cast<float*>(buf) + boff * c->dim, nullptr, 0, 0, 1.0f, false, s);
        if (rc) return rc;
        if (clear_dirty && c->tabs[k].dirty)
            CU_CHECK(cudaMemsetAsync(c->tabs[k].dirty, 0, sizeof(uint32_t) * ((c->tabs[k].cache_rows + 31) / 32), s));
        cap_off += c->tabs[k].cache_rows;
        boff += h_counts[k];
    }
    return CDLRM_OK;
}
