// mlp.cu -- the bottom / top MLPs of DLRM_Net (create_mlp / forward, model_no_ddp.py:244-270,
// 306-316 of the reference: Linear + ReLU, Sigmoid on the last top layer) on the 5th-gen
// tensor cores, at FP32 accuracy.
//
// The reference trains in FP32 and the parity bar on the loss is 1e-5 relative, so a plain
// TF32 product (10-bit mantissa) is not an option.  Every FP32 operand x is split into
//     hi = x with the low 13 mantissa bits cleared   (exactly a TF32 number)
//     lo = (x - hi) with the low 13 bits cleared      (the next 11 bits)
// and a product is evaluated as  hi*hi + hi*lo + lo*hi  (3xTF32) with FP32 accumulation in
// TMEM: relative error ~2^-21 per product, the same order as an FP32 FMA chain.
//
// One GEMM kernel serves forward, data-gradient and weight-gradient:
//     D[M,N] = A[M,K] * B[N,K]^T
// Each operand is read either K-major (row-major [M|N, K], K contiguous) or MN-major (row-major
// [K, M|N], the M or N index contiguous: the transpose of a tensor that is stored row-major anyway).
// A_hi/A_lo/B_hi/B_lo are four tensors in HBM, moved by TMA (128-byte swizzle) into a
// 3-stage shared-memory ring; one elected thread of a persistent CTA issues tcgen05.mma.kind::tf32
// (128x128x8, 12 per 32-wide k-block: 4 k-steps x 3 products) into a 128-column TMEM
// accumulator; four epilogue warps read it back with tcgen05.ld and apply the fused
// epilogue (bias, ReLU / sigmoid, ReLU-backward mask, hi/lo split of the result row-major,
// per-32-row column sums of the result, or a split-K reduce-add for the weight gradient).
//   forward    Y  = act(X W^T + b)        A = X [B,K]   K-major,    B = W   [N,K]  K-major
//   dgrad      dX = (dZ W) * relu'(X)     A = dZ [B,N]  K-major,    B = W^T from W [N,K]  MN-major
//   wgrad      dW = dZ^T X                A = dZ^T from dZ [B,N]  MN-major,  B = X^T from X [B,K]  MN-major  (split-K)
// The bias gradient db = column sums of dZ is taken where dZ is produced (dgrad epilogue, split_kernel,
// narrow_bwd_kernel) as partial sums per 32 rows, reduced in a fixed order by unpack_batch_kernel.
#include <cuda.h>

#include "common.cuh"

namespace {

// Tile 128 x 128, k-blocks of BK = 32 fp32 (one 128-byte swizzle row) in a 3-stage ring.  BK = 16
// (64-byte swizzle, 6 stages) is supported by the code below and was measured 10 % slower.
constexpr int BM = 128, BN = 128, BK = 32;
constexpr int STAGES = 3;
constexpr int TILE_BYTES = BM * BK * 4;           // 16 KB per operand tile
constexpr int STAGE_BYTES = 4 * TILE_BYTES;       // A_hi, A_lo, B_hi, B_lo (B_lo right behind B_hi: one 256-row operand)
constexpr int EPI_WARPS = 8;                      // two per TMEM lane quarter, 64 columns each
constexpr int GEMM_THREADS = 64 + 32 * EPI_WARPS; // warp 0: TMA, warp 1: MMA + TMEM, warps 2-9: epilogue
constexpr int STG_BYTES = 4096;                   // one 32 x 32 fp32 result tile per epilogue warp
// TMEM: two accumulator buffers of 256 columns (hi*hi | cross terms), so that the epilogue of one
// K segment / tile overlaps the MMAs of the next.  The tensor core's FP32 accumulation is not
// round-to-nearest, so the error of one accumulator grows with the number of MMAs chained into it:
// the two small cross terms get their own accumulator, and K is cut into segments of `seg_kb`
// k-blocks whose partial results the epilogue warps add up in registers (round-to-nearest).
constexpr int TMEM_COLS = 512;
constexpr int GEMM_SMEM = STAGES * STAGE_BYTES + EPI_WARPS * STG_BYTES + 1024 /*align*/ + 256 /*barriers*/;
// What bounds the mainloop (tools/gemm_probe.py, tools/gemm_trace.py on B200): shared-memory
// bandwidth.  Per k-step of 8 the three MMAs read 3 x (4 + 4) KB of operands and the TMA writes
// 16 KB (hi and lo of A and B): 40 KB at 128 B/clk = 320 clk, against 3 x 64 clk of tensor-core
// time; measured 0.65-0.7 us per 32-wide k-block = 330-345 clk per k-step, whatever the ring
// depth, the k-block size or the number of TMA instructions.  (A_hi x [B_hi ; B_lo] as ONE
// 128 x 256 x 8 MMA -- hi*hi and hi*lo side by side in TMEM -- is what the issuer does; it
// saves an instruction, not the second read of A_hi.)
// kind::tf32, FP32 accumulate, M = 128, N = n; bits 15 / 16: A / B MN-major instead of K-major
__host__ __device__ constexpr uint32_t idesc_tf32(int n, int a_mn, int b_mn) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(n >> 3) << 17) |
           ((uint32_t)(BM >> 4) << 24);
}

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_SIGMOID = 2 };

struct Epi {
    int M, N, K;                 // GEMM extents: rows of A, rows of B, reduction length
    int kb_per_split;            // k-blocks per K split
    int splits;                  // K splits (units = tiles x splits)
    int seg_kb;                  // k-blocks chained into one TMEM accumulator before the register add
    int cluster;                 // CTAs per cluster along M (1 or 2): the pair shares every B tile (TMA multicast)
    long long* trace;            // measurement only (cdlrm_mlp_set_trace): CTA 0 writes %globaltimer stamps, [4][128]
    int dbg;                     // measurement only (cdlrm_mlp_set_option(3, .)): 1 no result stores, 4 no MMAs
    const float* bias;           // [N] added per column (or null)
    int act;                     // ACT_*
    const float* mask;           // relu-backward: result passes where mask[row, col] > 0 (or null)
    int64_t ld_mask;
    int out_c;                   // 1: fp32 result row-major through map_c (2: reduce-add into it, split-K)
    int out_split;               // 1: hi/lo split row-major through map_c_hi / map_c_lo
    int a_mn, b_mn;              // 1: the operand is MN-major (see make_mn_map), 0: K-major
    float* colsum;               // sums of the result over each group of 32 rows: colsum[(row / 32) * N + col] (or null)
};

// tensor maps of one launch: 2 operand maps (128-byte swizzle) and up to 3 result maps (box 32 x 32,
// 128-byte swizzle)
struct Maps {
    CUtensorMap a, b;            // operands, hi and lo as one tensor: K-major {K, rows, 2}, MN-major {32, K, MN / 32, 2}
    CUtensorMap b_half;          // B again with a {BK, BN/2, 1} box: one CTA's share of a multicast B tile
    CUtensorMap c, c_hi, c_lo;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// bounded wait: a protocol error becomes a trap (launch failure), never a hung GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 28)) __trap();
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
// one instruction for the hi and lo tiles of an operand: 3-D map {K, rows, 2 (hi, lo)}
__device__ __forceinline__ void tma_load_pair(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(0), "r"(smem_u32(bar))
        : "memory");
}
// MN-major operand tile: 4-D map {32, K, MN / 32, 2 (hi, lo)}, box {32, BK, 4, 2}; lands as hi then lo, each
// four 32-wide column blocks of BK rows x 128 bytes (128-byte swizzle, 32-byte atoms: make_smem_desc_mn)
__device__ __forceinline__ void tma_load_mn(uint32_t dst, const CUtensorMap* map, int k, int mn0, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
        ::"r"(dst), "l"(map), "r"(0), "r"(k), "r"(mn0 / 32), "r"(0), "r"(smem_u32(bar))
        : "memory");
}
// one half (BN/2 rows) of the hi (c2 = 0) or lo (c2 = 1) B tile, written to the same shared-memory offset of
// every CTA in `mask`; each destination CTA's barrier (same offset) receives the byte count
__device__ __forceinline__ void tma_load_3d_mc(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar,
                                               uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3, %4}], [%5], %6;"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)), "h"(mask)
        : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// the same arrive on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void tc_commit_mc(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accum)
        : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// K-major, swizzle width = one row of BK fp32 (64 or 128 bytes), 8-row groups 8 rows apart (SBO),
// LBO unused (1), descriptor version 1 (sm_100), layout type 2 = SWIZZLE_128B / 4 = SWIZZLE_64B
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fff);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((8 * BK * 4) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(BK == 32 ? 2 : 4) << 61;
    return d;
}
// MN-major: 32 MN elements (128 bytes) per row, one row per k.  For 32-bit (tf32) operands the tensor core takes
// MN-major data only in the 128-byte swizzle with 32-byte atomicity (layout type 1, SWIZZLE_128B_BASE32B: 32-byte
// chunks of a row XOR-ed with the row index mod 4; 4-row atoms), which the TMA writes with
// CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.  The plain 128-byte swizzle is read as a different layout.
// The 32-wide column blocks are one TMA box (BK rows) apart (LBO), 4-row groups along K 512 bytes apart (SBO);
// a k-step of 8 covers two atoms, so the next k-step starts 1024 bytes further on.
__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fff);
    d |= (uint64_t)((32 * BK * 4) >> 4) << 16;
    d |= (uint64_t)(4 * 128 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;
    return d;
}

// round-to-nearest TF32 (ties away from zero in magnitude): the residual x - hi is then signed and
// at most half a TF32 ulp, and the same rounding of the residual leaves an error <= 2^-24 |x|
__device__ __forceinline__ float tf32_rn(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }
__device__ __forceinline__ float tf32_tr(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }
__device__ int g_split_trunc = 0;       // test hook: 1 = truncating split (the first version)
__device__ __forceinline__ float tf32_hi(float x) { return g_split_trunc ? tf32_tr(x) : tf32_rn(x); }
__device__ __forceinline__ float tf32_lo(float x, float hi) { return g_split_trunc ? tf32_tr(x - hi) : tf32_rn(x - hi); }

__device__ __forceinline__ long long gtime() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define TRACE(role, idx) do { if (ep.trace && blockIdx.x == 0 && (idx) < 128) ep.trace[(role) * 128 + (idx)] = gtime(); } while (0)
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Persistent: CTA b works on units b, b + gridDim.x, ... ; a unit = (n tile, m tile, K split),
// n fastest so that the CTAs running together share the A row panel in L2.
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm3x_tf32_kernel(const __grid_constant__ Maps maps, const Epi ep) {
    constexpr int NCH = BN / 64;                                 // 32-column chunks per epilogue warp
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t pad = ((raw + 1023u) & ~1023u) - raw;
    uint8_t* smem = smem_raw + pad;                              // 1024-byte aligned tiles
    uint8_t* stg_base = smem + STAGES * STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(stg_base + EPI_WARPS * STG_BYTES);
    uint64_t* full_bar = bars;                                   // [STAGES]  TMA -> MMA
    uint64_t* empty_bar = bars + STAGES;                         // [STAGES]  MMA -> TMA
    uint64_t* tfull_bar = bars + 2 * STAGES;                     // [2]       MMA -> epilogue
    uint64_t* tempty_bar = bars + 2 * STAGES + 2;                // [2]       epilogue -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_n = (ep.N + BN - 1) / BN;
    const int num_kb_total = (ep.K + BK - 1) / BK;
    // Cluster mode (ep.cluster == 2, launched with cluster dims {2,1,1}): CTAs 2p and 2p+1 walk the same unit
    // list; a unit then covers TWO adjacent m tiles (one per CTA) of one n tile, so both need the same B tile:
    // each loads half of it and multicasts it into both shared memories.  The stage is free again when BOTH
    // CTAs' MMAs have read it (empty barrier count 2, multicast tcgen05.commit).
    const int cl = ep.cluster;                                   // 1 or 2
    const int cr = cl == 2 ? (int)(blockIdx.x & 1u) : 0;         // rank in the cluster
    const int u_first = cl == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int u_step = cl == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int tiles_m = ((ep.M + BM - 1) / BM + cl - 1) / cl;    // m tiles per unit column (pairs in cluster mode)
    const int units = tiles_n * tiles_m * ep.splits;
    const uint16_t cl_mask = (uint16_t)((1u << cl) - 1u);

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], (uint32_t)cl); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tfull_bar[b], 1); mbar_init(&tempty_bar[b], EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&maps.a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&maps.b) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (cl == 2) cluster_sync_all();        // the peer's barriers exist before anything of mine can arrive on them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_enter();            // everything above (barriers, TMEM, tensor-map prefetch) overlaps the previous kernel's tail
    if (threadIdx.x == 0) TRACE(3, 0);

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            uint32_t it = 0;                       // k-blocks issued so far (ring position)
            for (int u = u_first; u < units; u += u_step) {
                const int n0 = (u % tiles_n) * BN, m0 = (((u / tiles_n) % tiles_m) * cl + cr) * BM;
                const int kb0 = (u / (tiles_n * tiles_m)) * ep.kb_per_split;
                const int num_kb = min(num_kb_total, kb0 + ep.kb_per_split) - kb0;
                for (int i = 0; i < num_kb; ++i, ++it) {
                    const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
                    mbar_wait(&empty_bar[s], ph ^ 1u);
                    TRACE(0, it);
                    const uint32_t base = smem_u32(smem + s * STAGE_BYTES);
                    const int k = (kb0 + i) * BK;
                    mbar_arrive_expect_tx(&full_bar[s], STAGE_BYTES);      // A + the whole B tile (own half + the peer's)
                    if (ep.a_mn) tma_load_mn(base, &maps.a, k, m0, &full_bar[s]);
                    else tma_load_pair(base, &maps.a, k, m0, &full_bar[s]);
                    if (ep.b_mn) {
                        tma_load_mn(base + 2 * TILE_BYTES, &maps.b, k, n0, &full_bar[s]);
                    } else if (cl == 2) {
                        const uint32_t off = (uint32_t)cr * (TILE_BYTES / 2);
                        tma_load_3d_mc(base + 2 * TILE_BYTES + off, &maps.b_half, k, n0 + cr * (BN / 2), 0, &full_bar[s], cl_mask);
                        tma_load_3d_mc(base + 3 * TILE_BYTES + off, &maps.b_half, k, n0 + cr * (BN / 2), 1, &full_bar[s], cl_mask);
                    } else {
                        tma_load_pair(base + 2 * TILE_BYTES, &maps.b, k, n0, &full_bar[s]);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one thread =====
        if (lane == 0) {
            uint32_t it = 0, seg = 0;              // ring position; K segments issued so far (TMEM buffer)
            for (int u = u_first; u < units; u += u_step) {
                const int kb0 = (u / (tiles_n * tiles_m)) * ep.kb_per_split;
                const int num_kb = min(num_kb_total, kb0 + ep.kb_per_split) - kb0;
                for (int i0 = 0; i0 < num_kb; i0 += ep.seg_kb, ++seg) {
                    const uint32_t buf = seg & 1u, use = seg >> 1;
                    mbar_wait(&tempty_bar[buf], (use & 1u) ^ 1u);      // the epilogue has drained this buffer
                    tc_fence_after();
                    const uint32_t d_big = tmem_base + buf * 256u, d_small = d_big + 128u;
                    const int i1 = min(num_kb, i0 + ep.seg_kb);
                    for (int i = i0; i < i1; ++i, ++it) {
                        const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
                        mbar_wait(&full_bar[s], ph);
                        TRACE(1, it);
                        tc_fence_after();
                        const uint32_t base = smem_u32(smem + s * STAGE_BYTES);
                        const uint64_t a_hi = ep.a_mn ? make_smem_desc_mn(base) : make_smem_desc(base);
                        const uint64_t a_lo = ep.a_mn ? make_smem_desc_mn(base + TILE_BYTES) : make_smem_desc(base + TILE_BYTES);
                        const uint64_t b_hi = ep.b_mn ? make_smem_desc_mn(base + 2 * TILE_BYTES) : make_smem_desc(base + 2 * TILE_BYTES);
                        // per k-step of 8: 32 bytes along a K-major row, 8 rows of 128 bytes in an MN-major tile
                        const uint64_t step_a = ep.a_mn ? (8 * 128) >> 4 : (8 * 4) >> 4, step_b = ep.b_mn ? (8 * 128) >> 4 : (8 * 4) >> 4;
                        const uint32_t id_big = idesc_tf32(2 * BN, ep.a_mn, ep.b_mn), id_small = idesc_tf32(BN, ep.a_mn, ep.b_mn);
#pragma unroll
                        for (int k = 0; k < ((ep.dbg & 4) ? 0 : BK / 8); ++k) {
                            const uint32_t acc = (i > i0 || k > 0) ? 1u : 0u;
                            // [big | small] (+)= A_hi [B_hi ; B_lo]^T, then small += A_lo B_hi^T
                            tc_mma_tf32(d_big, a_hi + k * step_a, b_hi + k * step_b, id_big, acc);
                            tc_mma_tf32(d_small, a_lo + k * step_a, b_hi + k * step_b, id_small, 1u);
                        }
                        // the stage is free once these MMAs have read it -- in cluster mode the peer must know too
                        if (cl == 2) tc_commit_mc(&empty_bar[s], cl_mask);
                        else tc_commit(&empty_bar[s]);
                    }
                    tc_commit(&tfull_bar[buf]);        // this segment's accumulators are complete
                }
            }
        }
    } else {
        // ===== epilogue: warp w may touch TMEM lanes [32*(w%4), +32); two warps per quarter, 64 columns each =====
        // Results leave through shared memory and TMA stores (32 x 32 fp32 tiles in the 128-byte swizzle);
        // the TMA clips rows >= M and columns >= N.
        const int ew = warp - 2, q = warp & 3, half = ew >> 2;
        uint8_t* stg = stg_base + ew * STG_BYTES;
        const uint32_t stg_u32 = smem_u32(stg);
        const int sw = lane & 7;                                  // swizzle phase of this thread's row
        uint32_t seg = 0;
        bool store_pending = false;
        for (int u = u_first; u < units; u += u_step) {
            const int n0 = (u % tiles_n) * BN, m0 = (((u / tiles_n) % tiles_m) * cl + cr) * BM;
            const int kb0 = (u / (tiles_n * tiles_m)) * ep.kb_per_split;
            const int num_kb = min(num_kb_total, kb0 + ep.kb_per_split) - kb0;
            float v[NCH][32];
            for (int i0 = 0; i0 < num_kb; i0 += ep.seg_kb, ++seg) {
                const uint32_t buf = seg & 1u, use = seg >> 1;
                mbar_wait(&tfull_bar[buf], use & 1u);
                if (warp == 2 && lane == 0) TRACE(2, seg);
                tc_fence_after();
                const uint32_t tb = tmem_base + buf * 256u + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * (BN / 2));
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    float big[32];
                    tc_ld32(tb + c * 32, big);
                    {
                        float small[32];
                        tc_ld32(tb + 128 + c * 32, small);
#pragma unroll
                        for (int j = 0; j < 32; ++j) big[j] += small[j];
                    }
                    if (i0 == 0) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[c][j] = big[j];
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[c][j] += big[j];
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty_bar[buf]);
            }
            const int row = m0 + q * 32 + lane;
            const bool row_ok = row < ep.M;
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                const int col0 = n0 + half * (BN / 2) + c * 32;
                if (col0 >= ep.N || (ep.dbg & 1)) break;           // warp-uniform
                float* vv = v[c];
                if (ep.bias) {
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (col0 + j < ep.N) vv[j] += __ldg(ep.bias + col0 + j);
                }
                if (ep.act == ACT_RELU) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) vv[j] = fmaxf(vv[j], 0.f);
                } else if (ep.act == ACT_SIGMOID) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) vv[j] = 1.f / (1.f + expf(-vv[j]));
                }
                if (ep.mask && row_ok) {
                    const float* mrow = ep.mask + (int64_t)row * ep.ld_mask + col0;
                    if (col0 + 32 <= ep.ld_mask) {                    // rows are 16-byte aligned (ld multiple of 4)
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            const float4 mk = __ldg(reinterpret_cast<const float4*>(mrow + j));
                            if (!(mk.x > 0.f)) vv[j] = 0.f;
                            if (!(mk.y > 0.f)) vv[j + 1] = 0.f;
                            if (!(mk.z > 0.f)) vv[j + 2] = 0.f;
                            if (!(mk.w > 0.f)) vv[j + 3] = 0.f;
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (col0 + j < ep.N && !(__ldg(mrow + j) > 0.f)) vv[j] = 0.f;
                    }
                }
                const int r0 = m0 + q * 32;
                // one staging tile per warp: wait until the previous store has read it, fill, fence, store
                auto stage_begin = [&]() {
                    if (store_pending) {
                        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                        __syncwarp();
                    }
                };
                auto stage_end = [&](const CUtensorMap* map, int c0, int c1, bool reduce) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) {
                        if (reduce) tma_reduce_add_2d(map, stg_u32, c0, c1);
                        else tma_store_2d(map, stg_u32, c0, c1);
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    store_pending = true;
                };
                float4* t_row = reinterpret_cast<float4*>(stg + lane * 128);
                if (ep.out_c) {
                    stage_begin();
#pragma unroll
                    for (int j = 0; j < 8; ++j) t_row[j ^ sw] = make_float4(vv[4 * j], vv[4 * j + 1], vv[4 * j + 2], vv[4 * j + 3]);
                    stage_end(&maps.c, col0, r0, ep.out_c == 2);
                }
                // hi / lo are recomputed per output instead of being kept (register pressure at BN = 256)
                auto hi_of = [&](int j) { return tf32_hi(vv[j]); };
                auto lo_of = [&](int j) { return tf32_lo(vv[j], tf32_hi(vv[j])); };
                if (ep.out_split) {
                    stage_begin();
#pragma unroll
                    for (int j = 0; j < 8; ++j) t_row[j ^ sw] = make_float4(hi_of(4 * j), hi_of(4 * j + 1), hi_of(4 * j + 2), hi_of(4 * j + 3));
                    stage_end(&maps.c_hi, col0, r0, false);
                    stage_begin();
#pragma unroll
                    for (int j = 0; j < 8; ++j) t_row[j ^ sw] = make_float4(lo_of(4 * j), lo_of(4 * j + 1), lo_of(4 * j + 2), lo_of(4 * j + 3));
                    stage_end(&maps.c_lo, col0, r0, false);
                }
                if (ep.colsum && r0 < ep.M) {
                    // column sums over this warp's 32 rows: a butterfly reduce-scatter that halves the columns a
                    // lane keeps at every step, so that lane j ends with the sum of column col0 + j
                    if (!row_ok) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) vv[j] = 0.f;
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        const bool upper = (lane & o) != 0;
#pragma unroll
                        for (int j = 0; j < o; ++j) {
                            const float send = upper ? vv[j] : vv[j + o];
                            const float keep = upper ? vv[j + o] : vv[j];
                            vv[j] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                        }
                    }
                    if (col0 + lane < ep.N) ep.colsum[(int64_t)(r0 >> 5) * ep.N + col0 + lane] = vv[0];
                }
            }
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        __syncwarp();
        if (warp == 2 && lane == 0) TRACE(3, 1);
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
    if (cl == 2) cluster_sync_all();        // the peer's last commits arrive on my barriers: stay until it is done too
}

// ------------------------------------------------------------------------------------
// split: dst = f(src) as hi/lo TF32 pairs, row-major [rows, ld_o]; f is the identity or the
// activation derivative applied to an upstream gradient (relu': src * (y > 0), sigmoid':
// src * y * (1 - y)).  With colsum: the sums of dst over each 32-row block, colsum[(r / 32) * cols + c]
// (the bias gradient's partial sums when dst is a gradient w.r.t. a pre-activation).
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) split_kernel(const float* __restrict__ src, int64_t lds, int rows, int cols,
                                                    const float* __restrict__ y, int64_t ldy, int dmode,
                                                    float* __restrict__ hi, float* __restrict__ lo, int64_t ld_o,
                                                    float* __restrict__ colsum) {
    pdl_enter();
    __shared__ float s_sum[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = r0 + ty + 8 * i, c = c0 + tx;
        if (r < rows && c < cols) {
            float v = src[(int64_t)r * lds + c];
            if (dmode == ACT_RELU) v = y[(int64_t)r * ldy + c] > 0.f ? v : 0.f;
            else if (dmode == ACT_SIGMOID) { const float p = y[(int64_t)r * ldy + c]; v = v * p * (1.f - p); }
            const float h = tf32_hi(v);
            hi[(int64_t)r * ld_o + c] = h;
            lo[(int64_t)r * ld_o + c] = tf32_lo(v, h);
            sum += v;
        }
    }
    if (!colsum) return;                                          // kernel-uniform
    s_sum[ty][tx] = sum;
    __syncthreads();
    if (ty == 0 && c0 + tx < cols) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += s_sum[i][tx];
        colsum[(int64_t)blockIdx.y * cols + c0 + tx] = t;
    }
}

// all weight matrices of one MLP in ONE launch (they change together, at the optimizer step)
constexpr int MAX_LAYERS = 8;
struct SplitJob {
    const float* src; int64_t lds; int rows, cols;
    float *hi, *lo; int64_t ld_o;
    int tiles_x, tile0;          // 32 x 32 tiles per row of tiles, first global tile of this job
    const float* grad;           // SGD fused in front of the split: src <- src - lr * grad (dense, row stride lds); or null
};
struct SplitBatch {
    SplitJob job[MAX_LAYERS];
    int n;
    float lr;
    const float* d_lr;           // split_batch_kernel<true>: the learning rate is *d_lr, read after griddepcontrol.wait
    // trailing blocks (blockIdx.x >= tiles): plain SGD on a vector that needs no split (the biases)
    int tiles;
    float* vec; const float* vec_grad; int64_t vec_n;
};
template <bool DLR>
__global__ void __launch_bounds__(256) split_batch_kernel(const __grid_constant__ SplitBatch sb) {
    pdl_enter();
    float lr = sb.lr;
    if constexpr (DLR) lr = *sb.d_lr;
    if (sb.vec && (int)blockIdx.x >= sb.tiles) {
        const int64_t i = (int64_t)((int)blockIdx.x - sb.tiles) * 256 + threadIdx.x;
        if (i < sb.vec_n) sb.vec[i] = fmaf(-lr, sb.vec_grad[i], sb.vec[i]);
        return;
    }
    int j = 0;
#pragma unroll 1
    while (j + 1 < sb.n && (int)blockIdx.x >= sb.job[j + 1].tile0) ++j;
    const SplitJob& jb = sb.job[j];
    const int tile = blockIdx.x - jb.tile0;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int r0 = (tile / jb.tiles_x) * 32, c0 = (tile % jb.tiles_x) * 32;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = r0 + ty + 8 * i, c = c0 + tx;
        if (r < jb.rows && c < jb.cols) {
            float v = jb.src[(int64_t)r * jb.lds + c];
            if (jb.grad) {
                v = fmaf(-lr, jb.grad[(int64_t)r * jb.lds + c], v);
                const_cast<float*>(jb.src)[(int64_t)r * jb.lds + c] = v;
            }
            const float h = tf32_hi(v);
            jb.hi[(int64_t)r * jb.ld_o + c] = h;
            jb.lo[(int64_t)r * jb.ld_o + c] = tf32_lo(v, h);
        }
    }
}

// dW [N, K] of every layer out of the padded split-K accumulators and db [N] out of the partial column
// sums [parts, N] of dZ, ONE launch.  The first db_blocks blocks reduce 32 bias columns each (8 row groups of
// threads, then the 8 group sums in order: a fixed summation order, the same result on every run); the
// others copy dW.
struct UnpackJob {
    const float* acc; int64_t ldp; int N, K;
    float *dW, *db;
    const float* dbp;            // [parts, N] partial column sums of dZ
    int64_t e0;                  // first global dW element of this job
    int c0;                      // first global bias column of this job
};
struct UnpackBatch {
    UnpackJob job[MAX_LAYERS];
    int n;
    int64_t total;               // dW elements of all jobs
    int columns, parts;          // bias columns of all jobs; partial sums per column
    int db_blocks;
};
__global__ void __launch_bounds__(256) unpack_batch_kernel(const __grid_constant__ UnpackBatch ub) {
    pdl_enter();
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    if ((int)blockIdx.x < ub.db_blocks) {
        __shared__ float s_sum[8][33];
        const int gc = blockIdx.x * 32 + tx;
        int j = 0;
#pragma unroll 1
        while (j + 1 < ub.n && gc >= ub.job[j + 1].c0) ++j;
        const UnpackJob& jb = ub.job[j];
        const int c = gc - jb.c0;
        float t = 0.f;
        if (gc < ub.columns)
            for (int p = ty; p < ub.parts; p += 8) t += jb.dbp[(int64_t)p * jb.N + c];
        s_sum[ty][tx] = t;
        __syncthreads();
        if (ty == 0 && gc < ub.columns) {
            t = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) t += s_sum[i][tx];
            jb.db[c] = t;
        }
        return;
    }
    const int64_t stride = (int64_t)(gridDim.x - ub.db_blocks) * blockDim.x;
    for (int64_t i = (blockIdx.x - ub.db_blocks) * (int64_t)blockDim.x + threadIdx.x; i < ub.total; i += stride) {
        int j = 0;
#pragma unroll 1
        while (j + 1 < ub.n && i >= ub.job[j + 1].e0) ++j;
        const UnpackJob& jb = ub.job[j];
        const int64_t e = i - jb.e0;
        const int n = (int)(e / jb.K), k = (int)(e - (int64_t)n * jb.K);
        jb.dW[(int64_t)n * jb.K + k] = jb.acc[(int64_t)n * jb.ldp + k];
    }
}

// ------------------------------------------------------------------------------------
// Narrow last layer (ONE output column: the click probability of the top MLP, 256 -> 1).
// On the tensor-core path a 128 x 128 tile would carry one useful column (forward, data
// gradient) or one useful row (weight gradient): three GEMM launches plus a split for 4 MFLOP.
// Forward is a row-wise dot product, backward an outer product and a column reduction: SIMT,
// HBM-bound on the activations, FP32 throughout (x = x_hi + x_lo to 2^-22).
// ------------------------------------------------------------------------------------
__device__ __forceinline__ float act_apply(float z, int act) {
    if (act == ACT_RELU) return z > 0.f ? z : 0.f;
    if (act == ACT_SIGMOID) return 1.f / (1.f + expf(-z));
    return z;
}
__device__ __forceinline__ float act_grad(float dy, float y, int act) {
    if (act == ACT_RELU) return y > 0.f ? dy : 0.f;
    if (act == ACT_SIGMOID) return dy * y * (1.f - y);
    return dy;
}

// y[r] = act(sum_k x[r, k] W[k] + bias); one warp per row; written to the workspace copy (backward reads it)
// and to the caller's output
__global__ void __launch_bounds__(256) narrow_fwd_kernel(const float* __restrict__ x_hi, const float* __restrict__ x_lo,
                                                         int64_t ldx, int rows, int K, const float* __restrict__ W,
                                                         const float* __restrict__ bias, int act,
                                                         float* __restrict__ y_ws, int64_t ld_ws,
                                                         float* __restrict__ y, int64_t ldy) {
    pdl_enter();
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= rows) return;
    const float* h = x_hi + (int64_t)r * ldx;
    const float* l = x_lo + (int64_t)r * ldx;
    float acc = 0.f;
    const int K4 = ((uintptr_t)W & 15) == 0 ? (K & ~3) : 0;       // rows of x are 16-byte aligned (padded ld)
    for (int k = lane * 4; k < K4; k += 128) {
        const float4 a = *reinterpret_cast<const float4*>(h + k), b = *reinterpret_cast<const float4*>(l + k);
        const float4 w = __ldg(reinterpret_cast<const float4*>(W + k));
        acc = fmaf(a.x + b.x, w.x, acc); acc = fmaf(a.y + b.y, w.y, acc);
        acc = fmaf(a.z + b.z, w.z, acc); acc = fmaf(a.w + b.w, w.w, acc);
    }
    for (int k = K4 + lane; k < K; k += 32) acc = fmaf(h[k] + l[k], __ldg(W + k), acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
        const float v = act_apply(acc + __ldg(bias), act);
        y_ws[(int64_t)r * ld_ws] = v;
        y[(int64_t)r * ldy] = v;
    }
}

// g[r] = dy[r] * act'(y[r]);  dwp[k] += sum_r g[r] x[r, k] (weight gradient, split over row chunks, atomics into the
// zeroed accumulator);  dbp[r / 32] = sum of g over each 32-row block (bias gradient partials);  dZ[r, k] =
// g[r] W[k] * (x[r, k] > 0) as hi/lo split (the operands of the layer below) with its column sums per 32 rows in
// colsum[(r / 32) * K + k], or plain FP32 into dx when this is layer 0.
// Block = 32 columns x NARROW_ROWS rows (32 x 32 sub-tiles), 32 x 8 threads.
constexpr int NARROW_ROWS = 64;     // 8 x 128 CTAs at batch 8192, K = 256 (32 x 128 rows left half the SMs idle: ncu 18 us)
constexpr int NARROW_SUBS = NARROW_ROWS / 32;
__global__ void __launch_bounds__(256) narrow_bwd_kernel(const float* __restrict__ dy, int64_t lddy,
                                                         const float* __restrict__ y, int64_t ldy, int act,
                                                         const float* __restrict__ x_hi, const float* __restrict__ x_lo,
                                                         int64_t ldx, int rows, int K, const float* __restrict__ W,
                                                         int relu_mask, float* __restrict__ g_hi, float* __restrict__ g_lo,
                                                         int64_t ld_o, float* __restrict__ colsum, float* __restrict__ dx,
                                                         int64_t lddx, float* __restrict__ dwp, float* __restrict__ dbp) {
    pdl_enter();
    __shared__ float s_sum[1 + NARROW_SUBS][8][33], s_g[NARROW_ROWS];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * NARROW_ROWS;
    if (threadIdx.x < NARROW_ROWS) {
        const int r = r0 + threadIdx.x;
        s_g[threadIdx.x] = r < rows ? act_grad(dy[(int64_t)r * lddy], y[(int64_t)r * ldy], act) : 0.f;
    }
    __syncthreads();
    const int c = c0 + tx;
    const float w = c < K ? __ldg(W + c) : 0.f;
    float wsum = 0.f;
#pragma unroll
    for (int sub = 0; sub < NARROW_SUBS; ++sub) {
        float dsum = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int rl = sub * 32 + ty + 8 * i, r = r0 + rl;
            if (r < rows && c < K) {
                const float g = s_g[rl];
                const float xh = x_hi[(int64_t)r * ldx + c];
                wsum = fmaf(g, xh + x_lo[(int64_t)r * ldx + c], wsum);
                float v = g * w;
                if (relu_mask) v = xh > 0.f ? v : 0.f;
                if (dx) dx[(int64_t)r * lddx + c] = v;
                if (g_hi) {
                    const float h = tf32_hi(v);
                    g_hi[(int64_t)r * ld_o + c] = h;
                    g_lo[(int64_t)r * ld_o + c] = tf32_lo(v, h);
                }
                dsum += v;
            }
        }
        s_sum[1 + sub][ty][tx] = dsum;
    }
    // column sums over the 8 row groups of threads, in order: warp 0 the weight gradient, warp 1 + sub the dZ
    // partials of sub-tile sub; warp 1 + NARROW_SUBS the bias gradient partials (one column block does that)
    s_sum[0][ty][tx] = wsum;
    __syncthreads();
    if (ty <= NARROW_SUBS && c < K) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += s_sum[ty][i][tx];
        if (ty == 0) atomicAdd(dwp + c, t);
        else if (colsum && r0 + (ty - 1) * 32 < rows) colsum[(int64_t)(r0 / 32 + ty - 1) * K + c] = t;
    }
    if (blockIdx.x == 0 && ty == 1 + NARROW_SUBS) {
#pragma unroll
        for (int sub = 0; sub < NARROW_SUBS; ++sub) {
            float t = s_g[sub * 32 + tx];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
            if (tx == 0 && r0 + sub * 32 < rows) dbp[r0 / 32 + sub] = t;
        }
    }
}

// ------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// Tensors are [rows, inner] fp32 with a row stride of ld elements (multiple of 4); out-of-range box elements read as
// zero and are not written.
// K-major operand pair: hi at `hi`, lo at `lo` (same shape and row stride, lo behind hi) as one {inner, rows, 2} tensor;
// box = BK x box_rows x 2, swizzle width = one BK row
int make_pair_map(CUtensorMap* m, const float* hi, const float* lo, int64_t inner, int64_t rows, int64_t ld, int box_rows,
                  int box_depth = 2) {
    EncodeTiledFn enc = get_encode();
    if (!enc) {
        cdlrm_set_error("cuTensorMapEncodeTiled is not available from the driver");
        return CDLRM_ERR_CUDA;
    }
    const int64_t gap = (const char*)lo - (const char*)hi;
    if (((uintptr_t)hi & 15) || (ld & 3) || inner <= 0 || rows <= 0 || gap < rows * ld * 4 || (gap & 15)) {
        cdlrm_set_error("operand pair must be 16-byte aligned, row stride multiple of 4, lo behind hi (hi %p lo %p ld %lld)", (const void*)hi,
                        (const void*)lo, (long long)ld);
        return CDLRM_ERR_ARG;
    }
    cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)rows, 2};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)gap};
    cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)box_rows, (cuuint32_t)box_depth};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)hi, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     BK == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        cdlrm_set_error("cuTensorMapEncodeTiled (pair) failed (%d): inner %lld rows %lld ld %lld gap %lld", (int)r, (long long)inner,
                        (long long)rows, (long long)ld, (long long)gap);
        return CDLRM_ERR_CUDA;
    }
    return CDLRM_OK;
}

// MN-major operand pair: row-major [rows = K, ld] with the MN index contiguous, hi at `hi`, lo behind it, as one
// 4-D tensor {32, K, MN / 32, 2} (strides ld, 32 elements, lo - hi) whose box {32, BK, 4, 2} is a 128-wide tile
// of BK rows in four 32-wide column blocks, in the 128-byte swizzle with 32-byte atoms (make_smem_desc_mn).  The row stride must cover the 32-wide column
// blocks (ld >= 32 * ceil(mn / 32)): elements mn .. of the last block are the row's padding, and only reach
// results at rows / columns >= mn, which the stores clip.
int make_mn_map(CUtensorMap* m, const float* hi, const float* lo, int64_t mn, int64_t rows, int64_t ld) {
    EncodeTiledFn enc = get_encode();
    if (!enc) {
        cdlrm_set_error("cuTensorMapEncodeTiled is not available from the driver");
        return CDLRM_ERR_CUDA;
    }
    const int64_t gap = (const char*)lo - (const char*)hi, blocks = (mn + 31) / 32;
    if (((uintptr_t)hi & 15) || (ld & 3) || mn <= 0 || rows <= 0 || ld < 32 * blocks || gap < rows * ld * 4 || (gap & 15)) {
        cdlrm_set_error("MN-major operand pair must be 16-byte aligned, row stride a multiple of 4 covering whole 32-wide "
                        "column blocks, lo behind hi (hi %p lo %p mn %lld ld %lld)", (const void*)hi, (const void*)lo,
                        (long long)mn, (long long)ld);
        return CDLRM_ERR_ARG;
    }
    cuuint64_t dims[4] = {32, (cuuint64_t)rows, (cuuint64_t)blocks, 2};
    cuuint64_t strides[3] = {(cuuint64_t)ld * 4, 128, (cuuint64_t)gap};
    cuuint32_t box[4] = {32, (cuuint32_t)BK, (cuuint32_t)(BM / 32), 2};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)hi, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        cdlrm_set_error("cuTensorMapEncodeTiled (MN-major pair) failed (%d): mn %lld rows %lld ld %lld gap %lld", (int)r,
                        (long long)mn, (long long)rows, (long long)ld, (long long)gap);
        return CDLRM_ERR_CUDA;
    }
    return CDLRM_OK;
}

// result map: box 32 x 32, 128-byte swizzle
int make_map(CUtensorMap* m, const float* base, int64_t inner, int64_t rows, int64_t ld) {
    EncodeTiledFn enc = get_encode();
    if (!enc) {
        cdlrm_set_error("cuTensorMapEncodeTiled is not available from the driver");
        return CDLRM_ERR_CUDA;
    }
    if (((uintptr_t)base & 15) || (ld & 3) || inner <= 0 || rows <= 0) {
        cdlrm_set_error("tensor map operand must be 16-byte aligned with a row stride multiple of 4 (base %p ld %lld)", (const void*)base, (long long)ld);
        return CDLRM_ERR_ARG;
    }
    cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        cdlrm_set_error("cuTensorMapEncodeTiled failed (%d): inner %lld rows %lld ld %lld", (int)r, (long long)inner, (long long)rows, (long long)ld);
        return CDLRM_ERR_CUDA;
    }
    return CDLRM_OK;
}

// where the result of a GEMM goes
struct Out {
    float* c = nullptr;          // fp32 [M, N] row-major
    int64_t ldc = 0;
    bool reduce = false;         // add into c (split-K) instead of storing
    float* c_hi = nullptr;       // hi/lo split [M, N] row-major
    float* c_lo = nullptr;
    int64_t ld_split = 0;
};

int g_narrow = 1;    // 1: a last layer with one output column runs on the SIMT narrow kernels; cdlrm_mlp_set_option(2, .)
// 2: CTA pairs share their B tiles through TMA multicast where the m tile count is even (cdlrm_mlp_set_option(4, .)).
// Parity-green but measured 5 % SLOWER on B200 (tools/gemm_cluster_ab.py: 34.7 vs 32.8 us for 8192 x 512 x 512, top MLP
// 335 vs 323 us): the multicast cuts L2 -> SM traffic by 25 % but every CTA still receives its 64 KB per k-block, so the
// shared-memory write + operand-read bandwidth that bounds the mainloop is unchanged and the pair now runs in lockstep.
int g_cluster = 1;
int g_wgrad_side = 1;   // 1: weight-gradient GEMMs run on a side stream beside the dgrad chain; cdlrm_mlp_set_option(5, .)
int g_seg_kb = 8;    // K segment (k-blocks of 32) per TMEM accumulation chain; cdlrm_mlp_set_option(1, .)
int g_num_sms = 0;
int g_dbg = 0;
long long* g_trace = nullptr;

// A and B as hi/lo pairs with row stride lda / ldb: K-major unless ep.a_mn / ep.b_mn
int launch_gemm(const float* a_hi, const float* a_lo, int64_t lda, const float* b_hi, const float* b_lo, int64_t ldb,
                Epi ep, const Out& o, int splits, cudaStream_t s) {
    if (!g_num_sms) {
        int dev = 0, n = 0;
        CU_CHECK(cudaGetDevice(&dev));
        CU_CHECK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
        g_num_sms = n > 0 ? n : 148;
    }
    CU_CHECK(cdlrm_smem_optin((const void*)gemm3x_tf32_kernel, GEMM_SMEM));
    const int64_t tiles_m = (ep.M + BM - 1) / BM, tiles_n = (ep.N + BN - 1) / BN;
    if (splits == 0) splits = (int)(g_num_sms / (tiles_m * tiles_n));      // split-K sized to one round of the persistent grid
    Maps mp;
    memset(&mp, 0, sizeof(mp));
    int rc;
    static_assert(BM == BN && BK == 32, "an MN-major tile is one box of four 32-wide column blocks of BK rows");
    if ((rc = ep.a_mn ? make_mn_map(&mp.a, a_hi, a_lo, ep.M, ep.K, lda) : make_pair_map(&mp.a, a_hi, a_lo, ep.K, ep.M, lda, BM))) return rc;
    if ((rc = ep.b_mn ? make_mn_map(&mp.b, b_hi, b_lo, ep.N, ep.K, ldb) : make_pair_map(&mp.b, b_hi, b_lo, ep.K, ep.N, ldb, BN))) return rc;
    ep.out_c = o.c ? (o.reduce ? 2 : 1) : 0;
    ep.out_split = o.c_hi ? 1 : 0;
    if (ep.out_c && ep.out_split) {
        cdlrm_set_error("a GEMM writes either the fp32 result or its hi/lo split row-major, not both");
        return CDLRM_ERR_ARG;
    }
    if (o.c && (rc = make_map(&mp.c, o.c, ep.N, ep.M, o.ldc))) return rc;
    if (o.c_hi) {
        if ((rc = make_map(&mp.c_hi, o.c_hi, ep.N, ep.M, o.ld_split))) return rc;
        if ((rc = make_map(&mp.c_lo, o.c_lo, ep.N, ep.M, o.ld_split))) return rc;
    }
    const int num_kb = (ep.K + BK - 1) / BK;
    if (splits < 1) splits = 1;
    if (splits > num_kb) splits = num_kb;
    ep.kb_per_split = (num_kb + splits - 1) / splits;
    splits = (num_kb + ep.kb_per_split - 1) / ep.kb_per_split;      // no empty split
    if (splits > 1 && ep.out_c != 2) {
        cdlrm_set_error("split-K needs the reduce-add output");
        return CDLRM_ERR_ARG;
    }
    ep.splits = splits;
    ep.dbg = g_dbg;
    ep.trace = g_trace;
    ep.seg_kb = g_seg_kb > 0 ? g_seg_kb * (32 / BK) : num_kb;      // the option counts k-blocks of 32
    // optional: CTA pairs along M share the B tile of every k-block (half each, multicast): 25 % less L2 -> SM traffic.
    // K-major B only (the half-tile map is K-major).
    ep.cluster = (g_cluster == 2 && !ep.b_mn && tiles_m % 2 == 0 && g_num_sms >= 2) ? 2 : 1;
    int grid;
    if (ep.cluster == 2) {
        if ((rc = make_pair_map(&mp.b_half, b_hi, b_lo, ep.K, ep.N, ldb, BN / 2, 1))) return rc;
        const int64_t pair_units = tiles_n * (tiles_m / 2) * splits;
        const int64_t pairs = pair_units < g_num_sms / 2 ? pair_units : g_num_sms / 2;
        grid = (int)(2 * pairs);
    } else {
        const int64_t units = tiles_n * tiles_m * splits;
        grid = (int)(units < g_num_sms ? units : g_num_sms);
    }
    cdlrm_prof_mark(K_MLP_GEMM, s, 0);
    cdlrm_launch_pdl_cluster(gemm3x_tf32_kernel, dim3(grid), dim3(GEMM_THREADS), GEMM_SMEM, s, ep.cluster, mp, ep);
    cdlrm_prof_mark(K_MLP_GEMM, s, 1);
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

int launch_split(const float* src, int64_t lds, int rows, int cols, const float* y, int64_t ldy, int dmode, float* hi,
                 float* lo, int64_t ld_o, float* colsum, cudaStream_t s) {
    if (rows <= 0 || cols <= 0) return CDLRM_OK;
    dim3 grid((cols + 31) / 32, (rows + 31) / 32);
    LAUNCH_PDL(K_MLP_SPLIT, s, split_kernel, grid, 256, 0, src, lds, rows, cols, y, ldy, dmode, hi, lo, ld_o, colsum);
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

inline int64_t pad4(int64_t v) { return (v + 3) & ~(int64_t)3; }
// row stride of the hi/lo splits of weights, activations and gradients: whole 32-wide blocks, so that every
// MN-major box stays inside its row (make_mn_map)
inline int64_t pad32(int64_t v) { return (v + 31) & ~(int64_t)31; }
inline int64_t parts32(int64_t rows) { return (rows + 31) / 32; }
inline int64_t align256(int64_t v) { return (v + 255) & ~(int64_t)255; }

}  // namespace

// One MLP (bottom or top): dims[0..L], batch capacity, the layer that ends in a sigmoid.
// Workspace carve-up (all fp32, every region 256-byte aligned):
//   per layer l:  w_hi/w_lo [N_l, pad32(K_l)]
//   per level i = 0..L (activation entering layer i; level L is the output):
//        x_hi/x_lo [cap, pad32(D_i)]   (i < L)
//        g_hi/g_lo [cap, pad32(D_i)]   (i > 0, gradient w.r.t. the pre-activation)
//   y_out [cap, pad4(D_L)]  fp32 output of the last layer (activation derivative input)
//   per layer l:  dwp [N_l, pad4(K_l)]  split-K accumulator of dW (back to back: one memset)
//   per layer l:  dbp [ceil(cap / 32), N_l]  column sums of g_{l+1} per 32 rows (db partials)
// The weight-gradient GEMM reads g and x MN-major and the data-gradient GEMM reads w MN-major: no
// transposed copy of any of them exists.
struct cdlrm_mlp {
    int device = 0;
    int L = 0;
    int cap = 0;
    int sigmoid_layer = -1;
    std::vector<int> D;
    std::vector<float*> w_hi, w_lo;
    std::vector<float*> x_hi, x_lo, g_hi, g_lo;
    std::vector<float*> dwp;     // per layer: split-K accumulator [N_l, pad4(K_l)]
    std::vector<float*> dbp;     // per layer: partial bias gradients [ceil(cap / 32), N_l]
    float* y_out = nullptr;
    int64_t dwp_bytes = 0;       // the dwp regions are carved back to back
    int last_batch = 0;
    bool last_narrow = false;    // the last forward ran its final layer on the narrow kernels
    const float* last_W = nullptr;   // FP32 weights of that layer (the narrow backward reads them)
    bool w_presplit = false;     // cdlrm_mlp_sgd_split left the splits of the CURRENT weights behind: the next forward skips its own
    int num_sms = 148;
    // weight-gradient GEMMs on a stream of their own beside the data-gradient chain (cdlrm_mlp_backward)
    cudaStream_t s2 = nullptr;
    cudaEvent_t ev_g = nullptr, ev_done = nullptr;
    bool defer_join = false;     // cdlrm_mlp_set_defer_join: the caller joins with cdlrm_mlp_join
    bool pending_join = false;
};

static int64_t mlp_carve(cdlrm_mlp* m, char* base) {
    int64_t off = 0;
    auto take = [&](int64_t elems) {
        float* p = base ? reinterpret_cast<float*>(base + off) : nullptr;
        off += align256(elems * 4);
        return p;
    };
    const int L = m->L;
    const int64_t cap = m->cap;
    m->w_hi.assign(L, nullptr); m->w_lo.assign(L, nullptr);
    for (int l = 0; l < L; ++l) {
        const int64_t K = m->D[l], N = m->D[l + 1];
        m->w_hi[l] = take(N * pad32(K)); m->w_lo[l] = take(N * pad32(K));
    }
    m->x_hi.assign(L + 1, nullptr); m->x_lo.assign(L + 1, nullptr);
    m->g_hi.assign(L + 1, nullptr); m->g_lo.assign(L + 1, nullptr);
    for (int i = 0; i <= L; ++i) {
        const int64_t Di = m->D[i];
        if (i < L) { m->x_hi[i] = take(cap * pad32(Di)); m->x_lo[i] = take(cap * pad32(Di)); }
        if (i > 0) { m->g_hi[i] = take(cap * pad32(Di)); m->g_lo[i] = take(cap * pad32(Di)); }
    }
    m->y_out = take(cap * pad4(m->D[L]));
    m->dwp.assign(L, nullptr);
    const int64_t dwp0 = off;
    for (int l = 0; l < L; ++l) m->dwp[l] = take((int64_t)m->D[l + 1] * pad4(m->D[l]));
    m->dwp_bytes = off - dwp0;
    m->dbp.assign(L, nullptr);
    for (int l = 0; l < L; ++l) m->dbp[l] = take(parts32(cap) * m->D[l + 1]);
    return off;
}

extern "C" int64_t cdlrm_mlp_workspace_bytes(int n_layers, const int32_t* h_dims, int32_t batch_cap) {
    if (n_layers < 1 || n_layers > MAX_LAYERS || !h_dims || batch_cap < 1) return -1;
    cdlrm_mlp m;
    m.L = n_layers;
    m.cap = batch_cap;
    m.D.assign(h_dims, h_dims + n_layers + 1);
    for (int v : m.D)
        if (v < 1) return -1;
    return mlp_carve(&m, nullptr);
}

extern "C" int cdlrm_mlp_create(cdlrm_mlp** out, int device, int n_layers, const int32_t* h_dims, int32_t batch_cap,
                                int sigmoid_layer, void* workspace, int64_t workspace_bytes) {
    ARG_CHECK(out && h_dims && workspace);
    ARG_CHECK(n_layers >= 1 && n_layers <= MAX_LAYERS && batch_cap >= 1);
    ARG_CHECK(((uintptr_t)workspace & 255) == 0);
    CU_CHECK(cudaSetDevice(device));
    cdlrm_mlp* m = new cdlrm_mlp();
    m->device = device;
    m->L = n_layers;
    m->cap = batch_cap;
    m->sigmoid_layer = sigmoid_layer;
    m->D.assign(h_dims, h_dims + n_layers + 1);
    for (int v : m->D) {
        if (v < 1) {
            delete m;
            cdlrm_set_error("layer width must be positive");
            return CDLRM_ERR_ARG;
        }
    }
    const int64_t need = mlp_carve(m, (char*)workspace);
    if (need > workspace_bytes) {
        delete m;
        cdlrm_set_error("MLP workspace too small: %lld < %lld bytes", (long long)workspace_bytes, (long long)need);
        return CDLRM_ERR_ARG;
    }
    if (cudaDeviceGetAttribute(&m->num_sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || m->num_sms <= 0) m->num_sms = 148;
    {   // side stream of the weight-gradient GEMMs (created here, not lazily: the first backward may be under capture)
        int lo = 0, hi = 0;
        if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess ||
            cudaStreamCreateWithPriority(&m->s2, cudaStreamNonBlocking, hi) != cudaSuccess ||
            cudaEventCreateWithFlags(&m->ev_g, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&m->ev_done, cudaEventDisableTiming) != cudaSuccess) {
            cudaGetLastError();
            m->s2 = nullptr;        // no device (CPU-only build check) or out of resources: in-line weight gradients
        }
    }
    *out = m;
    return CDLRM_OK;
}

// key 4: CTAs per cluster along M (2 = pairs multicast their shared B tiles; 1 = no clusters, default: faster)
// key 2: 1 (default) = a last layer with a single output column uses the SIMT narrow kernels, 0 = tensor-core GEMMs
// key 0: split rounding (0 = round to nearest, 1 = truncate); key 1: k-blocks (of 32) chained into one TMEM
// accumulator before the partial result is added in registers (0 = the whole K; default 8)
extern "C" int cdlrm_mlp_set_option(int key, int value) {
    if (key == 0) {
        const int v = value ? 1 : 0;
        CU_CHECK(cudaMemcpyToSymbol(g_split_trunc, &v, sizeof(int)));
    } else if (key == 1) {
        ARG_CHECK(value >= 0 && value <= 4096);
        g_seg_kb = value;
    } else if (key == 2) {
        g_narrow = value ? 1 : 0;
    } else if (key == 4) {
        ARG_CHECK(value == 1 || value == 2);
        g_cluster = value;
    } else if (key == 3) {
        g_dbg = value;
    } else if (key == 5) {
        g_wgrad_side = value ? 1 : 0;
    } else {
        ARG_CHECK(false && "unknown option");
    }
    return CDLRM_OK;
}

// measurement hook: device buffer of 4 x 128 int64 that CTA 0 of every following GEMM fills with
// %globaltimer stamps (0: TMA issue per k-block, 1: operands landed per k-block, 2: accumulator
// ready per K segment, 3: [0] prologue done, [1] last store done); null switches it off
extern "C" int cdlrm_mlp_set_trace(void* d_buf) {
    g_trace = reinterpret_cast<long long*>(d_buf);
    return CDLRM_OK;
}

extern "C" int cdlrm_mlp_destroy(cdlrm_mlp* m) {
    if (m) {
        if (m->s2) { cudaStreamSynchronize(m->s2); cudaStreamDestroy(m->s2); }
        if (m->ev_g) cudaEventDestroy(m->ev_g);
        if (m->ev_done) cudaEventDestroy(m->ev_done);
    }
    delete m;
    return CDLRM_OK;
}

extern "C" int cdlrm_mlp_set_defer_join(cdlrm_mlp* m, int on) {
    ARG_CHECK(m);
    m->defer_join = on != 0;
    return CDLRM_OK;
}

extern "C" int cdlrm_mlp_join(cdlrm_mlp* m, cdlrm_stream stream) {
    ARG_CHECK(m);
    if (m->pending_join) {
        CU_CHECK(cudaStreamWaitEvent((cudaStream_t)stream, m->ev_done, 0));
        m->pending_join = false;
    }
    return CDLRM_OK;
}

// SGD step of the weight matrices of up to two MLPs fused with the hi/lo split of the UPDATED weights, plus plain SGD on one extra vector (the biases): ONE launch instead of the optimizer's axpy and one
// split launch at the head of each forward -- which sat on the critical path of the step (before the bottom MLP's
// first GEMM, and between the interaction and the top MLP).  DLR: the learning rate is *d_lr (device), not lr.
template <bool DLR>
static int sgd_split_launch(int n_mlps, cdlrm_mlp* const* mlps, float* const* h_W, const float* const* h_dW, float lr,
                            const float* d_lr, float* vec, const float* vec_grad, int64_t vec_n, cdlrm_stream stream) {
    ARG_CHECK(n_mlps >= 1 && n_mlps <= 2 && mlps && h_W && h_dW && vec_n >= 0 && (vec_n == 0 || (vec && vec_grad)));
    ARG_CHECK(!DLR || d_lr);
    cudaStream_t s = (cudaStream_t)stream;
    SplitBatch sb = {};
    int tiles = 0, j = 0;
    for (int a = 0; a < n_mlps; ++a) {
        cdlrm_mlp* m = mlps[a];
        ARG_CHECK(m);
        for (int l = 0; l < m->L; ++l, ++j) {
            ARG_CHECK(j < MAX_LAYERS && h_W[j] && h_dW[j]);
            const int K = m->D[l], N = m->D[l + 1];
            SplitJob& jb = sb.job[j];
            jb.src = h_W[j]; jb.grad = h_dW[j]; jb.lds = K; jb.rows = N; jb.cols = K;
            jb.hi = m->w_hi[l]; jb.lo = m->w_lo[l]; jb.ld_o = pad32(K);
            jb.tiles_x = (K + 31) / 32; jb.tile0 = tiles;
            tiles += jb.tiles_x * ((N + 31) / 32);
        }
    }
    CU_CHECK(cudaSetDevice(mlps[0]->device));
    sb.n = j;
    sb.lr = lr;
    sb.d_lr = d_lr;
    sb.tiles = tiles;
    sb.vec = vec_n ? vec : nullptr; sb.vec_grad = vec_grad; sb.vec_n = vec_n;
    const int blocks = tiles + (int)((vec_n + 255) / 256);
    LAUNCH_PDL(K_MLP_SPLIT, s, split_batch_kernel<DLR>, blocks, 256, 0, sb);
    CU_CHECK(cudaGetLastError());
    for (int a = 0; a < n_mlps; ++a) mlps[a]->w_presplit = true;
    return CDLRM_OK;
}

extern "C" int cdlrm_mlp_sgd_split(int n_mlps, cdlrm_mlp* const* mlps, float* const* h_W, const float* const* h_dW, float lr,
                                   float* vec, const float* vec_grad, int64_t vec_n, cdlrm_stream stream) {
    return sgd_split_launch<false>(n_mlps, mlps, h_W, h_dW, lr, nullptr, vec, vec_grad, vec_n, stream);
}

extern "C" int cdlrm_mlp_sgd_split_dlr(int n_mlps, cdlrm_mlp* const* mlps, float* const* h_W, const float* const* h_dW,
                                       const float* d_lr, float* vec, const float* vec_grad, int64_t vec_n,
                                       cdlrm_stream stream) {
    return sgd_split_launch<true>(n_mlps, mlps, h_W, h_dW, 0.f, d_lr, vec, vec_grad, vec_n, stream);
}

// the weights were changed by something else than cdlrm_mlp_sgd_split: the next forward splits them again
extern "C" int cdlrm_mlp_invalidate_split(cdlrm_mlp* m) {
    ARG_CHECK(m);
    m->w_presplit = false;
    return CDLRM_OK;
}

extern "C" int cdlrm_mlp_forward(cdlrm_mlp* m, const float* x, int64_t ldx, int32_t batch, const float* const* h_W,
                                 const float* const* h_b, float* y, int64_t ldy, cdlrm_stream stream) {
    ARG_CHECK(m && x && h_W && h_b && y);
    ARG_CHECK(batch >= 0 && batch <= m->cap && ldx >= m->D[0] && ldy >= m->D[m->L]);
    if (batch == 0) return CDLRM_OK;
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(m->device));
    const int L = m->L;
    int rc;
    if (m->pending_join) {      // weight-gradient GEMMs of the last backward still read the activations
        CU_CHECK(cudaStreamWaitEvent(s, m->ev_done, 0));
        m->pending_join = false;
    }
    // weights: W [N,K] -> hi/lo (K-major for the forward, MN-major for the dgrad), all layers in one launch --
    // unless the optimizer step that produced these weights already did it (cdlrm_mlp_sgd_split)
    if (m->w_presplit) {
        for (int l = 0; l < L; ++l) ARG_CHECK(h_W[l] && h_b[l]);
        m->w_presplit = false;
    } else {
        SplitBatch sb = {};
        int tiles = 0;
        for (int l = 0; l < L; ++l) {
            ARG_CHECK(h_W[l] && h_b[l]);
            const int K = m->D[l], N = m->D[l + 1];
            SplitJob& jb = sb.job[l];
            jb.src = h_W[l]; jb.grad = nullptr; jb.lds = K; jb.rows = N; jb.cols = K;
            jb.hi = m->w_hi[l]; jb.lo = m->w_lo[l]; jb.ld_o = pad32(K);
            jb.tiles_x = (K + 31) / 32; jb.tile0 = tiles;
            tiles += jb.tiles_x * ((N + 31) / 32);
        }
        sb.n = L;
        sb.tiles = tiles;
        LAUNCH_PDL(K_MLP_SPLIT, s, split_batch_kernel<false>, tiles, 256, 0, sb);
        CU_CHECK(cudaGetLastError());
    }
    // input
    if ((rc = launch_split(x, ldx, batch, m->D[0], nullptr, 0, ACT_NONE, m->x_hi[0], m->x_lo[0], pad32(m->D[0]), nullptr, s))) return rc;
    for (int l = 0; l < L; ++l) {
        const int K = m->D[l], N = m->D[l + 1];
        Epi ep = {};
        Out o;
        ep.M = batch; ep.N = N; ep.K = K;
        ep.bias = h_b[l];
        ep.act = (l == m->sigmoid_layer) ? ACT_SIGMOID : ((m->sigmoid_layer == -2 && l == L - 1) ? ACT_NONE : ACT_RELU);
        if (l + 1 < L) {
            o.c_hi = m->x_hi[l + 1]; o.c_lo = m->x_lo[l + 1]; o.ld_split = pad32(N);
        } else {
            o.c = m->y_out; o.ldc = pad4(N);
        }
        if (l == L - 1 && N == 1 && g_narrow) {      // narrow last layer: row-wise dot products, writes y_out and y
            LAUNCH_PDL(K_MLP_SPLIT, s, narrow_fwd_kernel, (batch + 7) / 8, 256, 0, m->x_hi[l], m->x_lo[l], pad32(K), batch, K,
                       h_W[l], h_b[l], ep.act, m->y_out, pad4(N), y, ldy);
            CU_CHECK(cudaGetLastError());
            m->last_batch = batch;
            m->last_narrow = true;
            m->last_W = h_W[l];
            return CDLRM_OK;
        }
        if ((rc = launch_gemm(m->x_hi[l], m->x_lo[l], pad32(K), m->w_hi[l], m->w_lo[l], pad32(K), ep, o, 1, s))) return rc;
    }
    CU_CHECK(cudaMemcpy2DAsync(y, ldy * 4, m->y_out, pad4(m->D[L]) * 4, (size_t)m->D[L] * 4, batch, cudaMemcpyDeviceToDevice, s));
    m->last_batch = batch;
    m->last_narrow = false;
    return CDLRM_OK;
}

extern "C" int cdlrm_mlp_backward(cdlrm_mlp* m, const float* dy, int64_t lddy, float* dx, int64_t lddx, float* const* h_dW,
                                  float* const* h_db, cdlrm_stream stream) {
    ARG_CHECK(m && dy && h_dW && h_db);
    const int batch = m->last_batch;
    if (batch <= 0) {
        cdlrm_set_error("cdlrm_mlp_backward without a preceding forward");
        return CDLRM_ERR_STATE;
    }
    ARG_CHECK(lddy >= m->D[m->L] && (dx == nullptr || lddx >= m->D[0]));
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(m->device));
    const int L = m->L;
    int rc;
    if (m->pending_join) {      // a deferred join nobody asked for: the previous backward's dW must be complete
        CU_CHECK(cudaStreamWaitEvent(s, m->ev_done, 0));
        m->pending_join = false;
    }
    // The weight-gradient GEMMs are leaves of the backward: they run on a stream of their own, each behind the
    // event that marks its dZ ready, so that their CTAs fill the SMs the data-gradient chain (the critical path)
    // leaves idle at its tile-count tails and launch gaps.  Legal inside a stream capture (fork / join by events).
    // db_l = column sums of g_{l+1}: whatever writes g_{l+1} (this split, the narrow kernel or the data-gradient
    // epilogue of layer l + 1) also writes its partial sums per 32 rows into dbp[l]; the unpack reduces them.
    const bool side = g_wgrad_side != 0 && m->s2 != nullptr;
    cudaStream_t sw = side ? m->s2 : s;
    // gradient w.r.t. the last pre-activation: dy * act'(y), as hi/lo
    const int last_act = (L - 1 == m->sigmoid_layer) ? ACT_SIGMOID : (m->sigmoid_layer == -2 ? ACT_NONE : ACT_RELU);
    const bool narrow = m->last_narrow;
    if (!narrow && (rc = launch_split(dy, lddy, batch, m->D[L], m->y_out, pad4(m->D[L]), last_act, m->g_hi[L], m->g_lo[L], pad32(m->D[L]),
                                      m->dbp[L - 1], s))) return rc;
    CU_CHECK(cudaMemsetAsync(m->dwp[0], 0, (size_t)m->dwp_bytes, s));      // every layer's split-K accumulator
    for (int l = L - 1; l >= 0; --l) {
        const int K = m->D[l], N = m->D[l + 1];
        ARG_CHECK(h_dW[l] && h_db[l]);
        if (narrow && l == L - 1) {
            // activation derivative, weight / bias gradient and the data gradient (masked + split for the layer
            // below, or plain into dx for a one-layer MLP) of the single-column layer in one SIMT launch
            dim3 grid((K + 31) / 32, (batch + NARROW_ROWS - 1) / NARROW_ROWS);
            const bool below = l > 0;
            LAUNCH_PDL(K_MLP_SPLIT, s, narrow_bwd_kernel, grid, 256, 0, dy, lddy, m->y_out, pad4(N), last_act, m->x_hi[l],
                       m->x_lo[l], pad32(K), batch, K, m->last_W, below ? 1 : 0, below ? m->g_hi[l] : nullptr,
                       below ? m->g_lo[l] : nullptr, pad32(K), below ? m->dbp[l - 1] : nullptr, below ? nullptr : dx, lddx,
                       m->dwp[l], m->dbp[l]);
            CU_CHECK(cudaGetLastError());
            continue;
        }
        // wgrad: dW = dZ^T X with both operands read MN-major out of the row-major dZ [B, N] and X [B, K]: split-K
        // over the batch, TMA reduce-add into a zeroed padded accumulator, then unpacked into the dense dW the
        // optimizer sees
        {
            Epi ep = {};
            Out o;
            ep.M = N; ep.N = K; ep.K = batch;
            ep.a_mn = 1; ep.b_mn = 1;
            o.c = m->dwp[l]; o.ldc = pad4(K); o.reduce = true;
            if (side) {         // dZ of this layer (and, the first time, the zeroed accumulators) are ready on s
                CU_CHECK(cudaEventRecord(m->ev_g, s));
                CU_CHECK(cudaStreamWaitEvent(sw, m->ev_g, 0));
            }
            if ((rc = launch_gemm(m->g_hi[l + 1], m->g_lo[l + 1], pad32(N), m->x_hi[l], m->x_lo[l], pad32(K), ep, o, 0 /*auto split-K*/, sw))) return rc;
        }
        // dgrad: dX = dZ W with W read MN-major, then the ReLU mask of the layer below -> its dZ (split) and the
        // partial column sums of that dZ (the bias gradient of layer l - 1)
        if (l > 0) {
            Epi ep = {};
            Out o;
            ep.M = batch; ep.N = K; ep.K = N;
            ep.b_mn = 1;
            ep.mask = m->x_hi[l]; ep.ld_mask = pad32(K);    // x_l = relu(...) > 0  <=>  its hi part > 0
            ep.colsum = m->dbp[l - 1];
            o.c_hi = m->g_hi[l]; o.c_lo = m->g_lo[l]; o.ld_split = pad32(K);
            if ((rc = launch_gemm(m->g_hi[l + 1], m->g_lo[l + 1], pad32(N), m->w_hi[l], m->w_lo[l], pad32(K), ep, o, 1, s))) return rc;
        } else if (dx) {
            Epi ep = {};
            Out o;
            ep.M = batch; ep.N = K; ep.K = N;
            ep.b_mn = 1;
            o.c = dx; o.ldc = lddx;
            if ((rc = launch_gemm(m->g_hi[l + 1], m->g_lo[l + 1], pad32(N), m->w_hi[l], m->w_lo[l], pad32(K), ep, o, 1, s))) return rc;
        }
    }
    // the dense dW / db the optimizer sees, all layers in one launch
    {
        UnpackBatch ub;
        int64_t total = 0;
        int columns = 0;
        for (int l = 0; l < L; ++l) {
            UnpackJob& jb = ub.job[l];
            jb.acc = m->dwp[l]; jb.ldp = pad4(m->D[l]); jb.N = m->D[l + 1]; jb.K = m->D[l];
            jb.dW = h_dW[l]; jb.db = h_db[l]; jb.dbp = m->dbp[l];
            jb.e0 = total; jb.c0 = columns;
            total += (int64_t)jb.N * jb.K;
            columns += jb.N;
        }
        ub.n = L;
        ub.total = total;
        ub.columns = columns;
        ub.parts = (int)parts32(batch);
        ub.db_blocks = (columns + 31) / 32;
        int blocks = (int)((total + 255) / 256);
        if (blocks > 1184) blocks = 1184;
        blocks += ub.db_blocks;
        // the unpack reads the db partials and the narrow layer's accumulator (written on s) and the GEMMs'
        // split-K accumulators (on sw)
        const bool deferred = side && m->defer_join;
        if (side) {
            if (deferred) {
                CU_CHECK(cudaEventRecord(m->ev_g, s));
                CU_CHECK(cudaStreamWaitEvent(sw, m->ev_g, 0));
            } else {
                CU_CHECK(cudaEventRecord(m->ev_done, sw));
                CU_CHECK(cudaStreamWaitEvent(s, m->ev_done, 0));
            }
        }
        cudaStream_t su = deferred ? sw : s;
        LAUNCH_PDL(K_MLP_SPLIT, su, unpack_batch_kernel, blocks, 256, 0, ub);
        CU_CHECK(cudaGetLastError());
        if (deferred) {         // dW / db become visible to the caller's stream at cdlrm_mlp_join
            CU_CHECK(cudaEventRecord(m->ev_done, sw));
            m->pending_join = true;
        }
    }
    return CDLRM_OK;
}

// ------------------------------------------------------------------------------------
// Loss of the training step (main_no_ddp.py:355-369,403-405: torch.nn.BCELoss(reduction="mean") on the
// sigmoid output of the top MLP) fused with its own derivative: stock PyTorch spends five launches on
// 8192 numbers (loss, mean, ones, backward, scale).  One CTA:
//   loss = mean( -(t log p + (1 - t) log(1 - p)) ), logs clamped at -100 as torch does,
//   dz   = (p - t) / max(p (1 - p), 1e-12) / n          (d loss / d p)
// ------------------------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(1024) bce_mean_kernel(const float* __restrict__ z, int64_t ldz, const float* __restrict__ t,
                                                        int64_t ldt, int n, float* __restrict__ loss, float* __restrict__ dz) {
    pdl_enter();
    __shared__ float s_red[32];
    const float inv_n = 1.f / (float)n;
    float acc = 0.f;
    for (int i = threadIdx.x; i < n; i += 1024) {
        const float p = z[(int64_t)i * ldz], y = t[(int64_t)i * ldt];
        const float lp = fmaxf(logf(p), -100.f), lq = fmaxf(log1pf(-p), -100.f);
        acc += (y - 1.f) * lq - y * lp;
        dz[i] = (p - y) / fmaxf((1.f - p) * p, 1e-12f) * inv_n;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        acc = s_red[threadIdx.x];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (threadIdx.x == 0) *loss = acc * inv_n;
    }
}
}  // namespace

extern "C" int cdlrm_bce_mean(int device, const float* z, int64_t ldz, const float* t, int64_t ldt, int32_t n, float* loss,
                              float* dz, cdlrm_stream stream) {
    ARG_CHECK(z && t && loss && dz && n > 0 && ldz >= 1 && ldt >= 1);
    CU_CHECK(cudaSetDevice(device));
    cudaStream_t s = (cudaStream_t)stream;
    LAUNCH_PDL(K_MISC, s, bce_mean_kernel, 1, 1024, 0, z, ldz, t, ldt, (int)n, loss, dz);
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}
