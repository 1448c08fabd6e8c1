// rng.cu -- host-side victim-way random stream, bit-compatible with the torch CPU
// generator the reference consumes through torch.distributions.Categorical(...).sample()
// (main_no_ddp.py:183-185): torch.multinomial's fast path draws
// q = empty(rows, ways).exponential_(1) and takes argmax(probs / q).
//   exponential_(1) on float32 == float32(-log1p(-u)),  u = (r64 & (2^53-1)) * 2^-53,
//   r64 = (mt32() << 32) | mt32(),  mt19937 seeded with init_genrand(seed).
// mt19937 is sequential, so the raw stream is produced by the calling thread while a
// small pool of threads applies the (expensive) log1p transform block by block.
#include <math.h>

#include <random>
#include <thread>

#include "common.cuh"
#define MT_JUMP_QUAL __constant__
#include "mt_jump_table.h"

struct cdlrm_rng {
    std::mt19937 gen;
    uint64_t draws = 0;
    std::vector<uint64_t> raw[2];
};

static inline float transform(uint64_t r) {
    const double u = (double)(r & ((1ull << 53) - 1ull)) * (1.0 / 9007199254740992.0);
    return (float)(-log1p(-u));
}

extern "C" int cdlrm_rng_create(cdlrm_rng** out, uint64_t seed) {
    ARG_CHECK(out);
    cdlrm_rng* r = new cdlrm_rng();
    r->gen.seed((uint32_t)(seed & 0xffffffffull));  // torch: mt19937(seed) truncates to 32 bits
    *out = r;
    return CDLRM_OK;
}

extern "C" int cdlrm_rng_destroy(cdlrm_rng* r) {
    delete r;
    return CDLRM_OK;
}

extern "C" uint64_t cdlrm_rng_draws(const cdlrm_rng* r) { return r ? r->draws : 0; }

extern "C" int cdlrm_rng_exponential(cdlrm_rng* r, float* out, int64_t n, int threads) {
    ARG_CHECK(r && n >= 0 && (out || n == 0));
    if (threads < 1) threads = 1;
    constexpr int64_t BLOCK = 1 << 20;
    if (n < (1 << 16) || threads == 1) {
        for (int64_t i = 0; i < n; ++i) {
            uint64_t hi = r->gen(), lo = r->gen();
            out[i] = transform((hi << 32) | lo);
        }
        r->draws += (uint64_t)n;
        return CDLRM_OK;
    }
    r->raw[0].resize(BLOCK);
    r->raw[1].resize(BLOCK);
    auto fill = [&](int buf, int64_t cnt) {
        uint64_t* p = r->raw[buf].data();
        for (int64_t i = 0; i < cnt; ++i) {
            uint64_t hi = r->gen(), lo = r->gen();
            p[i] = (hi << 32) | lo;
        }
    };
    const int64_t nblk = (n + BLOCK - 1) / BLOCK;
    fill(0, n < BLOCK ? n : BLOCK);
    for (int64_t b = 0; b < nblk; ++b) {
        const int64_t base = b * BLOCK;
        const int64_t cnt = n - base < BLOCK ? n - base : BLOCK;
        const uint64_t* src = r->raw[b & 1].data();
        float* dst = out + base;
        std::vector<std::thread> pool;
        const int nt = threads - 1 > 0 ? threads - 1 : 1;
        const int64_t per = (cnt + nt - 1) / nt;
        for (int t = 0; t < nt; ++t) {
            const int64_t lo = t * per, hi = lo + per < cnt ? lo + per : cnt;
            if (lo >= hi) break;
            pool.emplace_back([=]() {
                for (int64_t i = lo; i < hi; ++i) dst[i] = transform(src[i]);
            });
        }
        if (b + 1 < nblk) {  // overlap: produce the next raw block while the pool transforms this one
            const int64_t nb = (b + 1) * BLOCK;
            fill((b + 1) & 1, n - nb < BLOCK ? n - nb : BLOCK);
        }
        for (auto& th : pool) th.join();
    }
    r->draws += (uint64_t)n;
    return CDLRM_OK;
}

// =================================================================================================
// Device-resident victim stream.  The same mt19937 sequence, generated ON the GPU by one CTA:
// the recurrence x[k+624] = x[k+397] ^ f(x[k], x[k+1]) leaves 227 / 227 / 170 independent
// elements per regeneration, so a 256-thread CTA refreshes the 624-word state in three
// barrier-separated phases (~4 G words/s) -- an order of magnitude faster than a host core and
// with no PCIe traffic for the draws.  The exponential transform (expdraw.cuh) is applied by
// whoever consumes the raw words (the planner's select kernel, or the kernel below).
// =================================================================================================
#include "expdraw.cuh"

struct cdlrm_rngdev {
    int device = 0;
    uint32_t* d_state = nullptr;   // x[624], pos
    uint32_t* d_states = nullptr;  // [MT_MAX_CHUNKS][624]: start states of the chunks of one parallel generation
    uint64_t draws = 0;
};

namespace {

constexpr int MT_N = 624, MT_M = 397;

__device__ __forceinline__ uint32_t mt_twist(uint32_t a, uint32_t b, uint32_t c) {
    const uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
    return c ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}

__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

// next block of 624 words in place (three dependent phases of up to 227 independent words); every thread of the
// 256-thread CTA calls it; all reads of the old block by the caller must be complete (barrier) before the call
__device__ __forceinline__ void mt_regen(uint32_t* x, int tid) {
    uint32_t v = 0;
    if (tid < 227) v = mt_twist(x[tid], x[tid + 1], x[tid + MT_M]);
    __syncthreads();
    if (tid < 227) x[tid] = v;
    __syncthreads();
    if (tid < 227) v = mt_twist(x[227 + tid], x[228 + tid], x[tid]);
    __syncthreads();
    if (tid < 227) x[227 + tid] = v;
    __syncthreads();
    if (tid < 170) v = mt_twist(x[454 + tid], x[tid == 169 ? 0 : 455 + tid], x[227 + tid]);
    __syncthreads();
    if (tid < 170) x[454 + tid] = v;
    __syncthreads();
}

// ---- parallel generation of ONE sequential stream: jump-ahead ----------------------------------------------
// mt19937 is sequential by construction (0.75 G words/s on one CTA: 0.4 s per Terabyte window on one GPU, 3.6 s
// for the 8-GPU global window -- longer than the window trains).  The state J words ahead is a fixed GF(2)-linear
// function of the state: with g(x) = x^J mod phi(x) (tools/gen_mt_jump.py derives phi and the g's, and checks them
// against sequential generation),   s[n + J] = XOR_{i : g_i = 1} s[n + i]   word-wise.  A long request is cut into
// chunks of MT_JUMP_BLOCKS_PER_CHUNK blocks; the start state of chunk j comes from chunk j - 2^m by the level-m
// polynomial (log2(chunks) launches, all chunks of a level in parallel), then every chunk is generated by its own
// CTA.  Output and final state are bit-identical to the sequential kernel (tests/test_gpu_parity.py).
constexpr int MT_SEQ_BLOCKS = 33;                 // s[0 .. 33 * 624) covers i + k <= 19936 + 623
constexpr int MT_MAX_CHUNKS = 1 << MT_JUMP_LEVELS;

// states[lo + b] = states[b] advanced by MT_JUMP_CHUNK_WORDS * 2^level words, b = blockIdx.x.  (The low 31 bits of the
// first word of a state are not state -- the recurrence only reads its top bit -- and come out arbitrary: a chunk's
// start state is only ever the PREDECESSOR of the first block that is output.)
__global__ void __launch_bounds__(256) mt_jump_kernel(uint32_t* __restrict__ states, int lo, int level) {
    extern __shared__ uint32_t seq[];              // [MT_SEQ_BLOCKS * 624]
    const int tid = threadIdx.x;
    const uint32_t* src = states + (size_t)blockIdx.x * MT_N;
    for (int i = tid; i < MT_N; i += 256) seq[i] = src[i];
    __syncthreads();
    for (int b = 1; b < MT_SEQ_BLOCKS; ++b) {
        uint32_t* nb = seq + b * MT_N;
        for (int i = tid; i < MT_N; i += 256) nb[i] = nb[i - MT_N];
        __syncthreads();
        mt_regen(nb, tid);
    }
    uint32_t a0 = 0, a1 = 0, a2 = 0;
    const bool third = tid + 512 < MT_N;
    for (int w = 0; w < MT_JUMP_POLY_WORDS; ++w) {
        uint32_t bits = mt_jump_poly[level][w];       // uniform: constant cache
        while (bits) {
            const int i = w * 32 + __ffs(bits) - 1;
            bits &= bits - 1;
            a0 ^= seq[i + tid];
            a1 ^= seq[i + tid + 256];
            if (third) a2 ^= seq[i + tid + 512];
        }
    }
    uint32_t* dst = states + (size_t)(lo + blockIdx.x) * MT_N;
    dst[tid] = a0;
    dst[tid + 256] = a1;
    if (third) dst[tid + 512] = a2;
}

// chunk j = blockIdx.x: the pending words of the current block (chunk 0 only), then blocks j*CB + 1 .. (j+1)*CB after
// it, tempered, at their position in the stream; the chunk that produces the last block leaves the generator state
__global__ void __launch_bounds__(256) mt_chunks_kernel(const uint32_t* __restrict__ states, uint32_t* __restrict__ state,
                                                        uint32_t* __restrict__ out, int pos, long long n_words, long long nb) {
    __shared__ uint32_t x[MT_N];
    const int tid = threadIdx.x;
    const long long j = blockIdx.x;
    for (int i = tid; i < MT_N; i += 256) x[i] = states[(size_t)j * MT_N + i];
    __syncthreads();
    const int r0 = MT_N - pos;
    if (j == 0)
        for (int i = tid; i < r0; i += 256) out[i] = mt_temper(x[pos + i]);
    __syncthreads();
    const long long q0 = j * MT_JUMP_BLOCKS_PER_CHUNK + 1;
    const long long q1 = (j + 1) * MT_JUMP_BLOCKS_PER_CHUNK < nb ? (j + 1) * MT_JUMP_BLOCKS_PER_CHUNK : nb;
    for (long long q = q0; q <= q1; ++q) {
        mt_regen(x, tid);
        const long long base = r0 + (q - 1) * MT_N;
        const long long left = n_words - base;
        const int cnt = left < MT_N ? (int)left : MT_N;
        for (int i = tid; i < cnt; i += 256) out[base + i] = mt_temper(x[i]);
        __syncthreads();
    }
    if (q1 == nb && q0 <= q1) {
        for (int i = tid; i < MT_N; i += 256) state[i] = x[i];
        if (tid == 0) state[MT_N] = (uint32_t)(n_words - (r0 + (nb - 1) * MT_N));
    }
}

__global__ void __launch_bounds__(256) mt_generate_kernel(uint32_t* __restrict__ state, uint32_t* __restrict__ out,
                                                          long long n_words) {
    __shared__ uint32_t x[MT_N];
    const int tid = threadIdx.x;
    for (int i = tid; i < MT_N; i += 256) x[i] = state[i];
    int pos = (int)state[MT_N];
    __syncthreads();
    long long done = 0;
    while (done < n_words) {
        if (pos == MT_N) {  // uniform across the CTA
            uint32_t v = 0;
            if (tid < 227) v = mt_twist(x[tid], x[tid + 1], x[tid + MT_M]);
            __syncthreads();
            if (tid < 227) x[tid] = v;
            __syncthreads();
            if (tid < 227) v = mt_twist(x[227 + tid], x[228 + tid], x[tid]);
            __syncthreads();
            if (tid < 227) x[227 + tid] = v;
            __syncthreads();
            if (tid < 170) v = mt_twist(x[454 + tid], x[tid == 169 ? 0 : 455 + tid], x[227 + tid]);
            __syncthreads();
            if (tid < 170) x[454 + tid] = v;
            __syncthreads();
            pos = 0;
        }
        const long long left = n_words - done;
        const int cnt = (MT_N - pos) < left ? (MT_N - pos) : (int)left;
        for (int i = tid; i < cnt; i += 256) out[done + i] = mt_temper(x[pos + i]);
        done += cnt;
        pos += cnt;
        __syncthreads();  // emit reads of x[] complete before the next regeneration writes
    }
    for (int i = tid; i < MT_N; i += 256) state[i] = x[i];
    if (tid == 0) state[MT_N] = (uint32_t)pos;
}

__global__ void exp_from_raw_kernel(const uint2* __restrict__ raw, float* __restrict__ out, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = exp_draw_from_raw(raw[i]);
}

}  // namespace

static long long g_mt_parallel_min_words = 0;     // requests of two or more chunks (5.1 M words) go parallel

extern "C" int cdlrm_rngdev_create(cdlrm_rngdev** out, int device, uint64_t seed) {
    ARG_CHECK(out);
    CU_CHECK(cudaSetDevice(device));
    cdlrm_rngdev* r = new cdlrm_rngdev();
    r->device = device;
    uint32_t h[MT_N + 1];
    h[0] = (uint32_t)(seed & 0xffffffffull);  // init_genrand, as torch.manual_seed(seed) does
    for (int i = 1; i < MT_N; ++i) h[i] = 1812433253u * (h[i - 1] ^ (h[i - 1] >> 30)) + (uint32_t)i;
    h[MT_N] = MT_N;  // first use regenerates
    CU_CHECK(cudaMalloc(&r->d_state, sizeof(h)));
    CU_CHECK(cudaMemcpy(r->d_state, h, sizeof(h), cudaMemcpyHostToDevice));
    CU_CHECK(cudaMalloc(&r->d_states, (size_t)MT_MAX_CHUNKS * MT_N * sizeof(uint32_t)));
    CU_CHECK(cudaFuncSetAttribute(mt_jump_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  MT_SEQ_BLOCKS * MT_N * (int)sizeof(uint32_t)));
    *out = r;
    return CDLRM_OK;
}

extern "C" int cdlrm_rngdev_destroy(cdlrm_rngdev* r) {
    if (!r) return CDLRM_OK;
    cudaSetDevice(r->device);
    cudaFree(r->d_state);
    cudaFree(r->d_states);
    delete r;
    return CDLRM_OK;
}

extern "C" uint64_t cdlrm_rngdev_draws(const cdlrm_rngdev* r) { return r ? r->draws : 0; }

extern "C" int cdlrm_rngdev_raw(cdlrm_rngdev* r, uint32_t* d_out, int64_t n_draws, cdlrm_stream stream) {
    ARG_CHECK(r && n_draws >= 0);
    if (n_draws == 0) return CDLRM_OK;
    ARG_CHECK(d_out && ((uintptr_t)d_out & 7) == 0);
    CU_CHECK(cudaSetDevice(r->device));
    cudaStream_t s = (cudaStream_t)stream;
    const long long n_words = (long long)n_draws * 2;
    // the host knows where the stream stands: `pos` words of the current block are used up
    const uint64_t before = r->draws * 2;
    const int pos = before == 0 ? MT_N : (int)((before - 1) % MT_N) + 1;
    const int r0 = MT_N - pos;
    const long long nb = n_words > r0 ? (n_words - r0 + MT_N - 1) / MT_N : 0;          // blocks after the current one
    const long long n_chunks = (nb + MT_JUMP_BLOCKS_PER_CHUNK - 1) / MT_JUMP_BLOCKS_PER_CHUNK;
    if (g_mt_parallel_min_words >= 0 && n_words >= g_mt_parallel_min_words && n_chunks >= 2 && n_chunks <= MT_MAX_CHUNKS) {
        CU_CHECK(cudaMemcpyAsync(r->d_states, r->d_state, MT_N * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s));
        for (int m = 0; (1LL << m) < n_chunks; ++m) {
            const long long lo = 1LL << m, hi = (2LL << m) < n_chunks ? (2LL << m) : n_chunks;
            LAUNCH(K_RNG_MT, s, (mt_jump_kernel<<<(int)(hi - lo), 256, MT_SEQ_BLOCKS * MT_N * sizeof(uint32_t), s>>>(r->d_states, (int)lo, m)));
        }
        LAUNCH(K_RNG_MT, s, (mt_chunks_kernel<<<(int)n_chunks, 256, 0, s>>>(r->d_states, r->d_state, d_out, pos, n_words, nb)));
    } else {
        LAUNCH(K_RNG_MT, s, mt_generate_kernel<<<1, 256, 0, s>>>(r->d_state, d_out, n_words));
    }
    CU_CHECK(cudaGetLastError());
    r->draws += (uint64_t)n_draws;
    return CDLRM_OK;
}

// key 0: smallest request (in 32-bit words) that is generated chunk-parallel with jump-ahead; -1 = always sequential
extern "C" int cdlrm_rngdev_set_option(int key, int64_t value) {
    ARG_CHECK(key == 0);
    g_mt_parallel_min_words = (long long)value;
    return CDLRM_OK;
}

extern "C" int cdlrm_exp_from_raw(const uint32_t* d_raw, float* d_out, int64_t n, cdlrm_stream stream) {
    ARG_CHECK(n >= 0);
    if (n == 0) return CDLRM_OK;
    ARG_CHECK(d_raw && d_out && ((uintptr_t)d_raw & 7) == 0);
    cudaStream_t s = (cudaStream_t)stream;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    LAUNCH(K_RNG_EXP, s, exp_from_raw_kernel<<<(int)blocks, 256, 0, s>>>(reinterpret_cast<const uint2*>(d_raw), d_out, (long long)n));
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

extern "C" int cdlrm_rngdev_exponential(cdlrm_rngdev* r, float* d_out, int64_t n, uint32_t* d_raw_scratch,
                                        cdlrm_stream stream) {
    ARG_CHECK(r && n >= 0);
    if (n == 0) return CDLRM_OK;
    ARG_CHECK(d_out && d_raw_scratch);
    int rc = cdlrm_rngdev_raw(r, d_raw_scratch, n, stream);
    if (rc) return rc;
    return cdlrm_exp_from_raw(d_raw_scratch, d_out, n, stream);
}

// Checkpoint of the device stream.  It keeps x[624] and pos (words of the current block already used) in HBM, and the host keeps the
// number of draws, from which cdlrm_rngdev_raw derives pos: the two must agree.
static int pos_of_draws(uint64_t draws) { return draws == 0 ? MT_N : (int)((draws * 2 - 1) % MT_N) + 1; }

extern "C" int cdlrm_rngdev_get_state(cdlrm_rngdev* r, uint32_t* h_state, uint64_t* h_draws, cdlrm_stream stream) {
    ARG_CHECK(r && h_state && h_draws);
    CU_CHECK(cudaSetDevice(r->device));
    CU_CHECK(cudaMemcpyAsync(h_state, r->d_state, sizeof(uint32_t) * (MT_N + 1), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    *h_draws = r->draws;
    return CDLRM_OK;
}

extern "C" int cdlrm_rngdev_set_state(cdlrm_rngdev* r, const uint32_t* h_state, uint64_t draws, cdlrm_stream stream) {
    ARG_CHECK(r && h_state);
    if ((int)h_state[MT_N] != pos_of_draws(draws)) {
        cdlrm_set_error("rngdev state: position %u does not match %llu draws (expected %d)", h_state[MT_N],
                        (unsigned long long)draws, pos_of_draws(draws));
        return CDLRM_ERR_ARG;
    }
    CU_CHECK(cudaSetDevice(r->device));
    CU_CHECK(cudaMemcpyAsync(r->d_state, h_state, sizeof(uint32_t) * (MT_N + 1), cudaMemcpyHostToDevice, (cudaStream_t)stream));
    r->draws = draws;
    return CDLRM_OK;
}
