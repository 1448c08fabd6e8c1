// eval.cu -- metrics of an evaluation pass over any number of batches: sample, class and correct counts, the BCE
// sum in fp64 and the exact ROC AUC (Mann-Whitney U, ties counted 1/2).
//
// accumulate (per batch, capturable): one pass over (z, t) writes a 4-byte record key << 1 | label per sample, where
// key is the fp32 bit pattern of z (for z in [0, 1] ordered as an unsigned integer, at most 0x3F800000 < 2^30), adds
// integer counts with integer atomics and adds the loss of every chunk of EV_CHUNK samples (aligned to the global
// sample index) into its own fp64 partial.
//
// result: 2U = sum over positives of (2 * #negatives with a lower key + #negatives with an equal key) needs only the
// counts per distinct key, so no full sort: a counting-sort scatter by the key's high 16 bits (bucket), then per
// bucket a shared-memory histogram of the low 14 bits by label and a scan over it.  A bucket holding more than one
// slice of samples is histogrammed by several CTAs whose integer histograms are merged in global memory first.
// Everything is integer arithmetic, so 2U is exact and deterministic.  The loss partials are summed in a fixed
// order by one CTA.  Memory: 8 bytes per sample (records + scattered records) and < 64 MB fixed.
#include "common.cuh"

namespace {

constexpr int EV_NT = 256;
constexpr int EV_CHUNK = 1024;              // samples per loss partial
constexpr int LO_BITS = 14;                 // key bits resolved by the per-bucket histogram
constexpr int NBINS = 1 << LO_BITS;
constexpr int HIST = 2 * NBINS;             // record & 0x7fff = (key & 0x3fff) << 1 | label
constexpr int NBUCKETS = 1 << 16;           // key >> 14 <= 0xFE00
constexpr int MAX_BIG = 384;                // merged histograms of buckets larger than a slice (128 KB each)
constexpr int64_t MAX_SAMPLES = (int64_t)1 << 30;
constexpr int SCAN_NT = 1024;
constexpr int SCAN_PER = NBUCKETS / SCAN_NT;
constexpr int HB_PER = NBINS / EV_NT;       // bins per thread in the contribution scan

struct DevStats {
    unsigned long long n;          // samples accumulated
    unsigned long long positives;
    unsigned long long correct;
    unsigned long long two_u;
    double loss;
    unsigned int flags;            // bit0 z outside [0, 1] or NaN, bit1 t not in {0, 1}, bit2 more than max_samples
    unsigned int pad;
};

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// sum over the CTA (any blockDim that is a multiple of 32, at most 1024), result in thread 0
__device__ __forceinline__ unsigned long long block_sum_u64(unsigned long long v, unsigned long long* s_red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    v = warp_sum_u64(v);
    __syncthreads();
    if (lane == 0) s_red[warp] = v;
    __syncthreads();
    unsigned long long r = 0;
    if (threadIdx.x == 0)
        for (int i = 0; i < nw; ++i) r += s_red[i];
    return r;
}

// exclusive prefix sum over the CTA; *total = the sum of all values
__device__ __forceinline__ unsigned long long block_excl_scan_u64(unsigned long long v, unsigned long long* s_red,
                                                                  unsigned long long* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    unsigned long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long x = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += x;
    }
    __syncthreads();
    if (lane == 31) s_red[warp] = inc;
    __syncthreads();
    unsigned long long before = 0, all = 0;
    for (int i = 0; i < nw; ++i) {
        if (i < warp) before += s_red[i];
        all += s_red[i];
    }
    *total = all;
    return before + inc - v;
}

__global__ void __launch_bounds__(EV_NT) eval_accum_kernel(const float* __restrict__ z, int64_t ldz,
                                                           const float* __restrict__ t, int64_t ldt, int n,
                                                           uint32_t* __restrict__ rec, double* __restrict__ part,
                                                           DevStats* __restrict__ st, int64_t cap) {
    pdl_enter();
    __shared__ double s_loss[EV_NT];
    __shared__ unsigned long long s_red[EV_NT / 32];
    const unsigned long long base = st->n;          // eval_commit_kernel (the next launch) advances it
    if (base + (unsigned long long)n > (unsigned long long)cap) {
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(&st->flags, 4u);
        return;
    }
    const long long c = (long long)(base / EV_CHUNK) + blockIdx.x;
    const long long lo = max((long long)base, c * EV_CHUNK);
    const long long hi = min((long long)base + n, (c + 1) * EV_CHUNK);
    if (lo >= hi) return;
    double loss = 0.0;
    unsigned int pos = 0, ok = 0, bad = 0;
    for (long long g = lo + threadIdx.x; g < hi; g += EV_NT) {
        const int64_t i = g - (long long)base;
        const float zf = z[i * ldz], tf = t[i * ldt];
        const bool z_in = zf >= 0.f && zf <= 1.f;                  // false for NaN
        const bool t_in = tf == 0.f || tf == 1.f;
        bad |= (z_in ? 0u : 1u) | (t_in ? 0u : 2u);
        const uint32_t key = (z_in && zf != 0.f) ? __float_as_uint(zf) : 0u;   // -0 and 0 are one key
        const uint32_t lab = tf == 1.f ? 1u : 0u;
        rec[g] = key << 1 | lab;
        pos += lab;
        ok += rintf(zf) == tf ? 1u : 0u;                            // round half to even, as torch.round
        const double zd = zf, td = tf;
        loss -= td * fmax(log(zd), -100.0) + (1.0 - td) * fmax(log(1.0 - zd), -100.0);
    }
    s_loss[threadIdx.x] = loss;
    __syncthreads();
#pragma unroll
    for (int w = EV_NT / 2; w > 0; w >>= 1) {                       // fixed tree: the same sum on every run
        if (threadIdx.x < w) s_loss[threadIdx.x] += s_loss[threadIdx.x + w];
        __syncthreads();
    }
    const unsigned long long p = block_sum_u64(pos, s_red);
    const unsigned long long k = block_sum_u64(ok, s_red);
    const unsigned int f = (__syncthreads_or(bad & 1u) ? 1u : 0u) | (__syncthreads_or(bad & 2u) ? 2u : 0u);
    if (threadIdx.x == 0) {
        part[c] += s_loss[0];                                       // a chunk split over two calls: stream order
        if (p) atomicAdd(&st->positives, p);
        if (k) atomicAdd(&st->correct, k);
        if (f) atomicOr(&st->flags, f);
    }
}

__global__ void eval_commit_kernel(DevStats* __restrict__ st, int n, int64_t cap) {
    pdl_enter();
    if (st->n + (unsigned long long)n <= (unsigned long long)cap) st->n += n;
}

// per bucket: samples and negatives (warp-aggregated atomics: heavy ties hit one counter)
__global__ void __launch_bounds__(EV_NT) eval_hist_kernel(const uint32_t* __restrict__ rec,
                                                          const DevStats* __restrict__ st,
                                                          uint32_t* __restrict__ bcnt, uint32_t* __restrict__ bneg) {
    pdl_enter();
    const long long n = (long long)st->n;
    const int lane = threadIdx.x & 31;
    for (long long b0 = (long long)blockIdx.x * EV_NT; b0 < n; b0 += (long long)gridDim.x * EV_NT) {
        const long long i = b0 + threadIdx.x;
        const bool in = i < n;
        const uint32_t mask = __ballot_sync(0xffffffffu, in);
        if (!in) continue;
        const uint32_t r = rec[i];
        const uint32_t b = r >> (LO_BITS + 1);
        const uint32_t peers = __match_any_sync(mask, b);
        const uint32_t negs = __ballot_sync(mask, (r & 1u) == 0) & peers;
        if (lane == __ffs(peers) - 1) {
            atomicAdd(bcnt + b, (uint32_t)__popc(peers));
            if (negs) atomicAdd(bneg + b, (uint32_t)__popc(negs));
        }
    }
}

struct BucketView {
    uint32_t* cnt;       // [NBUCKETS] samples per bucket
    uint32_t* neg;       // [NBUCKETS] negatives per bucket
    uint32_t* off;       // [NBUCKETS + 1] first scattered record of the bucket
    uint32_t* negbelow;  // [NBUCKETS] negatives in lower buckets
    uint32_t* cur;       // [NBUCKETS] scatter cursors
    uint32_t* soff;      // [NBUCKETS + 1] first slice of the bucket
    int32_t* bigid;      // [NBUCKETS] merged-histogram index, -1 for a bucket of one slice
    int32_t* bigb;       // [MAX_BIG] bucket of merged histogram k
    uint32_t* nbig;      // [1]
};

// one CTA: offsets, negatives below, slices and merged-histogram indices of every bucket
__global__ void __launch_bounds__(SCAN_NT) eval_scan_kernel(BucketView v, uint32_t slice) {
    pdl_enter();
    __shared__ unsigned long long s_red[SCAN_NT / 32];
    const int b0 = threadIdx.x * SCAN_PER;
    unsigned long long c = 0, ng = 0, sl = 0, bg = 0;
    for (int q = 0; q < SCAN_PER; ++q) {
        const uint32_t x = v.cnt[b0 + q];
        c += x;
        ng += v.neg[b0 + q];
        sl += (x + slice - 1) / slice;
        bg += x > slice ? 1 : 0;
    }
    unsigned long long tc, tn, ts, tb;
    unsigned long long rc = block_excl_scan_u64(c, s_red, &tc);
    unsigned long long rn = block_excl_scan_u64(ng, s_red, &tn);
    unsigned long long rs = block_excl_scan_u64(sl, s_red, &ts);
    unsigned long long rb = block_excl_scan_u64(bg, s_red, &tb);
    for (int q = 0; q < SCAN_PER; ++q) {
        const int b = b0 + q;
        const uint32_t x = v.cnt[b];
        v.off[b] = (uint32_t)rc;
        v.negbelow[b] = (uint32_t)rn;
        v.soff[b] = (uint32_t)rs;
        if (x > slice) {
            v.bigid[b] = (int32_t)rb;
            v.bigb[rb] = b;
            ++rb;
        } else {
            v.bigid[b] = -1;
        }
        rc += x;
        rn += v.neg[b];
        rs += (x + slice - 1) / slice;
    }
    if (threadIdx.x == SCAN_NT - 1) {
        v.off[NBUCKETS] = (uint32_t)tc;
        v.soff[NBUCKETS] = (uint32_t)ts;
        *v.nbig = (uint32_t)tb;
    }
}

// counting-sort scatter: the low 15 bits of every record, grouped by bucket (order inside a bucket is irrelevant)
__global__ void __launch_bounds__(EV_NT) eval_scatter_kernel(const uint32_t* __restrict__ rec,
                                                             const DevStats* __restrict__ st, BucketView v,
                                                             uint32_t* __restrict__ out) {
    pdl_enter();
    const long long n = (long long)st->n;
    const int lane = threadIdx.x & 31;
    for (long long b0 = (long long)blockIdx.x * EV_NT; b0 < n; b0 += (long long)gridDim.x * EV_NT) {
        const long long i = b0 + threadIdx.x;
        const bool in = i < n;
        const uint32_t mask = __ballot_sync(0xffffffffu, in);
        if (!in) continue;
        const uint32_t r = rec[i];
        const uint32_t b = r >> (LO_BITS + 1);
        const uint32_t peers = __match_any_sync(mask, b);
        const int leader = __ffs(peers) - 1;
        uint32_t first = 0;
        if (lane == leader) first = atomicAdd(v.cur + b, (uint32_t)__popc(peers));
        first = __shfl_sync(mask, first, leader);
        out[v.off[b] + first + __popc(peers & ((1u << lane) - 1u))] = r & (HIST - 1);
    }
}

// 2U contribution of one bucket from its histogram h (h[2 bin] negatives, h[2 bin + 1] positives); thread 0 returns it
__device__ unsigned long long bucket_two_u(const uint32_t* h, uint32_t negbelow, unsigned long long* s_red) {
    const int bin0 = threadIdx.x * HB_PER;
    unsigned long long negs = 0;
    for (int q = 0; q < HB_PER; ++q) negs += h[2 * (bin0 + q)];
    unsigned long long total;
    unsigned long long run = negbelow + block_excl_scan_u64(negs, s_red, &total);
    unsigned long long acc = 0;
    for (int q = 0; q < HB_PER; ++q) {
        const uint32_t ng = h[2 * (bin0 + q)], ps = h[2 * (bin0 + q) + 1];
        acc += (unsigned long long)ps * (2ull * run + ng);
        run += ng;
    }
    return block_sum_u64(acc, s_red);
}

// persistent: CTA loops over slices; a one-slice bucket is finished here, a larger one merged into its histogram
__global__ void __launch_bounds__(EV_NT) eval_slice_kernel(const uint32_t* __restrict__ sorted, BucketView v,
                                                           uint32_t slice, uint32_t* __restrict__ big,
                                                           DevStats* __restrict__ st) {
    pdl_enter();
    extern __shared__ uint32_t h[];                 // [HIST]
    __shared__ unsigned long long s_red[EV_NT / 32];
    const uint32_t n_slices = v.soff[NBUCKETS];
    const int lane = threadIdx.x & 31;
    for (uint32_t s = blockIdx.x; s < n_slices; s += gridDim.x) {
        int lo = 0, hi = NBUCKETS - 1;              // the bucket b with soff[b] <= s < soff[b + 1]
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (v.soff[mid + 1] <= s) lo = mid + 1; else hi = mid;
        }
        const int b = lo;
        const uint32_t beg = v.off[b] + (s - v.soff[b]) * slice;
        const uint32_t end = min(v.off[b + 1], beg + slice);
        for (int i = threadIdx.x; i < HIST; i += EV_NT) h[i] = 0;
        __syncthreads();
        for (uint32_t i0 = beg; i0 < end; i0 += EV_NT) {
            const uint32_t i = i0 + threadIdx.x;
            const bool in = i < end;
            const uint32_t mask = __ballot_sync(0xffffffffu, in);
            if (!in) continue;
            const uint32_t r = sorted[i];
            const uint32_t peers = __match_any_sync(mask, r);
            if (lane == __ffs(peers) - 1) atomicAdd(h + r, (uint32_t)__popc(peers));
        }
        __syncthreads();
        const int k = v.bigid[b];
        if (k < 0) {
            const unsigned long long u = bucket_two_u(h, v.negbelow[b], s_red);
            if (threadIdx.x == 0 && u) atomicAdd(&st->two_u, u);
        } else {
            uint32_t* g = big + (int64_t)k * HIST;
            for (int i = threadIdx.x; i < HIST; i += EV_NT)
                if (h[i]) atomicAdd(g + i, h[i]);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(EV_NT) eval_big_kernel(const uint32_t* __restrict__ big, BucketView v,
                                                         DevStats* __restrict__ st) {
    pdl_enter();
    __shared__ unsigned long long s_red[EV_NT / 32];
    const uint32_t nb = *v.nbig;
    for (uint32_t k = blockIdx.x; k < nb; k += gridDim.x) {
        const unsigned long long u = bucket_two_u(big + (int64_t)k * HIST, v.negbelow[v.bigb[k]], s_red);
        if (threadIdx.x == 0 && u) atomicAdd(&st->two_u, u);
        __syncthreads();
    }
}

// the loss partials in a fixed order: thread i sums partials i, i + 256, ... then a fixed tree
__global__ void __launch_bounds__(EV_NT) eval_loss_kernel(const double* __restrict__ part, DevStats* __restrict__ st) {
    pdl_enter();
    __shared__ double s[EV_NT];
    const long long nch = (long long)((st->n + EV_CHUNK - 1) / EV_CHUNK);
    double a = 0.0;
    for (long long c = threadIdx.x; c < nch; c += EV_NT) a += part[c];
    s[threadIdx.x] = a;
    __syncthreads();
#pragma unroll
    for (int w = EV_NT / 2; w > 0; w >>= 1) {
        if (threadIdx.x < w) s[threadIdx.x] += s[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) st->loss = s[0];
}

}  // namespace

struct cdlrm_eval {
    int device = 0;
    int num_sms = 148;
    int64_t cap = 0;
    uint32_t slice = 0;             // records per CTA of the histogram pass
    int max_big = 0;
    uint32_t* rec = nullptr;        // [cap] key << 1 | label, accumulation order
    uint32_t* sorted = nullptr;     // [cap] low 15 bits of the records, grouped by bucket
    double* part = nullptr;         // [cap / EV_CHUNK + 2] loss partial per chunk
    DevStats* st = nullptr;
    DevStats* h_st = nullptr;       // pinned
    uint32_t* bucket_mem = nullptr;
    BucketView bv = {};
    uint32_t* big = nullptr;        // [max_big][HIST]
};

static void eval_free(cdlrm_eval* e) {
    cudaFree(e->rec);
    cudaFree(e->sorted);
    cudaFree(e->part);
    cudaFree(e->st);
    cudaFree(e->bucket_mem);
    cudaFree(e->big);
    if (e->h_st) cudaFreeHost(e->h_st);
    delete e;
}

extern "C" int cdlrm_eval_create(cdlrm_eval** out, int device, int64_t max_samples) {
    ARG_CHECK(out);
    ARG_CHECK(max_samples > 0 && max_samples <= MAX_SAMPLES);
    int ndev = 0;
    CU_CHECK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) {
        cdlrm_set_error("device %d not available (%d CUDA devices); there is no CPU fallback", device, ndev);
        return CDLRM_ERR_CUDA;
    }
    CU_CHECK(cudaSetDevice(device));
    cdlrm_eval* e = new cdlrm_eval();
    e->device = device;
    e->cap = max_samples;
    if (cudaDeviceGetAttribute(&e->num_sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || e->num_sms <= 0)
        e->num_sms = 148;
    // fewer than cap / slice buckets can hold more than a slice: at most MAX_BIG merged histograms
    const int64_t sl = (max_samples + MAX_BIG - 1) / MAX_BIG;
    e->slice = (uint32_t)(sl > 65536 ? sl : 65536);
    e->max_big = (int)(max_samples / e->slice);
    const size_t nb = NBUCKETS;
    const size_t words = 7 * nb + 2 + 2 + MAX_BIG + 1;
    cudaError_t err = cudaMalloc(&e->rec, sizeof(uint32_t) * max_samples);
    if (err == cudaSuccess) err = cudaMalloc(&e->sorted, sizeof(uint32_t) * max_samples);
    if (err == cudaSuccess) err = cudaMalloc(&e->part, sizeof(double) * (max_samples / EV_CHUNK + 2));
    if (err == cudaSuccess) err = cudaMalloc(&e->st, sizeof(DevStats));
    if (err == cudaSuccess) err = cudaMalloc(&e->bucket_mem, sizeof(uint32_t) * words);
    if (err == cudaSuccess && e->max_big > 0) err = cudaMalloc(&e->big, sizeof(uint32_t) * HIST * (size_t)e->max_big);
    if (err == cudaSuccess) err = cudaMallocHost(&e->h_st, sizeof(DevStats));
    if (err == cudaSuccess) err = cudaMemset(e->st, 0, sizeof(DevStats));
    if (err == cudaSuccess) err = cudaMemset(e->part, 0, sizeof(double) * (max_samples / EV_CHUNK + 2));
    if (err != cudaSuccess) {
        cdlrm_set_error("cdlrm_eval_create(%lld samples): %s", (long long)max_samples, cudaGetErrorString(err));
        eval_free(e);
        return CDLRM_ERR_CUDA;
    }
    uint32_t* p = e->bucket_mem;
    BucketView& v = e->bv;
    v.cnt = p; p += nb;
    v.neg = p; p += nb;
    v.cur = p; p += nb;                  // cnt, neg, cur: cleared together by one memset
    v.off = p; p += nb + 1;
    v.negbelow = p; p += nb;
    v.soff = p; p += nb + 1;
    v.bigid = reinterpret_cast<int32_t*>(p); p += nb;
    v.bigb = reinterpret_cast<int32_t*>(p); p += MAX_BIG;
    v.nbig = p;
    *out = e;
    return CDLRM_OK;
}

extern "C" int cdlrm_eval_destroy(cdlrm_eval* ev) {
    if (!ev) return CDLRM_OK;
    cudaSetDevice(ev->device);
    cudaDeviceSynchronize();
    eval_free(ev);
    return CDLRM_OK;
}

extern "C" int cdlrm_eval_reset(cdlrm_eval* ev, cdlrm_stream stream) {
    ARG_CHECK(ev);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(ev->device));
    CU_CHECK(cudaMemsetAsync(ev->st, 0, sizeof(DevStats), s));
    CU_CHECK(cudaMemsetAsync(ev->part, 0, sizeof(double) * (ev->cap / EV_CHUNK + 2), s));
    return CDLRM_OK;
}

extern "C" int cdlrm_eval_accumulate(cdlrm_eval* ev, const float* z, int64_t ldz, const float* t, int64_t ldt,
                                     int32_t n, cdlrm_stream stream) {
    ARG_CHECK(ev && n >= 0);
    if (n == 0) return CDLRM_OK;
    ARG_CHECK(z && t && ldz > 0 && ldt > 0);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(ev->device));
    const int grid = n / EV_CHUNK + 2;           // chunks a batch of n samples can touch
    LAUNCH_PDL(K_EVAL, s, eval_accum_kernel, grid, EV_NT, 0, z, ldz, t, ldt, (int)n, ev->rec, ev->part, ev->st, ev->cap);
    LAUNCH_PDL(K_EVAL, s, eval_commit_kernel, 1, 1, 0, ev->st, (int)n, ev->cap);
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

extern "C" int cdlrm_eval_result(cdlrm_eval* ev, cdlrm_eval_stats* h_stats, cdlrm_stream stream) {
    ARG_CHECK(ev && h_stats);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(ev->device));
    const int smem = HIST * (int)sizeof(uint32_t);
    CU_CHECK(cdlrm_smem_optin((const void*)eval_slice_kernel, smem));
    CU_CHECK(cudaMemsetAsync(ev->bv.cnt, 0, sizeof(uint32_t) * 3 * NBUCKETS, s));
    CU_CHECK(cudaMemsetAsync(&ev->st->two_u, 0, sizeof(unsigned long long), s));
    if (ev->big) CU_CHECK(cudaMemsetAsync(ev->big, 0, sizeof(uint32_t) * HIST * (size_t)ev->max_big, s));
    const int grid = ev->num_sms * 4;
    LAUNCH_PDL(K_EVAL, s, eval_hist_kernel, grid, EV_NT, 0, ev->rec, ev->st, ev->bv.cnt, ev->bv.neg);
    LAUNCH_PDL(K_EVAL, s, eval_scan_kernel, 1, SCAN_NT, 0, ev->bv, ev->slice);
    LAUNCH_PDL(K_EVAL, s, eval_scatter_kernel, grid, EV_NT, 0, ev->rec, ev->st, ev->bv, ev->sorted);
    LAUNCH_PDL(K_EVAL, s, eval_slice_kernel, ev->num_sms, EV_NT, smem, ev->sorted, ev->bv, ev->slice, ev->big, ev->st);
    if (ev->big) LAUNCH_PDL(K_EVAL, s, eval_big_kernel, ev->max_big, EV_NT, 0, ev->big, ev->bv, ev->st);
    LAUNCH_PDL(K_EVAL, s, eval_loss_kernel, 1, EV_NT, 0, ev->part, ev->st);
    CU_CHECK(cudaGetLastError());
    CU_CHECK(cudaMemcpyAsync(ev->h_st, ev->st, sizeof(DevStats), cudaMemcpyDeviceToHost, s));
    CU_CHECK(cudaStreamSynchronize(s));
    const DevStats& d = *ev->h_st;
    h_stats->samples = (int64_t)d.n;
    h_stats->positives = (int64_t)d.positives;
    h_stats->negatives = (int64_t)(d.n - d.positives);
    h_stats->correct = (int64_t)d.correct;
    h_stats->loss_sum = d.loss;
    h_stats->auc_2u = d.two_u;
    h_stats->flags = d.flags;
    h_stats->reserved = 0;
    return CDLRM_OK;
}
