// ctx.cu -- context, geometry and bindings of libcdlrm_b200.
// Replaces Embedding_Table_Cache_Group.__init__ and helpers (model_no_ddp.py:102-147,
// :319-331 of the reference).
#include <stdarg.h>
#include <string.h>

#include <stdlib.h>

#include <map>
#include <mutex>
#include <utility>

#include "common.cuh"

cudaError_t cdlrm_smem_optin(const void* func, int bytes) {
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, int> done;     // (function, device) -> bytes opted in
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(mu);
    auto key = std::make_pair(func, dev);
    auto it = done.find(key);
    if (it != done.end() && it->second >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) done[key] = bytes;
    return e;
}

static thread_local char g_err[1024] = "";

void cdlrm_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* cdlrm_last_error(void) { return g_err; }
extern "C" int cdlrm_abi_version(void) { return CDLRM_ABI_VERSION; }

// model_no_ddp.py:319-331 -- deliberately NOT a correct primality test: divisors
// start at 3 (so even n pass) and stop at i*i < n (so squares of primes pass).
extern "C" int cdlrm_is_prime_ref(int64_t n) {
    if (n == 1 || n == 2) return 0;
    for (int64_t i = 3; i * i < n; ++i)
        if (n % i == 0) return 0;
    return 1;
}

// model_no_ddp.py:122-125
extern "C" int64_t cdlrm_find_next_prime(int64_t c) {
    for (int64_t i = c; i < 2 * c; ++i)
        if (cdlrm_is_prime_ref(i)) return i;
    return -1;
}

extern "C" int cdlrm_ctx_create(cdlrm_ctx** out, int device, int T, int dim, int ways, int64_t aux,
                                const int64_t* n_rows, int64_t max_cache_size) {
    ARG_CHECK(out && n_rows);
    ARG_CHECK(T > 0 && dim > 0 && aux >= 0);
    ARG_CHECK(ways > 0 && ways <= CDLRM_MAX_WAYS);
    int64_t mcs = cdlrm_find_next_prime(max_cache_size);
    if (mcs < 0) {
        cdlrm_set_error("find_next_prime(%lld) found nothing in [c, 2c)", (long long)max_cache_size);
        return CDLRM_ERR_ARG;
    }
    int ndev = 0;
    CU_CHECK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) {
        cdlrm_set_error("device %d not available (%d CUDA devices); there is no CPU fallback", device, ndev);
        return CDLRM_ERR_CUDA;
    }
    CU_CHECK(cudaSetDevice(device));
    cdlrm_ctx* c = new cdlrm_ctx();
    c->device = device;
    if (cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || c->num_sms <= 0) c->num_sms = 148;
    c->T = T;
    c->dim = dim;
    c->ways = ways;
    c->aux = aux;
    c->max_cache_size = mcs;
    c->tabs.resize(T);
    int64_t word_off = 0;
    for (int k = 0; k < T; ++k) {
        TableDesc& t = c->tabs[k];
        memset(&t, 0, sizeof(t));
        ARG_CHECK(n_rows[k] > 0);
        t.n_rows = n_rows[k];
        t.num_sets = n_rows[k] < mcs ? n_rows[k] : mcs;     // model_no_ddp.py:136
        t.cache_rows = (int64_t)ways * t.num_sets + aux;    // :138
        if (t.cache_rows >= (int64_t)1 << 31) {
            cdlrm_set_error("table %d: %lld cache rows do not fit int32 slots", k, (long long)t.cache_rows);
            delete c;
            return CDLRM_ERR_ARG;
        }
        t.dirty_word_off = word_off;
        word_off += (t.cache_rows + 31) / 32;
    }
    CU_CHECK(cudaMalloc(&c->d_tabs, sizeof(TableDesc) * T));
    CU_CHECK(cudaMalloc(&c->d_flags, sizeof(uint32_t)));
    CU_CHECK(cudaMemset(c->d_flags, 0, sizeof(uint32_t)));
    CU_CHECK(cudaMalloc(&c->p_counts, sizeof(int64_t) * T * 8));
    c->last_uniq.assign(T, 0);
    c->tabs_dirty = true;
    *out = c;
    return CDLRM_OK;
}

extern "C" int cdlrm_ctx_destroy(cdlrm_ctx* c) {
    if (!c) return CDLRM_OK;
    cudaSetDevice(c->device);
    cudaFree(c->d_tabs);
    cudaFree(c->d_flags);
    cudaFree(c->d_missmap);
    cudaFree(c->d_losers);
    cudaFree(c->d_lbucket);
    if (c->h_losers) cudaFreeHost(c->h_losers);
    cudaFree(c->p_counts);
    cudaFree(c->d_ptabs);
    delete c;
    return CDLRM_OK;
}

extern "C" int cdlrm_ctx_geometry(const cdlrm_ctx* c, int64_t* num_sets, int64_t* cache_rows) {
    ARG_CHECK(c);
    for (int k = 0; k < c->T; ++k) {
        if (num_sets) num_sets[k] = c->tabs[k].num_sets;
        if (cache_rows) cache_rows[k] = c->tabs[k].cache_rows;
    }
    return CDLRM_OK;
}

extern "C" int cdlrm_ctx_bind_cache(cdlrm_ctx* c, float* const* w, int64_t* const* tags) {
    ARG_CHECK(c && w && tags);
    for (int k = 0; k < c->T; ++k) {
        ARG_CHECK(w[k] && tags[k]);
        ARG_CHECK(((uintptr_t)w[k] & 15) == 0);
        c->tabs[k].weight = w[k];
        c->tabs[k].tags = tags[k];
        if (!c->tabs[k].plan_tags) c->tabs[k].plan_tags = tags[k];
    }
    c->tabs_dirty = true;
    return CDLRM_OK;
}

extern "C" int cdlrm_ctx_bind_plan_tags(cdlrm_ctx* c, int64_t* const* pt) {
    ARG_CHECK(c && pt);
    for (int k = 0; k < c->T; ++k) {
        ARG_CHECK(pt[k]);
        c->tabs[k].plan_tags = pt[k];
    }
    c->tabs_dirty = true;
    return CDLRM_OK;
}

extern "C" int cdlrm_ctx_bind_master(cdlrm_ctx* c, float* const* m) {
    ARG_CHECK(c && m);
    for (int k = 0; k < c->T; ++k) {
        ARG_CHECK(m[k]);
        ARG_CHECK(((uintptr_t)m[k] & 15) == 0 || (c->dim & 3) != 0);
        c->tabs[k].master = m[k];
    }
    c->tabs_dirty = true;
    return CDLRM_OK;
}

extern "C" int cdlrm_ctx_bind_dirty(cdlrm_ctx* c, uint32_t* const* d) {
    ARG_CHECK(c && d);
    for (int k = 0; k < c->T; ++k) c->tabs[k].dirty = d[k];
    c->tabs_dirty = true;
    return CDLRM_OK;
}

extern "C" int cdlrm_stream_create(int device, int priority, cdlrm_stream* out) {
    ARG_CHECK(out);
    CU_CHECK(cudaSetDevice(device));
    int lo = 0, hi = 0;                     // numerically lowest = highest priority
    CU_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    cudaStream_t s = nullptr;
    CU_CHECK(cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, priority < 0 ? hi : lo));
    *out = (cdlrm_stream)s;
    return CDLRM_OK;
}

extern "C" int cdlrm_stream_destroy(int device, cdlrm_stream stream) {
    if (!stream) return CDLRM_OK;
    CU_CHECK(cudaSetDevice(device));
    CU_CHECK(cudaStreamDestroy((cudaStream_t)stream));
    return CDLRM_OK;
}

int cdlrm_sync_tabs(cdlrm_ctx* c, cudaStream_t s) {
    if (!c->tabs_dirty) return CDLRM_OK;
    // Synchronous copy on purpose: bindings change only at set-up time, and a
    // pageable-source async copy would not be legal inside graph capture anyway.
    CU_CHECK(cudaStreamSynchronize(s));
    CU_CHECK(cudaMemcpy(c->d_tabs, c->tabs.data(), sizeof(TableDesc) * c->T, cudaMemcpyHostToDevice));
    c->tabs_dirty = false;
    return CDLRM_OK;
}

extern "C" int cdlrm_ctx_reserve(cdlrm_ctx* c, int64_t max_idx) {
    ARG_CHECK(c && max_idx >= 0);
    CU_CHECK(cudaSetDevice(c->device));
    if (max_idx <= c->scratch_max_idx && c->d_missmap) return CDLRM_OK;
    if (c->d_missmap) {
        CU_CHECK(cudaDeviceSynchronize());
        CU_CHECK(cudaFree(c->d_missmap));
        c->d_missmap = nullptr;
    }
    int64_t words = (max_idx + 31) / 32 + 1;
    CU_CHECK(cudaMalloc(&c->d_missmap, sizeof(uint32_t) * c->T * words));
    c->scratch_max_idx = max_idx;
    return CDLRM_OK;
}

__global__ void fill_i64_kernel(int64_t* p, int64_t n, int64_t v) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) p[i] = v;
}

extern "C" int cdlrm_tags_reset(cdlrm_ctx* c, cdlrm_stream stream) {
    ARG_CHECK(c);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    for (int k = 0; k < c->T; ++k) {
        const TableDesc& t = c->tabs[k];
        ARG_CHECK(t.tags);
        int64_t n = t.num_sets * c->ways;
        int grid = (int)((n + 255) / 256 < 2368 ? (n + 255) / 256 : 2368);
        fill_i64_kernel<<<grid, 256, 0, s>>>(t.tags, n, -1);
        if (t.plan_tags && t.plan_tags != t.tags) fill_i64_kernel<<<grid, 256, 0, s>>>(t.plan_tags, n, -1);
    }
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

extern "C" int cdlrm_ctx_check(cdlrm_ctx* c, cdlrm_stream stream, uint32_t* h_flags) {
    ARG_CHECK(c && h_flags);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    CU_CHECK(cudaMemcpyAsync(h_flags, c->d_flags, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CU_CHECK(cudaMemsetAsync(c->d_flags, 0, sizeof(uint32_t), s));
    CU_CHECK(cudaStreamSynchronize(s));
    return CDLRM_OK;
}

// ---- launch accounting / per-kernel timing -----------------------------------------------------
#include <atomic>
#include <mutex>

static std::atomic<long long> g_launches{0};
static std::atomic<int> g_prof_on{0};
static std::mutex g_prof_mu;
struct ProfRec { int id; cudaEvent_t b, e; };
static std::vector<ProfRec> g_prof;
static const char* const g_knames[K_COUNT] = {
    "embed_fwd", "embed_miss", "pool", "bwd_plan", "bwd_sgd", "bwd_sgd_multi", "interact_fwd", "interact_bwd",
    "plan_bitmap_set", "plan_compact", "plan_probe", "plan_surv", "plan_select", "plan_lists",
    "move_evict", "move_gather", "move_fill", "move_scatter", "agg_mark", "agg_or", "agg_collect",
    "agg_pack", "agg_unpack", "misc", "rng_mt19937", "rng_exp", "mlp_gemm", "mlp_split", "embed_fwd_eval", "eval_metrics",
    "lr_schedule", "null", "embed_victim", "move_carry"};

void cdlrm_prof_mark(int id, cudaStream_t s, int end) {
    if (!end) g_launches.fetch_add(1, std::memory_order_relaxed);
    if (!g_prof_on.load(std::memory_order_relaxed)) return;
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &st) != cudaSuccess || st != cudaStreamCaptureStatusNone) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (!end) {
        ProfRec r{id, nullptr, nullptr};
        cudaEventCreate(&r.b);
        cudaEventCreate(&r.e);
        cudaEventRecord(r.b, s);
        g_prof.push_back(r);
    } else {
        for (size_t i = g_prof.size(); i-- > 0;)
            if (g_prof[i].id == id) {
                cudaEventRecord(g_prof[i].e, s);
                break;
            }
    }
}

// programmatic dependent launch of the per-step kernels (common.cuh); CDLRM_PDL=0 disables it
int g_cdlrm_pdl = [] {
    const char* e = getenv("CDLRM_PDL");
    return (e && e[0] == '0') ? 0 : 1;
}();

extern "C" int cdlrm_set_pdl(int on) {
    g_cdlrm_pdl = on ? 1 : 0;
    return CDLRM_OK;
}

// an empty kernel through the same launch + event-pair path as every other kernel: what cdlrm_prof_report
// returns for it is the overhead the event pair adds to a measured duration
__global__ void null_kernel() {}
extern "C" int cdlrm_prof_null(cdlrm_stream stream) {
    cudaStream_t s = (cudaStream_t)stream;
    LAUNCH(K_NULL, s, (null_kernel<<<1, 32, 0, s>>>()));
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

extern "C" int cdlrm_prof_enable(int on) {
    g_prof_on.store(on ? 1 : 0);
    return CDLRM_OK;
}

extern "C" int64_t cdlrm_prof_launches(int reset) {
    return reset ? g_launches.exchange(0) : g_launches.load();
}

extern "C" int cdlrm_prof_num_kernels(void) { return K_COUNT; }

extern "C" const char* cdlrm_prof_kernel_name(int id) { return (id >= 0 && id < K_COUNT) ? g_knames[id] : ""; }

extern "C" int cdlrm_prof_report(double* h_ms, int64_t* h_calls, int n) {
    ARG_CHECK(h_ms && h_calls && n >= K_COUNT);
    CU_CHECK(cudaDeviceSynchronize());
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (int i = 0; i < n; ++i) { h_ms[i] = 0.0; h_calls[i] = 0; }
    size_t failed = 0;
    cudaError_t first = cudaSuccess;
    for (auto& r : g_prof) {
        float ms = 0.f;
        const cudaError_t e = cudaEventElapsedTime(&ms, r.b, r.e);
        if (e == cudaSuccess) {
            h_ms[r.id] += ms;
            h_calls[r.id] += 1;
        } else {
            if (!failed++) first = e;
            cudaGetLastError();
        }
        cudaEventDestroy(r.b);
        cudaEventDestroy(r.e);
    }
    cudaGetLastError();
    // not an error of the call: cdlrm_last_error() carries the tally for the caller's log
    cdlrm_set_error("prof_report: %zu records, %zu without a duration (%s)", g_prof.size(), failed,
                    failed ? cudaGetErrorString(first) : "-");
    g_prof.clear();
    return CDLRM_OK;
}
