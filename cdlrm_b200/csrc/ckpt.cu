// ckpt.cu -- the list of valid cache lines that a checkpoint or an export of the trained tables walks
// (cdlrm_cache_collect_valid; the state of the victim stream is read and restored in rng.cu).  No reference
// counterpart: the reference's --save-model / --load-model are parsed and never used, and its cache rows are lost at
// exit.
#include "common.cuh"
#include "compact.cuh"

namespace {

// word w of the bitmap covers slots [32 w, 32 w + 32) of the cache region (slot = S * way + set): bit set when the
// line holds an id (live tag >= 0) and its set lies in [set_lo, set_hi)
__global__ void __launch_bounds__(256) valid_bitmap_kernel(TableDesc T, int ways, int64_t set_lo, int64_t set_hi,
                                                           uint32_t* __restrict__ bitmap, int64_t nwords) {
    const int64_t S = T.num_sets, n_slots = S * ways;
    int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; w < nwords; w += stride) {
        uint32_t m = 0;
        int64_t slot = w * 32;
        int64_t way = slot / S, set = slot - way * S;
        for (int b = 0; b < 32 && slot < n_slots; ++b, ++slot) {
            if (set >= set_lo && set < set_hi && __ldg(T.tags + set * ways + way) >= 0) m |= 1u << b;
            if (++set == S) { set = 0; ++way; }
        }
        bitmap[w] = m;
    }
}

// ids[i] = live tag of slots[i], for i < *count (the count the scan left on the device)
__global__ void __launch_bounds__(256) ids_of_slots_kernel(TableDesc T, int ways, const int32_t* __restrict__ slots,
                                                           const unsigned long long* __restrict__ count,
                                                           int64_t* __restrict__ ids) {
    const int64_t n = (int64_t)*count;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const int64_t sl = slots[i];
        const int64_t way = sl / T.num_sets, set = sl - way * T.num_sets;
        ids[i] = T.tags[set * ways + way];
    }
}

}  // namespace

extern "C" int cdlrm_cache_collect_valid(cdlrm_ctx* c, int rank, int world, int32_t* slots, int64_t* ids,
                                         const int64_t* h_list_off, int64_t* h_counts, cdlrm_stream stream) {
    ARG_CHECK(c && world >= 1 && rank >= 0 && rank < world && slots && ids && h_list_off && h_counts);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(c->device));
    int64_t words_max = 0;
    for (int k = 0; k < c->T; ++k) {
        ARG_CHECK(c->tabs[k].tags && h_list_off[k] >= 0);
        const int64_t w = (c->tabs[k].num_sets * c->ways + 31) / 32;
        words_max = w > words_max ? w : words_max;
    }
    // scratch of the bitmap / popcount scan, grown on demand (a checkpoint is not on the training path)
    static thread_local uint32_t* bm = nullptr;
    static thread_local int32_t* bs = nullptr;
    static thread_local unsigned long long* d_counts = nullptr;
    static thread_local int64_t bm_cap = 0, bs_cap = 0, cnt_cap = 0;
    const int64_t nblk_max = (words_max + TILE - 1) / TILE;
    if (words_max > bm_cap) {
        if (bm) cudaFree(bm);
        CU_CHECK(cudaMalloc(&bm, sizeof(uint32_t) * words_max));
        bm_cap = words_max;
    }
    if (nblk_max + 1 > bs_cap) {
        if (bs) cudaFree(bs);
        CU_CHECK(cudaMalloc(&bs, sizeof(int32_t) * (nblk_max + 1)));
        bs_cap = nblk_max + 1;
    }
    if (c->T > cnt_cap) {
        if (d_counts) cudaFree(d_counts);
        CU_CHECK(cudaMalloc(&d_counts, sizeof(unsigned long long) * c->T));
        cnt_cap = c->T;
    }
    for (int k = 0; k < c->T; ++k) {
        const TableDesc& t = c->tabs[k];
        const int64_t S = t.num_sets;
        const int64_t lo = S * rank / world, hi = S * (rank + 1) / world;
        const int64_t nwords = (S * c->ways + 31) / 32;
        const int nblk = (int)((nwords + TILE - 1) / TILE);
        int64_t gb = (nwords + 255) / 256;
        if (gb > (int64_t)c->num_sms * 8) gb = (int64_t)c->num_sms * 8;
        LAUNCH(K_AGG_COLLECT, s, valid_bitmap_kernel<<<(int)gb, 256, 0, s>>>(t, c->ways, lo, hi, bm, nwords));
        LAUNCH(K_AGG_COLLECT, s, bitmap_count_kernel<<<nblk, 256, 0, s>>>(bm, nwords, bs));
        LAUNCH(K_AGG_COLLECT, s, scan_tiles_kernel<<<1, 1024, 0, s>>>(bs, nblk, d_counts + k));
        LAUNCH(K_AGG_COLLECT, s, (bitmap_emit_kernel<int32_t, false><<<nblk, 256, 0, s>>>(bm, nwords, bs, slots + h_list_off[k])));
        int64_t gi = (S * c->ways + 255) / 256;
        if (gi > (int64_t)c->num_sms * 8) gi = (int64_t)c->num_sms * 8;
        LAUNCH(K_AGG_COLLECT, s, ids_of_slots_kernel<<<(int)gi, 256, 0, s>>>(t, c->ways, slots + h_list_off[k], d_counts + k,
                                                                               ids + h_list_off[k]));
    }
    CU_CHECK(cudaGetLastError());
    CU_CHECK(cudaMemcpyAsync(h_counts, d_counts, sizeof(int64_t) * c->T, cudaMemcpyDeviceToHost, s));
    return CDLRM_OK;
}
