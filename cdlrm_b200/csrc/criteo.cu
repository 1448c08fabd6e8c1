// criteo.cu -- decode of MLPerf binary Criteo records on the device (data_loader_terabyte.py's CriteoBinDataset
// :195-235 reads them, _transform_features :68-87 turns them into a batch).
//
// A record is 1 + n_dense + n_sparse little-endian int32 fields: [label, dense..., categorical...].  Per record i:
//   T[i]           = (float)label
//   X[i][c]        = logf((float)dense_c + 1.0f)                       torch.log(x_int.float() + 1)
//   ids[k][i]      = (int64)cat_k, floor-modulo max_ind_range if > 0   (x_cat % max_ind_range).long().t()
// The kernel is memory-bound (160 B read, 264 B written per Criteo record): one CTA stages DECODE_ROWS records in
// shared memory with coalesced loads, then writes every output column coalesced -- a warp writes 32 consecutive
// int64 ids of one table.  Rows are padded to an odd word count, so the column reads of a warp (32 rows, one field)
// hit 32 different banks (40 words a row would give 8-way conflicts).
#include "common.cuh"

namespace {

constexpr int DECODE_ROWS = 128;
constexpr int DECODE_THREADS = 256;
constexpr int DECODE_MAX_FIELDS = 95;      // 128 rows x 96 padded words x 4 B = 48 KB: no shared-memory opt-in

__global__ void __launch_bounds__(DECODE_THREADS) criteo_decode_kernel(
        const int32_t* __restrict__ rec, int64_t n, int n_dense, int n_sparse, int64_t max_ind_range, int vec4,
        float* __restrict__ X, int64_t ld_x, int64_t* __restrict__ ids, int64_t ld_ids, float* __restrict__ T) {
    extern __shared__ int32_t tile[];
    const int R = 1 + n_dense + n_sparse;
    const int P = R | 1;                                   // padded row pitch (odd)
    const int64_t row0 = (int64_t)blockIdx.x * DECODE_ROWS;
    const int rows = (int)min((int64_t)DECODE_ROWS, n - row0);
    const int words = rows * R;
    const int32_t* src = rec + row0 * R;
    // stage: the tile's records are one contiguous run of `words` int32
    if (vec4) {                                            // src is 16-byte aligned (R % 4 == 0, rec aligned)
        const int n4 = words >> 2;
        const int4* src4 = reinterpret_cast<const int4*>(src);
        for (int i = threadIdx.x; i < n4; i += DECODE_THREADS) {
            const int4 v = __ldg(src4 + i);
            const int w = i << 2;
            const int r = w / R, c = w - r * R;            // R % 4 == 0: the 4 words share a row
            int32_t* d = tile + r * P + c;
            d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
        }
    } else {
        for (int w = threadIdx.x; w < words; w += DECODE_THREADS) {
            const int r = w / R;
            tile[r * P + (w - r * R)] = __ldg(src + w);
        }
    }
    __syncthreads();
    if (T) {
        for (int r = threadIdx.x; r < rows; r += DECODE_THREADS) T[row0 + r] = (float)tile[r * P];
    }
    if (X) {
        const int m = rows * n_dense;
        for (int e = threadIdx.x; e < m; e += DECODE_THREADS) {
            const int r = e / n_dense, c = e - r * n_dense;
            X[(row0 + r) * ld_x + c] = logf((float)tile[r * P + 1 + c] + 1.0f);
        }
    }
    if (ids) {
        const int m = rows * n_sparse;
        const int c0 = 1 + n_dense;
        for (int e = threadIdx.x; e < m; e += DECODE_THREADS) {
            const int k = e / rows, r = e - k * rows;
            const int32_t x = tile[r * P + c0 + k];
            int64_t v = (int64_t)x;
            if (max_ind_range > 0) {                       // torch's %: the result takes the divisor's sign
                if (max_ind_range <= 0x7fffffff) {
                    const int32_t m = (int32_t)max_ind_range, q = x % m;
                    v = (int64_t)(q < 0 ? q + m : q);
                } else {
                    v %= max_ind_range;
                    if (v < 0) v += max_ind_range;
                }
            }
            ids[(int64_t)k * ld_ids + row0 + r] = v;
        }
    }
}

}  // namespace

extern "C" int cdlrm_criteo_decode(int device, const int32_t* rec, int64_t n, int32_t n_dense, int32_t n_sparse,
                                   int64_t max_ind_range, float* X, int64_t ld_x, int64_t* ids, int64_t ld_ids,
                                   float* T, cdlrm_stream stream) {
    ARG_CHECK(n >= 0 && n_dense >= 0 && n_sparse >= 0);
    ARG_CHECK(1 + n_dense + n_sparse <= DECODE_MAX_FIELDS);
    ARG_CHECK(n == 0 || rec != nullptr);
    ARG_CHECK(((uintptr_t)rec & 3) == 0);
    ARG_CHECK(!X || (ld_x >= n_dense && ((uintptr_t)X & 3) == 0));
    ARG_CHECK(!ids || (ld_ids >= n && ((uintptr_t)ids & 7) == 0));
    ARG_CHECK(!T || ((uintptr_t)T & 3) == 0);
    ARG_CHECK((n + DECODE_ROWS - 1) / DECODE_ROWS <= 0x7fffffff);
    if (n == 0 || (!X && !ids && !T)) return CDLRM_OK;
    CU_CHECK(cudaSetDevice(device));
    const int R = 1 + n_dense + n_sparse;
    const int vec4 = (R % 4 == 0) && (((uintptr_t)rec & 15) == 0);
    const size_t smem = (size_t)DECODE_ROWS * (R | 1) * sizeof(int32_t);
    cudaStream_t s = (cudaStream_t)stream;
    const unsigned grid = (unsigned)((n + DECODE_ROWS - 1) / DECODE_ROWS);
    LAUNCH(K_MISC, s, criteo_decode_kernel<<<grid, DECODE_THREADS, smem, s>>>(
        rec, n, n_dense, n_sparse, max_ind_range, vec4, X, ld_x, ids, ld_ids, T));
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}
