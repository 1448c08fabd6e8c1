// lr.cu -- the learning rate of every training step as a value in device memory (cdlrm_lr_state), so that a captured
// step reads it when it runs instead of baking in the value of the step it was captured on.  The schedule is upstream
// DLRM's LRPolicyScheduler (dlrm_s_pytorch.py: --lr-num-warmup-steps, --lr-decay-start-step, --lr-num-decay-steps),
// evaluated on the device; cdlrm_b200.main_no_ddp.lr_policy is its host mirror, the same fp64 operations in the same
// order, rounded to fp32 once.
#include "common.cuh"

namespace {

__device__ __forceinline__ double warmup_lr(double b, int64_t c, int64_t W) {
    return b * (1.0 - (double)(W - c) / (double)W);
}

__device__ __forceinline__ double decay_lr(double b, int64_t c, int64_t D, int64_t N) {
    const double x = (double)(N - (c - D)) / (double)N;
    const double v = b * (x * x);
    return v > 1e-7 ? v : 1e-7;
}

// lr(c) for base b and step count c (1-based), see include/cdlrm_b200.h
__device__ double lr_policy(double b, int64_t c, int64_t W, int64_t D, int64_t N) {
    if (c < W) return warmup_lr(b, c, W);
    if (D <= c && c < D + N) return decay_lr(b, c, D, N);
    if (N == 0) return b;
    if (c >= D + N) return decay_lr(b, D + N - 1, D, N);     // held at the last decay value
    if (W >= 2) return warmup_lr(b, W - 1, W);               // between warmup and decay: held at the last warmup value
    return b;
}

__device__ __forceinline__ void write_lr(cdlrm_lr_state* st) {
    for (int g = 0; g < 2; ++g)
        st->lr[g] = (float)lr_policy(st->base[g], st->count, st->warmup_steps, st->decay_start_step, st->decay_steps);
}

__global__ void lr_set_kernel(cdlrm_lr_state* st, double base_dense, double base_sparse, int64_t W, int64_t D,
                              int64_t N, int64_t count) {
    pdl_enter();
    st->base[0] = base_dense;
    st->base[1] = base_sparse;
    st->warmup_steps = W;
    st->decay_start_step = D;
    st->decay_steps = N;
    st->count = count;
    write_lr(st);
}

__global__ void lr_advance_kernel(cdlrm_lr_state* st) {
    pdl_enter();
    st->count += 1;
    write_lr(st);
}

}  // namespace

extern "C" int cdlrm_lr_set(int device, cdlrm_lr_state* d_state, double base_dense, double base_sparse,
                            int64_t warmup_steps, int64_t decay_start_step, int64_t decay_steps, int64_t count,
                            cdlrm_stream stream) {
    ARG_CHECK(d_state);
    ARG_CHECK(warmup_steps >= 0 && decay_start_step >= 0 && decay_steps >= 0 && count >= 0);
    ARG_CHECK(decay_start_step >= warmup_steps);      // upstream: warmup must finish before the decay starts
    ARG_CHECK(decay_steps <= INT64_MAX - decay_start_step);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(device));
    LAUNCH_PDL(K_LR, s, lr_set_kernel, 1, 1, 0, d_state, base_dense, base_sparse, warmup_steps, decay_start_step,
               decay_steps, count);
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}

extern "C" int cdlrm_lr_advance(int device, cdlrm_lr_state* d_state, cdlrm_stream stream) {
    ARG_CHECK(d_state);
    cudaStream_t s = (cudaStream_t)stream;
    CU_CHECK(cudaSetDevice(device));
    LAUNCH_PDL(K_LR, s, lr_advance_kernel, 1, 1, 0, d_state);
    CU_CHECK(cudaGetLastError());
    return CDLRM_OK;
}
