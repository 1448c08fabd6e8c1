/* cdlrm_b200.h -- C ABI of libcdlrm_b200.so: the B200-native (sm_100a) look-ahead
 * embedding-cache hot path of cDLRM.
 *
 * The reference (lkp411/cDLRM) is pure Python on PyTorch and has no FFI layer; its
 * boundary for this path is the Python API of cache_manager.py / model_no_ddp.py /
 * main_no_ddp.py.  The same-named Python modules in cdlrm_b200/ keep that API and
 * call the entry points below through ctypes (see INTEGRATION.md).  Every entry
 * point cites the reference code it replaces as file:line in the reference tree.
 *
 * Conventions
 *  - plain C types only; pointers are DEVICE pointers unless the name starts with
 *    h_ (host).  "master" pointers are device-visible addresses of the host-pinned
 *    (cudaHostRegister/cudaHostAlloc mapped) master embedding tables, or plain
 *    device pointers when the master is kept in HBM.
 *  - every compute call enqueues work on `stream` (a cudaStream_t) and returns
 *    without synchronising unless stated.  Return value 0 = OK, <0 = error; the
 *    message is available from cdlrm_last_error() (thread-local).
 *  - one cdlrm_ctx per (process, device); a ctx is not thread-safe.
 *  - there is NO CPU fallback: without a CUDA device every compute call fails.
 *  - table-range calls take (table_begin, table_count) and strided per-table
 *    operands: operand of table k lives at base + (k - table_begin) * ld.
 *  - cache slot numbering is the reference's: slot = num_sets * way + set
 *    (model_no_ddp.py:174), aux (victim) slots start at num_sets * num_ways
 *    (model_no_ddp.py:177); tags are int64, -1 = empty (model_no_ddp.py:144-147).
 */
#ifndef CDLRM_B200_H
#define CDLRM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CDLRM_ABI_VERSION 1
#define CDLRM_MAX_WAYS 64          /* pin masks are 64-bit */
#define CDLRM_MAX_PEERS 8          /* ranks of one node that can share a sharded loser store */
#define CDLRM_IPC_HANDLE_BYTES 64  /* sizeof(cudaIpcMemHandle_t) */
#define CDLRM_SORT_MAX 16384       /* ids per table sorted by one CTA in the backward plan */

typedef struct cdlrm_ctx cdlrm_ctx;
typedef struct cdlrm_rng cdlrm_rng;
typedef struct cdlrm_rngdev cdlrm_rngdev;
typedef void* cdlrm_stream;        /* cudaStream_t */

/* ---- status -------------------------------------------------------------------- */
int cdlrm_abi_version(void);
const char* cdlrm_last_error(void);

/* ---- geometry: model_no_ddp.py:122-125 (find_next_prime), :319-331 (isPrime) ---- */
int cdlrm_is_prime_ref(int64_t n);
int64_t cdlrm_find_next_prime(int64_t max_cache_size);   /* -1 if none in [c, 2c) */

/* ---- context: Embedding_Table_Cache_Group.__init__/create_emb/
 *      create_occupancy_tables, model_no_ddp.py:102-147 -------------------------- */
int cdlrm_ctx_create(cdlrm_ctx** out, int device, int num_tables, int dim, int num_ways,
                     int64_t aux_rows, const int64_t* h_n_rows, int64_t max_cache_size);
int cdlrm_ctx_destroy(cdlrm_ctx* ctx);
/* h_num_sets[k] = min(n_rows[k], find_next_prime(max_cache_size)) (:113,136);
 * h_cache_rows[k] = num_ways * num_sets[k] + aux_rows (:138) */
int cdlrm_ctx_geometry(const cdlrm_ctx* ctx, int64_t* h_num_sets, int64_t* h_cache_rows);
/* storage is owned by the caller (PyTorch): weight[k] float32 [cache_rows[k], dim],
 * tags[k] int64 [num_sets[k], num_ways]; h_* are host arrays of device pointers */
int cdlrm_ctx_bind_cache(cdlrm_ctx* ctx, float* const* h_weight, int64_t* const* h_tags);
/* the planner's look-ahead copy of the tags (may equal the live tags) */
int cdlrm_ctx_bind_plan_tags(cdlrm_ctx* ctx, int64_t* const* h_plan_tags);
/* master tables: Embedding_Table_Group.emb_l[k].weight, model_no_ddp.py:21-98 */
int cdlrm_ctx_bind_master(cdlrm_ctx* ctx, float* const* h_master);
/* dirty-slot bitmaps for the table aggregation: ceil(cache_rows[k]/32) uint32 words */
int cdlrm_ctx_bind_dirty(cdlrm_ctx* ctx, uint32_t* const* h_dirty);
/* pre-size internal scratch for batches of up to max_idx ids per table (optional;
 * scratch otherwise grows on demand, which is not allowed during graph capture) */
int cdlrm_ctx_reserve(cdlrm_ctx* ctx, int64_t max_idx);
/* tags[k][:] = -1 for all tables (live and plan copies) */
int cdlrm_tags_reset(cdlrm_ctx* ctx, cdlrm_stream stream);
/* sticky device-side error flags (bit0: aux region overflow, model_no_ddp.py:177-179
 * would raise IndexError; bit1: id outside its table; bit2: a miss whose id is not in the bound loser store,
 * cdlrm_embed_victim_update); synchronises `stream`; clears the flags */
int cdlrm_ctx_check(cdlrm_ctx* ctx, cdlrm_stream stream, uint32_t* h_flags);

/* ---- forward: Embedding_Table_Cache_Group.forward, model_no_ddp.py:149-212 ------
 * per table k and id j: set = id mod num_sets; probe the tag line; hit ->
 * slot = num_sets*way+set; miss -> slot = num_sets*num_ways + ordinal (batch order),
 * weight[slot] = master[id]; out[b] = sum_{j in bag b} weight[slot_j].
 * offsets == NULL means one id per bag (Criteo, data_loader_terabyte.py:85).
 * out: float32 [n_bags, dim]; slots: int32 [n_idx]; n_miss: int32 [table_count];
 * bag_ids (optional, may be NULL): int32 [n_idx] bag index of every id (needed by
 * the backward when offsets != NULL). */
int cdlrm_embed_fwd(cdlrm_ctx* ctx, int table_begin, int table_count,
                    const int64_t* ids, int64_t ld_ids,
                    const int64_t* offsets, int64_t ld_off,
                    int32_t n_idx, int32_t n_bags,
                    float* out, int64_t ld_out,
                    int32_t* slots, int64_t ld_slots,
                    int32_t* n_miss,
                    int32_t* bag_ids, int64_t ld_bag,
                    cdlrm_stream stream);

/* Read-only lookup for evaluation, one id per bag: out[j] = the cache row of ids[j] when its set's tag line holds it,
 * else its row in the loser store of the installed window, else master[ids[j]] (zero-copy).  Writes out only (no
 * slots, aux rows, miss bitmap or dirty bits; no batch limit, no allocation).  An id outside its table raises flag 2
 * (cdlrm_ctx_check) and gets a zero row.  out: float32 [table_count][n_idx][dim], table stride ld_out. */
int cdlrm_embed_fwd_eval(cdlrm_ctx* ctx, int table_begin, int table_count, const int64_t* ids, int64_t ld_ids,
                         int32_t n_idx, float* out, int64_t ld_out, cdlrm_stream stream);

/* ---- backward + SGD: autograd of EmbeddingBag(sparse=True) followed by
 *      optimizer_embeds.step(), main_no_ddp.py:376,409,413 -------------------------
 * weight[slot] -= lr * sum_{j: slot_j == slot} d_out[bag(j)], duplicates merged by a
 * per-table sort (plain read-modify-write per slot; atomics only where the run of one slot
 * crosses a 32-entry range of the sorted order: hot rows, tiny tables).
 * d_out row of bag b of table k: d_out + (k-table_begin)*ld_dout + b*dout_row_stride.
 * Marks touched slots in the dirty bitmaps when bound.  */
int64_t cdlrm_embed_bwd_plan_bytes(int table_count, int32_t n_idx);
int cdlrm_embed_bwd_plan(cdlrm_ctx* ctx, int table_begin, int table_count,
                         const int32_t* slots, int64_t ld_slots, int32_t n_idx,
                         void* plan, cdlrm_stream stream);
/* key 0: thread-block cluster size of the backward plan's multi-CTA radix sort (1, 2, 4, 8; 0 = the one-CTA-per-table
 * kernel; -1 = default: environment CDLRM_PLAN_CLUSTER, else 8).  Same sorted run either way. */
int cdlrm_embed_set_option(int key, int value);
int cdlrm_embed_bwd_sgd(cdlrm_ctx* ctx, int table_begin, int table_count,
                        const void* plan, int32_t n_idx,
                        const int32_t* bag_ids, int64_t ld_bag,
                        const float* d_out, int64_t ld_dout, int64_t dout_row_stride,
                        float lr, cdlrm_stream stream);
/* The same update with the learning rate read from device memory when the kernels run (*d_lr, one float: a
 * cdlrm_lr_state's lr[1]), so that a CUDA graph replays whatever value the buffer holds; equal bit for bit to
 * cdlrm_embed_bwd_sgd with lr = *d_lr. */
int cdlrm_embed_bwd_sgd_dlr(cdlrm_ctx* ctx, int table_begin, int table_count,
                            const void* plan, int32_t n_idx,
                            const int32_t* bag_ids, int64_t ld_bag,
                            const float* d_out, int64_t ld_dout, int64_t dout_row_stride,
                            const float* d_lr, cdlrm_stream stream);

/* ---- update of the misses (--evict-victim-cache; the reference parses the flag and drops these updates) ----------
 * A miss of the step is a position j whose slot is an aux slot (>= num_sets * num_ways); its row came from the loser
 * store bound with cdlrm_ctx_bind_losers.  Per table and store row i:
 *     store[i] = fma(-lr, sum of d_out[bag(j)] over the misses j on i in ascending j, store[i])
 * (bag(j) = bag_ids[j], or j with bag_ids == NULL; d_out rows as in cdlrm_embed_bwd_sgd).  A miss whose id is not in
 * the store raises flag 4 (cdlrm_ctx_check) and is not applied.  Deterministic, capturable, allocates nothing; at most
 * CDLRM_SORT_MAX misses per table (min(aux_rows, n_idx) <= CDLRM_SORT_MAX). */
int cdlrm_embed_victim_update(cdlrm_ctx* ctx, int table_begin, int table_count,
                              const int32_t* slots, int64_t ld_slots, const int64_t* ids, int64_t ld_ids, int32_t n_idx,
                              const int32_t* bag_ids, int64_t ld_bag,
                              const float* d_out, int64_t ld_dout, int64_t dout_row_stride,
                              float lr, cdlrm_stream stream);
/* The same with the learning rate read from *d_lr when the kernel runs (a cdlrm_lr_state's lr[1]). */
int cdlrm_embed_victim_update_dlr(cdlrm_ctx* ctx, int table_begin, int table_count,
                                  const int32_t* slots, int64_t ld_slots, const int64_t* ids, int64_t ld_ids,
                                  int32_t n_idx, const int32_t* bag_ids, int64_t ld_bag,
                                  const float* d_out, int64_t ld_dout, int64_t dout_row_stride,
                                  const float* d_lr, cdlrm_stream stream);

/* ---- interaction: DLRM_Net.interact_features ("dot"), model_no_ddp.py:272-293 ---
 * feat[0] = x, feat[1..] = ly; h_feat is a host array of n_feat device pointers to
 * float32 [B, dim] matrices with row stride feat_row_stride (elements).
 * out[b] = [x[b], <T_i, T_j> for i in 0..n_feat-1 for j in 0..i-1 (+ j == i if itself)]
 * out row stride ld_out >= dim + n_pairs. */
/* kernel variant (process-wide): key 0, value 0 = CUDA-core kernels (default), 1 = mma.sync 3xTF32 tensor-core
 * kernels (measured slower on B200, kept for the comparison), 2 = the first CUDA-core forward (shuffle butterfly) */
/* key 1: 1 (default) = software-pipelined backward for dim 128 (persistent CTAs, bulk async copies into a two-stage
 * shared-memory ring; taken when d_out rows are 16-byte aligned, ld_dout % 4 == 0), 0 = the plain kernel;
 * key 2: pipelined forward variants (1 = two-stage rings, 2 = one-stage rings; default 0 = plain kernel: neither
 * variant is faster on B200) */
int cdlrm_interact_set_option(int key, int value);
int cdlrm_interact_fwd(int device, const float* const* h_feat, int n_feat, int64_t feat_row_stride,
                       int32_t batch, int dim, int itself, float* out, int64_t ld_out,
                       cdlrm_stream stream);
/* d_feat plane i (float32 [B, dim], contiguous) at d_feat + i*ld_dfeat receives the
 * gradient of feat[i] (plane 0 also receives d_out[:, :dim]). */
int cdlrm_interact_bwd(int device, const float* const* h_feat, int n_feat, int64_t feat_row_stride,
                       int32_t batch, int dim, int itself, const float* d_out, int64_t ld_dout,
                       float* d_feat, int64_t ld_dfeat, cdlrm_stream stream);

/* ---- dense MLPs: DLRM_Net.create_mlp / bot_l / top_l, model_no_ddp.py:244-270,306-316
 *      (SURVEY section 8(f) rank 4; the layers either side of the interaction) --------
 * Layer l: y = act(x W_l^T + b_l), W_l float32 [dims[l+1], dims[l]] (nn.Linear layout),
 * act = ReLU, or Sigmoid for l == sigmoid_layer (:262-265).  FP32 results (3xTF32 split
 * products with FP32 accumulation on the tensor cores; see csrc/mlp.cu).
 * The object keeps the activations of the last forward in the caller's workspace
 * (256-byte aligned, cdlrm_mlp_workspace_bytes) for the backward:
 *   dW_l = dZ_l^T x_l, db_l = column sums of dZ_l, dx = dZ_0 W_0 (optional, may be NULL),
 * with dZ the gradient w.r.t. the pre-activation.  h_W/h_b/h_dW/h_db are HOST arrays of
 * n_layers DEVICE pointers; dW_l [dims[l+1], dims[l]] and db_l [dims[l+1]] are dense. */
typedef struct cdlrm_mlp cdlrm_mlp;
int64_t cdlrm_mlp_workspace_bytes(int n_layers, const int32_t* h_dims, int32_t batch_cap);
int cdlrm_mlp_create(cdlrm_mlp** out, int device, int n_layers, const int32_t* h_dims,
                     int32_t batch_cap, int sigmoid_layer, void* workspace, int64_t workspace_bytes);
int cdlrm_mlp_destroy(cdlrm_mlp* mlp);
/* sigmoid_layer == -2: the last layer has no activation (plain affine layer; test hook).
 * Numerics knobs (process-wide; defaults are the accurate settings): key 0 = operand split
 * rounding (0 nearest, 1 truncate), key 1 = k-blocks of 32 chained into one TMEM accumulator
 * before the partial sum is added in registers (0 = whole K, default 8), key 2 = tile width
 * (0: 128 x 128, 1: 128 x 256, 2: by shape), key 3 = measurement switches (results invalid), key 5 = weight-gradient
 * GEMMs of the backward on a side stream beside the data-gradient chain (1, default) or in line (0). */
int cdlrm_mlp_set_option(int key, int value);
/* With key 5 on, cdlrm_mlp_backward joins the side stream before it returns, unless defer_join is set on the
 * object: then dW / db are complete on the caller's stream only after cdlrm_mlp_join(mlp, stream) -- which lets
 * the weight gradients of the top MLP run beside the interaction backward and the bottom MLP.  A forward or
 * backward of the same object joins implicitly. */
/* Optimizer step of the dense parameters (main_no_ddp.py:413, torch.optim.SGD.step on the MLPs) fused with the
 * operand split of the updated weights: for the n_mlps (1 or 2) objects in turn, layer by layer, W <- W - lr * dW
 * (h_W / h_dW: host arrays of device pointers, dense [dims[l+1], dims[l]]), written back AND as the hi / lo operand
 * copies the next forward needs (which then skips its own split launch); vec <- vec - lr * vec_grad (vec_n floats: the
 * biases) in the same launch.  The weights must not change between this call and the next forward of each object
 * (cdlrm_mlp_invalidate_split otherwise). */
int cdlrm_mlp_sgd_split(int n_mlps, cdlrm_mlp* const* mlps, float* const* h_W, const float* const* h_dW, float lr,
                        float* vec, const float* vec_grad, int64_t vec_n, cdlrm_stream stream);
/* The same step with the learning rate read from device memory when the kernel runs (*d_lr: a cdlrm_lr_state's
 * lr[0]); equal bit for bit to cdlrm_mlp_sgd_split with lr = *d_lr. */
int cdlrm_mlp_sgd_split_dlr(int n_mlps, cdlrm_mlp* const* mlps, float* const* h_W, const float* const* h_dW,
                            const float* d_lr, float* vec, const float* vec_grad, int64_t vec_n, cdlrm_stream stream);
int cdlrm_mlp_invalidate_split(cdlrm_mlp* mlp);
int cdlrm_mlp_set_defer_join(cdlrm_mlp* mlp, int on);
int cdlrm_mlp_join(cdlrm_mlp* mlp, cdlrm_stream stream);
/* measurement hook: CTA 0 of every following GEMM writes %globaltimer stamps into d_buf (4 x 128 int64); NULL = off */
int cdlrm_mlp_set_trace(void* d_buf);
int cdlrm_mlp_forward(cdlrm_mlp* mlp, const float* x, int64_t ldx, int32_t batch,
                      const float* const* h_W, const float* const* h_b,
                      float* y, int64_t ldy, cdlrm_stream stream);
int cdlrm_mlp_backward(cdlrm_mlp* mlp, const float* dy, int64_t lddy, float* dx, int64_t lddx,
                       float* const* h_dW, float* const* h_db, cdlrm_stream stream);

/* ---- learning-rate schedule: upstream DLRM's LRPolicyScheduler (dlrm_s_pytorch.py, --lr-num-warmup-steps W,
 *      --lr-decay-start-step D, --lr-num-decay-steps N), evaluated on the device --------------------------------
 * A caller-owned device buffer holds the learning rates of the current step, which the *_dlr update entry points
 * read, so that a captured training step follows the schedule and host-side changes of the base on replay.
 * For base b and the 1-based step count c, in fp64 rounded to fp32 once:
 *   c < W                    b * (1 - (W - c) / W)                               (warmup)
 *   D <= c < D + N           max(1e-7, b * x * x),  x = (N - (c - D)) / N         (decay)
 *   otherwise, N == 0        b
 *   otherwise, c >= D + N    the value at c = D + N - 1
 *   otherwise, W >= 2        the value at c = W - 1  (held between warmup and decay, as upstream does)
 *   otherwise                b */
typedef struct cdlrm_lr_state {
    float lr[2];                 /* [dense, sparse]: learning rates of the current step (step count `count`) */
    double base[2];              /* [dense, sparse]: base learning rates b */
    int64_t warmup_steps, decay_start_step, decay_steps;   /* W, D, N */
    int64_t count;               /* steps run so far */
} cdlrm_lr_state;
/* Writes bases, schedule and count, and lr[g] = lr(count) for both groups: with W = D = N = 0 that is fp32(base),
 * and nothing else needs to run per step.  A one-thread kernel in stream order (no host-to-device copy, which could
 * queue behind bulk copies on the copy engine).  Refuses W, D or N negative, D < W, a negative count. */
int cdlrm_lr_set(int device, cdlrm_lr_state* d_state, double base_dense, double base_sparse, int64_t warmup_steps,
                 int64_t decay_start_step, int64_t decay_steps, int64_t count, cdlrm_stream stream);
/* One step: count += 1, lr[g] = lr(count).  Capturable; launched at the start of every step when a schedule is set. */
int cdlrm_lr_advance(int device, cdlrm_lr_state* d_state, cdlrm_stream stream);

/* ---- window planner: Prefetcher.process_batch_slice (cache_manager.py:27-46, the
 *      torch.unique at :32) + the decision part of CacheEmbeddings
 *      (main_no_ddp.py:155-204) ---------------------------------------------------- */
/* bytes of planner workspace needed for windows of up to window_len ids per table */
int64_t cdlrm_plan_workspace_bytes(const cdlrm_ctx* ctx, int64_t window_len);
int cdlrm_plan_bind_workspace(cdlrm_ctx* ctx, void* workspace, int64_t bytes, int64_t window_len);
/* unique only (all tables): the torch.unique of cache_manager.py:32.  Writes
 * h_counts[k*4] = number of unique ids of table k (other three entries 0). */
int cdlrm_plan_unique(cdlrm_ctx* ctx, const int64_t* win_ids, int64_t ld, int64_t n,
                      int64_t* h_counts, cdlrm_stream stream);
/* Chunked window scan: OR the ids of a chunk (int64 [num_tables][n], table k at ids + k*ld) into the planner's id
 * bitmaps.  Any number of calls, in any order, then cdlrm_plan_phase_a with win_ids == NULL and n = the number of
 * ids marked per table (an upper bound of the distinct ids): the window never has to exist as one tensor. */
int cdlrm_plan_mark_ids(cdlrm_ctx* ctx, const int64_t* ids, int64_t ld, int64_t n, cdlrm_stream stream);
/* Data-parallel ranks: mark the ids of the window that THIS rank's own batches contain (any number of chunks, int64
 * [num_tables][n]).  The next cdlrm_plan_losers then lists only those un-cached ids -- the ones this rank's forwards will
 * miss on (model_no_ddp.py:176-179) -- instead of the union over all ranks, and clears the marks. */
int cdlrm_plan_mark_own_ids(cdlrm_ctx* ctx, const int64_t* ids, int64_t ld, int64_t n, cdlrm_stream stream);
/* Eviction lists of the following cdlrm_plan_phase_b* calls: on = 0 (default) one entry per claimant of a replaced
 * (set, way), flagged primary for the winner -- the reference's lists (main_no_ddp.py:190-199: `evicted` holds every
 * claimant's old tag); on = 1 only the winners (all primary): the rows the write-back (cache_manager.py:48-64) uses. */
int cdlrm_plan_set_primary_evictions(cdlrm_ctx* ctx, int on);
/* Scan sharded over the `world` ranks of a node (every rank marked its own share of the window with
 * cdlrm_plan_mark_ids): OR the id bitmaps of the other ranks into this rank's, reading them in place over NVLink.
 * h_peer_ws[r] = device address on THIS device of rank r's planner workspace (cdlrm_peer_alloc / cdlrm_peer_open;
 * the entry of `rank` itself is ignored).  The caller orders it between two host barriers: after every rank's marks
 * are complete, and before any rank's phase A (which clears the bitmaps) starts.  Replaces nothing in the reference
 * as code: cache_manager.py:27-46 scans the whole window in one worker pool; here the scan of an N-GPU job's global
 * window would otherwise be repeated on all N ranks. */
int cdlrm_plan_or_peer_bitmaps(cdlrm_ctx* ctx, const void* const* h_peer_ws, int world, int rank, cdlrm_stream stream);
/* phase A, all tables: unique ids of the window (ascending), probe against the plan
 * tags, pin hit ways, drop misses whose set is fully pinned, rank the survivors.
 * win_ids of table k at win_ids + k*ld (int64 [n]).  If h_uniq != NULL ids are taken
 * as already-unique ascending lists of length h_uniq_len[k] (the reference-API path).
 * Writes h_counts[k*4 + {0,1,2,3}] = {unique, hits, dropped, survivor rows}
 * (pinned host memory, valid after the stream is synchronised). */
int cdlrm_plan_phase_a(cdlrm_ctx* ctx, const int64_t* win_ids, int64_t ld, int64_t n,
                       const int64_t* h_uniq_len, int64_t* h_counts, cdlrm_stream stream);
/* phase B, all tables: q is the concatenation over tables of float32 [rows_k, num_ways]
 * exponential draws (main_no_ddp.py:183-185, see cdlrm_rng_*).  Chooses the way
 * argmax(probs/q) among un-pinned ways, resolves duplicate (set, way) claims
 * (last survivor wins), updates the plan tags and emits per table:
 *   evict_ids / evict_slots / evict_primary [E_k]  (survivor order, duplicates kept;
 *       primary = 1 for exactly one entry per distinct slot)
 *   fill_ids / fill_slots [F_k]                     (winners only, survivor order)
 * lists of table k start at element list_off[k] = sum_{j<k} rows_j of each output
 * array (rows_j from phase A).  h_counts2[k*2+{0,1}] = {E_k, F_k}. */
int cdlrm_plan_phase_b(cdlrm_ctx* ctx, const float* q, const int64_t* h_rows,
                       int64_t* evict_ids, int32_t* evict_slots, uint8_t* evict_primary,
                       int64_t* fill_ids, int32_t* fill_slots,
                       int64_t* h_counts2, cdlrm_stream stream);
/* phase B with the device-resident victim stream (cdlrm_rngdev_*): the draws of table k are
 * generated on the GPU into raw_scratch (uint32 pairs, capacity raw_draws >= max_k rows_k * num_ways
 * draws) right before table k's selection and transformed inside the select kernel; the stream
 * advances by exactly sum_k rows_k * num_ways draws, as the reference's generator does. */
int cdlrm_plan_phase_b_dev(cdlrm_ctx* ctx, cdlrm_rngdev* rng, uint32_t* raw_scratch, int64_t raw_draws,
                           const int64_t* h_rows,
                           int64_t* evict_ids, int32_t* evict_slots, uint8_t* evict_primary,
                           int64_t* fill_ids, int32_t* fill_slots,
                           int64_t* h_counts2, cdlrm_stream stream);
/* Loser list: ascending ids of the window that are NOT cached after the install (lost a contested
 * slot, main_no_ddp.py:204 last-wins, or dropped because their set was fully pinned, :173-180).
 * Call after phase B on the same stream.  h_uniq[k] = unique count of phase A; the list of table k
 * is written at loser_ids + h_off[k] (capacity dropped_k + rows_k); h_counts3[k] = its length. */
int cdlrm_plan_losers(cdlrm_ctx* ctx, const int64_t* h_uniq, const int64_t* h_off, int64_t* loser_ids,
                      int64_t* h_counts3, cdlrm_stream stream);
/* Loser store: per table the ascending loser ids and a copy of their master rows staged in HBM
 * (h_* are host arrays of device pointers / counts; NULL clears).  The forward's miss path
 * (model_no_ddp.py:176-179) then reads those rows from HBM instead of the host master; ids that
 * are not in the store still go to the master.  Takes effect in stream order. */
int cdlrm_ctx_bind_losers(cdlrm_ctx* ctx, const int64_t* const* h_ids, const float* const* h_rows,
                          const int64_t* h_n, cdlrm_stream stream);
/* unique ids of table k found by the last phase A (device pointer into the
 * workspace, ascending, h_counts[k*4] entries) */
const int64_t* cdlrm_plan_unique_ptr(const cdlrm_ctx* ctx, int table);
/* out[0..n) = first n unique ids of table k found by the last unique / phase A */
int cdlrm_plan_copy_unique(cdlrm_ctx* ctx, int table, int64_t* out, int64_t n, cdlrm_stream stream);

/* ---- mover: the data part of CacheEmbeddings (main_no_ddp.py:190-199,205-206) and
 *      Prefetcher.eviction_manager (cache_manager.py:48-64) ------------------------- */
/* rows_out[e] = weight[k][evict_slots[e]] (if rows_out != NULL); if write_master:
 * master[k][id] = row, or (master[k][id] + row)/2 when average_on_writeback
 * (primary entries only) */
int cdlrm_move_evict(cdlrm_ctx* ctx, int table, const int64_t* evict_ids, const int32_t* evict_slots,
                     const uint8_t* evict_primary, int64_t n, float* rows_out,
                     int write_master, int average_on_writeback, cdlrm_stream stream);
/* eviction_manager body for rows that are already packed (cache_manager.py:58-62):
 * master[k][ids[i]] = rows[i], or (master + rows[i]) / 2; ids must be distinct when
 * averaging */
int cdlrm_move_scatter_master(cdlrm_ctx* ctx, int table, const int64_t* ids, int64_t n, const float* rows,
                              int average_on_writeback, cdlrm_stream stream);
/* the same with a per-entry primary mask (may be NULL): entries with primary[i] == 0 are skipped
 * (an evict list keeps duplicates of a slot; they carry identical rows) */
int cdlrm_move_scatter_master2(cdlrm_ctx* ctx, int table, const int64_t* ids, const uint8_t* primary, int64_t n,
                               const float* rows, int average_on_writeback, cdlrm_stream stream);
/* rows_out[i] = master[k][ids[i]]: Embedding_Table_Group.fetch_unique_idx_slices,
 * model_no_ddp.py:80-87 (zero-copy gather over PCIe when the master is host-pinned) */
int cdlrm_move_gather_master(cdlrm_ctx* ctx, int table, const int64_t* ids, int64_t n,
                             float* rows_out, cdlrm_stream stream);
/* weight[k][fill_slots[i]] = rows[src_index ? src_index[i] : i] (rows == NULL: read
 * master[k][fill_ids[i]] directly); live tags[k][slot % S][slot / S] = fill_ids[i] */
int cdlrm_move_fill(cdlrm_ctx* ctx, int table, const int64_t* fill_ids, const int32_t* fill_slots,
                    int64_t n, const float* rows, const int64_t* src_index, cdlrm_stream stream);
/* rows_inout[i] = the row of ids[i] in the currently bound loser store of table k, for every ids[i] the store holds;
 * the other rows are left alone (--evict-victim-cache: the next window's prefetched rows of ids trained in this
 * window's store).  No store ever bound: nothing to do. */
int cdlrm_move_carry_losers(cdlrm_ctx* ctx, int table, const int64_t* ids, int64_t n, float* rows_inout,
                            cdlrm_stream stream);

/* ---- table aggregation: broadcast_and_aggregate, main_no_ddp.py:250-292 ---------
 * collect: ascending list of dirty slots per table (torch.unique(sorted=True) :270);
 *          slot_list int32 [sum cache_rows] capacity, d_counts int64 [num_tables]
 *          (device) and h_counts (pinned host, may be NULL).
 * pack:    buf[i] = weight[k][slot_i] / divisor (:273-281); unpack: weight[k][slot_i] = buf[i]
 *          (:292) and clears the dirty bits.  List of table k starts at h_list_off[k]. */
/* mark: set the dirty bit of every slot in idxs (int32 [table_count][n], table k at
 * idxs + k*ld) -- the reference's cache_group_idxs argument (main_no_ddp.py:251,268) */
int cdlrm_agg_mark(cdlrm_ctx* ctx, const int32_t* idxs, int64_t ld, int64_t n, cdlrm_stream stream);
int cdlrm_agg_or_bitmaps(cdlrm_ctx* ctx, const uint32_t* gathered, int world, int64_t words_total,
                         cdlrm_stream stream);
int cdlrm_agg_collect(cdlrm_ctx* ctx, int32_t* slot_list, int64_t* d_counts, int64_t* h_counts,
                      cdlrm_stream stream);
int cdlrm_agg_pack(cdlrm_ctx* ctx, const int32_t* slot_list, const int64_t* h_counts,
                   float divisor, float* buf, cdlrm_stream stream);
int cdlrm_agg_unpack(cdlrm_ctx* ctx, const int32_t* slot_list, const int64_t* h_counts,
                     const float* buf, int clear_dirty, cdlrm_stream stream);

/* ---- checkpoint / export of the trained tables (csrc/ckpt.cu).  No reference counterpart: the reference parses
 *      --save-model / --load-model and ignores them, and its cache rows never reach the master at exit. --------------
 * For every table k, the valid lines (live tag >= 0) whose set lies in rank `rank`'s share
 * [S_k * rank / world, S_k * (rank + 1) / world) of the sets, in ascending slot order (slot = S_k * way + set):
 * slots[h_list_off[k] + i] (int32) and ids[h_list_off[k] + i] (int64, the tag of that line), i < h_counts[k].
 * The list of table k needs room for num_ways * S_k entries.  h_counts: pinned host int64 [num_tables], valid after
 * `stream` is synchronised.  The shares of `world` ranks cover every valid line exactly once. */
int cdlrm_cache_collect_valid(cdlrm_ctx* ctx, int rank, int world, int32_t* slots, int64_t* ids,
                              const int64_t* h_list_off, int64_t* h_counts, cdlrm_stream stream);

/* ---- host memory: pin (cudaHostRegister, mapped + portable) a master table that lives
 *      in ordinary or shared host memory (emb_tables.share_memory(), main_no_ddp.py:621-622)
 *      and return its device-visible address ---------------------------------------- */
int cdlrm_host_register(int device, void* h_ptr, int64_t bytes, void** dev_ptr);
int cdlrm_host_unregister(void* h_ptr);

/* ---- measurement: every kernel launch of the library is counted; with profiling enabled
 *      each launch is additionally bracketed by CUDA events on its own stream ------------- */
/* ---- loss of the training step: torch.nn.BCELoss(reduction="mean") (main_no_ddp.py:355-369, 403-405) and its
 *      derivative in one launch: loss[0] = mean(-(t log z + (1-t) log(1-z))) (logs clamped at -100 as torch
 *      does), dz[i] = (z_i - t_i) / max(z_i (1 - z_i), 1e-12) / n.  z, t: n float32 values with element strides
 *      ldz / ldt; dz: n contiguous float32. */
int cdlrm_bce_mean(int device, const float* z, int64_t ldz, const float* t, int64_t ldt, int32_t n, float* loss,
                   float* dz, cdlrm_stream stream);

/* ---- host side of the copy-engine prefetch / write-back (csrc/hostio.cu) -----------------------------------------
 * The scattered half of a master <-> GPU transfer on host threads, against a contiguous (pinned) staging chunk that a
 * plain cudaMemcpyAsync then moves: cache_manager.py:34-43 (`weight[unique_idxs]` of the Prefetcher's workers) and
 * :58-62 (the eviction manager's `weight[idxs] = rows` / `(weight[idxs] + rows) / 2`).  All pointers are HOST pointers.
 * gather: dst[i] = master[ids[i]];  scatter: master[ids[i]] = src[i] (mean of the two with `average`) for every i whose
 * primary[i] != 0 (primary == NULL: all).  `threads` host threads share the rows. */
int cdlrm_host_gather_rows(const float* master, int64_t n_rows, int dim, const int64_t* ids, int64_t n, float* dst,
                           int threads);
int cdlrm_host_scatter_rows(float* master, int64_t n_rows, int dim, const int64_t* ids, const uint8_t* primary,
                            int64_t n, const float* src, int average, int threads);
/* cudaMemcpyAsync of a staging chunk on `stream` (copy engine): kind 1 = host to device, 2 = device to host */
int cdlrm_copy_async(int device, void* dst, const void* src, int64_t bytes, int kind, cdlrm_stream stream);
/* Whole transfers in one call (the chunk loop is native: the caller's interpreter lock is dropped once; host threads
 * come from a persistent pool).  n_jobs lists (one per table): HOST ids / primary flags, DEVICE rows.
 * prefetch (cache_manager.py:34-43): dst_j[i] = masters[j][ids_j[i]] -- host threads gather chunk c into one of the two
 * pinned staging chunks (chunk_rows x dim floats each) while cudaMemcpyAsync moves chunk c-1 into HBM; returns when the
 * last copy has finished.  writeback (cache_manager.py:48-64): masters[j][ids_j[i]] = src_j[i] (mean of the two with
 * `average`) where primary_j[i] != 0 (primary or primary[j] NULL: all) -- cudaMemcpyAsync brings chunk c out of HBM while
 * the host threads scatter chunk c-1; returns when every row is in the master. */
int cdlrm_host_prefetch_rows(int device, int n_jobs, const float* const* masters, const int64_t* n_rows, int dim,
                             const int64_t* const* ids, const int64_t* counts, float* const* dst, float* chunk0,
                             float* chunk1, int64_t chunk_rows, int threads, cdlrm_stream stream);
int cdlrm_host_writeback_rows(int device, int n_jobs, float* const* masters, const int64_t* n_rows, int dim,
                              const int64_t* const* ids, const uint8_t* const* primary, const int64_t* counts,
                              const float* const* src, float* chunk0, float* chunk1, int64_t chunk_rows, int average,
                              int threads, cdlrm_stream stream);

/* ---- peer-readable device buffers (CUDA IPC over NVLink / NVSwitch) and the SHARDED loser store ----------------
 * No reference counterpart as code: the reference fetches every forward miss from the CPU master table
 * (model_no_ddp.py:176-179).  Here the un-cacheable ids of a window (identical on every rank: same deterministic
 * plan) are prefetched into HBM, 1/world of the rows per rank, and a missing row is read from the rank that holds it.
 * alloc: cudaMalloc + IPC handle (CDLRM_IPC_HANDLE_BYTES bytes, to be sent to the peers); open / close: map / unmap a
 * peer's buffer on `device`; free: release a buffer made by alloc. */
int cdlrm_peer_alloc(int device, int64_t bytes, void** d_ptr, void* handle_out);
int cdlrm_peer_open(int device, const void* handle, void** d_ptr);
int cdlrm_peer_close(int device, void* d_ptr);
int cdlrm_peer_free(int device, void* d_ptr);
/* Sharded variant of cdlrm_ctx_bind_losers: table k has h_n[k] ascending ids at h_ids[k]; index i of that list is
 * row i % h_shard[k] of rank i / h_shard[k], whose shard of table k starts at h_peer[k * world + rank]. */
int cdlrm_ctx_bind_losers_sharded(cdlrm_ctx* ctx, const int64_t* const* h_ids, const int64_t* h_n,
                                  const int64_t* h_shard, int world, const float* const* h_peer, cdlrm_stream stream);

/* ---- synthetic Criteo-shaped sparse ids (SURVEY 8f.3: synthetic train_ld + cache_ld twin; replaces the role of
 *      dlrm_data_pytorch.py:386-547 for measurement, the reference's random mode main_no_ddp.py:539-547 cannot run).
 * out[(k - table_begin) * ld + s * nb + b] = id of table k, global step step0 + s, sample b0 + b of the global batch
 * (batch_global samples per step): a pure function of (seed, k, step, sample), so the trainers' batches and the
 * look-ahead planner's window scan can be generated independently, in chunks, on any rank.  uniform != 0: uniform
 * over [0, n_k); else a bounded power law with exponent zipf_a over ranks 1..n_k, scrambled over the id space. */
int cdlrm_synth_ids(int device, int table_begin, int table_count, const int64_t* h_n_rows, uint64_t seed,
                    int64_t batch_global, int64_t step0, int32_t n_steps, int64_t b0, int32_t nb,
                    int uniform, double zipf_a, int64_t* out, int64_t ld, cdlrm_stream stream);

/* A CUDA stream of the library's own (cudaStreamNonBlocking; priority 0 = default, -1 = highest).  PyTorch hands out
 * streams from a round-robin pool of 32 per priority, so two torch.cuda.Stream objects can be the SAME stream: the
 * look-ahead planner's side stream must never alias the stream a training-step graph is captured on.  The host
 * mirror wraps these with torch.cuda.ExternalStream.  No reference counterpart: stream plumbing. */
int cdlrm_stream_create(int device, int priority, cdlrm_stream* out);
int cdlrm_stream_destroy(int device, cdlrm_stream stream);

/* Programmatic dependent launch of the per-step kernels (on by default; environment CDLRM_PDL=0 or
 * cdlrm_set_pdl(0) falls back to plain stream order).  No reference counterpart: launch plumbing. */
int cdlrm_set_pdl(int on);
int cdlrm_prof_enable(int on);
/* launches an empty kernel through the same accounting: its reported duration ("null") is the overhead the
 * event pair adds to every measured launch */
int cdlrm_prof_null(cdlrm_stream stream);
int64_t cdlrm_prof_launches(int reset);          /* launches since the last reset */
int cdlrm_prof_num_kernels(void);
const char* cdlrm_prof_kernel_name(int id);
/* synchronises the device; h_ms[id] = summed duration, h_calls[id] = launches; clears */
int cdlrm_prof_report(double* h_ms, int64_t* h_calls, int n);

/* ---- victim-way RNG (host): the torch CPU mt19937 stream consumed by
 *      torch.distributions.Categorical(...).sample(), main_no_ddp.py:183-185 -------
 * out[i] = float32(-log1p(-u_i)), u_i = (r64 & (2^53-1)) * 2^-53,
 * r64 = (mt32() << 32) | mt32(), mt19937 seeded by init_genrand(seed)
 * == torch.manual_seed(seed); torch.empty(n).exponential_(1). */
int cdlrm_rng_create(cdlrm_rng** out, uint64_t seed);
int cdlrm_rng_destroy(cdlrm_rng* rng);
int cdlrm_rng_exponential(cdlrm_rng* rng, float* h_out, int64_t n, int threads);
uint64_t cdlrm_rng_draws(const cdlrm_rng* rng);

/* ---- victim-way RNG (device): the same mt19937 stream generated on the GPU by one CTA
 *      (three-phase parallel state refresh), state resident in HBM.  raw: 2 uint32 words
 *      {hi, lo} per draw; exponential: float32(-log1p(-u)) with glibc's log1p restated
 *      bit-exactly in IEEE double intrinsics (csrc/expdraw.cuh).  d_raw_scratch: 2*n uint32. */
int cdlrm_rngdev_create(cdlrm_rngdev** out, int device, uint64_t seed);
int cdlrm_rngdev_destroy(cdlrm_rngdev* rng);
int cdlrm_rngdev_raw(cdlrm_rngdev* rng, uint32_t* d_out, int64_t n_draws, cdlrm_stream stream);
int cdlrm_rngdev_exponential(cdlrm_rngdev* rng, float* d_out, int64_t n, uint32_t* d_raw_scratch,
                             cdlrm_stream stream);
uint64_t cdlrm_rngdev_draws(const cdlrm_rngdev* rng);
/* Checkpoint of the stream: h_state = 625 host words {x[624], pos}.  get: copies the state in stream order
 * (cudaMemcpyAsync on `stream`: pinned h_state is valid once the stream has reached the copy) and writes the
 * number of draws enqueued so far to *h_draws.  set: replaces the state in stream order; pos must be the one that
 * `draws` implies (an error otherwise). */
int cdlrm_rngdev_get_state(cdlrm_rngdev* rng, uint32_t* h_state, uint64_t* h_draws, cdlrm_stream stream);
int cdlrm_rngdev_set_state(cdlrm_rngdev* rng, const uint32_t* h_state, uint64_t draws, cdlrm_stream stream);
/* key 0: smallest request (32-bit words) generated chunk-parallel by mt19937 jump-ahead (default 0: every request of
 * two or more chunks of 2.56 M words); -1 = always the sequential single-CTA kernel.  Same stream either way. */
int cdlrm_rngdev_set_option(int key, int64_t value);
/* d_out[i] = exponential draw of the raw word pair {d_raw[2i], d_raw[2i+1]} (the transform alone) */
int cdlrm_exp_from_raw(const uint32_t* d_raw, float* d_out, int64_t n, cdlrm_stream stream);

/* ---- evaluation metrics (csrc/eval.cu): predictions z in [0, 1] and labels t in {0, 1} of any number of
 *      batches -> counts, BCE sum and the exact ROC AUC ------------------------------------------------------------
 * correct: round_half_even(z) == t.  loss_sum: sum of -(t max(log z, -100) + (1 - t) max(log(1 - z), -100)) in fp64
 * from the fp32 z, in a fixed order.  auc_2u: 2U = sum over positives of (2 #negatives with a lower z + #negatives
 * with an equal z), exact; AUC = auc_2u / (2 positives negatives).  flags: bit0 a z outside [0, 1] or NaN, bit1 a t
 * outside {0, 1}, bit2 more samples than max_samples (the batch that overflowed is dropped).
 * Memory: 8 bytes per sample of max_samples (<= 2^30) plus < 64 MB. */
typedef struct cdlrm_eval cdlrm_eval;
typedef struct cdlrm_eval_stats {
    int64_t samples;
    int64_t positives;
    int64_t negatives;
    int64_t correct;
    double loss_sum;
    uint64_t auc_2u;
    uint32_t flags;
    uint32_t reserved;
} cdlrm_eval_stats;
int cdlrm_eval_create(cdlrm_eval** out, int device, int64_t max_samples);
int cdlrm_eval_destroy(cdlrm_eval* ev);
/* forget every accumulated sample (stream order) */
int cdlrm_eval_reset(cdlrm_eval* ev, cdlrm_stream stream);
/* add samples z[i * ldz], t[i * ldt], i < n (float32 device arrays); capturable, allocates nothing */
int cdlrm_eval_accumulate(cdlrm_eval* ev, const float* z, int64_t ldz, const float* t, int64_t ldt, int32_t n,
                          cdlrm_stream stream);
/* metrics of everything accumulated since the last reset; synchronises `stream`; leaves the samples in place */
int cdlrm_eval_result(cdlrm_eval* ev, cdlrm_eval_stats* h_stats, cdlrm_stream stream);

/* ---- MLPerf binary Criteo records (csrc/criteo.cu): replaces the host decode of data_loader_terabyte.py,
 *      CriteoBinDataset.__getitem__ :224-235 and _transform_features :68-87 (flag_input_torch_tensor=True) --------
 * rec: n device records of 1 + n_dense + n_sparse int32 fields [label, dense..., categorical...] (4-byte aligned).
 *   X[i * ld_x + c]     = logf((float)dense_c + 1.0f)         torch.log(x_int.float() + 1)
 *   ids[k * ld_ids + i] = (int64)cat_k, floor modulo max_ind_range when max_ind_range > 0 (torch's %: the result
 *                         takes the divisor's sign)           (x_cat % max_ind_range).long().t()
 *   T[i]                = (float)label                        y.float()
 * Any output may be NULL (not written); n == 0 launches nothing.  Ids are not range-checked here (the forward and
 * the planner flag an id outside its table).  At most 95 fields per record. */
int cdlrm_criteo_decode(int device, const int32_t* rec, int64_t n, int32_t n_dense, int32_t n_sparse,
                        int64_t max_ind_range, float* X, int64_t ld_x, int64_t* ids, int64_t ld_ids, float* T,
                        cdlrm_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* CDLRM_B200_H */
