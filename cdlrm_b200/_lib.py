"""ctypes binding of libcdlrm_b200.so (the C ABI declared in include/cdlrm_b200.h).

There is no fallback: if the shared library is missing this module raises, and every
compute entry point fails without a CUDA device."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcdlrm_b200.so")

c_i64p = C.POINTER(C.c_int64)
c_i32p = C.POINTER(C.c_int32)
c_u32p = C.POINTER(C.c_uint32)
c_f32p = C.POINTER(C.c_float)
vp = C.c_void_p

# name -> (restype, argtypes); mirrors include/cdlrm_b200.h one to one
SIGNATURES = {
    "cdlrm_abi_version": (C.c_int, []),
    "cdlrm_last_error": (C.c_char_p, []),
    "cdlrm_is_prime_ref": (C.c_int, [C.c_int64]),
    "cdlrm_find_next_prime": (C.c_int64, [C.c_int64]),
    "cdlrm_ctx_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, c_i64p, C.c_int64]),
    "cdlrm_ctx_destroy": (C.c_int, [vp]),
    "cdlrm_ctx_geometry": (C.c_int, [vp, c_i64p, c_i64p]),
    "cdlrm_ctx_bind_cache": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp)]),
    "cdlrm_ctx_bind_plan_tags": (C.c_int, [vp, C.POINTER(vp)]),
    "cdlrm_ctx_bind_master": (C.c_int, [vp, C.POINTER(vp)]),
    "cdlrm_ctx_bind_dirty": (C.c_int, [vp, C.POINTER(vp)]),
    "cdlrm_ctx_reserve": (C.c_int, [vp, C.c_int64]),
    "cdlrm_tags_reset": (C.c_int, [vp, vp]),
    "cdlrm_ctx_check": (C.c_int, [vp, vp, c_u32p]),
    "cdlrm_embed_fwd": (C.c_int, [vp, C.c_int, C.c_int, vp, C.c_int64, vp, C.c_int64, C.c_int32, C.c_int32,
                                  vp, C.c_int64, vp, C.c_int64, vp, vp, C.c_int64, vp]),
    "cdlrm_embed_fwd_eval": (C.c_int, [vp, C.c_int, C.c_int, vp, C.c_int64, C.c_int32, vp, C.c_int64, vp]),
    "cdlrm_embed_bwd_plan_bytes": (C.c_int64, [C.c_int, C.c_int32]),
    "cdlrm_embed_bwd_plan": (C.c_int, [vp, C.c_int, C.c_int, vp, C.c_int64, C.c_int32, vp, vp]),
    "cdlrm_embed_bwd_sgd": (C.c_int, [vp, C.c_int, C.c_int, vp, C.c_int32, vp, C.c_int64, vp, C.c_int64,
                                      C.c_int64, C.c_float, vp]),
    "cdlrm_embed_set_option": (C.c_int, [C.c_int, C.c_int]),
    "cdlrm_interact_set_option": (C.c_int, [C.c_int, C.c_int]),
    "cdlrm_interact_fwd": (C.c_int, [C.c_int, C.POINTER(vp), C.c_int, C.c_int64, C.c_int32, C.c_int, C.c_int,
                                     vp, C.c_int64, vp]),
    "cdlrm_interact_bwd": (C.c_int, [C.c_int, C.POINTER(vp), C.c_int, C.c_int64, C.c_int32, C.c_int, C.c_int,
                                     vp, C.c_int64, vp, C.c_int64, vp]),
    "cdlrm_mlp_workspace_bytes": (C.c_int64, [C.c_int, c_i32p, C.c_int32]),
    "cdlrm_mlp_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, c_i32p, C.c_int32, C.c_int, vp, C.c_int64]),
    "cdlrm_mlp_destroy": (C.c_int, [vp]),
    "cdlrm_mlp_set_option": (C.c_int, [C.c_int, C.c_int]),
    "cdlrm_mlp_set_trace": (C.c_int, [vp]),
    "cdlrm_mlp_sgd_split": (C.c_int, [C.c_int, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.c_float, vp, vp, C.c_int64, vp]),
    "cdlrm_mlp_invalidate_split": (C.c_int, [vp]),
    "cdlrm_mlp_set_defer_join": (C.c_int, [vp, C.c_int]),
    "cdlrm_mlp_join": (C.c_int, [vp, vp]),
    "cdlrm_mlp_forward": (C.c_int, [vp, vp, C.c_int64, C.c_int32, C.POINTER(vp), C.POINTER(vp), vp, C.c_int64, vp]),
    "cdlrm_mlp_backward": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int64, C.POINTER(vp), C.POINTER(vp), vp]),
    "cdlrm_plan_workspace_bytes": (C.c_int64, [vp, C.c_int64]),
    "cdlrm_plan_bind_workspace": (C.c_int, [vp, vp, C.c_int64, C.c_int64]),
    "cdlrm_plan_unique": (C.c_int, [vp, vp, C.c_int64, C.c_int64, vp, vp]),
    "cdlrm_plan_mark_ids": (C.c_int, [vp, vp, C.c_int64, C.c_int64, vp]),
    "cdlrm_plan_mark_own_ids": (C.c_int, [vp, vp, C.c_int64, C.c_int64, vp]),
    "cdlrm_plan_set_primary_evictions": (C.c_int, [vp, C.c_int]),
    "cdlrm_plan_or_peer_bitmaps": (C.c_int, [vp, C.POINTER(vp), C.c_int, C.c_int, vp]),
    "cdlrm_synth_ids": (C.c_int, [C.c_int, C.c_int, C.c_int, c_i64p, C.c_uint64, C.c_int64, C.c_int64, C.c_int32,
                                  C.c_int64, C.c_int32, C.c_int, C.c_double, vp, C.c_int64, vp]),
    "cdlrm_plan_phase_a": (C.c_int, [vp, vp, C.c_int64, C.c_int64, c_i64p, vp, vp]),
    "cdlrm_plan_phase_b": (C.c_int, [vp, vp, c_i64p, vp, vp, vp, vp, vp, vp, vp]),
    "cdlrm_plan_unique_ptr": (vp, [vp, C.c_int]),
    "cdlrm_plan_copy_unique": (C.c_int, [vp, C.c_int, vp, C.c_int64, vp]),
    "cdlrm_move_evict": (C.c_int, [vp, C.c_int, vp, vp, vp, C.c_int64, vp, C.c_int, C.c_int, vp]),
    "cdlrm_move_scatter_master": (C.c_int, [vp, C.c_int, vp, C.c_int64, vp, C.c_int, vp]),
    "cdlrm_move_scatter_master2": (C.c_int, [vp, C.c_int, vp, vp, C.c_int64, vp, C.c_int, vp]),
    "cdlrm_plan_losers": (C.c_int, [vp, c_i64p, c_i64p, vp, vp, vp]),
    "cdlrm_ctx_bind_losers": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), c_i64p, vp]),
    "cdlrm_peer_alloc": (C.c_int, [C.c_int, C.c_int64, C.POINTER(vp), vp]),
    "cdlrm_peer_open": (C.c_int, [C.c_int, vp, C.POINTER(vp)]),
    "cdlrm_peer_close": (C.c_int, [C.c_int, vp]),
    "cdlrm_peer_free": (C.c_int, [C.c_int, vp]),
    "cdlrm_ctx_bind_losers_sharded": (C.c_int, [vp, C.POINTER(vp), c_i64p, c_i64p, C.c_int, C.POINTER(vp), vp]),
    "cdlrm_host_gather_rows": (C.c_int, [vp, C.c_int64, C.c_int, vp, C.c_int64, vp, C.c_int]),
    "cdlrm_host_scatter_rows": (C.c_int, [vp, C.c_int64, C.c_int, vp, vp, C.c_int64, vp, C.c_int, C.c_int]),
    "cdlrm_copy_async": (C.c_int, [C.c_int, vp, vp, C.c_int64, C.c_int, vp]),
    "cdlrm_host_prefetch_rows": (C.c_int, [C.c_int, C.c_int, C.POINTER(vp), c_i64p, C.c_int, C.POINTER(vp), c_i64p,
                                           C.POINTER(vp), vp, vp, C.c_int64, C.c_int, vp]),
    "cdlrm_host_writeback_rows": (C.c_int, [C.c_int, C.c_int, C.POINTER(vp), c_i64p, C.c_int, C.POINTER(vp), C.POINTER(vp),
                                            c_i64p, C.POINTER(vp), vp, vp, C.c_int64, C.c_int, C.c_int, vp]),
    "cdlrm_host_register": (C.c_int, [C.c_int, vp, C.c_int64, C.POINTER(vp)]),
    "cdlrm_host_unregister": (C.c_int, [vp]),
    "cdlrm_agg_mark": (C.c_int, [vp, vp, C.c_int64, C.c_int64, vp]),
    "cdlrm_move_gather_master": (C.c_int, [vp, C.c_int, vp, C.c_int64, vp, vp]),
    "cdlrm_move_fill": (C.c_int, [vp, C.c_int, vp, vp, C.c_int64, vp, vp, vp]),
    "cdlrm_agg_or_bitmaps": (C.c_int, [vp, vp, C.c_int, C.c_int64, vp]),
    "cdlrm_agg_collect": (C.c_int, [vp, vp, vp, vp, vp]),
    "cdlrm_agg_pack": (C.c_int, [vp, vp, c_i64p, C.c_float, vp, vp]),
    "cdlrm_agg_unpack": (C.c_int, [vp, vp, c_i64p, vp, C.c_int, vp]),
    "cdlrm_stream_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(vp)]),
    "cdlrm_stream_destroy": (C.c_int, [C.c_int, vp]),
    "cdlrm_set_pdl": (C.c_int, [C.c_int]),
    "cdlrm_bce_mean": (C.c_int, [C.c_int, vp, C.c_int64, vp, C.c_int64, C.c_int32, vp, vp, vp]),
    "cdlrm_prof_enable": (C.c_int, [C.c_int]),
    "cdlrm_prof_null": (C.c_int, [vp]),
    "cdlrm_prof_launches": (C.c_int64, [C.c_int]),
    "cdlrm_prof_num_kernels": (C.c_int, []),
    "cdlrm_prof_kernel_name": (C.c_char_p, [C.c_int]),
    "cdlrm_prof_report": (C.c_int, [C.POINTER(C.c_double), c_i64p, C.c_int]),
    "cdlrm_rng_create": (C.c_int, [C.POINTER(vp), C.c_uint64]),
    "cdlrm_rng_destroy": (C.c_int, [vp]),
    "cdlrm_rng_exponential": (C.c_int, [vp, vp, C.c_int64, C.c_int]),
    "cdlrm_rng_draws": (C.c_uint64, [vp]),
    "cdlrm_rngdev_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_uint64]),
    "cdlrm_rngdev_destroy": (C.c_int, [vp]),
    "cdlrm_rngdev_raw": (C.c_int, [vp, vp, C.c_int64, vp]),
    "cdlrm_rngdev_exponential": (C.c_int, [vp, vp, C.c_int64, vp, vp]),
    "cdlrm_rngdev_draws": (C.c_uint64, [vp]),
    "cdlrm_rngdev_get_state": (C.c_int, [vp, vp, C.POINTER(C.c_uint64), vp]),
    "cdlrm_rngdev_set_state": (C.c_int, [vp, vp, C.c_uint64, vp]),
    "cdlrm_cache_collect_valid": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, c_i64p, vp, vp]),
    "cdlrm_rngdev_set_option": (C.c_int, [C.c_int, C.c_int64]),
    "cdlrm_exp_from_raw": (C.c_int, [vp, vp, C.c_int64, vp]),
    "cdlrm_plan_phase_b_dev": (C.c_int, [vp, vp, vp, C.c_int64, c_i64p, vp, vp, vp, vp, vp, vp, vp]),
    "cdlrm_eval_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int64]),
    "cdlrm_eval_destroy": (C.c_int, [vp]),
    "cdlrm_eval_reset": (C.c_int, [vp, vp]),
    "cdlrm_eval_accumulate": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int64, C.c_int32, vp]),
    "cdlrm_eval_result": (C.c_int, [vp, vp, vp]),
}


class EvalStats(C.Structure):
    """cdlrm_eval_stats (include/cdlrm_b200.h)."""
    _fields_ = [("samples", C.c_int64), ("positives", C.c_int64), ("negatives", C.c_int64), ("correct", C.c_int64),
                ("loss_sum", C.c_double), ("auc_2u", C.c_uint64), ("flags", C.c_uint32), ("reserved", C.c_uint32)]


class CdlrmError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise CdlrmError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C cdlrm_b200/csrc`.  There is no CPU/PyTorch fallback for the cache hot path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export the symbol
        fn.restype = res
        fn.argtypes = args
    if lib.cdlrm_abi_version() != 1:
        raise CdlrmError("libcdlrm_b200.so ABI version mismatch")
    return lib


lib = _load()


def check(rc):
    if rc != 0:
        raise CdlrmError(f"libcdlrm_b200 error {rc}: {lib.cdlrm_last_error().decode()}")


def ptr_array(ptrs):
    arr = (vp * len(ptrs))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr


def i64_array(vals):
    arr = (C.c_int64 * len(vals))()
    for i, v in enumerate(vals):
        arr[i] = int(v)
    return arr


def new_stream(device, priority=0):
    """A torch.cuda.ExternalStream over a stream of the library's own (cdlrm_stream_create): never one of
    PyTorch's pooled streams (32 per priority, handed out round-robin), so it cannot alias another
    torch.cuda.Stream of the process -- in particular not the stream a training-step CUDA graph is captured
    on.  Meant for SIDE streams (planner, lookup): work is sent to it through the C ABI, event record / wait and
    ``with torch.cuda.stream(...)`` allocations.  Do not make it the current stream of autograd work or of a graph
    capture: the engine falls back to the legacy default stream for streams it does not own.  The handful of
    streams a process creates live until it exits."""
    import torch
    dev = torch.device(device)
    if os.environ.get("CDLRM_POOL_STREAMS", "0") == "1":        # A/B switch: PyTorch's pooled streams
        return torch.cuda.Stream(dev, priority=int(priority))
    h = vp()
    check(lib.cdlrm_stream_create(dev.index, int(priority), C.byref(h)))
    return torch.cuda.ExternalStream(h.value, device=dev)
