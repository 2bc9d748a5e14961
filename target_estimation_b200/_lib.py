"""ctypes binding of include/te_pool.h (the thin extern "C" CUDA layer).  No fallback of any kind:
if the shared library was not built the import fails loudly."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
lib_path = os.path.join(_HERE, "lib", "libte_pool.so")


class TeError(RuntimeError):
    pass


if not os.path.exists(lib_path):
    raise ImportError(
        "target_estimation_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(nvcc, sm_100a).  There is no CPU fallback." % lib_path)

lib = C.CDLL(lib_path, mode=C.RTLD_GLOBAL)

_p = C.c_void_p
_ll = C.c_longlong
_d = C.c_double
_i = C.c_int
_u32 = C.c_uint32
_sz = C.c_size_t

# name -> (restype, argtypes); mirrors include/te_pool.h line by line
SIGNATURES = {
    "te_last_error": (C.c_char_p, []),
    "te_device_count": (_i, []),
    "te_model_dims": (_i, [_i, _p, _p]),
    "te_model_bytes_per_step": (_sz, [_i]),
    "te_pool_create": (_p, [_i, _i, _p]),
    "te_pool_destroy": (None, [_p]),
    "te_pool_set_stream": (_i, [_p, _p]),
    "te_pool_sync": (_i, [_p]),
    "te_pool_set_variant": (_i, [_p, _i]),
    "te_pool_set_grid_cap": (_i, [_p, _i]),
    "te_pool_reserve": (_i, [_p, _sz]),
    "te_pool_size": (_ll, [_p]),
    "te_pool_device_bytes": (_sz, [_p]),
    "te_pool_register_class": (_i, [_p, _p, _p, _p]),
    "te_pool_class_count": (_i, [_p]),
    "te_pool_get_class": (_i, [_p, _i, _p, _p, _p]),
    "te_pool_add_batch": (_ll, [_p, _ll, _p, _p, _p, _p, _p, _p, _p]),
    "te_pool_erase_batch": (_ll, [_p, _ll, _p]),
    "te_pool_ids": (_ll, [_p, _p, _ll]),
    "te_pool_contains": (_i, [_p, _u32]),
    "te_pool_class_of": (_i, [_p, _u32]),
    "te_pool_step_dense": (_i, [_p, _d, _p, _i, _p, _i]),
    "te_pool_step_dense_ticks": (_i, [_p, _i, _d, _p, _i, _p, _i]),
    "te_pool_step_dense_host": (_i, [_p, _d, _p, _i, _p, _i]),
    "te_pool_tick_host": (_i, [_p, _d, _p, _i, _p, _i, _p]),
    "te_pool_step_ids": (_ll, [_p, _ll, _p, _p, _d, _p, _p]),
    "te_pool_predict_all": (_i, [_p, _d]),
    "te_pool_read_state": (_i, [_p, _ll, _p, _p, _p, _p, _p, _p, _p]),
    "te_pool_read_estimates": (_i, [_p, _ll, _p, _p, _p, _p, _p, _p, _p]),
    "te_pool_estimates_dev": (_i, [_p, _p]),
    "te_pool_dev_ids": (_p, [_p]),
    "te_pool_set_stamps": (_i, [_p, _ll, _p, _p, _p]),
    "te_pool_stamp_dense": (_i, [_p, _p, _i, _u32, _u32]),
    "te_pool_expire": (_ll, [_p, _u32, _u32, _d, _p, _ll]),
    "te_pool_step_dense_expire": (_ll, [_p, _d, _p, _i, _p, _i, _u32, _u32, _u32, _u32, _d, _p, _ll]),
    "te_host_register": (_i, [_p, C.c_size_t]),
    "te_host_unregister": (_i, [_p]),
    "te_pool_mailbox_ingest": (_i, [_p, _ll, _p, _p, _p, _p]),
    "te_pool_mailbox_ingest_dev": (_i, [_p, _ll, _p, _p, _p, _p]),
    "te_pool_mailbox_prefetch": (_i, [_p, _ll, _p, _p, _p, _p]),
    "te_pool_mailbox_ingest_prefetched": (_i, [_p]),
    "te_pool_mailbox_tick": (_ll, [_p, _d, _d, _i, _u32, _u32, _d, _p, _ll, _p, _ll, _p]),
    "te_pool_mailbox_count": (_ll, [_p]),
    "te_pool_mailbox_bound": (_ll, [_p]),
    "te_pool_mailbox_dev_pose": (_p, [_p]),
    "te_pool_mailbox_dev_action": (_p, [_p]),
    "te_isolver_create": (_p, [_p, _ll, C.c_uint]),
    "te_isolver_destroy": (None, [_p]),
    "te_isolver_query": (_i, [_p, _ll, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "te_isolver_query_dense": (_i, [_p, _p, _p, _p, _d, _d, _p, _p, _p]),
    "te_pool_earliest_intersections": (_ll, [_p, _ll, _p, _p, _p, _ll, _p, _p, _p]),
    "te_pool_nearest_targets": (_ll, [_p, _ll, _p, _p, _p, _ll, _p, _p, _p]),
    "te_pool_gated_targets": (_ll, [_p, _ll, _p, _p, _p, _ll, _p, _p, _p]),
    "te_pool_associate": (_ll, [_p, _d, _ll, _p, _d, _i, _i, _p, _p, _p]),
    "te_pool_gated_candidates": (_ll, [_p, _d, _ll, _p, _d, _i, _p, _p, _p]),
    "te_assign_greedy": (_ll, [_p, _ll, _i, _p, _p, _p, _p]),
    "te_pool_update_at": (_ll, [_p, _ll, _p, _d, _p]),
    "te_pool_assoc_stats": (_i, [_p, _p]),
    "te_isolver_move_streams": (_i, [_p, _p, _ll, _p]),
    "te_pool_tick_host_async": (_i, [_p, _d, _p, _i, _p, _i, _p]),
    "te_pool_tick_host_wait": (_i, [_p, _i]),
    "te_diag_device_peaks": (_i, [_i, _p, _p]),
    "te_pool_live_begin": (_i, [_p, _i, _d, _p, _i, _p, _i, _p]),
    "te_pool_live_release": (_i, [_p, _i]),
    "te_pool_live_push": (_i, [_p, _p, _p]),
    "te_pool_live_wait": (_i, [_p, _i]),
    "te_pool_live_end": (_i, [_p]),
    "te_group_create": (_p, [_i, _p]),
    "te_group_destroy": (None, [_p]),
    "te_group_size": (_i, [_p]),
    "te_group_uses_nccl": (_i, [_p]),
    "te_group_allgather_estimates": (_ll, [_p, _p, _p]),
    "te_group_sync": (_i, [_p]),
    "te_group_dev_records": (_p, [_p, _i]),
    "te_group_dev_ids": (_p, [_p, _i]),
    "te_group_fetch": (_ll, [_p, _i, _p, _p, _ll]),
    "te_group_last_gather_ms": (_d, [_p]),
    "te_group_route_records": (_ll, [_p, _p, _ll, _p, _p, _p, _p, _p]),
    "te_group_routed": (_i, [_p, _i, _p, _p, _p, _p, _p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _f = getattr(lib, _name)   # AttributeError here = header and library out of sync
    _f.restype = _res
    _f.argtypes = _args


def last_error():
    s = lib.te_last_error()
    return s.decode() if s else ""


def check(rc):
    if rc is None or rc < 0:
        raise TeError(last_error())
    return rc
