"""ctypes binding of libkpapa.so (C ABI in include/kmerpapa_b200.h)."""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KP_LIBKPAPA") or os.path.join(_PKG, "libkpapa.so")   # override: A/B of experimental builds
_lib = None


class KpError(RuntimeError):
    pass


KP_OK, KP_ERR, KP_ERR_CAPACITY = 0, 1, 2   # return codes of include/kmerpapa_b200.h


class PlanInfo(ctypes.Structure):
    _fields_ = [
        ("npat", ctypes.c_uint64), ("nkmer", ctypes.c_uint64), ("ntiles", ctypes.c_uint64),
        ("table_elems", ctypes.c_uint64), ("kept_elems", ctypes.c_uint64), ("expanded_elems", ctypes.c_uint64),
        ("backtrack_ws_bytes", ctypes.c_uint64),
        ("k", ctypes.c_uint32), ("nlevels", ctypes.c_uint32), ("tile_cells", ctypes.c_uint32),
        ("tile_stride", ctypes.c_uint32), ("tile_kmers", ctypes.c_uint32), ("low_positions", ctypes.c_uint32),
        ("register_radix", ctypes.c_uint32), ("rows", ctypes.c_uint32), ("rounds", ctypes.c_uint32),
        ("warps_per_cta", ctypes.c_uint32), ("high_levels", ctypes.c_uint32), ("sm_count", ctypes.c_uint32),
    ]


class ShardInfo(ctypes.Structure):
    _fields_ = [
        ("local_tiles", ctypes.c_uint64), ("table_elems", ctypes.c_uint64), ("kept_elems", ctypes.c_uint64),
        ("d_best", ctypes.c_uint64), ("d_kept", ctypes.c_uint64),
        ("rank", ctypes.c_uint32), ("world", ctypes.c_uint32), ("nwaves", ctypes.c_uint32), ("top_digits", ctypes.c_uint32),
        ("replicate", ctypes.c_uint32), ("reserved", ctypes.c_uint32),
    ]


# every symbol include/kmerpapa_b200.h declares: name -> (restype, argtypes)
_vp, _u64, _i64, _dbl, _int, _cp = (ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int64, ctypes.c_double, ctypes.c_int,
                                   ctypes.c_char_p)
SYMBOLS = {
    "kp_last_error": (_cp, []),
    "kp_version": (_int, []),
    "kp_plan_create": (_int, [_cp, _int, ctypes.POINTER(_vp)]),
    "kp_plan_create_lite": (_int, [_cp, _int, ctypes.POINTER(_vp)]),
    "kp_plan_destroy": (_int, [_vp]),
    "kp_plan_get_info": (_int, [_vp, ctypes.POINTER(PlanInfo)]),
    "kp_pack_counts": (_int, [_vp, _vp, _vp, _vp, _u64, _vp, _vp, _vp]),
    "kp_expand_counts": (_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "kp_dp_single": (_int, [_vp, _vp, _vp, _u64, _dbl, _dbl, _dbl, _vp, _vp, _vp]),
    "kp_backtrack_ws_bytes": (_u64, [_u64]),
    "kp_backtrack": (_int, [_vp, _vp, _vp, _vp, _u64, _u64, _vp, ctypes.POINTER(_u64), _vp]),
    "kp_split_codes": (_int, [_vp, _vp, _vp, _vp, _u64, _vp, _vp]),
    "kp_gather_table": (_int, [_vp, _vp, _u64, _u64, _vp, _vp]),
    "kp_gather_kept": (_int, [_vp, _vp, _u64, _u64, _vp, _vp]),
    "kp_gather_patterns": (_int, [_vp, _vp, _vp, _vp, _u64, _vp, _vp, _vp, _vp]),
    "kp_dp_cv_job": (_int, [_vp, _vp, _vp, _vp, _vp, _u64, _dbl, _dbl, _dbl, _vp, _vp, _vp, _u64, _vp, _vp]),
    "kp_cv_stage_bytes": (_u64, [_u64]),
    "kp_cv_job_enqueue": (_int, [_vp, _vp, _vp, _vp, _vp, _u64, _dbl, _dbl, _dbl, _vp, _vp, _vp, _u64, _vp, _vp]),
    "kp_cv_job_finish": (_int, [_vp, _u64, _vp]),
    "kp_cv_heldout": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _dbl, _dbl, _dbl, _u64, _vp, _u64, _vp, _vp]),
    "kp_pattern_counts": (_int, [_vp, _vp, _vp, _vp, _u64, _vp, _vp, _vp]),
    "kp_partition_assign": (_int, [_vp, _vp, _u64, _vp, ctypes.POINTER(_u64), ctypes.POINTER(_u64), _vp]),
    "kp_partition_score": (_int, [_vp, _vp, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "kp_kmer_rates": (_int, [_vp, _vp, _vp, _u64, _vp, _vp]),
    "kp_seq_scan": (_int, [_vp, _vp, _u64, _u64, _u64, _u64, _u64, _int, _vp, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "kp_region_sums": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u64, _vp, _vp, _vp]),
    "kp_snv_counts": (_int, [_vp, _vp, _u64, _u64, _u64, _u64, _u64, _int, _vp, _vp, _u64, _vp, _vp, _vp, _vp, _vp]),
    "kp_pattern_offset":(_int, [_vp, _u64, ctypes.POINTER(_u64), ctypes.POINTER(_u64), ctypes.POINTER(ctypes.c_uint32)]),
    "kp_plan_launch_count": (_u64, [_vp]),
    "kp_dp_kernel_name": (_cp, [_vp, _int]),
    "kp_shard_assignment": (_int, [_vp, _int, _vp, _vp]),
    "kp_shard_create": (_int, [_vp, _int, _int, _int, ctypes.POINTER(_vp)]),
    "kp_shard_destroy": (_int, [_vp]),
    "kp_shard_get_info": (_int, [_vp, ctypes.POINTER(ShardInfo)]),
    "kp_shard_set_peer": (_int, [_vp, _int, _vp, _vp]),
    "kp_ipc_export": (_int, [_vp, _vp]),
    "kp_ipc_open": (_int, [_int, _vp, ctypes.POINTER(_vp)]),
    "kp_ipc_close": (_int, [_int, _vp]),
    "kp_shard_dp_wave": (_int, [_vp, _int, _vp, _vp, _u64, _dbl, _dbl, _dbl, _vp]),
    "kp_shard_cv_wave": (_int, [_vp, _int, _vp, _vp, _vp, _vp, _u64, _dbl, _dbl, _dbl, _vp]),
    "kp_shard_cv_heldout": (_int, [_vp, _vp, _vp, _vp, _vp, _dbl, _dbl, _dbl, _u64, _vp, _u64, _vp, _vp]),
    "kp_shard_backtrack":(_int, [_vp, _vp, _u64, _u64, _vp, ctypes.POINTER(_u64), _vp]),
    "kp_shard_gather": (_int, [_vp, _vp, _u64, _vp, _vp, _vp, _vp]),
    "kp_greedy_ws_bytes": (_u64, [_u64]),
    "kp_greedy": (_int, [_vp, _vp, _vp, _vp, _vp, _dbl, _dbl, _dbl, _vp, _u64, _vp, _vp, _vp, ctypes.POINTER(_u64),
                         ctypes.POINTER(_dbl), _vp]),
    "kp_kmer_fold_terms": (_int, [_int, _vp, _vp, _vp, _vp, _vp, _u64, _dbl, _vp, _vp]),
    "kp_debug_log": (_int, [_int, _vp, _vp, _u64]),
    "kp_debug_leaf_score": (_int, [_int, _vp, _vp, _u64, _dbl, _dbl, _dbl, _vp]),
    "kp_debug_self_score": (_int, [_int, _vp, _vp, _vp, _vp, _vp, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp]),
}


def lib():
    """Load libkpapa.so.  Fails loudly when it has not been built: there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise KpError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(kmerpapa_b200 has no CPU implementation of the DP)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().kp_last_error()
        raise KpError(f"{what}: {msg.decode() if msg else 'error ' + str(rc)}")
