"""ctypes binding of libmsamtools_b200.so (include/msamtools_b200.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is
present, every entry point fails loudly (ImportError / MsgError).  Nothing in this
package touches the CPU checker kept outside it.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmsamtools_b200.so")

MSG_ABI_VERSION = 2
MSG_OK, MSG_EINVAL, MSG_ENODEV, MSG_ECUDA, MSG_ENOMEM = 0, -1, -2, -3, -4
MSG_ENOTAG, MSG_ENOAS, MSG_EFORMAT, MSG_ERANGE, MSG_ENCCL, MSG_ESTATE = -5, -6, -7, -8, -9, -10
HIT_NONE, HIT_BEST, HIT_UNIQUE = 0, 1, 2
MULTI_ALL, MULTI_EQUAL, MULTI_PROPORTIONAL, MULTI_IGNORE = 1, 2, 3, 4
MSG_COLLATE_RANKS = 2       # msg_config.collate: group by QNAME across the ranks of a multi-GPU run


class MsgConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32),
        ("do_filter", C.c_uint8), ("hit_mode", C.c_uint8), ("invert", C.c_uint8), ("keep_unmapped", C.c_uint8),
        ("rescore", C.c_uint8), ("collate", C.c_uint8), ("exact", C.c_uint8), ("reserved0", C.c_uint8 * 1),
        ("min_length", C.c_int32), ("ppt", C.c_int32), ("max_clip", C.c_int32),
        ("want_kept", C.c_uint8), ("want_records", C.c_uint8), ("want_profile", C.c_uint8), ("want_coverage", C.c_uint8),
        ("want_stats", C.c_uint8), ("share_type", C.c_uint8), ("debug_force_slow", C.c_uint8), ("coverage_summary", C.c_uint8),
        ("n_targets", C.c_int32), ("n_features", C.c_int32),
        ("fmap", C.POINTER(C.c_int32)), ("target_len", C.POINTER(C.c_uint32)),
        ("device", C.c_int32), ("n_ranks", C.c_int32), ("rank", C.c_int32),
        ("nccl_unique_id", C.c_void_p),
    ]


class MsgProfileStats(C.Structure):
    _fields_ = [
        ("mapped_inserts", C.c_uint32), ("uniq_mapper_count", C.c_uint32), ("multi_mapper_count", C.c_uint32),
        ("purged_insert_count", C.c_uint32), ("em_iterations", C.c_int32), ("em_converged", C.c_int32),
        ("em_delta", C.c_double * 20), ("multi_lists", C.c_uint64), ("multi_entries", C.c_uint64),
    ]


class MsgTiming(C.Structure):
    _fields_ = [
        ("decode_ms", C.c_double), ("decode_launches", C.c_uint64), ("total_ms", C.c_double),
        ("kernel_launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
        ("alg_bytes", C.c_uint64), ("slow_records", C.c_uint64), ("fused_chunks", C.c_uint64), ("fused_fallbacks", C.c_uint64),
        ("zero_copy_chunks", C.c_uint64),
    ]


# every symbol include/msamtools_b200.h declares (tests check the library exports them all)
EXPORTS = [
    "msg_create", "msg_destroy", "msg_last_error", "msg_abi_version", "msg_device_count",
    "msg_index_records", "msg_split_point",
    "msg_push", "msg_push_device", "msg_push_async", "msg_push_device_async", "msg_wait", "msg_device_alloc", "msg_device_free", "msg_device_upload", "msg_sync", "msg_reset",
    "msg_kept_count", "msg_pull_kept", "msg_pull_records", "msg_pull_stats", "msg_pull_counts",
    "msg_finish_profile", "msg_finish_coverage", "msg_pull_coverage", "msg_get_timing", "msg_nccl_unique_id",
    "msg_mark", "msg_elapsed_ms", "msg_host_alloc", "msg_host_free",
]

_lib = None


def load():
    """Load the CUDA library; raises ImportError with build instructions if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `make` (nvcc, sm_100a). "
            "msamtools_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, sz, u8p, u64p, u32p, i32p = C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p
    lib.msg_create.argtypes = [C.POINTER(MsgConfig), C.POINTER(vp)]
    lib.msg_destroy.argtypes = [vp]; lib.msg_destroy.restype = None
    lib.msg_last_error.argtypes = [vp]; lib.msg_last_error.restype = C.c_char_p
    lib.msg_abi_version.argtypes = []
    lib.msg_device_count.argtypes = []
    lib.msg_index_records.argtypes = [u8p, sz, u64p, sz, C.POINTER(sz), C.POINTER(sz), C.c_int]
    lib.msg_split_point.argtypes = [u8p, u64p, sz, sz]; lib.msg_split_point.restype = sz
    lib.msg_push.argtypes = [vp, u8p, sz, u64p, sz]
    lib.msg_push_device.argtypes = [vp, vp, sz, vp, sz]
    lib.msg_push_async.argtypes = [vp, u8p, sz, u64p, sz]
    lib.msg_push_device_async.argtypes = [vp, vp, sz, vp, sz]
    lib.msg_wait.argtypes = [vp]
    lib.msg_device_alloc.argtypes = [vp, sz, C.POINTER(vp)]
    lib.msg_device_free.argtypes = [vp, vp]
    lib.msg_device_upload.argtypes = [vp, vp, vp, sz]
    lib.msg_sync.argtypes = [vp]
    lib.msg_reset.argtypes = [vp]
    lib.msg_kept_count.argtypes = [vp, C.POINTER(sz)]
    lib.msg_pull_kept.argtypes = [vp, u32p, sz, C.POINTER(sz)]
    lib.msg_pull_records.argtypes = [vp, u8p, sz, C.POINTER(sz), C.POINTER(sz)]
    lib.msg_pull_stats.argtypes = [vp, sz, i32p, i32p, i32p, i32p, i32p, u8p]
    lib.msg_pull_counts.argtypes = [vp, u32p, vp]
    lib.msg_finish_profile.argtypes = [vp, vp, C.POINTER(MsgProfileStats)]
    lib.msg_finish_coverage.argtypes = [vp, u8p, vp, vp]
    lib.msg_pull_coverage.argtypes = [vp, C.c_int32, i32p]
    lib.msg_get_timing.argtypes = [vp, C.POINTER(MsgTiming), C.c_int]
    lib.msg_nccl_unique_id.argtypes = [vp]
    lib.msg_mark.argtypes = [vp, C.c_int]
    lib.msg_host_alloc.argtypes = [C.c_int, sz, C.POINTER(vp)]
    lib.msg_host_free.argtypes = [vp]
    lib.msg_elapsed_ms.argtypes = [vp, C.c_int, C.c_int, C.POINTER(C.c_double)]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("msg_destroy", "msg_last_error", "msg_split_point"):
            fn.restype = C.c_int
    _lib = lib
    return lib
