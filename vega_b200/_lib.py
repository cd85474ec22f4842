"""ctypes binding of libvega_b200.so (include/vega_b200.h).

The shared library is the product; this file only declares its C ABI.  There is no
Python/CPU fallback: if the library is missing, importing fails loudly, and without a
CUDA device every compute entry raises VegaB200Error(VB_ERR_CUDA).
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VEGA_B200_LIB") or os.path.join(_PKG, "libvega_b200.so")   # env override: A/B builds only

VB_OK, VB_ERR_INVALID, VB_ERR_CUDA, VB_ERR_OOM, VB_ERR_STATE, VB_ERR_UNSUPPORTED, VB_ERR_TOO_LARGE = 0, -1, -2, -3, -4, -5, -6
VB_U64, VB_I64, VB_F64 = 0, 1, 2
VB_AGG_GROUP, VB_AGG_SUM, VB_AGG_MIN, VB_AGG_MAX, VB_AGG_COUNT, VB_AGG_COGROUP, VB_AGG_SORT = range(7)
VB_PART_HASH_METRO64, VB_PART_RANGE = 0, 1
VB_HOST, VB_DEVICE, VB_DEVICE_BORROWED = 0, 1, 2
VB_GEN_UNIFORM, VB_GEN_ZIPF, VB_GEN_UNIQUE = 0, 1, 2
VB_XCHG_AUTO, VB_XCHG_NCCL, VB_XCHG_P2P = 0, 1, 2
VB_JOIN_LEFT_OUTER, VB_JOIN_RIGHT_OUTER, VB_JOIN_FULL_OUTER = 1, 2, 3
VB_JOIN_HAS_V, VB_JOIN_HAS_W = 1, 2
VB_UNIQUE_ID_BYTES = 128

KERNEL_CLASSES = ["hash_agg", "dict", "merge", "rp_hist", "rp_scan", "rp_scatter", "misc", "join"]


class VegaB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"vega_b200 error {code}: {msg}")
        self.code = code


class vb_stats(ctypes.Structure):
    _fields_ = [
        ("rows_in", ctypes.c_uint64), ("rows_out", ctypes.c_uint64), ("kernel_launches", ctypes.c_uint64),
        ("h2d_bytes", ctypes.c_uint64), ("d2h_bytes", ctypes.c_uint64), ("table_slots", ctypes.c_uint64),
        ("table_restarts", ctypes.c_uint64), ("hot_kernel_ms", ctypes.c_double),
        ("hot_kernel_launches", ctypes.c_uint64), ("hot_kernel_rows", ctypes.c_uint64),
        ("map_ms", ctypes.c_double), ("seal_ms", ctypes.c_double), ("hot_kernel_variant", ctypes.c_uint64),
    ]


class vb_xstats(ctypes.Structure):
    _fields_ = [("sent_rows", ctypes.c_uint64), ("recv_rows", ctypes.c_uint64), ("exchanges", ctypes.c_uint64),
                ("exchange_ms", ctypes.c_double), ("kind", ctypes.c_int32), ("pad", ctypes.c_int32),
                ("prepare_wall_ms", ctypes.c_double), ("counts_wall_ms", ctypes.c_double), ("post_wall_ms", ctypes.c_double)]


# name -> (restype, argtypes); also the list of symbols include/vega_b200.h declares
_vp, _u64, _u32, _i32, _dbl = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int32, ctypes.c_double
_pvp, _pu64 = ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_uint64)
SYMBOLS = {
    "vb_ctx_create": (_i32, [_i32, _pvp]),
    "vb_ctx_destroy": (_i32, [_vp]),
    "vb_ctx_synchronize": (_i32, [_vp]),
    "vb_ctx_set_profile": (_i32, [_vp, _i32]),
    "vb_ctx_device": (_i32, [_vp]),
    "vb_ctx_stream": (_vp, [_vp]),
    "vb_ctx_mem_info": (_i32, [_vp, _pu64, _pu64]),
    "vb_shuffle_create": (_i32, [_vp, _u64, _u32, _u32, _i32, _i32, _i32, _i32, _pvp]),
    "vb_shuffle_set_key_width": (_i32, [_vp, _u32]),
    "vb_shuffle_set_hint": (_i32, [_vp, _u64]),
    "vb_shuffle_set_dist": (_i32, [_vp, _u32, _u32]),
    "vb_shuffle_map_aos": (_i32, [_vp, _u32, _vp, _u64, _i32]),
    "vb_shuffle_map_soa": (_i32, [_vp, _u32, _vp, _vp, _u64, _i32]),
    "vb_shuffle_export_prepare": (_i32, [_vp, _pu64]),
    "vb_shuffle_export_buffers": (_i32, [_vp, _pvp, _pvp]),
    "vb_shuffle_import": (_i32, [_vp, _vp, _vp, _pu64]),
    "vb_ctx_arena_reserve": (_i32, [_vp, _u64, _vp, _pu64]),
    "vb_ctx_peer_open": (_i32, [_vp, _u32, _vp, _u64, _i32]),
    "vb_shuffle_export_counts": (_i32, [_vp, _pu64]),
    "vb_shuffle_export_direct": (_i32, [_vp, _pu64, _pu64]),
    "vb_shuffle_import_arena": (_i32, [_vp, _pu64]),
    "vb_ctx_arena_release_retired": (_i32, [_vp]),
    "vb_ctx_trim": (_i32, [_vp, _u64]),
    "vb_comm_unique_id": (_i32, [_vp]),
    "vb_ctx_comm_init": (_i32, [_vp, _vp, _u32, _u32]),
    "vb_ctx_comm_destroy": (_i32, [_vp]),
    "vb_ctx_comm_info": (_i32, [_vp, ctypes.POINTER(_u32), ctypes.POINTER(_u32), ctypes.POINTER(_i32)]),
    "vb_shuffle_exchange": (_i32, [_vp, _i32]),
    "vb_shuffle_exchange_stats": (_i32, [_vp, ctypes.POINTER(vb_xstats)]),
    "vb_shuffle_seal": (_i32, [_vp]),
    "vb_shuffle_is_sealed": (_i32, [_vp]),
    "vb_shuffle_reduce_size": (_i32, [_vp, _u32, _pu64, _pu64]),
    "vb_shuffle_reduce": (_i32, [_vp, _u32, _vp, _vp, _vp, _vp, _i32]),
    "vb_join_size": (_i32, [_vp, _vp, _u32, _pu64]),
    "vb_join": (_i32, [_vp, _vp, _u32, _vp, _vp, _vp, _i32]),
    "vb_cogroup_size": (_i32, [_vp, _vp, _u32, _pu64, _pu64, _pu64]),
    "vb_cogroup": (_i32, [_vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _i32]),
    "vb_join_outer_size": (_i32, [_vp, _vp, _u32, _i32, _pu64]),
    "vb_join_outer": (_i32, [_vp, _vp, _u32, _i32, _vp, _vp, _vp, _vp, _i32]),
    "vb_shuffle_reduce_blob_size": (_i32, [_vp, _u32, _pu64]),
    "vb_shuffle_reduce_blob": (_i32, [_vp, _u32, _vp, _i32]),
    "vb_shuffle_map_blob": (_i32, [_vp, _u32, _vp, _u64, _i32]),
    "vb_shuffle_free": (_i32, [_vp]),
    "vb_shuffle_stats": (_i32, [_vp, ctypes.POINTER(vb_stats)]),
    "vb_shuffle_kernel_time": (_i32, [_vp, _i32, ctypes.POINTER(_dbl), _pu64]),
    "vb_last_error": (ctypes.c_char_p, []),
    "vb_hash_key": (_u64, [_u64, _u32]),
    "vb_get_partition": (_u32, [_u64, _u32, _u32]),
    "vb_slice": (_u64, [_u64, _u64, _vp]),
    "vb_range_len": (_u64, [_u64, _u64, _u64]),
    "vb_range": (_i32, [_vp, _vp, _u64, _u64, _u64]),
    "vb_gen_pairs": (_i32, [_vp, _vp, _vp, _vp, _u64, _u64, _i32, _u64, _u64, _u64, _u64, _dbl]),
    "vb_version": (ctypes.c_char_p, []),
}

_lib = None


def lib():
    """Load libvega_b200.so (built in-tree by __graft_entry__.build()).  Fails loudly."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C vega_b200/csrc`). vega_b200 has no CPU fallback.")
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)      # AttributeError if the library does not export it
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def check(rc):
    if rc != VB_OK:
        raise VegaB200Error(rc, lib().vb_last_error().decode(errors="replace"))
    return rc
