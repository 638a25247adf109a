"""ctypes binding of include/spl.h (libspalinalg_b200.so).  This is the only way the Python host
mirror reaches the device; there is no fallback: if the library is missing or no CUDA device is
present, imports succeed but every operation raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libspalinalg_b200.so")

SPL_OK, SPL_ERR_SHAPE, SPL_ERR_INVALID, SPL_ERR_CUDA, SPL_ERR_UNSUPPORTED, SPL_ERR_OOM, SPL_ERR_ARG = range(7)
SPL_CSR, SPL_CSC = 0, 1
SPL_F32, SPL_F64 = 0, 1
SPL_SPMV_AUTO, SPL_SPMV_VECTOR, SPL_SPMV_MERGE, SPL_SPMV_SPLIT, SPL_SPMV_SLICED, SPL_SPMV_STREAM, SPL_SPMV_SCATTER = 0, 1, 2, 3, 4, 5, 6
SPL_MAX_PEERS, SPL_IPC_HANDLE_BYTES = 8, 64

STATUS_NAMES = {0: "SPL_OK", 1: "SPL_ERR_SHAPE", 2: "SPL_ERR_INVALID", 3: "SPL_ERR_CUDA",
                4: "SPL_ERR_UNSUPPORTED", 5: "SPL_ERR_OOM", 6: "SPL_ERR_ARG"}

_vp, _u64, _i = C.c_void_p, C.c_uint64, C.c_int
_pp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); must list every symbol include/spl.h declares
SIGNATURES = {
    "spl_ctx_create": (_i, [_i, _vp, _pp]),
    "spl_ctx_destroy": (_i, [_vp]),
    "spl_ctx_sync": (_i, [_vp]),
    "spl_ctx_trim": (_i, [_vp]),
    "spl_host_alloc": (_i, [_u64, _pp]),
    "spl_host_free": (_i, [_vp]),
    "spl_host_register": (_i, [_vp, _u64]),
    "spl_host_unregister": (_i, [_vp]),
    "spl_last_error": (C.c_char_p, [_vp]),
    "spl_invalid_reason": (_i, [_vp]),
    "spl_launch_count": (_u64, [_vp]),
    "spl_mat_from_coo": (_i, [_vp, _i, _i, _u64, _u64, _u64, _vp, _vp, _vp, _i, _i, _pp]),
    "spl_mat_from_coo_dev": (_i, [_vp, _i, _i, _u64, _u64, _u64, _vp, _vp, _vp, _i, _i, _pp]),
    "spl_mat_from_compressed": (_i, [_vp, _i, _i, _u64, _u64, _u64, _vp, _u64, _vp, _u64, _vp, _pp]),
    "spl_mat_from_compressed_dev": (_i, [_vp, _i, _i, _u64, _u64, _u64, _vp, _vp, _vp, _i, _pp]),
    "spl_mat_from_compressed_dev64": (_i, [_vp, _i, _i, _u64, _u64, _u64, _vp, _vp, _vp, _i, _pp]),
    "spl_mat_device_ptr64": (_i, [_vp, _pp]),
    "spl_mat_eye": (_i, [_vp, _i, _i, _u64, _pp]),
    "spl_mat_convert": (_i, [_vp, _vp, _i, _pp]),
    "spl_mat_transpose": (_i, [_vp, _vp, _pp]),
    "spl_mat_add": (_i, [_vp, _vp, _vp, _pp]),
    "spl_mat_sub": (_i, [_vp, _vp, _vp, _pp]),
    "spl_mat_mul": (_i, [_vp, _vp, _vp, _pp]),
    "spl_mat_neg": (_i, [_vp, _vp, _pp]),
    "spl_spmv": (_i, [_vp, _vp, _vp, _vp]),
    "spl_spmv_ex": (_i, [_vp, _vp, _vp, _vp, _i]),
    "spl_spmv_host": (_i, [_vp, _vp, _vp, _vp]),
    "spl_spmv_choice": (_i, [_vp, _vp, C.POINTER(_i), C.POINTER(_i)]),
    "spl_mat_info": (_i, [_vp, C.POINTER(_i), C.POINTER(_i), C.POINTER(_u64), C.POINTER(_u64),
                          C.POINTER(_u64)]),
    "spl_mat_download": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "spl_mat_set_values": (_i, [_vp, _vp, _vp]),
    "spl_mat_device_ptrs": (_i, [_vp, _pp, _pp, _pp]),
    "spl_mat_to_coo": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "spl_mat_to_coo_dev": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "spl_mat_read_entries": (_i, [_vp, _vp, _u64, _u64, _vp, _vp, _vp]),
    "spl_mat_free": (_i, [_vp, _vp]),
    "spl_coo_route_dev": (_i, [_vp, _i, _i, _u64, _u64, _u64, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "spl_coo_route_count_dev": (_i, [_vp, _i, _u64, _u64, _u64, _vp, _vp, _i, _vp, _vp]),
    "spl_coo_route_peers_dev": (_i, [_vp, _i, _i, _u64, _u64, _u64, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "spl_mat_from_packed_dev": (_i, [_vp, _i, _i, _u64, _u64, _u64, _vp, _vp, _i, _i, _pp]),
    "spl_peer_alloc": (_i, [_vp, _u64, _pp, _vp]),
    "spl_peer_open": (_i, [_vp, _vp, _pp]),
    "spl_peer_close": (_i, [_vp, _vp]),
    "spl_peer_free": (_i, [_vp, _vp]),
    "spl_peer_barrier": (_i, [_vp, _i, _i, _vp, C.c_uint32, C.c_uint32]),
    "spl_peer_barrier_halo": (_i, [_vp, _i, _i, _vp, C.c_uint32, C.c_uint32, _i, _vp, _vp, _u64, _u64]),
    "spl_spmv_window": (_i, [_vp, _vp, _vp, _u64, _u64, _vp]),
    "spl_spmv_footprint": (_i, [_vp, _vp, C.POINTER(_u64), C.POINTER(_u64)]),
    "spl_spmv_transpose_window": (_i, [_vp, _vp, _vp, _vp]),
    "spl_peer_reduce_windows": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp, C.c_uint32, C.c_uint32, _vp]),
    "spl_peer_pull": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp]),
    "spl_peer_barrier_status": (_i, [_vp, C.POINTER(_i)]),
    "spl_peer_gather_rows": (_i, [_vp, _i, _i, _u64, _u64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _pp]),
    "spl_spmv_peer": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "spl_spmv_gather_fused": (_i, [_vp, _i, _u64, _i, _i, _vp, _vp, _i, _vp, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp, C.c_uint32, _u64, _vp,
                              C.c_uint32, C.c_uint32, _vp]),
    "spl_spmv_peer_host": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp]),
    "spl_coo_create": (_i, [_vp, _i, _u64, _u64, _u64, _pp]),
    "spl_coo_free": (_i, [_vp]),
    "spl_coo_last_error": (C.c_char_p, [_vp]),
    "spl_coo_push": (_i, [_vp, _u64, _u64, _vp]),
    "spl_coo_extend": (_i, [_vp, _u64, _vp, _vp, _vp]),
    "spl_coo_reserve": (_i, [_vp, _u64]),
    "spl_coo_truncate": (_i, [_vp, _u64]),
    "spl_coo_len": (_u64, [_vp]),
    "spl_coo_capacity": (_u64, [_vp]),
    "spl_coo_streamed": (_u64, [_vp]),
    "spl_coo_invalidate": (_i, [_vp, _u64]),
    "spl_coo_host_ptrs": (_i, [_vp, _pp, _pp, _pp]),
    "spl_mat_from_coo_builder": (_i, [_vp, _vp, _i, _i, _i, _pp]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library; raises if it has not been built (python -m spalinalg_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA library has not been built and there is no CPU "
                "fallback.  Run `python -m spalinalg_b200.build`.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)      # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
