"""ctypes binding of ``libevs.so`` (C ABI in ``include/evs.h``).  Fails loudly when the library is
missing: there is no Python, PyTorch or CPU fallback for any compute entry point."""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libevs.so")

EVS_OK, EVS_EINVAL, EVS_ENODEV, EVS_ECUDA, EVS_ENOMEM, EVS_EIO, EVS_EFORMAT, EVS_ELIMIT, EVS_ETIMEOUT = 0, -1, -2, -3, -4, -5, -6, -7, -8
EVS_F32, EVS_F16, EVS_BF16 = 0, 1, 2
EVS_STORE_F32, EVS_STORE_BF16_F32 = 0, 1
EVS_MAX_K = 112
EVS_MAX_K_LARGE = 2048
EVS_IPC_HANDLE_BYTES = 64

_c = ctypes
_vp, _i, _i64, _u64 = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_uint64
_pi, _pi64, _pf = _c.POINTER(_c.c_int), _c.POINTER(_c.c_int64), _c.POINTER(_c.c_float)

# name -> (restype, argtypes): every symbol include/evs.h declares
SIGNATURES = {
    "evs_version": (_i, []),
    "evs_last_error": (_c.c_char_p, []),
    "evs_device_count": (_i, [_pi]),
    "evs_index_create": (_i, [_i, _i, _i, _c.POINTER(_vp)]),
    "evs_index_free": (_i, [_vp]),
    "evs_index_d": (_i, [_vp, _pi]),
    "evs_index_ntotal": (_i, [_vp, _pi64]),
    "evs_index_device": (_i, [_vp, _pi]),
    "evs_index_storage": (_i, [_vp, _pi]),
    "evs_index_set_id_base": (_i, [_vp, _i64]),
    "evs_index_id_base": (_i, [_vp, _pi64]),
    "evs_index_reserve": (_i, [_vp, _i64]),
    "evs_index_add": (_i, [_vp, _i64, _vp]),
    "evs_index_add_dev": (_i, [_vp, _i64, _vp, _i, _vp]),
    "evs_index_add_synth": (_i, [_vp, _i64, _u64, _i]),
    "evs_index_add_rows_from": (_i, [_vp, _vp, _i64, _vp]),
    "evs_index_get_rows": (_i, [_vp, _i64, _i64, _vp]),
    "evs_index_search": (_i, [_vp, _i64, _vp, _i64, _vp, _vp]),
    "evs_index_search_dev": (_i, [_vp, _i64, _vp, _i64, _vp, _vp, _vp]),
    "evs_index_search_partial_dev": (_i, [_vp, _i64, _vp, _i64, _vp, _vp, _vp]),
    "evs_merge_partials_dev": (_i, [_i, _i, _i64, _i64, _vp, _vp, _i64, _vp, _vp, _vp]),
    "evs_index_last_margins": (_i, [_vp, _i64, _vp]),
    "evs_index_write": (_i, [_vp, _c.c_char_p]),
    "evs_index_read": (_i, [_c.c_char_p, _i, _i, _c.POINTER(_vp)]),
    "evs_l2_normalize_dev": (_i, [_i, _vp, _i64, _i, _i, _vp]),
    "evs_l2_normalize": (_i, [_i, _vp, _i64, _i]),
    "evs_f32_to_bf16_dev": (_i, [_i, _vp, _vp, _i64, _vp]),
    "evs_set_option": (_i, [_c.c_char_p, _i64]),
    "evs_get_option": (_i, [_c.c_char_p, _pi64]),
    "evs_kernel_launches": (_i64, []),
    "evs_index_time_scan": (_i, [_vp, _i64, _vp, _i64, _i, _pf]),
    "evs_index_scan_profile": (_i, [_vp, _pi64, _c.POINTER(_c.c_double)]),
    "evs_index_tc_max_queries": (_i, [_vp, _pi]),
    "evs_index_tc_x3_max_queries": (_i, [_vp, _pi]),
    "evs_index_tc_scores_dev": (_i, [_vp, _i64, _vp, _vp, _pi, _vp]),
    "evs_exchange_create": (_i, [_i, _i, _i, _i64, _i64, _c.POINTER(_vp)]),
    "evs_exchange_handle": (_i, [_vp, _vp, _i64]),
    "evs_exchange_connect": (_i, [_vp, _vp, _i64]),
    "evs_exchange_status": (_i, [_vp, _pi, _pi64]),
    "evs_exchange_free": (_i, [_vp]),
    "evs_index_search_exchange_dev": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp]),
    "evs_index_search_exchange": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _vp]),
    "evs_index_set_storage": (_i, [_vp, _i]),
    "evs_index_max_row_norm": (_i, [_vp, _pf]),
    "evs_index_guard_stats": (_i, [_vp, _pi64, _pi64]),
    "evs_index_shadow_stats": (_i, [_vp, _pi64, _pf, _pi64]),
    "evs_index_large_k_stats": (_i, [_vp, _pi64, _pi64]),
    "evs_index_coalesce_stats": (_i, [_vp, _pi64, _pi64, _pi64]),
    "evs_index_read_rows": (_i, [_c.c_char_p, _i, _i, _i64, _i64, _c.POINTER(_vp), _pi64]),
    "evs_index_file_info": (_i, [_c.c_char_p, _pi, _pi64]),
    "evs_index_scan_clocks": (_i, [_vp, _vp, _i64, _pi64]),
}

_lib = None


class EvsError(RuntimeError):
    """A libevs call failed (faiss raises RuntimeError from FaissException the same way)."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"libevs error {code}: {msg}")
        self.code = code


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  evo-ssearch_b200 has no fallback path without its CUDA library.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError here = header and library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().evs_last_error()
        raise EvsError(rc, msg.decode("utf-8", "replace") if msg else "")


_c_char = ctypes.c_char


def host_ptr(a) -> int:
    """Address of a C-contiguous numpy array's data.  ``a.ctypes.data_as(...)`` builds a helper object per call (~5 us, three
    of them per search: a third of the 10k-row search's end-to-end time); the buffer protocol is ~6 times cheaper."""
    try:
        return ctypes.addressof(_c_char.from_buffer(a))
    except (TypeError, ValueError, BufferError):  # read-only or empty arrays
        return a.ctypes.data


def device_count() -> int:
    n = ctypes.c_int(0)
    check(lib().evs_device_count(ctypes.byref(n)))
    return n.value


def set_option(name: str, value: int) -> None:
    check(lib().evs_set_option(name.encode(), int(value)))


def get_option(name: str) -> int:
    v = ctypes.c_int64(0)
    check(lib().evs_get_option(name.encode(), ctypes.byref(v)))
    return v.value


def kernel_launches() -> int:
    return int(lib().evs_kernel_launches())
