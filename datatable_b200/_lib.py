"""
ctypes binding of the C-ABI (include/dtb200.h).  The library is built in-tree
by `__graft_entry__.build()` (datatable_b200/csrc/Makefile) into
datatable_b200/lib/libdtb200.so.  There is no fallback: if the library is
missing, importing this module raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libdtb200.so")

# -- constants mirrored from include/dtb200.h ---------------------------------
ABI_VERSION = 1
BOOL, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64, DATE32, TIME64 = 1, 2, 3, 4, 5, 6, 7, 17, 18
FLAG_NONE, FLAG_DESCENDING, FLAG_SORT_ONLY = 0, 2, 4
NA_FIRST, NA_LAST, NA_REMOVE = 1, 2, 3
OP_SUM, OP_MEAN, OP_MIN, OP_MAX, OP_COUNT, OP_COUNTNA, OP_NROWS = 1, 2, 3, 4, 5, 6, 7
OP_FIRST, OP_LAST, OP_SD, OP_MEDIAN, OP_NUNIQUE = 8, 9, 10, 11, 12
SET_UNION, SET_INTERSECT, SET_SETDIFF, SET_SYMDIFF = 0, 1, 2, 3
WIN_CUMSUM, WIN_CUMPROD, WIN_CUMMIN, WIN_CUMMAX, WIN_CUMCOUNT, WIN_NGROUP, WIN_FILLNA, WIN_SHIFT = 1, 2, 3, 4, 5, 6, 7, 8
OK, EINVAL, ENOTIMPL, ECUDA, ENOMEM, ENOSPACE = 0, -1, -2, -3, -4, -5

EXPORTS = [
    "dtb_last_error", "dtb_abi_version", "dtb_stype_size", "dtb_reduce_out_stype", "dtb_init",
    "dtb_group", "dtb_group64", "dtb_groupby_create", "dtb_groupby_create_reduce", "dtb_groupby_reduced", "dtb_groupby_norder", "dtb_groupby_ngroups",
    "dtb_groupby_order", "dtb_groupby_offsets", "dtb_groupby_destroy", "dtb_groupby_reduce", "dtb_reduce",
    "dtb_groupby_reduce_begin", "dtb_groupby_reduce_add", "dtb_groupby_reduce_end", "dtb_slice_groups",
    "dtb_gather", "dtb_memcpy", "dtb_set_option", "dtb_get_option", "dtb_last_call_stats",
    "dtb_profile_count", "dtb_profile_get", "dtb_profile_reset",
    "dtb_dense_scatter", "dtb_dense_compact",
    "dtb_sort_grouped", "dtb_set_select", "dtb_largest_group", "dtb_join", "dtb_cache_begin", "dtb_cache_end", "dtb_lower_bound",
    "dtb_window_out_stype", "dtb_window",
]


class dtb_col(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("stype", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class dtb_reduce_spec(ctypes.Structure):
    _fields_ = [("op", ctypes.c_int32), ("reserved", ctypes.c_int32), ("value", dtb_col)]


class dtb_call_stats(ctypes.Structure):
    _fields_ = [("kernels_launched", ctypes.c_int32), ("radix_passes", ctypes.c_int32),
                ("key_bits", ctypes.c_int32), ("cache_hits", ctypes.c_int32),
                ("scratch_bytes", ctypes.c_int64)]


class DtbError(RuntimeError):
    """Base of the engine's exceptions (mirrors dt::Error, utils/exceptions.h:43)."""
    code = None


class DtbValueError(DtbError, ValueError):
    code = EINVAL


class DtbNotImplError(DtbError, NotImplementedError):
    code = ENOTIMPL


class DtbCudaError(DtbError):
    code = ECUDA


class DtbMemoryError(DtbError, MemoryError):
    code = ENOMEM


_ERR = {EINVAL: DtbValueError, ENOTIMPL: DtbNotImplError, ECUDA: DtbCudaError,
        ENOMEM: DtbMemoryError, ENOSPACE: DtbValueError}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA extension first "
            "(python -c 'import __graft_entry__ as g; g.build()'). "
            "datatable_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    c = ctypes
    lib.dtb_last_error.restype = c.c_char_p
    lib.dtb_abi_version.restype = c.c_int
    lib.dtb_stype_size.argtypes = [c.c_int]
    lib.dtb_reduce_out_stype.argtypes = [c.c_int, c.c_int]
    lib.dtb_init.argtypes = [c.c_int]
    lib.dtb_group.argtypes = [c.POINTER(dtb_col), c.c_int, c.POINTER(c.c_int), c.c_int, c.c_int64,
                              c.c_void_p, c.c_void_p, c.c_void_p, c.c_int64,
                              c.POINTER(c.c_int64), c.POINTER(c.c_int64)]
    lib.dtb_group64.argtypes = lib.dtb_group.argtypes
    lib.dtb_groupby_create.argtypes = [c.POINTER(dtb_col), c.c_int, c.POINTER(c.c_int), c.c_int,
                                       c.c_int64, c.c_void_p, c.POINTER(c.c_void_p)]
    lib.dtb_groupby_create_reduce.argtypes = [c.POINTER(dtb_col), c.c_int, c.POINTER(c.c_int), c.c_int,
                                              c.c_int64, c.c_void_p, c.POINTER(dtb_reduce_spec), c.c_int,
                                              c.POINTER(c.c_void_p)]
    lib.dtb_groupby_reduced.restype = c.c_void_p
    lib.dtb_groupby_reduced.argtypes = [c.c_void_p, c.c_int]
    for fn in ("dtb_groupby_norder", "dtb_groupby_ngroups"):
        getattr(lib, fn).restype = c.c_int64
        getattr(lib, fn).argtypes = [c.c_void_p]
    for fn in ("dtb_groupby_order", "dtb_groupby_offsets"):
        getattr(lib, fn).restype = c.c_void_p
        getattr(lib, fn).argtypes = [c.c_void_p]
    lib.dtb_groupby_destroy.argtypes = [c.c_void_p, c.c_void_p]
    lib.dtb_groupby_reduce.argtypes = [c.c_void_p, c.c_int, dtb_col, c.c_int64, c.c_void_p, c.c_void_p]
    lib.dtb_groupby_reduce_begin.argtypes = [c.c_void_p, c.c_int, c.c_int, c.c_void_p, c.POINTER(c.c_void_p)]
    lib.dtb_groupby_reduce_add.argtypes = [c.c_void_p, c.c_void_p, c.c_int64, c.c_int64, c.c_void_p]
    lib.dtb_groupby_reduce_end.argtypes = [c.c_void_p, c.c_void_p, c.c_void_p]
    lib.dtb_slice_groups.argtypes = [c.c_void_p, c.c_int64, c.c_int64, c.c_int64, c.c_int64, c.c_void_p, c.c_void_p, c.c_int64,
                                     c.c_void_p, c.POINTER(c.c_int64), c.POINTER(c.c_int64)]
    lib.dtb_reduce.argtypes = [c.c_int, dtb_col, c.c_int64, c.c_void_p, c.c_int, c.c_void_p,
                               c.c_int64, c.c_void_p, c.c_void_p]
    lib.dtb_gather.argtypes = [dtb_col, c.c_int64, c.c_void_p, c.c_int, c.c_int64, c.c_void_p, c.c_void_p]
    lib.dtb_dense_scatter.argtypes = [c.c_void_p, c.c_int, c.c_void_p, c.c_int64, c.c_int64, c.c_int64,
                                      c.c_void_p, c.c_void_p, c.c_void_p]
    lib.dtb_dense_compact.argtypes = [c.c_void_p, c.c_void_p, c.c_int64, c.c_int64, c.c_int, c.c_void_p, c.c_void_p,
                                      c.POINTER(c.c_int64), c.c_void_p]
    lib.dtb_sort_grouped.argtypes = [dtb_col, c.c_int64, c.c_void_p, c.c_void_p, c.c_int64, c.c_void_p, c.c_void_p]
    lib.dtb_set_select.argtypes = [c.c_int, c.c_void_p, c.c_void_p, c.c_int64, c.POINTER(c.c_int64), c.c_int,
                                   c.c_void_p, c.c_void_p, c.POINTER(c.c_int64)]
    lib.dtb_largest_group.argtypes = [c.c_void_p, c.c_int64, c.c_int64, c.c_void_p, c.POINTER(c.c_int64),
                                      c.POINTER(c.c_int64)]
    lib.dtb_join.argtypes = [c.POINTER(dtb_col), c.POINTER(dtb_col), c.c_int, c.c_int64, c.c_int64, c.c_void_p,
                             c.c_void_p]
    lib.dtb_lower_bound.argtypes = [dtb_col, c.c_int64, dtb_col, c.c_int64, c.c_void_p, c.c_void_p]
    lib.dtb_window_out_stype.argtypes = [c.c_int, c.c_int]
    lib.dtb_window.argtypes = [c.c_int, c.c_int64, dtb_col, c.c_int64, c.c_void_p, c.c_void_p, c.c_int64, c.c_void_p,
                               c.c_void_p]
    lib.dtb_memcpy.argtypes = [c.c_void_p, c.c_void_p, c.c_int64, c.c_void_p]
    lib.dtb_set_option.argtypes = [c.c_char_p, c.c_int64]
    lib.dtb_get_option.argtypes = [c.c_char_p, c.POINTER(c.c_int64)]
    lib.dtb_last_call_stats.argtypes = [c.POINTER(dtb_call_stats)]
    lib.dtb_profile_get.argtypes = [c.c_int, c.c_char_p, c.c_int, c.POINTER(c.c_double)]
    if lib.dtb_abi_version() != ABI_VERSION:
        raise ImportError("libdtb200.so ABI version mismatch")
    return lib


lib = _load()


def check(rc):
    if rc == OK:
        return
    msg = lib.dtb_last_error().decode("utf-8", "replace")
    raise _ERR.get(rc, DtbError)(msg)


def last_call_stats():
    st = dtb_call_stats()
    check(lib.dtb_last_call_stats(ctypes.byref(st)))
    return {"kernels_launched": st.kernels_launched, "radix_passes": st.radix_passes,
            "key_bits": st.key_bits, "cache_hits": st.cache_hits, "scratch_bytes": st.scratch_bytes}


def profile_records(reset=True):
    """[(kernel family, ms), ...] collected while option "profile" is on."""
    out = []
    buf = ctypes.create_string_buffer(64)
    ms = ctypes.c_double(0)
    for i in range(lib.dtb_profile_count()):
        check(lib.dtb_profile_get(i, buf, 64, ctypes.byref(ms)))
        out.append((buf.value.decode(), ms.value))
    if reset:
        lib.dtb_profile_reset()
    return out
