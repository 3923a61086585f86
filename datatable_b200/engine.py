"""
Functional host layer over the C-ABI: group() / reduce() / gather() on raw
columns.  Mirrors the reference's internal seam (SURVEY.md 8b):

    RiGb group(columns, flags, na_pos)              src/core/sort.h:56-58
    reducer columns materialised over a Groupby     src/core/column/reduce_unary.h:30-68
    ArrayView gather                                src/core/column/view.cc:88-155

Columns are numpy arrays (host; staged by the engine) or torch CUDA tensors
(device-resident; zero-copy).  Results come back in the same kind of memory.
Everything is computed by libdtb200.so on the GPU; there is no CPU fallback.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import (BOOL, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64, DATE32, TIME64, FLAG_DESCENDING,
                   FLAG_SORT_ONLY, NA_FIRST, NA_LAST, NA_REMOVE, check, dtb_col, lib)

try:  # torch is plumbing only: device memory + streams
    import torch
except Exception:  # pragma: no cover
    torch = None

_NP2ST = {np.dtype(np.bool_): BOOL, np.dtype(np.int8): INT8, np.dtype(np.int16): INT16,
          np.dtype(np.int32): INT32, np.dtype(np.int64): INT64,
          np.dtype(np.float32): FLOAT32, np.dtype(np.float64): FLOAT64}
_ST2NP = {BOOL: np.int8, INT8: np.int8, INT16: np.int16, INT32: np.int32, INT64: np.int64,
          FLOAT32: np.float32, FLOAT64: np.float64, DATE32: np.int32, TIME64: np.int64}


def _torch_dtype(st):
    return {BOOL: torch.int8, INT8: torch.int8, INT16: torch.int16, INT32: torch.int32,
            INT64: torch.int64, FLOAT32: torch.float32, FLOAT64: torch.float64, DATE32: torch.int32,
            TIME64: torch.int64}[st]


def is_tensor(x):
    return torch is not None and isinstance(x, torch.Tensor)


class Col:
    """A material fixed-width column handed to the engine: pointer + stype + nrows."""

    def __init__(self, data, stype=None):
        if isinstance(data, Col):
            self.__dict__.update(data.__dict__)
            return
        if is_tensor(data):
            if not data.is_contiguous():
                data = data.contiguous()
            self.data = data
            self.on_device = data.is_cuda
            self.ptr = data.data_ptr()
            self.nrows = data.numel()
            npdt = np.dtype(str(data.dtype).replace("torch.", "")) if data.dtype != torch.bool else np.dtype(np.bool_)
        else:
            data = np.ascontiguousarray(data)
            self.data = data
            self.on_device = False
            self.ptr = data.ctypes.data
            self.nrows = data.shape[0]
            npdt = data.dtype
        if stype is None:
            if npdt not in _NP2ST:
                raise _lib.DtbNotImplError(f"Unable to sort Column of dtype {npdt}")
            stype = _NP2ST[npdt]
        self.stype = stype

    @classmethod
    def from_ptr(cls, ptr, stype, nrows, on_device=True, owner=None):
        """Wrap a raw pointer (e.g. the HBM-resident RowIndex of a Groupby handle) without copying."""
        self = cls.__new__(cls)
        self.data, self.on_device, self.ptr, self.nrows, self.stype = owner, on_device, ptr, nrows, stype
        return self

    def c(self):
        return dtb_col(ctypes.c_void_p(self.ptr), self.stype, 0)


def _stream():
    if torch is not None and torch.cuda.is_available():
        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    return ctypes.c_void_p(0)


def _alloc(n, st, device):
    """Output buffer: torch CUDA tensor for device results, numpy otherwise."""
    if device:
        t = torch.empty(max(n, 0), dtype=_torch_dtype(st), device="cuda")
        return t, t.data_ptr()
    a = np.empty(max(n, 0), dtype=_ST2NP[st])
    return a, a.ctypes.data


def group(cols, flags=None, na_pos=NA_FIRST):
    """group() of the reference: returns (order, offsets, ngroups).

    order   : int32 RowIndex (ARR32) -- stable order of the rows
    offsets : int32[ngroups+1] Groupby offsets, or None when flags[0] has SORT_ONLY
    """
    cols = [Col(c) for c in cols]
    nk = len(cols)
    if nk == 0:
        raise _lib.DtbValueError("group() needs at least one key column")
    n = cols[0].nrows
    for c in cols:
        if c.nrows != n:
            raise _lib.DtbValueError("key columns have different numbers of rows")
    flags = list(flags) if flags is not None else [0] * nk
    device = all(c.on_device for c in cols)
    do_groups = not (flags[0] & FLAG_SORT_ONLY)
    ckeys = (dtb_col * nk)(*[c.c() for c in cols])
    cflags = (ctypes.c_int * nk)(*flags)
    order, optr = _alloc(n, INT32, device)
    offs, fptr = (_alloc(n + 1, INT32, device) if do_groups else (None, 0))
    ng = ctypes.c_int64(-1)
    no = ctypes.c_int64(0)
    check(lib.dtb_group(ckeys, nk, cflags, na_pos, n, _stream(), ctypes.c_void_p(optr),
                        ctypes.c_void_p(fptr), n + 1 if do_groups else 0,
                        ctypes.byref(ng), ctypes.byref(no)))
    order = order[:no.value]
    if ng.value < 0:
        return order, None, None
    return order, offs[:ng.value + 1], ng.value


def group64(cols, flags=None, na_pos=NA_FIRST):
    """group() with the ARR64 layout (dtb_group64): int64 RowIndex and int64 Groupby offsets; for frames of
    more than INT32_MAX rows (up to 2^32 on one GPU) or callers that want 64-bit indices."""
    cols = [Col(c) for c in cols]
    nk = len(cols)
    n = cols[0].nrows
    flags = list(flags) if flags is not None else [0] * nk
    device = all(c.on_device for c in cols)
    do_groups = not (flags[0] & FLAG_SORT_ONLY)
    ckeys = (dtb_col * nk)(*[c.c() for c in cols])
    cflags = (ctypes.c_int * nk)(*flags)
    order, optr = _alloc(n, INT64, device)
    ng = ctypes.c_int64(-1)
    no = ctypes.c_int64(0)
    if do_groups:
        # the number of groups is not known in advance: a first sizing pass is avoided by allocating n + 1
        offs, fptr = _alloc(n + 1, INT64, device)
    else:
        offs, fptr = None, 0
    check(lib.dtb_group64(ckeys, nk, cflags, na_pos, n, _stream(), ctypes.c_void_p(optr),
                          ctypes.c_void_p(fptr), n + 1 if do_groups else 0, ctypes.byref(ng), ctypes.byref(no)))
    order = order[:no.value]
    if ng.value < 0:
        return order, None, None
    return order, offs[:ng.value + 1], ng.value


class Groupby:
    """Device-resident result of group(): owns the RowIndex and the Groupby offsets in HBM
    (dtb_groupby handle).  Mirrors the pair the reference keeps in EvalContext
    (src/core/expr/eval_context.cc:278-280)."""

    def __init__(self, cols, flags=None, na_pos=NA_FIRST, reducers=None):
        """reducers: optional [(op, value column or None), ...] evaluated inside the same call
        (dtb_groupby_create_reduce): with a small key domain they overlap the sort on a side stream."""
        cols = [Col(c) for c in cols]
        nk = len(cols)
        n = cols[0].nrows
        flags = list(flags) if flags is not None else [0] * nk
        ckeys = (dtb_col * nk)(*[c.c() for c in cols])
        cflags = (ctypes.c_int * nk)(*flags)
        h = ctypes.c_void_p(0)
        self._red = []
        if reducers:
            specs = (_lib.dtb_reduce_spec * len(reducers))()
            for i, (op, val) in enumerate(reducers):
                if op == _lib.OP_NROWS or val is None:
                    v = None
                    specs[i] = _lib.dtb_reduce_spec(_lib.OP_NROWS, 0, dtb_col(None, INT8, 0))
                    self._red.append((_lib.OP_NROWS, INT64, None))
                else:
                    v = Col(val)
                    out_st = lib.dtb_reduce_out_stype(op, v.stype)
                    if not out_st:
                        raise _lib.DtbValueError(f"Invalid column of stype {v.stype} in reducer {op}")
                    specs[i] = _lib.dtb_reduce_spec(op, 0, v.c())
                    self._red.append((op, out_st, v))
            check(lib.dtb_groupby_create_reduce(ckeys, nk, cflags, na_pos, n, _stream(), specs, len(reducers),
                                                ctypes.byref(h)))
        else:
            check(lib.dtb_groupby_create(ckeys, nk, cflags, na_pos, n, _stream(), ctypes.byref(h)))
        self._h = h
        self._keys = cols            # the handle may re-read the key columns (direct-address reducers)
        self.norder = lib.dtb_groupby_norder(h)
        self.ngroups = lib.dtb_groupby_ngroups(h)
        self.order_ptr = lib.dtb_groupby_order(h)
        self.offsets_ptr = lib.dtb_groupby_offsets(h)

    def reduce(self, op, value, out=None):
        if op == _lib.OP_NROWS:
            v = Col(torch.empty(0, dtype=torch.int8, device="cuda"), INT8)
            out_st = INT64
        else:
            v = Col(value)
            out_st = lib.dtb_reduce_out_stype(op, v.stype)
        if not out_st:
            raise _lib.DtbValueError(f"Invalid column of stype {v.stype} in reducer {op}")
        if out is None:
            out, optr = _alloc(self.ngroups, out_st, v.on_device)
        else:
            optr = out.data_ptr() if is_tensor(out) else out.ctypes.data
        check(lib.dtb_groupby_reduce(self._h, op, v.c(), v.nrows, _stream(), ctypes.c_void_p(optr)))
        return out

    def reduce_pieces(self, op, stype, pieces):
        """The reducer fed piecewise (dtb_groupby_reduce_begin / _add / _end).  pieces: [(CUDA tensor with rows
        [row0, row0 + len), row0, CUDA event to wait for or None), ...] covering every row once.  Returns the result
        (CUDA tensor) or None when the handle has no streaming path for this reducer (use reduce())."""
        out_st = lib.dtb_reduce_out_stype(op, stype)
        if not out_st:
            raise _lib.DtbValueError(f"Invalid column of stype {stype} in reducer {op}")
        st = ctypes.c_void_p(0)
        rc = lib.dtb_groupby_reduce_begin(self._h, op, stype, _stream(), ctypes.byref(st))
        if rc == _lib.ENOTIMPL:
            return None
        check(rc)
        cur = torch.cuda.current_stream()
        try:
            for t, row0, ev in pieces:
                if ev is not None:
                    cur.wait_event(ev)
                check(lib.dtb_groupby_reduce_add(st, ctypes.c_void_p(t.data_ptr()), int(row0), t.numel(), _stream()))
        except Exception:
            lib.dtb_groupby_reduce_end(st, _stream(), None)          # frees the state
            raise
        out = torch.empty(max(self.ngroups, 0), dtype=_torch_dtype(out_st), device="cuda")
        check(lib.dtb_groupby_reduce_end(st, _stream(), ctypes.c_void_p(out.data_ptr())))
        return out

    def reduced(self, i):
        """Result of the i-th reducer passed to the constructor (CUDA tensor, ngroups elements)."""
        op, out_st, _ = self._red[i]
        t = torch.empty(max(self.ngroups, 0), dtype=_torch_dtype(out_st), device="cuda")
        if self.ngroups > 0:
            _memcpy_d2d(t.data_ptr(), lib.dtb_groupby_reduced(self._h, i), t.numel() * t.element_size())
        return t

    def sort_grouped(self, value):
        """RowIndex with the rows of every group ordered by `value` (NA first): what median / nunique read."""
        v = Col(value)
        t = torch.empty(self.norder, dtype=torch.int32, device="cuda")
        if self.norder:
            check(lib.dtb_sort_grouped(v.c(), v.nrows, ctypes.c_void_p(self.order_ptr), ctypes.c_void_p(self.offsets_ptr),
                                       self.ngroups, _stream(), ctypes.c_void_p(t.data_ptr())))
        return t

    def reduce_ordered(self, op, value, order):
        """Reducer over the handle's groups but another RowIndex (the output of sort_grouped)."""
        v = Col(value)
        out_st = lib.dtb_reduce_out_stype(op, v.stype)
        if not out_st:
            raise _lib.DtbValueError(f"Invalid column of stype {v.stype} in reducer {op}")
        out, optr = _alloc(self.ngroups, out_st, True)
        check(lib.dtb_reduce(op, v.c(), v.nrows, ctypes.c_void_p(order.data_ptr()), 0, ctypes.c_void_p(self.offsets_ptr),
                             self.ngroups, _stream(), ctypes.c_void_p(optr)))
        return out

    def window(self, op, value, param=0):
        """Window function over the handle's RowIndex and Groupby (CUDA tensor, one value per row of the RowIndex)."""
        return window(op, value, self.order_col(), self.offsets_col(), param)

    def order_col(self):
        """The RowIndex as a zero-copy column view (valid while the handle lives)."""
        return Col.from_ptr(self.order_ptr, INT32, self.norder, owner=self)

    def offsets_col(self, drop_last=False):
        return Col.from_ptr(self.offsets_ptr, INT32, self.ngroups + (0 if drop_last else 1), owner=self)

    def first_rows(self):
        """Row id of the first row of every group: order[offsets[:-1]] (eval_context.cc:124-135)."""
        return gather(self.order_col(), self.offsets_col(drop_last=True))

    def order(self):
        t = torch.empty(self.norder, dtype=torch.int32, device="cuda")
        if self.norder:
            _memcpy_d2d(t.data_ptr(), self.order_ptr, 4 * self.norder)
        return t

    def offsets(self):
        if self.ngroups < 0:
            return None
        t = torch.empty(self.ngroups + 1, dtype=torch.int32, device="cuda")
        _memcpy_d2d(t.data_ptr(), self.offsets_ptr, 4 * (self.ngroups + 1))
        return t

    def close(self):
        if self._h:
            lib.dtb_groupby_destroy(self._h, _stream())
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _memcpy_d2d(dst, src, nbytes):
    check(lib.dtb_memcpy(ctypes.c_void_p(dst), ctypes.c_void_p(src), nbytes, _stream()))


def reduce_out_stype(op, stype):
    return lib.dtb_reduce_out_stype(op, stype)


def reduce(op, value, order, offsets, stype=None):
    """Per-group reducer over `value` viewed through RowIndex `order` (None = identity)."""
    ngroups = int(offsets.shape[0]) - 1
    if op == _lib.OP_NROWS:
        v = None
        vst, vptr, vn, vdev = INT8, 0, 0, is_tensor(offsets) and offsets.is_cuda
    else:
        v = Col(value, stype)
        vst, vptr, vn, vdev = v.stype, v.ptr, v.nrows, v.on_device
    out_st = lib.dtb_reduce_out_stype(op, vst)
    if not out_st:
        raise _lib.DtbValueError(f"Invalid column of stype {vst} in reducer {op}")
    out, optr = _alloc(ngroups, out_st, vdev)
    o = None if order is None else Col(order)
    f = Col(offsets)
    is64 = 0
    if o is not None:
        if o.stype == INT64:
            is64 = 1
        elif o.stype != INT32:
            raise _lib.DtbValueError("order must be int32 or int64")
    check(lib.dtb_reduce(op, dtb_col(ctypes.c_void_p(vptr), vst, 0), vn,
                         ctypes.c_void_p(o.ptr) if o is not None else None, is64,
                         ctypes.c_void_p(f.ptr), ngroups, _stream(), ctypes.c_void_p(optr)))
    return out


def window_out_stype(op, stype):
    return lib.dtb_window_out_stype(op, stype)


def window(op, value, order, offsets, param=0, stype=None):
    """Grouped cumulative / window function (dtb_window): one value per position of the grouped frame given by
    RowIndex `order` (None = identity) and Groupby `offsets`.  param: `reverse` for WIN_CUMSUM .. WIN_FILLNA, the
    shift n for WIN_SHIFT.  `value` is ignored (may be None) for WIN_CUMCOUNT / WIN_NGROUP.  The result lives where
    the value column (or, without one, the offsets) lives."""
    f = Col(offsets)
    ngroups = f.nrows - 1
    if op in (_lib.WIN_CUMCOUNT, _lib.WIN_NGROUP):
        vst, vptr, vn, device = INT8, 0, 0, f.on_device
    else:
        v = Col(value, stype)
        vst, vptr, vn, device = v.stype, v.ptr, v.nrows, v.on_device
    out_st = lib.dtb_window_out_stype(op, vst)
    if not out_st:
        raise _lib.DtbValueError(f"Invalid column of stype {vst} in window op {op}")
    o = None if order is None else Col(order)
    if o is not None and o.stype != INT32:
        raise _lib.DtbValueError("order must be int32")
    if ngroups <= 0:
        n = 0
    elif isinstance(offsets, Col):
        n = _offsets_total(f)
    else:
        last = offsets[-1]
        n = int(last.item() if is_tensor(last) else last)
    out, optr = _alloc(n, out_st, device)
    check(lib.dtb_window(op, int(param), dtb_col(ctypes.c_void_p(vptr), vst, 0), vn,
                         ctypes.c_void_p(o.ptr) if o is not None else None, ctypes.c_void_p(f.ptr), ngroups,
                         _stream(), ctypes.c_void_p(optr)))
    return out


def _offsets_total(f):
    """offsets[ngroups] of an offsets column given as a Col (e.g. the HBM-resident offsets of a Groupby handle)."""
    n = ctypes.c_int32(0)
    check(lib.dtb_memcpy(ctypes.byref(n), ctypes.c_void_p(f.ptr + 4 * (f.nrows - 1)), 4, _stream()))
    return n.value


def gather(src, order, stype=None):
    """Materialise `src` through RowIndex `order` (negative index -> NA)."""
    s = Col(src, stype)
    o = Col(order)
    if o.stype not in (INT32, INT64):
        raise _lib.DtbValueError("order must be int32 or int64")
    n = o.nrows
    device = s.on_device and o.on_device
    out, optr = _alloc(n, s.stype, device)
    if not device and s.stype == BOOL and isinstance(s.data, np.ndarray) and s.data.dtype == np.bool_:
        out = out.view(np.bool_)
    check(lib.dtb_gather(s.c(), s.nrows, ctypes.c_void_p(o.ptr), 1 if o.stype == INT64 else 0, n,
                         _stream(), ctypes.c_void_p(optr)))
    return out


def sort_grouped(value, order, offsets, stype=None):
    """Column::sort_grouped (sort.cc:1499-1530): reorder the rows inside every group of (order, offsets)
    by `value` ascending, NA first, stable.  Returns the new int32 RowIndex (median / nunique read it)."""
    v = Col(value, stype)
    f = Col(offsets)
    ngroups = f.nrows - 1
    o = None if order is None else Col(order)
    if o is not None and o.stype != INT32:
        raise _lib.DtbValueError("order must be int32")
    n = int(offsets[-1].item()) if is_tensor(offsets) else int(offsets[-1])
    device = v.on_device and f.on_device and (o is None or o.on_device)
    out, optr = _alloc(n, INT32, device)
    check(lib.dtb_sort_grouped(v.c(), v.nrows, ctypes.c_void_p(o.ptr) if o is not None else None,
                               ctypes.c_void_p(f.ptr), ngroups, _stream(), ctypes.c_void_p(optr)))
    return out


def set_select(mode, order, offsets, cum_sizes):
    """Group selection of union / intersect / setdiff / symdiff (set_funcs.cc:126-456): the first-row
    indices of the groups the operation keeps (int32, same memory kind as `order`)."""
    o, f = Col(order), Col(offsets)
    ngroups = f.nrows - 1
    device = o.on_device and f.on_device
    out, optr = _alloc(max(ngroups, 0), INT32, device)
    K = len(cum_sizes)
    cs = (ctypes.c_int64 * K)(*[int(x) for x in cum_sizes])
    nout = ctypes.c_int64(0)
    check(lib.dtb_set_select(int(mode), ctypes.c_void_p(o.ptr), ctypes.c_void_p(f.ptr), ngroups, cs, K,
                             _stream(), ctypes.c_void_p(optr), ctypes.byref(nout)))
    return out[:nout.value]


def largest_group(offsets, skip=0):
    """(index, size) of the first largest group among groups [skip, ngroups) -- mode / nmodal (stats.cc:984-991)."""
    f = Col(offsets)
    idx, size = ctypes.c_int64(-1), ctypes.c_int64(0)
    check(lib.dtb_largest_group(ctypes.c_void_p(f.ptr), f.nrows - 1, int(skip), _stream(),
                                ctypes.byref(idx), ctypes.byref(size)))
    return idx.value, size.value


SLICE_NA = -2**63


def slice_groups(offsets, start=None, stop=None, step=None):
    """An integer slice applied inside every group (the `i` node under by() / sort(), dtb_slice_groups;
    expr/fexpr_literal_sliceint.cc:82-170).  Returns (positions into the RowIndex of group(), offsets of the
    groups that remain); in HBM when `offsets` is."""
    f = Col(offsets)
    ng = f.nrows - 1
    st, sp, se = [SLICE_NA if x is None else int(x) for x in (start, stop, step)]
    if ng > 0:
        last = offsets[-1]
        nrows = int(last.item() if is_tensor(last) else last)
    else:
        nrows = 0
    cap = nrows if se != 0 else ng * (sp if sp != SLICE_NA and sp > 0 else 0)
    rows, rptr = _alloc(cap, INT32, f.on_device)
    offs, optr = _alloc(ng + 1, INT32, f.on_device)
    ngo, nro = ctypes.c_int64(0), ctypes.c_int64(0)
    check(lib.dtb_slice_groups(ctypes.c_void_p(f.ptr), ng, st, sp, se, _stream(), ctypes.c_void_p(rptr), cap,
                               ctypes.c_void_p(optr), ctypes.byref(ngo), ctypes.byref(nro)))
    if ng == 0:
        offs[:1] = 0
    return rows[:nro.value], offs[:ngo.value + 1]


def join_index(xcols, jcols):
    """natural_join (frame/join.cc:392-470): for every X row the row of J (sorted by its key columns) with
    equal key, or the NA index; int32, in HBM when every column is."""
    xs, js = [Col(c) for c in xcols], [Col(c) for c in jcols]
    if len(xs) != len(js) or not xs:
        raise _lib.DtbValueError("join needs the same number (>= 1) of key columns on both sides")
    nx, nj = xs[0].nrows, js[0].nrows
    device = all(c.on_device for c in xs + js)
    out, optr = _alloc(nx, INT32, device)
    nk = len(xs)
    cx = (dtb_col * nk)(*[c.c() for c in xs])
    cj = (dtb_col * nk)(*[c.c() for c in js])
    check(lib.dtb_join(cx, cj, nk, nx, nj, _stream(), ctypes.c_void_p(optr)))
    return out


def set_option(name, value):
    check(lib.dtb_set_option(name.encode(), int(value)))


def get_option(name):
    v = ctypes.c_int64(0)
    check(lib.dtb_get_option(name.encode(), ctypes.byref(v)))
    return v.value
