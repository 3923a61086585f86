"""
Host-side mirror of the reference's Python surface for the DT[i, j, by(), sort()] path:
Frame, f, by(), sort(), sum/mean/min/max/count.  Only what the hot path needs -- no fread,
no general expression engine (SURVEY.md 8: out of scope).

    reference                                   here
    ---------                                   ----
    dt.Frame                 src/datatable/frame.py:23 / src/core/frame/      Frame
    f.A, f["A"], -f.A        src/datatable/expr/                               f / ColRef
    by(...), sort(...)       src/core/expr/py_by.cc, py_sort.cc:40-110         by / sort
    dt.sum/mean/min/max/count  src/datatable/expr/reduce.py:49-153             sum_/mean/min_/max_/count
    dt.cumsum/.../shift/fillna  src/core/expr/fexpr_cumsumprod.cc, ...        cumsum .. fillna (Window)
    DT[i, j, by, sort]       src/core/frame/__getitem__.cc:47-194,
                             src/core/expr/eval_context.cc:144-288, 473-520    Frame.__getitem__

Evaluation follows EvalContext: group() on the by/sort columns -> (RowIndex, Groupby);
reducers are evaluated over (value column, RowIndex, Groupby); plain columns are gathered
through the RowIndex; group keys are the first row of every group
(eval_context.cc:473-485).  All of it runs in libdtb200.so on the GPU.
"""
import numpy as np

from . import _lib, engine
from ._lib import (BOOL, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64, DATE32, TIME64, FLAG_DESCENDING,
                   FLAG_SORT_ONLY, NA_FIRST, NA_LAST, NA_REMOVE)

try:
    import torch
except Exception:  # pragma: no cover
    torch = None

_NA_POS = {"first": NA_FIRST, "last": NA_LAST, "remove": NA_REMOVE}
_NA_VALUE = {INT8: -2**7, INT16: -2**15, INT32: -2**31, INT64: -2**63, BOOL: -128, DATE32: -2**31, TIME64: -2**63}


# ---------------------------------------------------------------------------
# f-expressions (only column references, their negation, and reducers)
# ---------------------------------------------------------------------------
class ColRef:
    def __init__(self, name, negated=False):
        self.name = name
        self.negated = negated

    def __neg__(self):            # sort(-f.A) / by(-f.A): DESCENDING flag, not arithmetic (fexpr_list.cc:346-358)
        return ColRef(self.name, not self.negated)

    def __repr__(self):
        return f"{'-' if self.negated else ''}f.{self.name}"


class _FNamespace:
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return ColRef(name)

    def __getitem__(self, name):
        return ColRef(name)


f = _FNamespace()


class Reducer:
    def __init__(self, op, name, arg):
        self.op, self.opname, self.arg = op, name, arg


def sum(x): return Reducer(_lib.OP_SUM, "sum", x)          # noqa: A001  (mirrors dt.sum)
def mean(x): return Reducer(_lib.OP_MEAN, "mean", x)
def min(x): return Reducer(_lib.OP_MIN, "min", x)          # noqa: A001
def max(x): return Reducer(_lib.OP_MAX, "max", x)          # noqa: A001
def countna(x): return Reducer(_lib.OP_COUNTNA, "countna", x)
# within-group ordered reducers (src/core/expr/head_reduce_unary.cc:544-558; SURVEY.md 8f)
def first(x): return Reducer(_lib.OP_FIRST, "first", x)
def last(x): return Reducer(_lib.OP_LAST, "last", x)
def sd(x): return Reducer(_lib.OP_SD, "sd", x)
def median(x): return Reducer(_lib.OP_MEDIAN, "median", x)
def nunique(x): return Reducer(_lib.OP_NUNIQUE, "nunique", x) if isinstance(x, (ColRef, str)) else _frame_nunique(x)


def count(x=None):
    return Reducer(_lib.OP_NROWS if x is None else _lib.OP_COUNT, "count", x)


class Window:
    """A grouped cumulative / window function: one value per row of its group (the reference's GtoALL columns)."""

    def __init__(self, op, name, arg, param=0):
        self.op, self.opname, self.arg, self.param = op, name, arg, param

    def __repr__(self):
        if self.op == _lib.WIN_SHIFT:
            return f"shift({self.arg!r}, n={self.param})"
        arg = "" if self.arg is None else f"{self.arg!r}, "
        return f"{self.opname}({arg}reverse={bool(self.param)})"


def _window(op, name, x, param):
    if isinstance(x, (list, tuple)):                 # cumsum([f.a, f.b]): one column per argument
        return [Window(op, name, _as_ref(a), param) for a in _flatten(x)]
    return Window(op, name, _as_ref(x), param)


# grouped cumulative functions (column/cumsumprod.h, cumminmax.h, cumcountngroup.h) and shift / fillna
# (expr/head_func_shift.cc, fexpr_fillna.cc); under by() they restart in every group
def cumsum(x, reverse=False): return _window(_lib.WIN_CUMSUM, "cumsum", x, int(bool(reverse)))
def cumprod(x, reverse=False): return _window(_lib.WIN_CUMPROD, "cumprod", x, int(bool(reverse)))
def cummin(x, reverse=False): return _window(_lib.WIN_CUMMIN, "cummin", x, int(bool(reverse)))
def cummax(x, reverse=False): return _window(_lib.WIN_CUMMAX, "cummax", x, int(bool(reverse)))
def cumcount(reverse=False): return Window(_lib.WIN_CUMCOUNT, "cumcount", None, int(bool(reverse)))
def ngroup(reverse=False): return Window(_lib.WIN_NGROUP, "ngroup", None, int(bool(reverse)))


def shift(x, n=1):
    """Value n rows earlier in the group (n < 0: later), NA where that row is outside the group."""
    if not isinstance(n, int) or isinstance(n, bool):
        raise TypeError(f"Argument n in shift() should be an integer, instead got {type(n)}")
    if not -2**31 <= n < 2**31:
        raise ValueError(f"Value is too large to fit in an int32: {n}")
    return Window(_lib.WIN_SHIFT, "shift", _as_ref(x), n)


def fillna(x, value=None, reverse=False):
    """Forward fill inside the group (backward with reverse=True).  Filling with a value is elementwise and not on
    the GPU path."""
    if value is not None:
        raise NotImplementedError("fillna(value=...) is an elementwise expression, outside the GPU hot path")
    return _window(_lib.WIN_FILLNA, "fillna", x, int(bool(reverse)))


class by:
    def __init__(self, *cols):
        self.cols = [_as_ref(c) for c in _flatten(cols)]


class join:
    """join(J): natural join with the keyed frame J (src/core/expr/py_join.cc; frame/join.cc:392-470)."""

    def __init__(self, frame):
        if not isinstance(frame, Frame):
            raise TypeError("The argument to join() must be a Frame")
        if not frame.key:
            raise ValueError("The join frame is not keyed")
        self.frame = frame


class sort:
    """sort(*cols, reverse=False, na_position="first") -- py_sort.cc:40-110."""

    def __init__(self, *cols, reverse=False, na_position="first"):
        self.cols = [_as_ref(c) for c in _flatten(cols)]
        n = len(self.cols)
        if isinstance(reverse, (list, tuple)):
            if len(reverse) != n:
                raise ValueError(f"number of elements (nflags={len(reverse)}) in the reverse flag list "
                                 f"does not match the number of sort columns ({n})")
            self.reverse = [bool(r) for r in reverse]
        elif isinstance(reverse, bool):
            self.reverse = [reverse] * n
        else:
            raise TypeError("reverse should be a boolean or a list of booleans")
        if na_position not in _NA_POS:
            raise ValueError(f"na position value `{na_position}` is not supported")
        self.na_position = na_position


def _flatten(cols):
    out = []
    for c in cols:
        if isinstance(c, (list, tuple)):
            out.extend(_flatten(c))
        else:
            out.append(c)
    return out


def _as_ref(c):
    if isinstance(c, ColRef):
        return c
    if isinstance(c, str):
        return ColRef(c)
    raise TypeError(f"Unsupported key expression {c!r}: only column references are on the GPU path")


# ---------------------------------------------------------------------------
# Frame
# ---------------------------------------------------------------------------
class Frame:
    """Column store: every column is a numpy array (host) or a torch CUDA tensor (HBM) plus an stype.
    Bool columns with NAs are int8 with -128 (the reference's bool8 layout)."""

    def __init__(self, data=None, stypes=None, **kwargs):
        self._cols = {}
        self._stypes = {}
        self._key = ()
        if data is None:
            data = kwargs
        if isinstance(data, Frame):
            self._cols, self._stypes = dict(data._cols), dict(data._stypes)
            return
        if not isinstance(data, dict):
            data = {"C0": data}
        n = None
        for name, col in data.items():
            st = None if stypes is None else stypes.get(name)
            if isinstance(col, (list, tuple)):
                col, st2 = _from_list(col)
                st = st or st2
            c = engine.Col(col, st)
            if n is None:
                n = c.nrows
            elif c.nrows != n:
                raise ValueError("columns have different numbers of rows")
            self._cols[name] = c.data
            self._stypes[name] = c.stype
        self._nrows = n or 0

    # -- metadata ---------------------------------------------------------------
    @property
    def names(self): return tuple(self._cols.keys())
    @property
    def nrows(self): return self._nrows
    @property
    def ncols(self): return len(self._cols)
    @property
    def shape(self): return (self.nrows, self.ncols)
    @property
    def stypes(self): return tuple(self._stypes[n] for n in self._cols)

    def _col(self, name):
        if name not in self._cols:
            raise KeyError(f"Column `{name}` does not exist in the Frame")
        return engine.Col(self._cols[name], self._stypes[name])

    def column(self, name):
        """Raw storage of a column (numpy array or CUDA tensor)."""
        return self._cols[name]

    def to_numpy(self, name=None):
        if name is None:
            return {n: self.to_numpy(n) for n in self._cols}
        c = self._cols[name]
        return c.cpu().numpy() if engine.is_tensor(c) else c

    def to_list(self):
        out = []
        for n in self._cols:
            a = self.to_numpy(n)
            st = self._stypes[n]
            if st in (FLOAT32, FLOAT64):
                out.append([None if np.isnan(x) else float(x) for x in a.tolist()])
            elif st == BOOL:
                out.append([None if x == -128 else bool(x) for x in a.tolist()])
            else:
                na = _NA_VALUE[st]
                out.append([None if x == na else int(x) for x in a.tolist()])
        return out

    def to_dict(self):
        return dict(zip(self.names, self.to_list()))

    # -- Arrow ingest / export (the reference reads Arrow through Frame(pa.Table), frame/__init__.cc; here the
    #    fixed-width columns become the NA-sentinel buffers the engine consumes, SURVEY.md 8f rank 4) -----------
    @classmethod
    def from_arrow(cls, table):
        """pyarrow.Table / RecordBatch -> Frame: bool/int8-64/float32-64 columns, nulls -> the reference's NA
        sentinels (bool8 = int8 with -128).  Zero-copy for null-free numeric columns."""
        import pyarrow as pa
        cols, sts = {}, {}
        for name, col in zip(table.column_names, table.columns):
            arr = col.combine_chunks() if isinstance(col, pa.ChunkedArray) else col
            t = arr.type
            if pa.types.is_boolean(t):
                a = np.asarray(arr.cast(pa.int8()).fill_null(-128).to_numpy(zero_copy_only=False), dtype=np.int8)
                st = BOOL
            elif pa.types.is_integer(t) and t.bit_width <= 64 and pa.types.is_signed_integer(t):
                st = {8: INT8, 16: INT16, 32: INT32, 64: INT64}[t.bit_width]
                a = arr.fill_null(_NA_VALUE[st]).to_numpy(zero_copy_only=False) if arr.null_count else arr.to_numpy()
            elif pa.types.is_floating(t) and t.bit_width in (32, 64):
                st = FLOAT32 if t.bit_width == 32 else FLOAT64
                a = arr.to_numpy(zero_copy_only=False)          # nulls become NaN == NA
            else:
                raise _lib.DtbNotImplError(f"Arrow column `{name}` of type {t} is outside the GPU hot path")
            cols[name], sts[name] = np.ascontiguousarray(a), st
        return cls(cols, stypes=sts)

    def to_jay(self, path):
        """Frame -> Jay file the reference opens with dt.fread (src/core/jay/save_jay.cc); see datatable_b200/jay.py."""
        from .jay import save_jay
        save_jay(self, path)

    def to_arrow(self):
        """Frame -> pyarrow.Table with NA sentinels turned back into nulls."""
        import pyarrow as pa
        out = {}
        for n in self._cols:
            a, st = self.to_numpy(n), self._stypes[n]
            if st in (FLOAT32, FLOAT64):
                out[n] = pa.array(a, mask=np.isnan(a))
            elif st == BOOL:
                out[n] = pa.array(a.astype(np.bool_), mask=(a == -128))
            else:
                out[n] = pa.array(a, mask=(a == _NA_VALUE[st]))
        return pa.table(out)

    def to_device(self):
        """Copy every column into HBM (the analogue of a device-backed Buffer, SURVEY.md 8f rank 4)."""
        fr = Frame()
        for n, c in self._cols.items():
            fr._cols[n] = c if engine.is_tensor(c) else torch.from_numpy(np.ascontiguousarray(c)).cuda()
            fr._stypes[n] = self._stypes[n]
        fr._nrows = self._nrows
        return fr

    # -- DT.key (frame/key.cc:118-180): sort by the key columns, require unique rows, key columns first
    @property
    def key(self):
        return tuple(self._key)

    @key.setter
    def key(self, val):
        names = [val] if isinstance(val, str) else list(val or [])
        if not names:
            self._key = ()
            return
        for nm in names:
            if not isinstance(nm, str):
                raise TypeError("Key should be a list/tuple of column names")
            if nm not in self._cols:
                raise KeyError(f"Column `{nm}` does not exist in the Frame")
        if len(set(names)) != len(names):
            raise ValueError("A column is specified multiple times within the key")
        if self._nrows:
            order, offsets, ng = engine.group([self._col(nm) for nm in names], [0] * len(names), NA_FIRST)
            if ng < self._nrows:
                raise ValueError("Cannot set a key: the values are not unique")
        rest = [nm for nm in self._cols if nm not in names]
        cols, sts = {}, {}
        for nm in names + rest:
            c = self._col(nm)
            if self._nrows:
                o = order if (engine.is_tensor(c.data) and c.data.is_cuda) == engine.is_tensor(order) else (
                    order.cpu().numpy() if engine.is_tensor(order) else torch.from_numpy(order).cuda())
                cols[nm] = engine.gather(c, o)
            else:
                cols[nm] = c.data
            sts[nm] = c.stype
        self._cols, self._stypes = cols, sts
        self._key = tuple(names)

    # -- column statistics that go through group() (stats.cc:955-1003) ---------------------------
    def nunique(self):
        return _frame_nunique(self)

    def mode(self):
        return _frame_mode(self)[0]

    def nmodal(self):
        return _frame_mode(self)[1]

    # -- DT.sort(cols) (sort.cc:1544-1574) ------------------------------------------
    def sort(self, *cols):
        return self[:, :, sort(*cols)]

    # -- DT[i, j, by, sort] -------------------------------------------------------------
    def __getitem__(self, item):
        if not isinstance(item, tuple):
            item = (slice(None), item)
        if len(item) < 2:
            raise ValueError("Frame[...] needs at least i and j")
        i, j = item[0], item[1]
        by_, sort_, join_ = None, None, None
        for m in item[2:]:
            if isinstance(m, by):
                by_ = m
            elif isinstance(m, sort):
                sort_ = m
            elif isinstance(m, join):
                join_ = m
            else:
                raise TypeError(f"Unsupported modifier {m!r}")
        isel = None
        if i is None:                                    # FExpr_Literal_None: every row (fexpr_literal_none.cc:88-96)
            i = slice(None)
        if not (isinstance(i, slice) and i == slice(None)):
            ok = (isinstance(i, int) and not isinstance(i, bool)) or (
                isinstance(i, slice) and all(x is None or (isinstance(x, int) and not isinstance(x, bool)) for x in (i.start, i.stop, i.step)))
            if not ok:
                raise NotImplementedError("row filters other than an integer or an integer slice are outside the GPU hot path")
            isel = i
        if join_ is not None:
            if by_ is not None or sort_ is not None or isel is not None:
                raise NotImplementedError("join() together with i / by() / sort() is outside the GPU hot path")
            return _evaluate_join(self, j, join_.frame)
        return _evaluate(self, j, by_, sort_, isel)


def _from_list(lst):
    """Python list -> (array, stype) with None as NA (bool8 / int32 / int64 / float64 like the reference)."""
    vals = [x for x in lst if x is not None]
    if vals and all(isinstance(x, bool) for x in vals):
        return np.array([-128 if x is None else int(x) for x in lst], dtype=np.int8), BOOL
    if all(isinstance(x, int) for x in vals):
        big = any(abs(x) > 2**31 - 1 for x in vals)
        dt_, na = (np.int64, -2**63) if big else (np.int32, -2**31)
        return np.array([na if x is None else x for x in lst], dtype=dt_), (INT64 if big else INT32)
    return np.array([np.nan if x is None else float(x) for x in lst], dtype=np.float64), FLOAT64


_COPY_STREAMS = {}


def _copy_stream():
    """One upload stream per device for the life of the process.  torch's caching allocator keeps freed blocks per
    stream: a fresh stream per query (the first version) could never reuse the previous query's staging buffers and
    cudaMalloc'ed every uploaded column again (12 GB per C2 query until the device was full)."""
    dev = torch.cuda.current_device()
    if dev not in _COPY_STREAMS:
        _COPY_STREAMS[dev] = torch.cuda.Stream()
    return _COPY_STREAMS[dev]


_PIECE_BYTES = 1 << 30        # host value columns of >= 2 GB are uploaded (and reduced) in 1 GB pieces


def _evaluate(DT, j, by_, sort_, isel=None):
    """EvalContext::evaluate (eval_context.cc:144-172) for the hot-path shapes.
    isel: an integer or integer slice for `i` -- applied inside every group under by() / sort()
    (iexpr_->evaluate_iby, eval_context.cc:154-158), to the rows otherwise (evaluate_i, :159-163)."""
    # Host columns are uploaded once (pinned memory -> DMA), the whole query then runs on
    # HBM-resident buffers, and only the result frame travels back.
    if torch is None or not torch.cuda.is_available():
        raise _lib.DtbCudaError("no usable CUDA device: datatable_b200 has no CPU fallback")
    host_frame = not any(engine.is_tensor(c) and c.is_cuda for c in DT._cols.values())
    cache = {}
    names, exprs = _resolve_j(DT, j)

    # Host columns: start every upload the query needs on a copy stream, key columns first, so
    # that the PCIe transfer of the value columns overlaps the sort of the keys; each column is
    # awaited (stream event) only where it is first used.
    needed = []
    for m in (by_, sort_):
        if m is not None:
            needed += [r.name for r in m.cols]
    for e in exprs:
        if isinstance(e, (Reducer, Window)):
            nm = None if e.arg is None else e.arg.name
        else:
            nm = e.name
        if nm is not None:
            needed.append(nm)
    copy_stream = None
    pending = {}
    pieces = {}               # large value columns travel in pieces, each with its own event (see the late path)
    keynames = set()
    for m in (by_, sort_):
        if m is not None:
            keynames.update(r.name for r in m.cols)
    for nm in dict.fromkeys(needed):
        c = DT._col(nm)
        t = c.data if engine.is_tensor(c.data) else torch.from_numpy(c.data)
        if t.is_cuda:
            continue
        if copy_stream is None:
            copy_stream = _copy_stream()
            copy_stream.wait_stream(torch.cuda.current_stream())    # buffers freed by earlier queries are reused in order
        with torch.cuda.stream(copy_stream):
            if nm not in keynames and t.dim() == 1 and t.numel() * t.element_size() >= _PIECE_BYTES * 2:
                d = torch.empty_like(t, device="cuda")
                step = _builtins.max(1, _PIECE_BYTES // t.element_size())
                pcs = []
                for a in range(0, t.numel(), step):
                    b = _builtins.min(a + step, t.numel())
                    d[a:b].copy_(t[a:b], non_blocking=True)
                    pev = torch.cuda.Event(); pev.record(copy_stream)
                    pcs.append((a, b, pev))
                pieces[nm] = pcs
                ev = pcs[-1][2]
            else:
                d = t.cuda(non_blocking=True)                       # pinned host memory -> async DMA
                ev = torch.cuda.Event(); ev.record(copy_stream)
        pending[nm] = (engine.Col(d, c.stype), ev)

    def dcol(name):
        if name not in cache:
            if name in pending:
                c, ev = pending[name]
                torch.cuda.current_stream().wait_event(ev)
                c.data.record_stream(torch.cuda.current_stream())
            else:
                c = DT._col(name)
                t = c.data if engine.is_tensor(c.data) else torch.from_numpy(c.data)
                if not t.is_cuda:
                    c = engine.Col(t.cuda(non_blocking=True), c.stype)
            cache[name] = c
        return cache[name]

    # ---- compute_groupby_and_sort (eval_context.cc:249-288) ----
    keycols, flags = [], []
    na_pos = NA_FIRST
    if by_ is not None:
        for ref in by_.cols:
            keycols.append(dcol(ref.name))
            flags.append(FLAG_DESCENDING if ref.negated else 0)
    if sort_ is not None:
        na_pos = _NA_POS[sort_.na_position]
        for ref, rev in zip(sort_.cols, sort_.reverse):
            keycols.append(dcol(ref.name))
            desc = (not rev) if ref.negated else rev                 # fexpr_list.cc:346-358
            flags.append((FLAG_DESCENDING if desc else 0) | FLAG_SORT_ONLY)
    order = offsets = None
    ngroups = None
    gb = None
    has_reducer = any(isinstance(e, Reducer) for e in exprs)
    # GtoALL (eval_context.cc:144-172): one output row per row of the grouped frame -- j holds a window function, or a
    # plain column next to a reducer under by(); reducers are then repeated on every row of their group
    gtoall = any(isinstance(e, Window) for e in exprs) or (
        by_ is not None and has_reducer and any(isinstance(e, ColRef) for e in exprs))
    for e in exprs:
        if isinstance(e, Window) and e.arg is not None:
            st_ = DT._col(e.arg.name).stype
            if not engine.window_out_stype(e.op, st_):
                raise TypeError(f"Invalid column of type {_STYPE_NAME.get(st_, st_)} in {e!r}")
    sliced = False
    if keycols and isel is not None:
        # i under by() / sort(): group() first, then the slice inside every group; its positions are composed with
        # the RowIndex (apply_rowindex) and the Groupby is replaced (replace_groupby)
        order, offsets, ngroups = engine.group(keycols, flags, na_pos)
        if offsets is None:                                            # sort() alone: Groupby::single_group
            offsets = torch.tensor([0, len(order)], dtype=torch.int32, device="cuda")
        if isinstance(isel, int):
            st_, sp_, se_ = isel, (isel + 1 if isel != -1 else None), 1     # fexpr_literal_int.cc:146-192 == the slice [i, i+1)
            if not -2**31 <= isel < 2**31:
                st_, sp_, se_ = 0, 0, 1
        else:
            st_, sp_, se_ = isel.start, isel.stop, isel.step
        sel, offsets = engine.slice_groups(offsets, st_, sp_, se_)
        order = engine.gather(order, sel)
        ngroups = len(offsets) - 1
        sliced = True
    elif isel is not None:
        # no by() / sort(): evaluate_i -- a plain row slice (python slice semantics; step 0 = repeat is not taken here)
        n_ = DT.nrows
        if isinstance(isel, int):
            if not -n_ <= isel < n_:
                raise ValueError(f"Row `{isel}` is invalid for a frame with {n_} row{'s' if n_ != 1 else ''}")
            rng_ = range(isel % n_, isel % n_ + 1)
        else:
            if isel.step == 0:
                raise NotImplementedError("repeat slices (step 0) without by() are outside the GPU hot path")
            rng_ = range(*isel.indices(n_))
        order = torch.arange(rng_.start, rng_.stop, rng_.step, dtype=torch.int32, device="cuda")
    elif keycols:
        if by_ is not None and has_reducer and not gtoall:
            # RowIndex + Groupby stay in HBM behind a handle; reducers go through it
            # the reducers of j are known before group() runs: hand them over so that the engine can
            # overlap them with the sort (dtb_groupby_create_reduce)
            # (median / nunique read the rows sorted inside their group: evaluated after group(), below)
            fused = [e for e in exprs if isinstance(e, Reducer) and e.op not in _SORTED_OPS]
            # Host frame whose value columns are still on their way over PCIe: group() first (the sort runs
            # under the upload), the reducers afterwards through the handle, each waiting only for its own
            # column.  Handing the reducers to group() would make the stream wait for every value column
            # before the sort starts.  Columns with several reducers keep the fused call (bucketed multi-reducer).
            args_pending = [e.arg.name for e in fused if e.arg is not None and e.arg.name in pending and e.arg.name not in cache]
            per_col = {nm: _builtins.sum(2 if e.op == _lib.OP_MEAN else 1 for e in fused if e.arg is not None and e.arg.name == nm)
                       for nm in args_pending}
            late = bool(args_pending) and all(c < 2 for c in per_col.values())
            late_results = {}
            early_keys = None
            if late:
                gb = engine.Groupby(keycols, flags, na_pos)
                # the group-key columns of the result (first row of every group, gathered, brought to the host)
                # depend on group() alone: done now, under the upload of the value columns
                first = gb.first_rows()
                early_keys = []
                for ref in by_.cols:
                    c = dcol(ref.name)
                    g_ = engine.gather(c, first)
                    early_keys.append((ref.name, g_.cpu().numpy() if host_frame and engine.is_tensor(g_) else g_, c.stype))
                for e in fused:
                    nm_ = None if e.arg is None else e.arg.name
                    res_ = None
                    if nm_ in pieces and nm_ not in cache:
                        # fold every piece of the column as soon as it has arrived (dtb_groupby_reduce_add): after
                        # the last byte only the last piece's share of the reducer is left
                        col_ = pending[nm_][0]
                        col_.data.record_stream(torch.cuda.current_stream())
                        res_ = gb.reduce_pieces(e.op, col_.stype, [(col_.data[a:b], a, pev) for a, b, pev in pieces[nm_]])
                    late_results[id(e)] = res_ if res_ is not None else gb.reduce(e.op, None if nm_ is None else dcol(nm_))
            else:
                reds = [(e.op, None if e.arg is None else dcol(e.arg.name)) for e in fused]
                gb = engine.Groupby(keycols, flags, na_pos, reducers=reds)
            ngroups = gb.ngroups
        else:
            order, offsets, ngroups = engine.group(keycols, flags, na_pos)

    # ---- j ----
    out = Frame()

    def add(name, data, st):
        base, k = name, 0
        while name in out._cols:
            k += 1
            name = f"{base}.{k - 1}"
        if host_frame and engine.is_tensor(data):
            data = data.cpu().numpy()
        out._cols[name] = data
        out._stypes[name] = st

    if gtoall:
        if offsets is None:                     # no by(): one group over the rows kept (Groupby::single_group)
            n_ = DT.nrows if order is None else len(order)
            offsets = torch.tensor([0, n_] if n_ else [0], dtype=torch.int32, device="cuda")
        _evaluate_gtoall(by_, names, exprs, dcol, add, order, offsets)
        out._nrows = DT.nrows if order is None else len(order)
        return out

    if by_ is not None:
        if has_reducer and sliced:
            first = engine.gather(order, offsets[:-1])
            for ref in by_.cols:
                c = dcol(ref.name)
                add(ref.name, engine.gather(c, first), c.stype)
            for name, e in zip(names, exprs):
                if not isinstance(e, Reducer):
                    raise NotImplementedError("mixing reducers and plain columns under by() is outside the hot path")
                add(name, _reduce(dcol, e, order, offsets), _red_stype(dcol, e))
            for n_ in out._cols:
                if out._stypes[n_] is None:
                    out._stypes[n_] = engine.Col(out._cols[n_]).stype
            out._nrows = ngroups
            return out
        if has_reducer:
            # group keys = first row of every group (get_group_rowindex, eval_context.cc:124-135)
            if early_keys is not None:
                for nm_, data_, st_ in early_keys:
                    add(nm_, data_, st_)
            else:
                first = gb.first_rows()
                for ref in by_.cols:
                    c = dcol(ref.name)
                    add(ref.name, engine.gather(c, first), c.stype)
            ired = 0
            for name, e in zip(names, exprs):
                if isinstance(e, Reducer) and e.op in _SORTED_OPS:
                    c = dcol(e.arg.name)                      # Median_ColumnImpl::pre_materialize_hook: sort_grouped first
                    add(name, gb.reduce_ordered(e.op, c, gb.sort_grouped(c)), _red_stype(dcol, e))
                elif isinstance(e, Reducer):
                    add(name, late_results[id(e)] if late else gb.reduced(ired), _red_stype(dcol, e))
                    ired += 1
                else:
                    raise NotImplementedError("mixing reducers and plain columns under by() is outside the hot path")
            for n_ in out._cols:
                if out._stypes[n_] is None:
                    out._stypes[n_] = engine.Col(out._cols[n_]).stype
            out._nrows = ngroups
            gb.close()
            return out
        # by() without reducers: every row, grouped order, key columns first
        bynames = [r.name for r in by_.cols]
        for ref in by_.cols:
            c = dcol(ref.name)
            add(ref.name, engine.gather(c, order), c.stype)
        for name, e in zip(names, exprs):
            if e.name in bynames and j_is_all(j):
                continue
            c = dcol(e.name)
            add(name, engine.gather(c, order), c.stype)
        out._nrows = len(order)
        return out

    if has_reducer:
        # reducers without by(): one group over all rows (Groupby::single_group, groupby.cc:60-68)
        nrows = DT.nrows if order is None else len(order)
        offs = torch.tensor([0, nrows], dtype=torch.int32, device="cuda")
        for name, e in zip(names, exprs):
            if not isinstance(e, Reducer):
                raise NotImplementedError("mixing reducers and plain columns is outside the hot path")
            add(name, _reduce(dcol, e, order, offs), _red_stype(dcol, e))
        out._nrows = 1
        return out

    for name, e in zip(names, exprs):
        if order is None:
            c = DT._col(e.name)
            out._cols[name] = c.data; out._stypes[name] = c.stype
        else:
            c = dcol(e.name)
            add(name, engine.gather(c, order), c.stype)
    out._nrows = DT.nrows if order is None else len(order)
    return out


def _evaluate_gtoall(by_, names, exprs, dcol, add, order, offsets):
    """j evaluated per row of the grouped frame (RowIndex `order`, None = identity; Groupby `offsets`): by-columns
    and plain columns gathered through the RowIndex, window functions from dtb_window, reducers computed per group
    and repeated on every row of the group (gathered through the group id of every row)."""
    def rows(c):
        return c.data if order is None else engine.gather(c, order)
    bynames = [] if by_ is None else [ref.name for ref in by_.cols]
    final = _unique_names(bynames + list(names))
    for ref, name in zip(by_.cols if by_ is not None else [], final):
        c = dcol(ref.name)
        add(name, rows(c), c.stype)
    gid = None
    for name, e in zip(final[len(bynames):], exprs):
        if isinstance(e, Window):
            c = None if e.arg is None else dcol(e.arg.name)
            st = engine.window_out_stype(e.op, INT8 if c is None else c.stype)
            add(name, engine.window(e.op, c, order, offsets, e.param), st)
        elif isinstance(e, Reducer):
            if gid is None:
                gid = engine.window(_lib.WIN_NGROUP, None, None, offsets)
            st = _red_stype(dcol, e)
            add(name, engine.gather(engine.Col(_reduce(dcol, e, order, offsets), st), gid), st)
        else:
            c = dcol(e.name)
            add(name, rows(c), c.stype)


def _unique_names(names):
    """Duplicate column names made unique the way the reference's Frame does it: a name that ends in digits counts
    on from them ("x9" -> "x10"), any other name gets ".0", ".1", ... ("v" -> "v.0")."""
    out, seen = [], set()
    for name in names:
        if name in seen:
            stem = name.rstrip("0123456789")
            if stem != name:
                k = int(name[len(stem):]) + 1
            else:
                stem, k = (stem if stem.endswith(".") else stem + "."), 0
            while f"{stem}{k}" in seen:
                k += 1
            name = f"{stem}{k}"
        seen.add(name)
        out.append(name)
    return out


def j_is_all(j):
    return isinstance(j, slice) and j == slice(None)


def _resolve_j(DT, j):
    if j_is_all(j):
        return list(DT.names), [ColRef(n) for n in DT.names]
    if isinstance(j, dict):
        return list(j.keys()), [_as_expr(v) for v in j.values()]
    if isinstance(j, (list, tuple)):
        es = [_as_expr(v) for v in _flatten(j)]
    else:
        es = [_as_expr(j)]
    names = []
    unnamed = 0
    for e in es:
        if isinstance(e, Reducer):
            names.append("count" if e.arg is None else e.arg.name)     # reducers keep the column's name
        elif isinstance(e, Window):
            if e.arg is None:                                           # cumcount / ngroup: C0, C1, ...
                names.append(f"C{unnamed}")
                unnamed += 1
            else:
                names.append(e.arg.name)
        else:
            names.append(e.name)
    return names, es


def _as_expr(v):
    if isinstance(v, (Reducer, ColRef, Window)):
        return v
    if isinstance(v, str):
        return ColRef(v)
    raise TypeError(f"Unsupported j expression {v!r}")


def _index_through(order, pos):
    """order[pos] -- composition of RowIndexes (rowindex.cc:246-250) done as a gather."""
    return engine.gather(engine.Col(order, INT32), pos)


def _red_stype(dcol, e):
    """Output stype of a reducer column (bool8 min/max stay bool8, fexpr_minmax.cc:50-72)."""
    if e.op == _lib.OP_NROWS or e.arg is None:
        return INT64
    return engine.reduce_out_stype(e.op, dcol(e.arg.name).stype)


_SORTED_OPS = (_lib.OP_MEDIAN, _lib.OP_NUNIQUE)
_STYPE_NAME = {BOOL: "bool8", INT8: "int8", INT16: "int16", INT32: "int32", INT64: "int64", FLOAT32: "float32",
               FLOAT64: "float64", DATE32: "date32", TIME64: "time64"}


def _reduce(dcol, e, order, offsets):
    if e.op == _lib.OP_NROWS:
        return engine.reduce(e.op, None, order, offsets)
    c = dcol(e.arg.name)
    if e.op in _SORTED_OPS:
        order = engine.sort_grouped(c, order, offsets)
    return engine.reduce(e.op, c, order, offsets)


# ---------------------------------------------------------------------------
# Callers of group() beyond DT[i, j, by, sort] (SURVEY.md 8f): set operations, column statistics, join
# ---------------------------------------------------------------------------
_INT_ORDER = [BOOL, INT8, INT16, INT32, INT64]
_TORCH_OF = {BOOL: "int8", INT8: "int8", INT16: "int16", INT32: "int32", INT64: "int64", FLOAT32: "float32", FLOAT64: "float64"}


def _dev(c):
    t = c.data if engine.is_tensor(c.data) else torch.from_numpy(np.ascontiguousarray(c.data))
    return t if t.is_cuda else t.cuda()


def _promote(cols):
    """Common stype of rbind-ed columns (the reference upcasts to the widest input type) with NA mapped."""
    sts = {c.stype for c in cols}
    if len(sts) == 1:
        return [_dev(c) for c in cols], cols[0].stype
    isf = any(st in (FLOAT32, FLOAT64) for st in sts)
    tgt = (FLOAT32 if sts <= {FLOAT32} else FLOAT64) if isf else builtins_max(sts, key=_INT_ORDER.index)
    out = []
    for c in cols:
        t = _dev(c)
        if c.stype != tgt:
            if c.stype in (FLOAT32, FLOAT64):
                t = t.to(getattr(torch, _TORCH_OF[tgt]))
            else:
                na = t == _NA_VALUE[c.stype]
                t = t.to(getattr(torch, _TORCH_OF[tgt]))
                t = torch.where(na, torch.full_like(t, float("nan") if isf else _NA_VALUE[tgt]), t)
        out.append(t)
    return out, tgt


import builtins as _builtins  # noqa: E402
builtins_max = _builtins.max


def _set_op(mode, frames):
    frames = [fr for fr in _flatten(frames)]
    for fr in frames:
        if not isinstance(fr, Frame):
            raise TypeError("set functions expect a list or sequence of Frames")
        if fr.ncols > 1:
            raise ValueError(f"Only single-column Frames are allowed, but received a Frame with {fr.ncols} columns")
    frames = [fr for fr in frames if fr.ncols == 1]
    if not frames:
        return Frame()
    name = frames[0].names[0]
    host = not any(engine.is_tensor(fr._cols[fr.names[0]]) and fr._cols[fr.names[0]].is_cuda for fr in frames)
    tens, st = _promote([fr._col(fr.names[0]) for fr in frames])
    if len(frames) <= 1:
        mode = _lib.SET_UNION                                  # set_funcs.cc:302-305, 356-359, 438-441
    cat = tens[0] if len(tens) == 1 else torch.cat(tens)
    cd = engine.Col(cat, st)
    out = Frame()
    if cat.numel() == 0:
        vals = cat
    else:
        order, offsets, ng = engine.group([cd], [0], NA_FIRST)
        rows = engine.set_select(mode, order, offsets, np.cumsum([t.numel() for t in tens]))
        vals = engine.gather(cd, rows)
    out._cols[name] = vals.cpu().numpy() if host else vals
    out._stypes[name] = st
    out._nrows = int(vals.shape[0])
    return out


def union(*frames): return _set_op(_lib.SET_UNION, frames)
def intersect(*frames): return _set_op(_lib.SET_INTERSECT, frames)
def setdiff(*frames): return _set_op(_lib.SET_SETDIFF, frames)
def symdiff(*frames): return _set_op(_lib.SET_SYMDIFF, frames)


def unique(frame):
    """dt.unique(frame): the sorted unique values (NA first) -- the union of the frame's columns
    (set_funcs.cc:203-216)."""
    cols = []
    for nm in frame.names:
        fr = Frame(); fr._cols[nm] = frame._cols[nm]; fr._stypes[nm] = frame._stypes[nm]; fr._nrows = frame.nrows
        cols.append(fr)
    return _set_op(_lib.SET_UNION, cols)


def _column_groups(frame, name):
    c = frame._col(name)
    cd = engine.Col(_dev(c), c.stype)
    if cd.nrows == 0:
        return cd, None, None, 0, False
    order, offsets, ng = engine.group([cd], [0], NA_FIRST)
    # the NA rows sort first: the column has NAs iff the first sorted row is NA (stats.cc:966-975)
    first = engine.gather(cd, order[:1]).cpu().numpy()
    has_na = bool(np.isnan(first[0])) if c.stype in (FLOAT32, FLOAT64) else bool(first[0] == _NA_VALUE[c.stype])
    return cd, order, offsets, ng, has_na


def _frame_nunique(frame):
    """Frame.nunique(): distinct non-NA values per column (stats.cc:955-979 via group())."""
    out = Frame()
    for name in frame.names:
        cd, order, offsets, ng, has_na = _column_groups(frame, name)
        out._cols[name] = np.array([ng - int(has_na)], dtype=np.int64)
        out._stypes[name] = INT64
    out._nrows = 1
    return out


def _frame_mode(frame):
    """(Frame.mode(), Frame.nmodal()): value and size of the first largest non-NA group (stats.cc:981-1003)."""
    mode, nmodal = Frame(), Frame()
    for name in frame.names:
        cd, order, offsets, ng, has_na = _column_groups(frame, name)
        idx, size = (-1, 0) if order is None else engine.largest_group(offsets, int(has_na))
        if size:
            val = engine.gather(cd, engine.gather(engine.Col(order, INT32), offsets[idx:idx + 1])).cpu().numpy()
        else:
            val = np.array([np.nan if cd.stype in (FLOAT32, FLOAT64) else _NA_VALUE[cd.stype]],
                           dtype=getattr(np, _TORCH_OF[cd.stype]))
        mode._cols[name] = val; mode._stypes[name] = cd.stype
        nmodal._cols[name] = np.array([size], dtype=np.int64); nmodal._stypes[name] = INT64
    mode._nrows = nmodal._nrows = 1
    return mode, nmodal


def _evaluate_join(X, j, J):
    """X[:, j, join(J)] (eval_context.cc add_join + natural_join, frame/join.cc:392-470): J's key columns are
    looked up by name in X; J's non-key columns are viewed through the resulting RowIndex."""
    keys = list(J.key)
    for nm in keys:
        if nm not in X._cols:
            raise ValueError(f"Key column `{nm}` does not exist in the left Frame")
    host = not any(engine.is_tensor(c) and c.is_cuda for c in X._cols.values())
    xk = [engine.Col(_dev(X._col(nm)), X._stypes[nm]) for nm in keys]
    jk = [engine.Col(_dev(J._col(nm)), J._stypes[nm]) for nm in keys]
    index = engine.join_index(xk, jk)
    out = Frame()
    wanted = None if j_is_all(j) else [e.name for e in _resolve_j_names(j)]
    for nm in X.names:
        if wanted is None or nm in wanted:
            out._cols[nm] = X._cols[nm]; out._stypes[nm] = X._stypes[nm]
    for nm in J.names:
        if nm in keys or (wanted is not None and nm not in wanted):
            continue
        c = J._col(nm)
        g = engine.gather(engine.Col(_dev(c), c.stype), index)
        name, k = nm, 0
        while name in out._cols:
            name = f"{nm}.{k}"; k += 1
        out._cols[name] = g.cpu().numpy() if host else g
        out._stypes[name] = c.stype
    out._nrows = X.nrows
    return out


def _resolve_j_names(j):
    es = j if isinstance(j, (list, tuple)) else [j]
    return [_as_ref(e) for e in es]
