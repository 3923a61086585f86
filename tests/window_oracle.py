"""
NumPy restatement of the reference's grouped cumulative and window functions: the serial per-group loops over a
value column viewed through the RowIndex.

    cumsum / cumprod     column/cumsumprod.h:48-95       NA counts as 0 / 1; integers in int64 (wrapping)
    cummin / cummax      column/cumminmax.h:48-110       NA skipped, a leading NA stays NA, ties -> current row
    cumcount / ngroup    column/cumcountngroup.h:52-70   row number inside the group / group number
    fillna               expr/fexpr_fillna.cc:86-118     last non-NA value so far
    shift                expr/head_func_shift.cc:41-62   value n rows earlier in the group (n < 0: later), else NA

`reverse` runs the loop from the end of every group.  Test infrastructure only: the tests and the golden generator
compare the engine against it.
"""
import numpy as np

CUMSUM, CUMPROD, CUMMIN, CUMMAX, CUMCOUNT, NGROUP, FILLNA, SHIFT = 1, 2, 3, 4, 5, 6, 7, 8
BOOL, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64, DATE32, TIME64 = 1, 2, 3, 4, 5, 6, 7, 17, 18
_NA = {BOOL: -128, INT8: -128, INT16: -2**15, INT32: -2**31, INT64: -2**63, DATE32: -2**31, TIME64: -2**63}


def na_mask(a, st):
    if st in (FLOAT32, FLOAT64):
        return np.isnan(a)
    return a == _NA[st]


def na_value(st):
    return np.nan if st in (FLOAT32, FLOAT64) else _NA[st]


def out_dtype(op, st, dtype):
    if op in (CUMCOUNT, NGROUP):
        return np.dtype(np.int64)
    if op in (CUMSUM, CUMPROD):
        if st in (DATE32, TIME64):
            return None                                       # TypeError in the reference
        return np.dtype(dtype) if st in (FLOAT32, FLOAT64) else np.dtype(np.int64)
    return np.dtype(dtype)


def _viewed(v, order, n):
    v = np.asarray(v)
    if order is None:
        return v[:n]
    return v[np.asarray(order, dtype=np.int64)]


def window(op, v, order, offsets, param=0, stype=None):
    """One value per position of the grouped frame (RowIndex `order`, None = identity; Groupby `offsets`)."""
    offsets = np.asarray(offsets, dtype=np.int64)
    ng = len(offsets) - 1
    n = int(offsets[-1]) if ng > 0 else 0
    if op == SHIFT:
        return shift(v, order, offsets, param, stype)
    rev = bool(param)
    if op in (CUMCOUNT, NGROUP):
        out = np.empty(n, dtype=np.int64)
        for g in range(ng):
            a, b = offsets[g], offsets[g + 1]
            if op == CUMCOUNT:
                out[a:b] = np.arange(b - a)[::-1] if rev else np.arange(b - a)
            else:
                out[a:b] = ng - 1 - g if rev else g
        return out
    x = _viewed(v, order, n)
    na = na_mask(x, stype)
    odt = out_dtype(op, stype, x.dtype)
    if odt is None:
        raise TypeError(f"Invalid column of stype {stype} in window op {op}")
    out = np.empty(n, dtype=odt)
    for g in range(ng):
        a, b = offsets[g], offsets[g + 1]
        idx = np.arange(b - 1, a - 1, -1) if rev else np.arange(a, b)
        if op in (CUMSUM, CUMPROD):
            ident = 0 if op == CUMSUM else 1
            if odt.kind == "f":
                seg = np.where(na[idx], ident, x[idx]).astype(odt)
            else:
                seg = np.where(na[idx], ident, x[idx].astype(np.int64)).astype(np.uint64)
            with np.errstate(over="ignore", invalid="ignore"):
                acc = np.cumsum(seg, dtype=seg.dtype) if op == CUMSUM else np.cumprod(seg, dtype=seg.dtype)
            out[idx] = acc.view(np.int64) if odt.kind != "f" else acc
            continue
        prev, have = None, False
        for i in idx:
            if not na[i]:
                val = x[i]
                if not have or op == FILLNA:
                    prev, have = val, True
                elif op == CUMMIN:
                    prev = prev if prev < val else val
                else:
                    prev = prev if prev > val else val
            out[i] = prev if have else na_value(stype)
    return out


def shift(v, order, offsets, n, stype=None):
    """compute_lag_rowindex (expr/head_func_shift.cc:41-62): out[p] = v[order[p - n]] when p - n is in p's group."""
    if not -2**31 <= n < 2**31:
        raise ValueError(f"Value is too large to fit in an int32: {n}")
    offsets = np.asarray(offsets, dtype=np.int64)
    ng = len(offsets) - 1
    total = int(offsets[-1]) if ng > 0 else 0
    x = _viewed(v, order, total)
    out = np.empty(total, dtype=x.dtype)
    for g in range(ng):
        a, b = offsets[g], offsets[g + 1]
        src = np.arange(a, b) - n
        ok = (src >= a) & (src < b)
        out[a:b] = na_value(stype)
        out[a:b][ok] = x[src[ok]]
    return out


def golden_array(G, ref):
    """A column of tests/golden/golden_v5.npz: ref = [dtype pool, offset, length] as the case's JSON records it."""
    pool, off, n = ref
    return G[pool][off:off + n]


# ---------------------------------------------------------------------------
# DT[i, j, by(), sort()] with window functions, restated over the CPU oracle's group() (oracle/oracle.py)
# ---------------------------------------------------------------------------
class _Capture:
    def __getitem__(self, item):
        return item


def namespace(mod):
    """Names a stored query uses, taken from module `mod` (datatable_b200 or a compatible one)."""
    return {"f": mod.f, "by": mod.by, "sort": mod.sort, "cumsum": mod.cumsum, "cumprod": mod.cumprod,
            "cummin": mod.cummin, "cummax": mod.cummax, "cumcount": mod.cumcount, "ngroup": mod.ngroup,
            "shift": mod.shift, "fillna": mod.fillna, "sum": mod.sum, "count": mod.count, "max": mod.max,
            "min": mod.min, "mean": mod.mean, "median": mod.median, "first": mod.first}


def evaluate(cols, stypes, query):
    """Evaluates `query` (source text over DT) on numpy columns with the oracle.  Returns (row ids in output order,
    [(name, stype, values, scale)]): `scale` is None where the engine must be bit-exact, else the magnitude its float
    error is measured against (running sum of |v| for cumsum, |result| otherwise)."""
    import datatable_b200 as d
    from datatable_b200 import frame as fr
    from oracle import oracle as orc
    item = eval(query, dict(namespace(d), DT=_Capture()))
    i, j, mods = item[0], item[1], item[2:]
    by_ = next((m for m in mods if isinstance(m, d.by)), None)
    sort_ = next((m for m in mods if isinstance(m, d.sort)), None)
    nrows = len(next(iter(cols.values())))
    keys, flags, na_pos = [], [], orc.NA_FIRST
    for ref in (by_.cols if by_ else []):
        keys.append(ref.name); flags.append(orc.DESCENDING if ref.negated else 0)
    if sort_ is not None:
        na_pos = {"first": orc.NA_FIRST, "last": orc.NA_LAST, "remove": orc.NA_REMOVE}[sort_.na_position]
        for ref, rev in zip(sort_.cols, sort_.reverse):
            keys.append(ref.name)
            flags.append((orc.DESCENDING if rev != ref.negated else 0) | orc.SORT_ONLY)
    whole = isinstance(i, slice) and i == slice(None)
    if keys:
        order, offsets, _ = orc.group([cols[k] for k in keys], flags, na_pos, stypes=[stypes[k] for k in keys])
        if offsets is None:
            offsets = np.array([0, len(order)], dtype=np.int32)
        if not whole:
            sel, offsets = (orc.int_groups(offsets, i) if isinstance(i, int)
                            else orc.slice_groups(offsets, i.start, i.stop, i.step))
            order = order[sel]
    else:
        order = np.arange(nrows, dtype=np.int32)
        if isinstance(i, int):
            order = order[i:i + 1] if i != -1 else order[-1:]
        elif not whole:
            order = order[i]
        offsets = np.array([0, len(order)] if len(order) else [0], dtype=np.int32)
    offsets = np.asarray(offsets, dtype=np.int32)
    gid = np.repeat(np.arange(len(offsets) - 1), np.diff(offsets))
    names, exprs = fr._resolve_j(None, j)
    out = []
    for ref in (by_.cols if by_ else []):
        out.append((ref.name, stypes[ref.name], cols[ref.name][order], None))
    for name, e in zip(names, exprs):
        if isinstance(e, fr.Window):
            x = None if e.arg is None else cols[e.arg.name]
            st = None if e.arg is None else stypes[e.arg.name]
            got = window(e.op, x, order, offsets, e.param, st)
            ost = INT64 if e.op in (CUMCOUNT, NGROUP) else (INT64 if got.dtype == np.int64 and st not in (INT64, TIME64) else st)
            scale = None
            if got.dtype.kind == "f" and e.op == CUMSUM:
                scale = window(CUMSUM, np.abs(x).astype(np.float64), order, offsets, e.param, FLOAT64)
            elif got.dtype.kind == "f" and e.op == CUMPROD:
                scale = np.abs(got).astype(np.float64)
            out.append((name, ost, got, scale))
        elif isinstance(e, fr.Reducer):
            if e.arg is None:
                red, st = np.diff(offsets).astype(np.int64), INT64
            else:
                x, st = cols[e.arg.name], stypes[e.arg.name]
                o = orc.sort_grouped(x, order, offsets, stype=st) if e.op in (orc.MEDIAN, orc.NUNIQUE) else order
                red = orc.reduce(e.op, x, o, offsets, stype=st)
                st = d.engine.reduce_out_stype(e.op, st)
            vals = red[gid]
            out.append((name, st, vals, np.abs(vals).astype(np.float64) if vals.dtype.kind == "f" else None))
        else:
            out.append((name, stypes[e.name], cols[e.name][order], None))
    names = fr._unique_names([o[0] for o in out])
    return order, [(nm,) + o[1:] for nm, o in zip(names, out)]


def assert_close(got, want, stype, scale, ctx=""):
    """Bit-exact (NaN == NaN, signs of zero included) where scale is None; else |got - want| <= tol * scale with tol
    1e-9 for float64 and 2e-4 for float32 (accumulated serially in float32 by the reference)."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{ctx}: shape {got.shape} != {want.shape}"
    if scale is None or got.dtype.kind != "f":
        if got.dtype.kind == "f":
            assert np.array_equal(got.view(f"u{got.itemsize}"), want.astype(got.dtype).view(f"u{got.itemsize}"))  \
                or (np.array_equal(np.isnan(got), np.isnan(want)) and
                    np.array_equal(got[~np.isnan(got)].view(f"u{got.itemsize}"),
                                   want.astype(got.dtype)[~np.isnan(want)].view(f"u{got.itemsize}"))), f"{ctx}: not bit-exact"
        else:
            assert np.array_equal(got.astype(np.int64), want.astype(np.int64)), f"{ctx}: integer mismatch"
        return
    tol = 2e-4 if stype == FLOAT32 else 1e-9
    nan_g, nan_w = np.isnan(got), np.isnan(want)
    assert np.array_equal(nan_g, nan_w), f"{ctx}: NA pattern differs"
    g, w, s = got[~nan_g].astype(np.float64), want[~nan_w].astype(np.float64), np.asarray(scale)[~nan_w]
    inf = np.isinf(w)
    assert np.array_equal(g[inf], w[inf]), f"{ctx}: infinities differ"
    err = np.abs(g[~inf] - w[~inf])
    assert np.all(err <= tol * s[~inf] + 1e-300), f"{ctx}: max err {err.max() if err.size else 0}"
