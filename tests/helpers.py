"""Shared helpers for parity tests (oracle and CUDA path use the same checks)."""
import numpy as np

BOOL, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64 = 1, 2, 3, 4, 5, 6, 7
DESCENDING, SORT_ONLY = 2, 4
NA_POS = {"first": 1, "last": 2, "remove": 3}
OPS = {"sum": 1, "mean": 2, "min": 3, "max": 4, "count": 5, "countna": 6, "nrows": 7}


def case_flags(case):
    """SortFlag per key column as the reference builds them (fexpr_list.cc:322-365, eval_context.cc:271-273)."""
    nk = len(case["kst"])
    nby = case["nby"]
    flags = []
    for i in range(nk):
        fl = DESCENDING if case["reverse"][i] else 0
        if nby is None or i >= nby:
            fl |= SORT_ONLY
        flags.append(fl)
    return flags


def assert_reducer_equal(got, want, op, vst, ctx=""):
    """Integers / counts / min / max bit-exact (NaN == NaN); float sums and means to 1e-6 relative
    (north_star tolerance; the reference's own helper uses 1e-7, tests/__init__.py:65-143)."""
    got = np.asarray(got); want = np.asarray(want)
    assert got.shape == want.shape, f"{ctx}: shape {got.shape} != {want.shape}"
    assert got.dtype == want.dtype, f"{ctx}: dtype {got.dtype} != {want.dtype}"
    if got.dtype.kind != "f":
        assert np.array_equal(got, want), f"{ctx}: integer mismatch"
        return
    nan_g, nan_w = np.isnan(got), np.isnan(want)
    assert np.array_equal(nan_g, nan_w), f"{ctx}: NA pattern differs"
    g, w = got[~nan_g].astype(np.float64), want[~nan_w].astype(np.float64)
    if op in ("min", "max"):
        assert np.array_equal(g, w), f"{ctx}: min/max must be exact"
        return
    rtol = 1e-6
    if vst == FLOAT32 and op == "sum":
        # the reference accumulates float32 sums sequentially in float32 (column/sumprod.h:47-54);
        # any other association differs by O(n * 2^-24)
        rtol = 2e-4
    inf = np.isinf(w)
    assert np.array_equal(g[inf], w[inf]), f"{ctx}: infinities differ"
    err = np.abs(g[~inf] - w[~inf])
    ok = err <= rtol * np.abs(w[~inf])
    assert np.all(ok), f"{ctx}: float mismatch, max rel err {np.max(err / np.maximum(np.abs(w[~inf]), 1e-300))}"


def hook_inputs(name):
    """The frames integration/check_hook.py ("group"), check_hook_reducers.py ("reducers") and check_hook_views.py
    ("views") build, as numpy columns (same seeds and sizes)."""
    if name == "group":
        rng = np.random.default_rng(7)
        n = 200_000
        return {"k": rng.integers(0, 1000, n).astype(np.int32), "x": rng.standard_normal(n), "v": rng.random(n),
                "idx": np.arange(n, dtype=np.int32)}
    rng = np.random.default_rng(3 if name == "reducers" else 11)
    n = 300_000 if name == "reducers" else 400_000
    k = rng.integers(0, 5000, n).astype(np.int32)
    v = rng.random(n); v[rng.random(n) < 0.05] = np.nan
    w = rng.integers(-1000, 1000, n).astype(np.int16)
    b = rng.random(n) < 0.3
    cols = {"k": k, "v": v, "w": w, "b": b}
    if name == "views":
        cols["x"] = rng.integers(-2**60, 2**60, n)
    return cols


def digest(a):
    """sha256 of a column's values (integers as int64, floats as float64 with one NaN pattern), for outputs too large
    to store."""
    import hashlib
    a = np.asarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a.astype(np.float64))
    else:
        a = a.astype(np.int64)
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
