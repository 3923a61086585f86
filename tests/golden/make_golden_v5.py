#!/usr/bin/env python
"""
Generates tests/golden/golden_v5.{npz,json} by running the *reference itself* (the unmodified build staged by
oracle/build_ref.sh) on the grouped cumulative and window functions of DT[i, j, by(), sort()]:

    PYTHONPATH=oracle/_ref python tests/golden/make_golden_v5.py

    cumsum / cumprod      column/cumsumprod.h:48-95
    cummin / cummax       column/cumminmax.h:48-110
    cumcount / ngroup     column/cumcountngroup.h:52-70
    fillna                expr/fexpr_fillna.cc:86-118
    shift                 expr/head_func_shift.cc:41-62
    GtoALL evaluation     expr/eval_context.cc:144-172 (reducers repeated on every row of their group)

Every case stores its input columns (each distinct column once), the query as Python source (evaluated against the reference here and against
datatable_b200 by the tests), and what the reference returned: names, stypes, the values of every column, and the
row ids `r` in output order.  sort(..., na_position="remove") is left out: the reference corrupts its heap on it
together with a cumulative function (eval_context.cc:283-286 builds single_group(nrows) over fewer rows).
"""
import hashlib
import json
import os

import numpy as np

import datatable as dt
from datatable import f, by, sort

HERE = os.path.dirname(os.path.abspath(__file__))
rng = np.random.default_rng(20261017)
pools, manifest, seen = {}, [], {}


def put(a, shared=False):
    """Appends `a` to the pool of its dtype; returns [pool, offset, length].  Every dtype has one array in the npz:
    a few large entries compress far better than one small entry per column.  shared: store equal arrays once."""
    key = hashlib.sha256(a.dtype.str.encode() + a.tobytes()).hexdigest()
    if shared and key in seen:
        return seen[key]
    pool = pools.setdefault(a.dtype.name, [])
    ref = [a.dtype.name, int(sum(len(x) for x in pool)), int(len(a))]
    pool.append(a)
    if shared:
        seen[key] = ref
    return ref

ST = {"bool8": 1, "int8": 2, "int16": 3, "int32": 4, "int64": 5, "float32": 6, "float64": 7, "date32": 17, "time64": 18}
NP = {1: np.int8, 2: np.int8, 3: np.int16, 4: np.int32, 5: np.int64, 6: np.float32, 7: np.float64, 17: np.int32,
      18: np.int64}
NA = {1: -128, 2: -128, 3: -2**15, 4: -2**31, 5: -2**63, 17: -2**31, 18: -2**63}
NS = {"f": f, "by": by, "sort": sort, "cumsum": dt.cumsum, "cumprod": dt.cumprod, "cummin": dt.cummin,
      "cummax": dt.cummax, "cumcount": dt.cumcount, "ngroup": dt.ngroup, "shift": dt.shift, "fillna": dt.fillna,
      "sum": dt.sum, "count": dt.count, "max": dt.max, "min": dt.min, "mean": dt.mean, "median": dt.median,
      "first": dt.first}


def to_dt(cols):
    """{name: (array with NA sentinels / NaN, stype code)} -> reference Frame"""
    data, stypes, casts = {}, {}, {}
    for nm, (a, st) in cols.items():
        if st in (6, 7):
            data[nm] = [None if np.isnan(x) else float(x) for x in a.tolist()]
        elif st == 1:
            data[nm] = [None if x == -128 else bool(x) for x in a.tolist()]
        else:
            data[nm] = [None if x == NA[st] else int(x) for x in a.tolist()]
        name = [k for k, v in ST.items() if v == st][0]
        if st in (17, 18):
            stypes[nm], casts[nm] = (dt.int32 if st == 17 else dt.int64), getattr(dt.stype, name)
        else:
            stypes[nm] = getattr(dt, name)
    DT = dt.Frame(data, stypes=stypes)
    for nm, s in casts.items():
        DT[nm] = s
    return DT


def column(R, i, st):
    a = R[:, i].to_numpy()[:, 0]
    fill = np.nan if st in (6, 7) else NA[st]
    if a.dtype.kind == "M":
        mask = np.isnat(a)
        a = a.view(np.int64)
        a = np.where(mask, fill, a)
    if isinstance(a, np.ma.MaskedArray):
        mask = np.ma.getmaskarray(a)
        a = np.where(mask, fill, a.data.astype(np.float64 if st in (6, 7) else np.int64))
    return np.asarray(a).astype(NP[st])


def add(name, cols, query, rquery):
    DT = to_dt(cols)
    R = eval(query, dict(NS, DT=DT))
    RR = eval(rquery, dict(NS, DT=DT))
    sts = [ST[str(s).split(".")[-1]] for s in R.stypes]
    case = {"name": name, "query": query, "cols": {nm: st for nm, (a, st) in cols.items()},
            "inputs": {nm: put(np.asarray(a).astype(NP[st]), shared=True) for nm, (a, st) in cols.items()},
            "nrows": int(R.nrows), "names": list(R.names), "stypes": sts,
            "outputs": [put(column(R, i, st)) for i, st in enumerate(sts)],
            "r": put(column(RR, list(RR.names).index("r"), 4))}
    manifest.append(case)


def with_na(a, st, frac=0.15):
    a = a.copy()
    m = rng.random(len(a)) < frac
    a[m] = np.nan if st in (6, 7) else NA[st]
    return a


def base(n, ngroups):
    k = rng.integers(0, ngroups, n).astype(np.int32)
    k[rng.random(n) < 0.08] = NA[4]
    sign = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    return {
        "k": (k, 4), "k2": (rng.integers(0, 3, n).astype(np.int8), 2), "r": (np.arange(n, dtype=np.int32), 4),
        "b": (with_na(rng.integers(0, 2, n).astype(np.int8), 1), 1),
        "i8": (with_na(rng.integers(-3, 4, n).astype(np.int8), 2), 2),
        "i16": (with_na(rng.integers(-300, 300, n).astype(np.int16), 3), 3),
        "i32": (with_na(rng.integers(-3, 4, n).astype(np.int32), 4), 4),
        "i64": (with_na(rng.integers(-2**40, 2**40, n).astype(np.int64), 5), 5),
        "f32": (with_na((sign * rng.uniform(0.5, 1.5, n)).astype(np.float32), 6), 6),
        "f64": (with_na(np.round(sign * rng.uniform(0.5, 1.5, n), 6), 7), 7),
        "d": (with_na(rng.integers(0, 20000, n).astype(np.int32), 17), 17),
        "t": (with_na(rng.integers(0, 2**50, n).astype(np.int64), 18), 18),
    }


B = base(200, 5)
ALL = "[f.b, f.i8, f.i16, f.i32, f.i64, f.f32, f.f64, f.d, f.t]"
NUM = "[f.b, f.i8, f.i16, f.i32, f.i64, f.f32, f.f64]"
RQ = "DT[{i}, [f.r, cumcount()]{m}]"


def q(name, j, i=":", m=", by(f.k)", cols=None):
    add(name, B if cols is None else cols, f"DT[{i}, {j}{m}]", RQ.format(i=i, m=m))


# every op and direction over every stype it accepts
for op in ("cumsum", "cumprod", "cummin", "cummax", "fillna"):
    for rev in (False, True):
        q(f"{op}.rev{int(rev)}", f"[f.r, {op}({NUM if op.startswith('cums') or op == 'cumprod' else ALL}, reverse={rev})]")
q("counts", "[cumcount(), cumcount(reverse=True), ngroup(), ngroup(reverse=True)]")
for sh in (0, 1, -1, 3, -3, 60, -400):
    q(f"shift.{sh}", "[f.r, " + ", ".join(f"shift({c}, {sh})" for c in ALL[1:-1].split(", ")) + "]")

# group layouts: by(k), by(-k), by(k1, k2), by + sort, sort alone (NA first and last), no by
MIX = "[f.r, cumsum(f.f64), cummax(f.i32), shift(f.i64, 2), fillna(f.f32, reverse=True), cumcount(), ngroup(reverse=True), cumprod(f.i8)]"
for nm, m in [("by", ", by(f.k)"), ("bydesc", ", by(-f.k)"), ("by2", ", by(f.k, f.k2)"), ("bysort", ", by(f.k), sort(f.i16)"),
              ("bysortlast", ", by(f.k), sort(-f.f64, na_position='last')"), ("sort", ", sort(f.i32)"),
              ("sortlast", ", sort(f.i32, na_position='last')"), ("sortdesc", ", sort(-f.f64)"), ("noby", "")]:
    q(f"layout.{nm}", MIX, m=m)

# integer and slice i inside the groups (and a plain row slice without by)
for nm, i in [("head", ":5"), ("step", "2::3"), ("rev", "::-1"), ("tail", "-3:"), ("revstep", "::-2"), ("mid", "5:1:-2"),
              ("int", "3"), ("intneg", "-1"), ("none", "40:"), ("rep", "1:4:0")]:
    q(f"iby.{nm}", MIX, i=i)
    q(f"isort.{nm}", MIX, i=i, m=", sort(f.i32)")
for nm, i in [("slice", "2:50"), ("revslice", "::-3"), ("int", "7")]:
    q(f"inoby.{nm}", MIX, i=i, m="")

# mixed j: plain columns, reducers repeated per row, window functions, dict names, list arguments
q("mixed.bcast", "[f.r, sum(f.f64)]")
q("mixed.all", "[f.r, cumsum(f.f64), sum(f.f64), count()]")
q("mixed.dict", "{'a': f.r, 's': sum(f.i32), 'c': cumsum(f.f64), 'n': count(), 'm': max(f.i16), 'x': cummin(f.d)}")
q("mixed.list", "[f.r, mean(f.f64), min(f.b), cumsum([f.i8, f.f32]), median(f.f64), first(f.r)]")
q("mixed.noby", "[sum(f.f64), cumsum(f.f64), count()]", m="")
q("mixed.sliced", "[f.r, sum(f.f64), cumcount(), max(f.i64)]", i="1::2")
q("mixed.key", "[f.k, cumsum(f.k), shift(f.k)]")

# special values: +-0, +-inf, int64 wrap of sums and products
zeros = np.array([-0.0, 0.0, -0.0, 0.0, np.inf, -np.inf, np.nan, 1.0, -np.inf, -0.0, np.nan, 0.0, np.inf, -0.0], np.float64)
ks = np.array([1, 1, 1, 1, 2, 2, 2, 2, 2, 3, 3, 3, 3, 3], np.int32)
SP = {"k": (ks, 4), "r": (np.arange(len(ks), dtype=np.int32), 4), "x": (zeros, 7), "y": (zeros.astype(np.float32), 6),
      "w": (np.array([2**62, 4, 3, -2**62, 2**62, 2**62, -2**63, 5, 2**61, 8, 7, 2**63 - 1, 2, 3], np.int64), 5)}
for rev in (False, True):
    q(f"special.rev{int(rev)}", f"[f.r, cummin([f.x, f.y], reverse={rev}), cummax([f.x, f.y], reverse={rev}), "
      f"fillna([f.x, f.y], reverse={rev}), cumsum([f.x, f.y, f.w], reverse={rev}), cumprod([f.x, f.w], reverse={rev})]", cols=SP)
    q(f"special.noby.rev{int(rev)}", f"[f.r, cummin(f.x, reverse={rev}), cummax(f.x, reverse={rev}), cumsum(f.w, reverse={rev}), "
      f"cumprod(f.w, reverse={rev}), shift(f.x, 1)]", m="", cols=SP)
q("special.wrap2", "cumprod(f.w)", m="", cols={"w": (np.array([2**62, 4], np.int64), 5), "r": (np.arange(2, dtype=np.int32), 4)})

# one group, every row its own group.  (The reference crashes on a cumulative function over an empty frame, with or
# without by(); tests/test_gpu_window.py checks that case against the oracle.)
one = dict(B); one["k"] = (np.full(200, 7, np.int32), 4)
q("onegroup", MIX, cols=one)
own = dict(B); own["k"] = (rng.permutation(200).astype(np.int32), 4)
q("owngroups", MIX, cols=own)

# float64 tolerance case: 10k rows, groups of ~1000
n = 10000
big = {"k": (rng.integers(0, 10, n).astype(np.int32), 4), "r": (np.arange(n, dtype=np.int32), 4),
       "v": (with_na(rng.standard_normal(n) * 1e3, 7), 7)}
q("big.f64", "[f.r, cumsum(f.v)]", cols=big)

np.savez_compressed(os.path.join(HERE, "golden_v5.npz"), **{k: np.concatenate(v) for k, v in pools.items()})
json.dump({"generator": "tests/golden/make_golden_v5.py", "datatable_version": dt.__version__, "cases": manifest},
          open(os.path.join(HERE, "golden_v5.json"), "w"), indent=0)
print(len(manifest), "cases")
