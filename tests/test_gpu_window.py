"""GPU: grouped cumulative and window functions (dtb_window) against the oracle's restatement
(tests/window_oracle.py) and against the reference's own results (tests/golden/golden_v5.*)."""
import json
import os

import numpy as np
import pytest

import window_oracle as wo

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
G = dict(np.load(os.path.join(HERE, "golden", "golden_v5.npz")))
CASES = json.load(open(os.path.join(HERE, "golden", "golden_v5.json")))["cases"]
TILE = 4096
SCANS = (wo.CUMSUM, wo.CUMPROD, wo.CUMMIN, wo.CUMMAX, wo.FILLNA)
ELEMS = (wo.CUMCOUNT, wo.NGROUP)
STYPES = (wo.BOOL, wo.INT8, wo.INT16, wo.INT32, wo.INT64, wo.FLOAT32, wo.FLOAT64, wo.DATE32, wo.TIME64)
NPT = {wo.BOOL: np.int8, wo.INT8: np.int8, wo.INT16: np.int16, wo.INT32: np.int32, wo.INT64: np.int64,
       wo.FLOAT32: np.float32, wo.FLOAT64: np.float64, wo.DATE32: np.int32, wo.TIME64: np.int64}


def values(rng, n, st, na=0.15):
    if st == wo.BOOL:
        a = rng.integers(0, 2, n).astype(np.int8)
    elif st in (wo.FLOAT32, wo.FLOAT64):
        a = (np.where(rng.random(n) < 0.5, -1.0, 1.0) * rng.uniform(0.9, 1.1, n)).astype(NPT[st])
        a[rng.random(n) < 0.02] = 0.0
    elif st in (wo.INT8, wo.INT32):
        a = rng.integers(-3, 4, n).astype(NPT[st])
    else:
        a = rng.integers(-1000, 1000, n).astype(NPT[st])
    a[rng.random(n) < na] = wo.na_value(st)
    return a


def layout(name, rng):
    """Groupby offsets of one group layout."""
    if name == "tile":
        sizes = [TILE] * 3 + [100]
    elif name == "edge":                 # groups ending exactly on a tile edge, a group of one at a tile start
        sizes = [TILE, 2 * TILE, 1, TILE - 1, 7, TILE - 7]
    elif name == "nohead":               # tiles without any head: one group spanning several tiles
        sizes = [5, 3 * TILE + 12, 40]
    elif name == "single":               # every row its own group
        sizes = [1] * 5000
    elif name == "ragged":               # n not a multiple of the tile
        sizes = rng.integers(1, 700, 60).tolist()
    else:                                # "empty"
        sizes = []
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)


def check(got, want, op, st, x, order, offsets, param, ctx):
    scale = None
    if want.dtype.kind == "f" and op == wo.CUMSUM:
        scale = wo.window(wo.CUMSUM, np.abs(x).astype(np.float64), order, offsets, param, wo.FLOAT64)
    elif want.dtype.kind == "f" and op == wo.CUMPROD:
        scale = np.abs(want).astype(np.float64)
    wo.assert_close(got, want, st, scale, ctx)


def run_engine(op, x, st, order, offsets, param, device):
    import torch
    from datatable_b200 import engine
    if device:
        x = torch.from_numpy(x).cuda()
        order = None if order is None else torch.from_numpy(order).cuda()
        offsets = torch.from_numpy(offsets).cuda()
    got = engine.window(op, x, order, offsets, param, stype=st)
    return got.cpu().numpy() if device else got


@pytest.mark.parametrize("st", STYPES)
@pytest.mark.parametrize("op", SCANS + ELEMS + (wo.SHIFT,))
def test_engine_every_op_and_stype(op, st):
    """every op x stype x direction on host and device buffers (ragged groups through a shuffled RowIndex)"""
    from datatable_b200 import engine
    rng = np.random.default_rng(op * 100 + st)
    offsets = layout("ragged", rng)
    n = int(offsets[-1])
    x = values(rng, n + 11, st)
    order = rng.permutation(n + 11)[:n].astype(np.int32)
    params = (-3, -1, 0, 1, 2, 700) if op == wo.SHIFT else (0, 1)
    for param in params:
        if not engine.window_out_stype(op, st):
            with pytest.raises(ValueError):
                engine.window(op, x, order, offsets, param, stype=st)
            continue
        want = wo.window(op, x, order, offsets, param, st)
        for device in (False, True):
            got = run_engine(op, x, st, order, offsets, param, device)
            check(got, want, op, st, x, order, offsets, param, f"op={op} st={st} param={param} device={device}")


@pytest.mark.parametrize("lay", ["tile", "edge", "nohead", "single", "ragged", "empty"])
@pytest.mark.parametrize("identity", [False, True])
def test_engine_group_layouts(lay, identity):
    rng = np.random.default_rng(7)
    offsets = layout(lay, rng)
    n = int(offsets[-1])
    for st in (wo.INT64, wo.FLOAT64, wo.FLOAT32, wo.INT16):
        x = values(rng, n, st)
        order = None if identity else rng.permutation(n).astype(np.int32)
        for op in SCANS + ELEMS + (wo.SHIFT,):
            for param in ((1, -TILE, 5) if op == wo.SHIFT else (0, 1)):
                if op in (wo.CUMSUM, wo.CUMPROD) and st == wo.INT16 and param:
                    continue
                want = wo.window(op, x, order, offsets, param, st)
                got = run_engine(op, x, st, order, offsets, param, True)
                check(got, want, op, st, x, order, offsets, param, f"{lay} op={op} st={st} param={param}")


def test_engine_one_group_of_1e7_rows():
    import torch
    from datatable_b200 import engine, _lib
    n = 10_000_000
    rng = np.random.default_rng(11)
    vi = rng.integers(0, 1 << 20, n).astype(np.int64)
    vf = rng.standard_normal(n)
    offsets = torch.tensor([0, n], dtype=torch.int32, device="cuda")
    di, df = torch.from_numpy(vi).cuda(), torch.from_numpy(vf).cuda()
    assert np.array_equal(engine.window(_lib.WIN_CUMSUM, di, None, offsets).cpu().numpy(), np.cumsum(vi))
    assert np.array_equal(engine.window(_lib.WIN_CUMSUM, di, None, offsets, 1).cpu().numpy(), np.cumsum(vi[::-1])[::-1])
    assert np.array_equal(engine.window(_lib.WIN_CUMMAX, di, None, offsets).cpu().numpy(), np.maximum.accumulate(vi))
    assert np.array_equal(engine.window(_lib.WIN_CUMMIN, di, None, offsets, 1).cpu().numpy(),
                          np.minimum.accumulate(vi[::-1])[::-1])
    assert np.array_equal(engine.window(_lib.WIN_CUMCOUNT, None, None, offsets).cpu().numpy(), np.arange(n))
    got = engine.window(_lib.WIN_CUMSUM, df, None, offsets).cpu().numpy()
    assert np.all(np.abs(got - np.cumsum(vf)) <= 1e-9 * np.cumsum(np.abs(vf)) + 1e-12)


# ---------------------------------------------------------------------------
# the Frame against the reference's results
# ---------------------------------------------------------------------------
def golden_frame(case):
    import datatable_b200 as d
    cols = {nm: wo.golden_array(G, case["inputs"][nm]) for nm in case["cols"]}
    return d.Frame(cols, stypes={nm: int(st) for nm, st in case["cols"].items()})


def run_query(DT, query):
    import datatable_b200 as d
    return eval(query, dict(wo.namespace(d), DT=DT))


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_frame_matches_reference(case):
    DT = golden_frame(case)
    R = run_query(DT, case["query"])
    assert R.nrows == case["nrows"]
    assert list(R.names) == case["names"]
    assert list(R.stypes) == case["stypes"]
    cols = {nm: wo.golden_array(G, case["inputs"][nm]) for nm in case["cols"]}
    _, want = wo.evaluate(cols, {nm: int(st) for nm, st in case["cols"].items()}, case["query"])
    for k, nm in enumerate(R.names):
        ref = wo.golden_array(G, case["outputs"][k])
        wo.assert_close(R.to_numpy(nm), ref, case["stypes"][k], want[k][3], ctx=f"{case['name']}:{nm}")


@pytest.mark.parametrize("case", [c for c in CASES if c["name"] in ("layout.bysort", "iby.revstep", "mixed.dict",
                                                                   "special.rev1", "cummin.rev0", "shift.-3")],
                         ids=lambda c: c["name"])
def test_host_and_device_frames_agree(case):
    DT = golden_frame(case)
    H = run_query(DT, case["query"])
    D = run_query(DT.to_device(), case["query"])
    assert H.names == D.names and H.stypes == D.stypes and H.nrows == D.nrows
    for nm in H.names:
        h, dv = H.to_numpy(nm), D.to_numpy(nm)
        assert h.tobytes() == dv.tobytes(), nm


def test_row_order_matches_reference():
    """the row ids of every case come out in the reference's order"""
    for case in CASES:
        DT = golden_frame(case)
        q = case["query"]
        head = q[:q.index(", ") + 2]                            # "DT[i, "
        rest = q[len(head):]
        mods = ""
        for m in (", by(", ", sort("):
            if m in rest:
                mods = rest[rest.index(m):-1] if not mods else mods
        R = run_query(DT, f"{head}[f.r, cumcount()]{mods}]")
        assert np.array_equal(R.to_numpy("r"), wo.golden_array(G, case["r"])), case["name"]


def test_na_remove_against_oracle():
    """sort(..., na_position="remove"): one group over the rows kept (the reference corrupts its heap here)"""
    import datatable_b200 as d
    case = next(c for c in CASES if c["name"] == "layout.by")
    cols = {nm: wo.golden_array(G, case["inputs"][nm]) for nm in case["cols"]}
    stypes = {nm: int(st) for nm, st in case["cols"].items()}
    DT = d.Frame(cols, stypes=stypes)
    for q in ("DT[:, [f.r, cumsum(f.f64), cummax(f.i32), shift(f.i16, 1), cumcount(), ngroup()], sort(f.f64, na_position='remove')]",
              "DT[:, [f.r, cumsum(f.f64, reverse=True), fillna(f.f32), sum(f.i64)], sort(f.k, f.i32, na_position='remove')]",
              "DT[2:9, [f.r, cumprod(f.i8), cumcount(reverse=True)], sort(f.i16, na_position='remove')]"):
        order, want = wo.evaluate(cols, stypes, q)
        R = run_query(DT, q)
        assert list(R.names) == [w[0] for w in want], q
        assert list(R.stypes) == [w[1] for w in want], q
        assert R.nrows == len(order)
        for nm, st, vals, scale in want:
            wo.assert_close(R.to_numpy(nm), vals, st, scale, ctx=f"{q}:{nm}")


def test_empty_frame_against_oracle():
    import datatable_b200 as d
    case = next(c for c in CASES if c["name"] == "layout.by")
    cols = {nm: wo.golden_array(G, case["inputs"][nm])[:0] for nm in case["cols"]}
    stypes = {nm: int(st) for nm, st in case["cols"].items()}
    DT = d.Frame(cols, stypes=stypes)
    for q in ("DT[:, [f.r, cumsum(f.f64), cumcount(), sum(f.i32)], by(f.k)]", "DT[:, [cumsum(f.f64), shift(f.i8)]]"):
        _, want = wo.evaluate(cols, stypes, q)
        R = run_query(DT, q)
        assert R.nrows == 0 and list(R.names) == [w[0] for w in want] and list(R.stypes) == [w[1] for w in want]


def test_errors():
    import datatable_b200 as d
    from datatable_b200 import f, by
    DT = d.Frame({"k": np.array([1, 1, 2], np.int32), "d": np.array([1, 2, 3], np.int32)}, stypes={"d": wo.DATE32})
    with pytest.raises(TypeError, match="Invalid column of type date32 in cumsum"):
        DT[:, d.cumsum(f.d), by(f.k)]
    R = DT[:, d.cummax(f.d), by(f.k)]
    assert list(R.stypes) == [wo.INT32, wo.DATE32]
    with pytest.raises(ValueError, match="too large to fit in an int32"):
        d.shift(f.d, 2**31)
    with pytest.raises(NotImplementedError):
        d.fillna(f.d, value=0)


# ---------------------------------------------------------------------------
# 1e8 rows in the C2 shape (int32 keys, ~1000 rows per group), device-resident
# ---------------------------------------------------------------------------
def test_c2_shape_1e8_rows():
    import torch
    import datatable_b200 as d
    from datatable_b200 import f, by
    n, nk = 100_000_000, 100_000
    rng = np.random.default_rng(5)
    k = rng.integers(0, nk, n).astype(np.int32)
    vi = rng.integers(0, 1 << 20, n).astype(np.int64)
    vf = rng.standard_normal(n)
    DT = d.Frame({"k": torch.from_numpy(k).cuda(), "vi": torch.from_numpy(vi).cuda(), "vf": torch.from_numpy(vf).cuda()})
    R = DT[:, [d.cumsum(f.vi), d.cummax(f.vi), d.shift(f.vi, 1), d.cumsum(f.vf), d.cumcount(), d.sum(f.vi), d.count()],
           by(f.k)]
    assert list(R.names) == ["k", "vi", "vi.0", "vi.1", "vf", "C0", "vi.2", "count"]
    order = np.argsort(k, kind="stable")
    ks = k[order]
    assert np.array_equal(R.to_numpy("k"), ks)
    head = np.ones(n, bool); head[1:] = ks[1:] != ks[:-1]
    starts = np.flatnonzero(head)
    gid = np.cumsum(head) - 1
    x = vi[order]
    cs = np.cumsum(x)
    want = cs - np.concatenate([[0], cs[starts[1:] - 1]])[gid]
    got = R.to_numpy("vi")
    assert np.array_equal(got, want)
    assert np.array_equal(R.to_numpy("vi.0"), np.maximum.accumulate(gid.astype(np.int64) << 21 | x) & ((1 << 21) - 1))
    sh = np.empty(n, np.int64); sh[1:] = x[:-1]; sh[head] = -2**63
    assert np.array_equal(R.to_numpy("vi.1"), sh)
    xf = vf[order]
    csf, csa = np.cumsum(xf), np.cumsum(np.abs(xf))
    base = np.concatenate([[0.0], csf[starts[1:] - 1]])[gid]
    basea = np.concatenate([[0.0], csa[starts[1:] - 1]])[gid]
    assert np.all(np.abs(R.to_numpy("vf") - (csf - base)) <= 1e-9 * (csa - basea) + 1e-15 * csa)
    ends = np.concatenate([starts[1:], [n]]) - 1
    assert np.array_equal(got[ends], R.to_numpy("vi.2")[ends])              # last cumsum of a group == sum()
    cc = R.to_numpy("C0")
    assert np.array_equal(cc[ends] + 1, R.to_numpy("count")[ends])          # max(cumcount) + 1 == count()
