"""GPU: seeded random parity against the oracle at growing sizes, plus size-independent
properties at sizes the oracle cannot reach in seconds."""
import numpy as np
import pytest

from helpers import (BOOL, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64, DESCENDING, SORT_ONLY,
                     OPS, assert_reducer_equal)

pytestmark = pytest.mark.gpu

NA = {INT8: -2**7, INT16: -2**15, INT32: -2**31, INT64: -2**63}
NPT = {BOOL: np.int8, INT8: np.int8, INT16: np.int16, INT32: np.int32, INT64: np.int64,
       FLOAT32: np.float32, FLOAT64: np.float64}


def make_col(rng, st, n, spread, na_frac):
    if st == BOOL:
        a = rng.integers(0, 2, n).astype(np.int8)
    elif st in (FLOAT32, FLOAT64):
        if spread == "few":
            a = (rng.integers(-50, 50, n) / 4).astype(NPT[st])
        elif spread == "unit":
            a = rng.random(n).astype(NPT[st])
        else:
            a = (rng.standard_normal(n) * 10.0 ** rng.integers(-30, 30, n)).astype(NPT[st])
    else:
        info = np.iinfo(NPT[st])
        if spread == "few":
            lo, hi = -20, 20
        elif spread == "unit":
            lo, hi = max(info.min + 1, -30000), min(info.max, 1000000)
        else:
            lo, hi = info.min + 1, info.max
        a = rng.integers(lo, hi, n, dtype=np.int64, endpoint=True).astype(NPT[st])
    if na_frac:
        m = rng.random(n) < na_frac
        if st in NA:
            a[m] = NA[st]
        elif st == BOOL:
            a[m] = -128
        else:
            a[m] = np.nan
    return a


@pytest.mark.parametrize("st", [BOOL, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64])
@pytest.mark.parametrize("n", [1000, 4097, 100_000, 1_000_003])
def test_single_key_sort_vs_oracle(st, n):
    from datatable_b200 import engine
    from oracle import oracle as orc
    rng = np.random.default_rng(n * 31 + st)
    for spread, na_frac, desc, na_pos in (("few", 0.1, False, 1), ("unit", 0.0, True, 2), ("wide", 0.05, False, 3),
                                          ("wide", 0.02, True, 1)):
        k = make_col(rng, st, n, spread, na_frac)
        fl = [SORT_ONLY | (DESCENDING if desc else 0)]
        want, _, _ = orc.group([k], fl, na_pos, stypes=[st])
        got, offs, ng = engine.group([engine.Col(k, st)], fl, na_pos)
        assert offs is None
        assert np.array_equal(got, want), f"st={st} n={n} {spread} desc={desc} na_pos={na_pos}"


@pytest.mark.parametrize("st", [INT8, INT32, INT64, FLOAT64])
@pytest.mark.parametrize("n", [5000, 300_000])
def test_groupby_reducers_vs_oracle(st, n):
    from datatable_b200 import engine
    from oracle import oracle as orc
    rng = np.random.default_rng(n + st)
    for spread in ("few", "unit"):
        k = make_col(rng, st, n, spread, 0.03)
        want_o, want_f, want_ng = orc.group([k], [0], 1, stypes=[st])
        got_o, got_f, got_ng = engine.group([engine.Col(k, st)], [0], 1)
        assert np.array_equal(got_o, want_o)
        assert np.array_equal(got_f, want_f) and got_ng == want_ng
        for vst in (BOOL, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64):
            v = make_col(rng, vst, n, "few" if vst == BOOL else "unit", 0.1)
            for op in ("sum", "mean", "min", "max", "count", "countna"):
                want = orc.reduce(OPS[op], v, want_o, want_f, stype=vst)
                got = engine.reduce(OPS[op], engine.Col(v, vst), got_o, got_f)
                assert_reducer_equal(got, want, op, vst, ctx=f"key st={st} {spread} {op} vst={vst}")
        got = engine.reduce(OPS["nrows"], None, got_o, got_f)
        assert np.array_equal(got, np.diff(want_f).astype(np.int64))


@pytest.mark.parametrize("sts", [(INT64, INT32), (INT8, FLOAT64, INT16), (FLOAT32, BOOL), (INT32, INT32, INT32, INT8)])
def test_multikey_vs_oracle(sts):
    from datatable_b200 import engine
    from oracle import oracle as orc
    n = 200_000
    rng = np.random.default_rng(len(sts) * 7 + sts[0])
    for trial in range(3):
        keys = [make_col(rng, st, n, "few", 0.05) for st in sts]
        flags = [DESCENDING if rng.integers(0, 2) else 0 for _ in sts]
        nby = len(sts) if trial == 0 else (len(sts) - 1 if trial == 1 else 0)
        for i in range(nby, len(sts)):
            flags[i] |= SORT_ONLY
        na_pos = 1 if trial < 2 else 2
        want_o, want_f, want_ng = orc.group(keys, flags, na_pos, stypes=list(sts))
        got_o, got_f, got_ng = engine.group([engine.Col(k, st) for k, st in zip(keys, sts)], flags, na_pos)
        assert np.array_equal(got_o, want_o), f"{sts} trial {trial}"
        if nby:
            assert np.array_equal(got_f, want_f) and got_ng == want_ng
        else:
            assert got_f is None


def test_c4_shape_keys_vs_oracle():
    """(int64 with 33 constant low bits, int32) keys: the composite key must shrink to ~20 bits."""
    from datatable_b200 import engine, _lib
    from oracle import oracle as orc
    n = 500_000
    rng = np.random.default_rng(44)
    k1 = rng.integers(0, 1000, n).astype(np.int64) << 33
    k2 = rng.integers(0, 1000, n).astype(np.int32)
    want_o, want_f, _ = orc.group([k1, k2], [0, 0], 1)
    got_o, got_f, _ = engine.group([k1, k2], [0, 0], 1)
    assert _lib.last_call_stats()["key_bits"] == 20
    assert np.array_equal(got_o, want_o) and np.array_equal(got_f, want_f)


@pytest.mark.parametrize("n", [20_000_000])
def test_large_device_properties(n):
    """Size-independent properties on device-resident data: the RowIndex is a permutation, the
    gathered keys are sorted, ties keep ascending row index, offsets match the key run lengths,
    and group sums add up to the column total."""
    import torch
    from datatable_b200 import engine
    g = torch.Generator(device="cuda"); g.manual_seed(7)
    k = torch.randint(0, 100_000, (n,), generator=g, device="cuda", dtype=torch.int32)
    v = torch.rand(n, generator=g, device="cuda", dtype=torch.float64)
    order, offsets, ng = engine.group([k], [0], 1)
    o64 = order.long()
    assert torch.equal(torch.sort(o64).values, torch.arange(n, device="cuda"))
    ks = k[o64]
    assert bool((ks[1:] >= ks[:-1]).all())
    same = ks[1:] == ks[:-1]
    assert bool((o64[1:][same] > o64[:-1][same]).all()), "ties must keep ascending row index"
    uniq, counts = torch.unique_consecutive(ks, return_counts=True)
    assert ng == uniq.numel()
    assert torch.equal(offsets.long(), torch.cat([torch.zeros(1, dtype=torch.long, device="cuda"), counts.cumsum(0)]))
    sums = engine.reduce(OPS["sum"], v, order, offsets)
    ref = torch.zeros(100_000, dtype=torch.float64, device="cuda").index_add_(0, k.long(), v)
    assert torch.allclose(sums, ref[uniq.long()], rtol=1e-9, atol=0)
    cnt = engine.reduce(OPS["count"], v, order, offsets)
    assert torch.equal(cnt, counts)


def test_large_float64_sort_properties():
    import torch
    from datatable_b200 import engine
    n = 10_000_000
    g = torch.Generator(device="cuda"); g.manual_seed(11)
    x = torch.randn(n, generator=g, device="cuda", dtype=torch.float64)
    x[::1000] = float("nan")
    x[1::1000] = 0.0
    x[2::1000] = -0.0
    order, offsets, ng = engine.group([x], [SORT_ONLY], 1)
    assert offsets is None
    xs = x[order.long()]
    nn = int(torch.isnan(x).sum())
    assert bool(torch.isnan(xs[:nn]).all()) and not bool(torch.isnan(xs[nn:]).any())   # NaN first
    body = xs[nn:]
    assert bool((body[1:] >= body[:-1]).all())
    bits = body.view(torch.int64)
    zero = body == 0
    zb = bits[zero]
    assert bool((zb[1:] >= zb[:-1]).all()), "-0.0 sorts before +0.0 (bit-pattern order)"
    assert torch.equal(torch.sort(order.long()).values, torch.arange(n, device="cuda"))


@pytest.mark.parametrize("kst", [INT8, INT32, INT64, FLOAT64])
def test_groupby_handle_direct_reducers_vs_oracle(kst):
    """Groupby handle on device-resident columns: small key domains take the direct-address
    (streaming + L2 atomics) reducers; results must equal the oracle's gather-based answer."""
    import torch
    from datatable_b200 import engine
    from oracle import oracle as orc
    n = 400_000
    rng = np.random.default_rng(900 + kst)
    for variant in ("uniform", "hot", "na"):
        k = make_col(rng, kst, n, "few" if kst != INT32 else "unit", 0.05 if variant == "na" else 0.0)
        if variant == "hot":
            k[rng.random(n) < 0.7] = k[0]                  # one key owns 70% of the rows
        want_o, want_f, want_ng = orc.group([k], [0], 1, stypes=[kst])
        kd = torch.from_numpy(k).cuda()
        gb = engine.Groupby([engine.Col(kd, kst)], [0], 1)
        assert gb.ngroups == want_ng
        assert np.array_equal(gb.order().cpu().numpy(), want_o)
        assert np.array_equal(gb.offsets().cpu().numpy(), want_f)
        for vst in (BOOL, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64):
            v = make_col(rng, vst, n, "few" if vst == BOOL else "unit", 0.1)
            vd = engine.Col(torch.from_numpy(v).cuda(), vst)
            for op in ("sum", "mean", "min", "max", "count", "countna"):
                want = orc.reduce(OPS[op], v, want_o, want_f, stype=vst)
                got = gb.reduce(OPS[op], vd).cpu().numpy()
                assert_reducer_equal(got, want, op, vst, ctx=f"direct key st={kst} {variant} {op} vst={vst}")
        got = gb.reduce(OPS["nrows"], None).cpu().numpy()
        assert np.array_equal(got, np.diff(want_f).astype(np.int64))
        gb.close()


def test_groupby_handle_multikey_direct():
    import torch
    from datatable_b200 import engine
    from oracle import oracle as orc
    n = 300_000
    rng = np.random.default_rng(77)
    k1 = make_col(rng, INT64, n, "few", 0.02) << 20
    k1[k1 == (NA[INT64] << 20)] = NA[INT64]
    k2 = make_col(rng, INT16, n, "few", 0.02)
    x = make_col(rng, FLOAT64, n, "unit", 0.0)
    v = make_col(rng, FLOAT64, n, "unit", 0.1)
    # by(k1, k2) + sort(x): groups come from the by-columns only
    flags = [0, DESCENDING, SORT_ONLY]
    want_o, want_f, want_ng = orc.group([k1, k2, x], flags, 1)
    gb = engine.Groupby([torch.from_numpy(a).cuda() for a in (k1, k2, x)], flags, 1)
    assert np.array_equal(gb.order().cpu().numpy(), want_o)
    assert np.array_equal(gb.offsets().cpu().numpy(), want_f)
    vd = torch.from_numpy(v).cuda()
    for op in ("sum", "mean", "min", "max", "count"):
        want = orc.reduce(OPS[op], v, want_o, want_f)
        got = gb.reduce(OPS[op], vd).cpu().numpy()
        assert_reducer_equal(got, want, op, FLOAT64, ctx=f"multikey direct {op}")
    gb.close()


def _check_direct_modes(k, kst, vals, ctx):
    """fused create_reduce and the handle's reduce against the oracle, every reducer, on one key column"""
    import torch
    from datatable_b200 import engine
    from oracle import oracle as orc
    want_o, want_f, want_ng = orc.group([k], [0], 1, stypes=[kst])
    kd = torch.from_numpy(k).cuda()
    ops = ("sum", "mean", "min", "max", "count", "countna")
    reds = [(op, v, vst) for v, vst in vals for op in ops]
    gb = engine.Groupby([engine.Col(kd, kst)], [0], 1,
                        reducers=[(OPS[op], engine.Col(torch.from_numpy(v).cuda(), vst)) for op, v, vst in reds])
    assert gb.ngroups == want_ng
    assert np.array_equal(gb.order().cpu().numpy(), want_o)
    assert np.array_equal(gb.offsets().cpu().numpy(), want_f)
    for i, (op, v, vst) in enumerate(reds):
        want = orc.reduce(OPS[op], v, want_o, want_f, stype=vst)
        assert_reducer_equal(gb.reduced(i).cpu().numpy(), want, op, vst, ctx=f"{ctx} fused {op} vst={vst}")
        got = gb.reduce(OPS[op], engine.Col(torch.from_numpy(v).cuda(), vst)).cpu().numpy()
        assert_reducer_equal(got, want, op, vst, ctx=f"{ctx} handle {op} vst={vst}")
    gb.close()


def test_direct_reducers_few_groups_in_sparse_domain():
    """<= 2048 groups whose keys are spread over a domain of millions: the rows fold into per-CTA
    shared-memory tables through a key -> group map (dtb_reduce.cu, plan_direct)."""
    rng = np.random.default_rng(4242)
    n = 700_000
    for ngroups, kst in ((3, INT32), (150, INT32), (2048, INT64), (2049, INT32)):
        domain = rng.choice(3_000_000, ngroups, replace=False).astype(NPT[kst]) - 1_000_000
        k = domain[rng.integers(0, ngroups, n)]
        k[:ngroups] = domain                                   # every key occurs
        if ngroups == 150:
            k[rng.random(n) < 0.02] = NA[kst]
        vals = [(make_col(rng, FLOAT64, n, "unit", 0.1), FLOAT64), (make_col(rng, INT32, n, "unit", 0.1), INT32),
                (make_col(rng, FLOAT32, n, "few", 0.1), FLOAT32)]
        _check_direct_modes(k, kst, vals, f"sparse ng={ngroups}")


def test_direct_reducers_skewed_group_sizes():
    """Thousands of groups, some of them huge: rows of the hot keys fold in a shared-memory cache (more hot
    keys than cache slots here, so the overflow path to the global table runs too), the rest go one atomic
    per row; one giant key on top."""
    rng = np.random.default_rng(777)
    hot = rng.choice(2_000_000, 3500, replace=False)
    cold = rng.choice(2_000_000, 10_000, replace=False)
    k = np.concatenate([np.repeat(hot, 1100), np.full(20_000, hot[0]), cold[rng.integers(0, len(cold), 300_000)]])
    k = k.astype(np.int32)
    rng.shuffle(k)
    n = len(k)
    k[rng.random(n) < 0.001] = NA[INT32]
    vals = [(make_col(rng, FLOAT64, n, "unit", 0.1), FLOAT64), (make_col(rng, INT64, n, "unit", 0.1), INT64)]
    _check_direct_modes(k, INT32, vals, "skewed")
    # half of the rows in one key, the rest spread out
    k2 = rng.integers(0, 1_000_000, 1_000_000).astype(np.int32)
    k2[rng.random(len(k2)) < 0.5] = 123_456
    vals2 = [(make_col(rng, FLOAT64, len(k2), "unit", 0.0), FLOAT64), (make_col(rng, INT8, len(k2), "unit", 0.2), INT8)]
    _check_direct_modes(k2, INT32, vals2, "half-hot")


@pytest.mark.parametrize("overlap", [0, 1])
@pytest.mark.parametrize("small_domain", [True, False])
def test_fused_create_reduce_vs_oracle(small_domain, overlap):
    """dtb_groupby_create_reduce: reducers evaluated inside the group() call (side-stream overlap for
    small key domains, RowIndex path otherwise) must equal separate group + reduce."""
    import torch
    from datatable_b200 import engine
    from oracle import oracle as orc
    n = 600_000
    engine.set_option("overlap_reducers", overlap)
    rng = np.random.default_rng(5 + small_domain)
    k = make_col(rng, INT32, n, "few" if small_domain else "wide", 0.03)
    v1 = make_col(rng, FLOAT64, n, "unit", 0.1)
    v2 = make_col(rng, INT16, n, "unit", 0.1)
    want_o, want_f, want_ng = orc.group([k], [0], 1)
    reds = [("sum", v1, FLOAT64), ("mean", v2, INT16), ("min", v1, FLOAT64), ("max", v2, INT16),
            ("count", v1, FLOAT64), ("nrows", None, None), ("sum", v2, INT16)]
    gb = engine.Groupby([torch.from_numpy(k).cuda()], [0], 1,
                        reducers=[(OPS[op], None if v is None else torch.from_numpy(v).cuda()) for op, v, _ in reds])
    assert gb.ngroups == want_ng
    assert np.array_equal(gb.order().cpu().numpy(), want_o)
    assert np.array_equal(gb.offsets().cpu().numpy(), want_f)
    for i, (op, v, vst) in enumerate(reds):
        got = gb.reduced(i).cpu().numpy()
        if op == "nrows":
            assert np.array_equal(got, np.diff(want_f).astype(np.int64))
        else:
            want = orc.reduce(OPS[op], v, want_o, want_f, stype=vst)
            assert_reducer_equal(got, want, op, vst, ctx=f"fused {op} small={small_domain}")
    gb.close()
    engine.set_option("overlap_reducers", 0)


def test_rows_beyond_2_pow_30():
    """n > 2^30 rows (the first look-back design was limited to 2^30): permutation + sortedness + group
    count + sum total on device-resident data, checked with engine kernels and cheap torch reductions."""
    import torch
    from datatable_b200 import engine
    torch.cuda.empty_cache()                                  # what earlier tests left cached is free HBM too
    engine.set_option("trim_scratch", 1)
    free, _ = torch.cuda.mem_get_info()
    n = 1_200_000_000
    if free < 80e9:
        pytest.skip("needs ~60 GB of free HBM")
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    k = torch.randint(-50_000, 50_000, (n,), generator=g, device="cuda", dtype=torch.int32)
    v = torch.ones(n, device="cuda", dtype=torch.float64)
    gb = engine.Groupby([k], [0], 1, reducers=[(OPS["sum"], v), (OPS["nrows"], None)])
    assert gb.ngroups == 100_000
    sums, cnt = gb.reduced(0), gb.reduced(1)
    assert torch.equal(sums.long(), cnt) and int(cnt.sum()) == n
    ks = engine.gather(k, gb.order_col())                     # keys in RowIndex order
    assert bool((ks[1:] >= ks[:-1]).all())
    offs = gb.offsets()
    assert int(offs[-1]) == n and bool((offs[1:] > offs[:-1]).all())
    heads = ks[offs[:-1].long()]
    assert torch.equal(heads, torch.arange(-50_000, 50_000, device="cuda", dtype=torch.int32))
    # stability: inside the first and the last group the row ids ascend
    o = gb.order()
    for a, b in ((0, int(offs[1])), (int(offs[-2]), n)):
        seg = o[a:b]
        assert bool((seg[1:] > seg[:-1]).all())
    del o, ks
    gb.close()


@pytest.mark.parametrize("bits", [4, 6, 7, 8])
def test_digit_width_option_gives_identical_results(bits):
    """The RowIndex / offsets must not depend on the digit width of the passes (6/7/8-ballot variants of
    the 256-bin kernel)."""
    from datatable_b200 import engine
    from oracle import oracle as orc
    rng = np.random.default_rng(bits)
    n = 300_007
    cases = [(make_col(rng, INT32, n, "unit", 0.02), INT32), (make_col(rng, FLOAT64, n, "wide", 0.02), FLOAT64),
             (make_col(rng, INT64, n, "wide", 0.0), INT64)]
    engine.set_option("radix_bits", bits)
    try:
        for k, st in cases:
            want_o, want_f, want_ng = orc.group([k], [0], 1, stypes=[st])
            got_o, got_f, got_ng = engine.group([engine.Col(k, st)], [0], 1)
            assert np.array_equal(got_o, want_o) and np.array_equal(got_f, want_f) and got_ng == want_ng
    finally:
        engine.set_option("radix_bits", 0)


def test_bucketed_multi_reducer_vs_oracle_and_plain():
    """Several reducers of one value column over a 2^12..2^20 key domain take the bucketed multi-reducer
    (dtb_bucket.cu): every value stype x every op against the oracle, and against the one-atomic-per-row path."""
    import torch
    from datatable_b200 import engine, _lib
    from oracle import oracle as orc
    rng = np.random.default_rng(991)
    n = 1_500_000
    k = rng.integers(0, 50_000, n).astype(np.int32)
    k[rng.random(n) < 0.01] = -2**31
    want_o, want_f, want_ng = orc.group([k], [0], orc.NA_FIRST)
    kd = torch.from_numpy(k).cuda()
    ops = [("sum", _lib.OP_SUM, orc.SUM), ("mean", _lib.OP_MEAN, orc.MEAN), ("min", _lib.OP_MIN, orc.MIN),
           ("max", _lib.OP_MAX, orc.MAX), ("count", _lib.OP_COUNT, orc.COUNT), ("countna", _lib.OP_COUNTNA, orc.COUNTNA)]
    for vst in (BOOL, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64):
        v = make_col(rng, vst, n, "few" if vst == BOOL else "unit", 0.1)
        vd = engine.Col(torch.from_numpy(v).cuda(), vst)
        results = {}
        for bucketed in (1, 0):
            engine.set_option("bucketed_reducers", bucketed)
            try:
                gb = engine.Groupby([kd], [0], _lib.NA_FIRST, reducers=[(op, vd) for _, op, _ in ops])
                assert gb.ngroups == want_ng
                results[bucketed] = [gb.reduced(i).cpu().numpy() for i in range(len(ops))]
                gb.close()
            finally:
                engine.set_option("bucketed_reducers", 1)
        for i, (name, _, oop) in enumerate(ops):
            want = orc.reduce(oop, v, want_o, want_f, stype=vst)
            assert_reducer_equal(results[1][i], want, name, vst, f"bucketed {name} vst={vst}")
            assert_reducer_equal(results[0][i], want, name, vst, f"plain {name} vst={vst}")


def test_group64_equals_group_and_crosses_int32():
    """dtb_group64 (ARR64 RowIndex + int64 offsets): identical to dtb_group below 2^31 rows, and a
    2^31 + 1e7-row frame (which no int32 RowIndex can address) checked by sortedness, stability,
    the permutation checksum and the Groupby invariants."""
    import torch
    from datatable_b200 import engine, _lib
    rng = np.random.default_rng(5)
    for n, sts in ((100_003, (INT32,)), (70_001, (INT64, FLOAT64))):
        cols = [make_col(rng, st, n, "few", 0.1) for st in sts]
        dcols = [engine.Col(torch.from_numpy(c).cuda(), st) for c, st in zip(cols, sts)]
        o32, f32, ng32 = engine.group(dcols, [0] * len(sts), _lib.NA_FIRST)
        o64, f64, ng64 = engine.group64(dcols, [0] * len(sts), _lib.NA_FIRST)
        assert o64.dtype == torch.int64 and f64.dtype == torch.int64 and ng64 == ng32
        assert torch.equal(o64, o32.long()) and torch.equal(f64, f32.long())
        oh, fh, ngh = engine.group64(cols, [_lib.FLAG_SORT_ONLY] * len(sts), _lib.NA_LAST)      # host buffers, sort only
        ow, _, _ = engine.group(cols, [_lib.FLAG_SORT_ONLY] * len(sts), _lib.NA_LAST)
        assert fh is None and np.array_equal(oh, ow.astype(np.int64))
    torch.cuda.empty_cache()                                  # what earlier tests left cached is free HBM too
    engine.set_option("trim_scratch", 1)
    free, _ = torch.cuda.mem_get_info()
    n = 2**31 + 10_000_000
    if free < 130 * 2**30:
        pytest.skip("needs ~110 GB of free HBM")
    g = torch.Generator(device="cuda"); g.manual_seed(9)
    k = torch.randint(0, 1000, (n,), generator=g, device="cuda", dtype=torch.int32)
    order, offs, ng = engine.group64([k], [0], _lib.NA_FIRST)
    assert ng == 1000 and order.numel() == n and int(offs[0]) == 0 and int(offs[-1]) == n
    assert bool((offs[1:] > offs[:-1]).all())
    total, prev_k, prev_o = 0, None, None
    step = 200_000_000
    for c0 in range(0, n, step):
        o = order[c0:c0 + step]
        assert int(o.min()) >= 0 and int(o.max()) < n
        ks = k[o]
        total += int(o.sum())
        ok = (ks[1:] > ks[:-1]) | ((ks[1:] == ks[:-1]) & (o[1:] > o[:-1]))
        assert bool(ok.all()), "not sorted / not stable"
        if prev_k is not None:
            assert int(ks[0]) > prev_k or (int(ks[0]) == prev_k and int(o[0]) > prev_o)
        prev_k, prev_o = int(ks[-1]), int(o[-1])
        del ks, ok
    assert total == n * (n - 1) // 2, "RowIndex is not a permutation of 0..n-1"
    # group boundaries: offsets[g] is where key g starts
    firsts = k[order[offs[:-1]]]
    assert torch.equal(firsts, torch.arange(1000, device="cuda", dtype=torch.int32))


def test_stage_keys_option_gives_identical_results():
    """Option stage_keys (materialise the normalised keys in the first count kernel, round-1 behaviour) and the
    default (normalise on the fly in count and scatter) must produce the same RowIndex / offsets."""
    import torch
    from datatable_b200 import engine, _lib
    rng = np.random.default_rng(12)
    n = 300_017
    for st in (INT8, INT16, INT32, INT64, FLOAT32, FLOAT64):
        k = make_col(rng, st, n, "wide" if st in (FLOAT32, FLOAT64) else "unit", 0.05)
        kd = engine.Col(torch.from_numpy(k).cuda(), st)
        res = []
        for sk in (0, 1):
            engine.set_option("stage_keys", sk)
            try:
                for fl, nap in (([0], _lib.NA_FIRST), ([_lib.FLAG_SORT_ONLY | _lib.FLAG_DESCENDING], _lib.NA_LAST)):
                    o, f, ng = engine.group([kd], fl, nap)
                    res.append((sk, o.cpu().numpy(), None if f is None else f.cpu().numpy()))
            finally:
                engine.set_option("stage_keys", 0)
        for a, b in zip(res[:2], res[2:]):
            assert np.array_equal(a[1], b[1]) and (a[2] is None) == (b[2] is None) and (a[2] is None or np.array_equal(a[2], b[2]))


def test_fused_stats_histogram_gives_identical_results():
    """Single-column keys: the statistics kernel's per-tile histogram of the low 8 bits folded into the first
    pass's digit counts (default) against the separate count kernel (option fuse_stats_hist = 0), and both
    against the oracle; includes keys with constant low bits (the fold does not apply) and an all-NA column."""
    import torch
    from datatable_b200 import engine, _lib
    from oracle import oracle as orc
    rng = np.random.default_rng(77)
    n = 200_003
    cols = [(st, make_col(rng, st, n, "wide" if st in (FLOAT32, FLOAT64) else "unit", 0.05))
            for st in (BOOL, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64)]
    k8 = (rng.integers(-5000, 5000, n) * 8).astype(np.int32); k8[::13] = np.iinfo(np.int32).min
    cols.append((INT32, k8))                                                     # three constant low bits
    cols.append((INT64, np.full(n, np.iinfo(np.int64).min, dtype=np.int64)))     # all NA
    cols.append((INT32, rng.integers(0, 1_000_000, n).astype(np.int32)))         # C2's shape: 20 bits, 7/7/6
    for st, k in cols:
        kd = engine.Col(torch.from_numpy(k).cuda(), st)
        for fl, nap in (([0], _lib.NA_FIRST), ([DESCENDING], _lib.NA_LAST), ([SORT_ONLY | DESCENDING], _lib.NA_FIRST)):
            res = []
            for fuse in (1, 0):
                engine.set_option("fuse_stats_hist", fuse)
                try:
                    o, f, ng = engine.group([kd], fl, nap)
                    res.append((o.cpu().numpy(), None if f is None else f.cpu().numpy()))
                finally:
                    engine.set_option("fuse_stats_hist", 1)
            assert np.array_equal(res[0][0], res[1][0]), (st, fl, nap)
            assert (res[0][1] is None) == (res[1][1] is None) and (res[0][1] is None or np.array_equal(res[0][1], res[1][1]))
            oo, of, _ = orc.group([k], fl, nap, stypes=[st])
            assert np.array_equal(res[0][0], oo), (st, fl, nap)
            if of is not None:
                assert np.array_equal(res[0][1], of)
