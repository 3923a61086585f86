"""GPU: the queries that integration/check_hook*.py send through the reference patched by integration/apply_hook.py
(options sort.b200 / sort.b200_reducers) must give, on the engine, the reference's own CPU results -- the drop-in
boundary seen from the reference's side.  The inputs are rebuilt from the scripts' seeds (helpers.hook_inputs); the
reference's answers are stored in tests/golden/golden_v4.* (tests/golden/make_golden_v4.py): small results in full,
RowIndex-sized exact ones as digests."""
import json
import os

import numpy as np
import pytest

from helpers import digest, hook_inputs

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
META = json.load(open(os.path.join(G, "golden_v4.json")))
ARR = np.load(os.path.join(G, "golden_v4.npz"))


def test_patched_reference_matches_its_own_cpu_path():
    """option sort.b200: the reference's group() through dtb_group"""
    import datatable_b200 as dt
    from datatable_b200 import f, by, sort
    DT = dt.Frame(**hook_inputs("group"))
    R = DT[:, {"s": dt.sum(f.v), "c": dt.count()}, by(f.k)]
    want = {nm: ARR[f"hook_group_sum_count__{nm}"] for nm in ("k", "s", "c")}
    assert np.array_equal(R.to_numpy("k"), want["k"]) and np.array_equal(R.to_numpy("c"), want["c"])
    assert np.allclose(R.to_numpy("s"), want["s"], rtol=1e-6, atol=0)
    R = DT[:, f.idx, sort(-f.x, na_position="last")]
    assert digest(R.to_numpy("idx")) == META["hook_group_sort_desc"]["idx"], "sort(-x) RowIndex differs"
    R = DT[:, f.idx, by(f.k), sort(f.x)]
    for nm, h in META["hook_group_by_sort"].items():
        assert digest(R.to_numpy(nm)) == h, f"by(k), sort(x): column {nm} differs"


def test_patched_reference_reducers_match_its_own_cpu_path():
    """option sort.b200_reducers: the reference's sum/mean/min/max/count through dtb_reduce, with group() on the engine
    too (the whole DT[:, reducers, by(k)])"""
    import datatable_b200 as dt
    from datatable_b200 import f, by
    DT = dt.Frame(**hook_inputs("reducers"))
    red = META["hook_reducers"]
    R = DT[:, {nm: getattr(dt, op)(f[c]) for nm, (op, c) in red.items()}, by(f.k)]
    assert np.array_equal(R.to_numpy("k"), ARR["hook_reducers__k"])
    for nm in red:
        a, c = R.to_numpy(nm), ARR[f"hook_reducers__{nm}"]
        if nm in ("sv", "mv", "mw"):
            assert np.allclose(a, c, rtol=1e-6, atol=0, equal_nan=True), nm
        else:
            assert np.array_equal(a, c, equal_nan=c.dtype.kind == "f"), nm
    assert len(red) == 10


def test_patched_reference_views_and_residency():
    """ArrayView_ColumnImpl::materialize through dtb_gather; the residency bracket (dtb_cache_begin / dtb_cache_end)
    the hook puts around evaluate(): the reducer finds the host RowIndex dtb_group just returned already in HBM"""
    import datatable_b200 as dt
    from datatable_b200 import engine, _lib, f, sort
    cols = hook_inputs("views")
    R = dt.Frame(**cols)[:, :, sort(f.k)]
    assert set(R.names) == set(META["hook_views_sorted"])
    for nm, h in META["hook_views_sorted"].items():
        assert digest(R.to_numpy(nm)) == h, f"sorted view column {nm} differs"
    _lib.check(_lib.lib.dtb_cache_begin())
    try:
        order, offsets, _ = engine.group([cols["k"]], [0], _lib.NA_FIRST)
        engine.reduce(_lib.OP_SUM, cols["v"], order, offsets)
        st = _lib.last_call_stats()
    finally:
        _lib.check(_lib.lib.dtb_cache_end())
    assert st["cache_hits"] >= 1, st
