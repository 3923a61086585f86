"""CPU: the oracle's restatement of the grouped cumulative and window functions (tests/window_oracle.py) and of their
GtoALL evaluation under by() / sort() / i against vectors produced by the reference itself
(tests/golden/make_golden_v5.py)."""
import json
import os

import numpy as np
import pytest

import window_oracle as wo

HERE = os.path.dirname(os.path.abspath(__file__))
G = dict(np.load(os.path.join(HERE, "golden", "golden_v5.npz")))
CASES = json.load(open(os.path.join(HERE, "golden", "golden_v5.json")))["cases"]


def inputs(case):
    cols = {nm: wo.golden_array(G, case["inputs"][nm]) for nm in case["cols"]}
    return cols, {nm: int(st) for nm, st in case["cols"].items()}


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_window_oracle_matches_reference(case):
    cols, stypes = inputs(case)
    order, out = wo.evaluate(cols, stypes, case["query"])
    assert np.array_equal(wo.golden_array(G, case["r"]), cols["r"][order])
    assert [o[0] for o in out] == case["names"]
    assert [o[1] for o in out] == case["stypes"]
    for k, (name, st, vals, scale) in enumerate(out):
        assert len(vals) == case["nrows"]
        wo.assert_close(vals, wo.golden_array(G, case["outputs"][k]), st, scale, ctx=f"{case['name']}:{name}")


def test_shift_range():
    with pytest.raises(ValueError, match="too large to fit in an int32"):
        wo.shift(np.zeros(3), None, np.array([0, 3]), 2**31)
