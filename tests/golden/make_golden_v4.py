"""
Stores what the checks that used to run the reference itself at test time compared against, so that the suite
needs nothing outside the repository.  Run with the reference (an unmodified build, staged by oracle/build_ref.sh)
on the path and the reference's source tree as the argument:

    PYTHONPATH=oracle/_ref python tests/golden/make_golden_v4.py <reference source tree>

golden_v4.json / golden_v4.npz
    hook_*   the queries of integration/check_hook.py, check_hook_reducers.py and check_hook_views.py on the
             reference's own CPU path (tests/test_gpu_reference_hook.py runs them on the engine); small results
             in full, large exact ones (RowIndex-sized columns) as digests (helpers.digest)
    anchors  for each anchor string integration/apply_hook.py inserts next to: its sha256 and how often it occurs in
             the reference's file (tests/test_bench_contract.py)
jay_written.jay
    datatable_b200's Jay writer applied to the fixed-width columns of jay_v1.jay, once the reference's reader has
    opened the file and found the same frame as in jay_v1.jay (tests/test_jay.py)
"""
import hashlib
import json
import os
import sys

import numpy as np
import datatable as dt
from datatable import f, by, sort

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from helpers import digest, hook_inputs  # noqa: E402

REDUCERS = {"sv": ("sum", "v"), "mv": ("mean", "v"), "lo": ("min", "v"), "hi": ("max", "v"), "cv": ("count", "v"),
            "sw": ("sum", "w"), "mw": ("mean", "w"), "lw": ("min", "w"), "hw": ("max", "w"), "sb": ("sum", "b")}


def col(R, name):
    return R[name].to_numpy()[:, 0]


def main(ref_src):
    meta, arr = {"reference": "h2oai/datatable @ 3611640 (1.2.0a), unmodified build (oracle/build_ref.sh)"}, {}

    DT = dt.Frame(**hook_inputs("group"))
    R = DT[:, {"s": dt.sum(f.v), "c": dt.count()}, by(f.k)]
    for nm in ("k", "s", "c"):
        arr[f"hook_group_sum_count__{nm}"] = col(R, nm)
    R = DT[:, f.idx, sort(-f.x, na_position="last")]
    meta["hook_group_sort_desc"] = {"idx": digest(col(R, "idx"))}
    R = DT[:, f.idx, by(f.k), sort(f.x)]
    meta["hook_group_by_sort"] = {nm: digest(col(R, nm)) for nm in ("k", "idx")}

    DT = dt.Frame(**hook_inputs("reducers"))
    R = DT[:, {nm: getattr(dt, op)(f[c]) for nm, (op, c) in REDUCERS.items()}, by(f.k)]
    for nm in ("k",) + tuple(REDUCERS):
        arr[f"hook_reducers__{nm}"] = col(R, nm)
    meta["hook_reducers"] = REDUCERS

    DT = dt.Frame(**hook_inputs("views"))
    R = DT[:, :, sort(f.k)]
    R.materialize()
    meta["hook_views_sorted"] = {nm: digest(col(R, nm)) for nm in R.names}

    sys.path.insert(0, os.path.join(ROOT, "integration"))
    import apply_hook as ah
    anchors = {}
    for rel, names in (("src/core/sort.cc", ("INCLUDE_ANCHOR", "OPTION_ANCHOR", "REGISTER_ANCHOR", "HOOK_ANCHOR")),
                       ("src/core/expr/fexpr_reduce_unary.cc", ("RED_INCLUDE_ANCHOR", "RED_HELPER_ANCHOR", "RED_LOOP_ANCHOR")),
                       ("ci/ext.py", ("EXT_ANCHOR",))):
        text = open(os.path.join(ref_src, rel)).read()
        for nm in names:
            a = getattr(ah, nm)
            anchors[nm] = {"file": rel, "sha256": hashlib.sha256(a.encode()).hexdigest(), "count": text.count(a)}
    meta["anchors"] = anchors

    from datatable_b200 import jay
    out = os.path.join(HERE, "jay_written.jay")
    jay.open_jay(os.path.join(HERE, "jay_v1.jay"), columns=["b", "i8", "i16", "i32", "i64", "f32", "f64", "d32"],
                 device=False).to_jay(out)
    A, B = dt.fread(out), dt.fread(os.path.join(HERE, "jay_v1.jay"))[:, :8]
    assert A.names == B.names and A.stypes == B.stypes and A.to_list() == B.to_list(), "the reference reads another frame"

    with open(os.path.join(HERE, "golden_v4.json"), "w") as fh:
        json.dump(meta, fh, indent=1, sort_keys=True)
    np.savez_compressed(os.path.join(HERE, "golden_v4.npz"), **arr)


if __name__ == "__main__":
    main(sys.argv[1])
