#!/usr/bin/env python
"""
Grouped cumulative / window functions at the C2 shape, device-resident: N rows (default 1e9), int32 keys in
[0, 1e6) (~1000 rows per group), float64 `v`, int64 `w`.

  * end to end: DT[:, cumsum(f.v), by(f.k)] per step (group() + window + by-column gather), CUDA events, median of
    --steps after --warmup;
  * the window call alone over a fixed RowIndex / Groupby, for cumsum (float64), cummax (int64), shift(1), cumcount
    and cumsum without by (one group: every row goes through the fix-up), next to dtb_gather of the same column
    through the same RowIndex, the yardstick: the scan moves the same bytes plus the leading-segment fix-up;
  * per-kernel times from the engine's "profile" option (window_scan / window_carry / window_fixup / window_shift /
    window_count), in a separate pass;
  * self-checks at full size on the timed outputs: the last cumsum of every group equals sum() of the group, and the
    last cumcount + 1 equals count().

Algorithmic traffic of a window kernel: 20 B/row (order 4 + value 8 + out 8).  The share of 7.7 TB/s (HBM3e, HGX B200
data sheet, one GPU) is reported, but the bound is the random 8-byte gather v[order[p]] (one 32-byte sector per
row), not the bytes.  Writes profiles/r4_window_n1.json (--out).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import datatable_b200 as d  # noqa: E402
from datatable_b200 import engine, _lib, f, by  # noqa: E402

PEAK_BPS = 7.7e12


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), [round(t, 4) for t in ts]


def profiled(fn):
    engine.set_option("profile", 1)
    _lib.profile_records(reset=True)
    fn()
    torch.cuda.synchronize()
    recs = _lib.profile_records(reset=True)
    engine.set_option("profile", 0)
    out = {}
    for name, ms in recs:
        if name.startswith("window"):
            out[name] = round(out.get(name, 0.0) + ms, 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=float, default=1e9)
    ap.add_argument("--keys", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_window_n1.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_window.py needs a CUDA device")
    n = int(args.rows)
    gpu, power = gpu_info()
    g = torch.Generator(device="cuda").manual_seed(1)
    k = torch.randint(0, args.keys, (n,), dtype=torch.int32, device="cuda", generator=g)
    v = torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    w = torch.randint(-2**40, 2**40, (n,), dtype=torch.int64, device="cuda", generator=g)
    DT = d.Frame({"k": k, "v": v, "w": w})

    res = {"gpu": gpu, "power_limit": power, "rows": n, "keys": args.keys, "steps": args.steps, "warmup": args.warmup,
           "bytes_per_row": 20, "peak_bps": PEAK_BPS,
           "bound": "random 8-byte gather v[order[p]] (one 32-byte sector per row), not the 20 algorithmic bytes"}
    ms, ts = timed(lambda: DT[:, d.cumsum(f.v), by(f.k)], args.steps, args.warmup)
    res["e2e_cumsum_by_ms"] = {"median": round(ms, 4), "all": ts}

    order, offsets, ng = engine.group([k])
    res["ngroups"] = int(ng)
    one = torch.tensor([0, n], dtype=torch.int32, device="cuda")
    calls = {
        "cumsum_f64": lambda: engine.window(_lib.WIN_CUMSUM, v, order, offsets),
        "cummax_i64": lambda: engine.window(_lib.WIN_CUMMAX, w, order, offsets),
        "shift1_f64": lambda: engine.window(_lib.WIN_SHIFT, v, order, offsets, 1),
        "cumcount": lambda: engine.window(_lib.WIN_CUMCOUNT, None, order, offsets),
        "cumsum_f64_noby": lambda: engine.window(_lib.WIN_CUMSUM, v, None, one),
        "gather_f64": lambda: engine.gather(v, order),
    }
    kern = {}
    for name, fn in calls.items():
        ms, ts = timed(fn, args.steps, args.warmup)
        entry = {"median_ms": round(ms, 4), "all": ts}
        if name != "cumcount":
            entry["gbps_20B"] = round(20 * n / (ms * 1e-3) / 1e9, 1)
            entry["share_of_7.7TBs"] = round(20 * n / (ms * 1e-3) / PEAK_BPS, 3)
        if name != "gather_f64":
            entry["kernels_ms"] = profiled(fn)
        kern[name] = entry
    res["window_calls"] = kern
    res["cumsum_over_gather"] = round(kern["cumsum_f64"]["median_ms"] / kern["gather_f64"]["median_ms"], 3)

    # self-checks on the timed outputs
    cs = engine.window(_lib.WIN_CUMSUM, v, order, offsets)
    ends = (offsets[1:] - 1).long()
    sums = engine.reduce(_lib.OP_SUM, v, order, offsets)
    asum = engine.reduce(_lib.OP_SUM, v.abs(), order, offsets)
    ok_sum = bool(((cs[ends] - sums).abs() <= 1e-9 * asum).all())
    cc = engine.window(_lib.WIN_CUMCOUNT, None, order, offsets)
    ok_cnt = bool(torch.equal(cc[ends] + 1, (offsets[1:] - offsets[:-1]).long()))
    cs1 = engine.window(_lib.WIN_CUMSUM, v, None, one)
    ok_one = bool(abs(cs1[-1].item() - v.sum().item()) <= 1e-9 * v.abs().sum().item())
    res["self_checks"] = {"group_end_equals_sum": ok_sum, "cumcount_end_plus1_equals_count": ok_cnt,
                          "one_group_end_equals_sum": ok_one}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))
    if not (ok_sum and ok_cnt and ok_one):
        raise SystemExit("self-check failed")


if __name__ == "__main__":
    main()
