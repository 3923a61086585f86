#!/usr/bin/env python
"""
bench.py -- BASELINE.json's metric on BASELINE.json's configs.

    metric  : rows/sec of DT[:, sum(f.v), by(f.k)]  (groupby-sum) ...
    config  : C2 = 1e9 rows, int32 key with 1e6 distinct values, float64 value, 1 x B200
              (N > 1: every rank owns its own 1e9-row partition -> weak scaling; the per-group
               partials are merged with an NCCL all-reduce of the dense per-key tables)
              ... "; sort HBM GB/s vs peak": C3 (1e9-row float64 sort -> RowIndex) and C4 (2-key
              groupby, 12 reducers) are timed at N = 1 in the same run and reported under
              `other_configs` on the same JSON line.

One "step" = one pass of the hot path over one batch:
    group() -> RowIndex + Groupby offsets, then the per-group SUM reducer.

    value    device-resident inputs, CUDA-event timed, max over ranks
    e2e      the public Frame API on pinned HOST columns: H2D of k and v, the query,
             D2H of the result frame, all inside the timed region
    roofline dominant kernel (radix scatter pass): algorithmic bytes / CUDA-event time
    cpu_baseline   the reference itself (oracle/_ref, an unmodified build of /root/reference staged by
             oracle/build_ref.sh) or, where that is absent, the CPU oracle port, on a bounded sample,
             timed on this box's host cores

`--impl reference` times the CPU implementation alone and prints the same line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "rows/sec groupby-sum 1e9 int32 keys"
UNIT = "rows/s"
WORKLOAD = "C2: int32 key (1e6 distinct), float64 value, DT[:, sum(v), by(k)]"


def config_of(args, world):
    """The same dict in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "rows_per_gpu": args.rows, "groups": args.groups,
            "outputs": "RowIndex int32[n] + Groupby offsets int32[ng+1] + float64 sums[ng]",
            "l2": "inputs (12 GB/GPU) exceed L2 (126 MB); no flush needed",
            "parallelism": f"row-partitioned x{world}, NCCL all-reduce of the dense per-key partial tables" if world > 1 else "single GPU"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=1_000_000_000, help="rows per GPU (C2 = 1e9)")
    ap.add_argument("--groups", type=int, default=1_000_000)
    ap.add_argument("--e2e-steps", type=int, default=9, help="end-to-end steps (the median step is reported, every step listed)")
    ap.add_argument("--cpu-rows", type=int, default=0,
                    help="rows per CPU step; 0 = the largest of 1e7/3e7/1e8/3e8/1e9 (<= --rows) whose run fits --cpu-budget")
    ap.add_argument("--cpu-budget", type=float, default=240.0, help="seconds the whole CPU arm may take")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the C3 / C4 sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float64), see dump_outputs()")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


# ---------------------------------------------------------------------------
# clocks: nvidia-smi sampled DURING the timed region
# ---------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[1])); smax.append(float(p[2]))
            except ValueError:
                continue
            for nm, val in zip(names, p[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------
# CPU side: the reference itself when oracle/_ref holds a build of it, else the oracle port
# ---------------------------------------------------------------------------
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def have_reference():
    return os.path.exists(os.path.join(REF_DIR, "datatable", "__init__.py"))


def host_cores():
    try:
        return max(1, min(len(os.sched_getaffinity(0)), 256))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_groupby_sum(k, v, sort_new=False):
    """Returns (seconds, kind, cores, ngroups) for DT[:, sum(v), by(k)] on host arrays."""
    if have_reference():
        if REF_DIR not in sys.path:
            sys.path.insert(0, REF_DIR)
        import datatable as rdt                         # the reference, built unmodified from /root/reference
        rdt.options.sort.new = bool(sort_new)
        try:
            DT = rdt.Frame(k=k, v=v)
            t0 = time.perf_counter()
            R = DT[:, rdt.sum(rdt.f.v), rdt.by(rdt.f.k)]
            R.materialize()
            dt = time.perf_counter() - t0
            return dt, "reference", int(rdt.options.nthreads), int(R.nrows)
        finally:
            rdt.options.sort.new = False
    from oracle import oracle as orc
    orc.build()
    cores = host_cores()
    orc.set_threads(cores)                              # chunk-parallel like the reference's own sort
    try:
        t0 = time.perf_counter()
        o, f, ng = orc.group([k], [0], orc.NA_FIRST)
        orc.reduce(orc.SUM, v, o, f)
        dt = time.perf_counter() - t0
    finally:
        orc.set_threads(1)
    return dt, "port", cores, int(ng)


def host_sample(rows, groups, seed):
    rng = np.random.default_rng(seed)
    k = rng.integers(0, groups, rows, dtype=np.int32)
    v = rng.random(rows)
    return k, v


LADDER = (10_000_000, 30_000_000, 100_000_000, 300_000_000, 1_000_000_000)


def pick_cpu_rows(args, nsteps, make):
    """Largest ladder size <= args.rows whose nsteps steps fit the CPU budget.  The reference's default
    sort is far from linear in the row count (SURVEY.md 3.5: 0.3 s at 1e7 rows, 13 s at 3e7 on 8 threads),
    so every size is probed once instead of extrapolating.  Returns (rows, probes)."""
    if args.cpu_rows > 0:
        return min(args.rows, args.cpu_rows), []
    t_start = time.perf_counter()
    probes, best = [], min(args.rows, LADDER[0])
    for rows in LADDER:
        if rows > args.rows:
            break
        k, v = make(rows)
        t, kind, cores, ng = cpu_groupby_sum(k, v)
        probes.append({"rows": rows, "seconds": round(t, 3)})
        spent = time.perf_counter() - t_start
        if t * nsteps > args.cpu_budget - spent:
            break
        best = rows
        # the next probe alone (>= 3x this one) must still leave room for the run at the current size
        if spent + 3.0 * t + t * nsteps > args.cpu_budget:
            break
    return best, probes


def run_reference(args, rank, world):
    if rank != 0:
        return
    nsteps = args.steps + args.warmup
    rows, probes = pick_cpu_rows(args, nsteps, lambda r: host_sample(r, args.groups, 42))
    k, v = host_sample(rows, args.groups, 42)
    kind, cores = "port", 1
    for _ in range(args.warmup):
        cpu_groupby_sum(k, v)
    ts = []
    for _ in range(args.steps):
        t, kind, cores, ng = cpu_groupby_sum(k, v)
        ts.append(t)
    ms = 1e3 * sum(ts) / len(ts)
    value = rows / (ms / 1e3)
    why = ("the full C2 input" if rows == args.rows else
           f"bounded sample: {nsteps} steps at the next ladder size do not fit the {args.cpu_budget:.0f} s CPU budget")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32 keys / float64 sums", "data": "synthetic",
        "config": config_of(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{rows} rows of the C2 workload per step (uniform keys in [0,{args.groups})); {why}",
                         "rows_per_step": rows, "probes": probes,
                         "implementation": ("h2oai/datatable built unmodified from /root/reference (oracle/build_ref.sh), "
                                            "default options (legacy SortContext path, nthreads = all cores)") if kind == "reference"
                                           else "oracle/dt_oracle.c (pthreads port of the reference's algorithm)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------
# the B200 arm
# ---------------------------------------------------------------------------
def cuda_ms(torch, fn, reps):
    ts, r = [], None
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); r = fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return sum(ts) / len(ts), r


def other_configs(torch, engine, _lib, n, peak):
    """C3 and C4 of BASELINE.json at N = 1, device-resident, CUDA-event timed (2 warm-up + 3 timed calls each),
    each with a size-independent correctness check (the bit-exact parity runs at <= 1e8 rows are in tests/)."""
    out = {}
    g = torch.Generator(device="cuda"); g.manual_seed(1)
    # ---- C3: float64 column sort -> RowIndex (ARR32; the reference emits ARR32 below 2^31 rows, SURVEY.md mismatch 2)
    x = torch.randn(n, generator=g, device="cuda", dtype=torch.float64)
    x[::1000] = float("nan")

    def c3():
        h = engine.Groupby([x], [_lib.FLAG_SORT_ONLY], _lib.NA_FIRST)
        return h
    for _ in range(2):
        c3().close()
    ms, h = cuda_ms(torch, lambda: (c3()), 1)
    st = _lib.last_call_stats()
    xs = engine.gather(x, h.order_col())
    nn = n // 1000 + (1 if n % 1000 else 0)
    ok = bool(torch.isnan(xs[:nn]).all()) and bool((xs[nn + 1:] >= xs[nn:-1]).all())
    h.close(); del xs
    ms, _ = cuda_ms(torch, lambda: c3().close(), 3)
    alg = 12.0 * n                                           # read the 8-byte key, write the 4-byte row id
    out["C3"] = {"workload": "C3: float64 column sort (sign-flip image), N(0,1) + 0.1 % NaN -> RowIndex ARR32",
                 "rows": n, "ms_per_step": ms, "rows_per_s": n / ms * 1e3,
                 "alg_bytes_per_row": 12, "achieved_GBps": alg / ms / 1e6, "frac_of_hbm_peak": alg / ms / 1e6 / peak,
                 "key_bits": st["key_bits"], "radix_passes": st["radix_passes"], "check_sorted_nan_first": ok}
    del x
    torch.cuda.empty_cache()
    # ---- C4: (int64, int32) keys, mean/min/max/count over 3 float64 columns
    k1 = torch.randint(0, 1000, (n,), generator=g, device="cuda", dtype=torch.int64) << 33
    k2 = torch.randint(0, 1000, (n,), generator=g, device="cuda", dtype=torch.int32)
    vs = [torch.randn(n, generator=g, device="cuda", dtype=torch.float64) for _ in range(3)]
    for v in vs:
        v[::100] = float("nan")
    ops = [_lib.OP_MEAN, _lib.OP_MIN, _lib.OP_MAX, _lib.OP_COUNT]

    def c4(keep=False):
        gb = engine.Groupby([k1, k2], [0, 0], _lib.NA_FIRST, reducers=[(op, v) for v in vs for op in ops])
        res = [gb.reduced(i) for i in range(12)] if keep else None
        ng = gb.ngroups
        gb.close()
        return ng, res
    c4()
    ng, res = c4(keep=True)
    valid0 = ~torch.isnan(vs[0])
    ok = int(res[3].sum()) == int(valid0.sum())
    ok = ok and float(torch.nan_to_num(res[2], nan=-1e300).max()) == float(vs[0][valid0].max())
    ok = ok and float(torch.nan_to_num(res[1], nan=1e300).min()) == float(vs[0][valid0].min())
    tot = float((res[0] * res[3]).sum()); want = float(vs[0][valid0].sum())
    ok = ok and abs(tot - want) <= 1e-6 * max(1.0, abs(want)) * 10
    del res, valid0
    ms, _ = cuda_ms(torch, lambda: c4(), 3)
    alg = 40.0 * n                                           # keys 8 + 4, three 8-byte value columns, 4-byte row id
    out["C4"] = {"workload": "C4: by(int64 id<<33, int32 < 1000) -> 1e6 groups; mean/min/max/count over 3 float64 columns (1 % NaN)",
                 "rows": n, "ms_per_step": ms, "rows_per_s": n / ms * 1e3, "ngroups": ng,
                 "alg_bytes_per_row": 40, "achieved_GBps": alg / ms / 1e6, "frac_of_hbm_peak": alg / ms / 1e6 / peak,
                 "checks_ok": bool(ok)}
    return out


def c5_record(torch, dist, engine, _lib, ddist, rank, world, steps=3):
    """BASELINE config C5 shape at N > 1: int64 keys (1e8 distinct), float64 values, 1.25e9 rows per GPU (1e10 rows
    at N = 8), groupby-sum with the rows left where they are: local group + reduce, then the per-group partials
    (key, sum) are range-partitioned over the ranks with one NCCL all-to-all and merged.  Returns the record (rank 0)."""
    rows, G = 1_250_000_000, 100_000_000
    gen = torch.Generator(device="cuda"); gen.manual_seed(7 + rank)
    k = torch.randint(0, G, (rows,), generator=gen, device="cuda", dtype=torch.int64)
    v = torch.rand(rows, generator=gen, device="cuda", dtype=torch.float64)

    def step():
        gb = engine.Groupby([k], [0], _lib.NA_FIRST, reducers=[(_lib.OP_SUM, v)])
        part = gb.reduced(0)
        gkeys = engine.gather(k, gb.first_rows())
        gb.close()
        return ddist.merge_partials_alltoall(gkeys, part, _lib.OP_SUM)
    step()
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a2a_ms = []
    e0.record()
    for _ in range(steps):
        mk, mv = step()
        a2a_ms.append(ddist.LAST_EXCHANGE_EVENTS)
    e1.record()
    dist.barrier(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    x_ms = sum(a.elapsed_time(b) for a, b in a2a_ms) / steps
    t = torch.tensor([ms, x_ms, float(ddist.LAST_EXCHANGE_BYTES), float(mv.sum()), float(v.sum()), float(mk.numel())],
                     dtype=torch.float64, device="cuda")
    tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    ms, x_ms, bytes_max = float(tmax[0]), float(tmax[1]), float(tmax[2])
    ok = abs(float(tsum[3]) - float(tsum[4])) <= 1e-6 * abs(float(tsum[4]))
    del k, v
    torch.cuda.empty_cache()
    return {"workload": "C5 shape: int64 key (1e8 distinct), float64 value, groupby-sum over a row-partitioned frame; "
                        "local group+reduce, NCCL all-to-all of the (key, partial) lists by key range, merge",
            "rows_per_gpu": rows, "rows_total": rows * world, "ms_per_step": ms, "rows_per_s": rows * world / ms * 1e3,
            "groups_total": int(float(tsum[5])),
            "alltoall": {"bytes_sent_per_rank": bytes_max, "ms": x_ms,
                         "GBps_per_direction": bytes_max / (x_ms / 1e3) / 1e9 if x_ms > 0 else None,
                         "nvlink5_peak_GBps_per_direction": 900.0},
            "check_sums_add_up": bool(ok), "steps": steps}


def bind_to_gpu_numa_node(torch, local_rank):
    """One process per GPU: run (and first-touch the pinned host buffers) on the CPU socket the GPU hangs off,
    so that the 12 GB/step of H2D traffic does not cross the inter-socket link.  Best effort; returns the node or None."""
    try:
        props = torch.cuda.get_device_properties(local_rank)
        if hasattr(props, "pci_bus_id"):
            bdf = f"{getattr(props, 'pci_domain_id', 0):04x}:{props.pci_bus_id:02x}:{getattr(props, 'pci_device_id', 0):02x}.0"
        else:
            out = subprocess.run(["nvidia-smi", f"--id={local_rank}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                 capture_output=True, text=True, timeout=10).stdout.strip()
            bdf = out[-12:]                                       # 00000000:1B:00.0 -> 0000:1B:00.0
        node = int(open(f"/sys/bus/pci/devices/{bdf.lower()}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception:
        pass
    return None


DUMP_BYTES = 64_000_000


def dump_outputs(torch, dirname, arrays):
    """Writes the arrays a caller of the timed path receives as DIR/<name>.npy in float64, so that two builds can be
    compared output for output (the inputs come from fixed seeds).  An array too long for DUMP_BYTES in all is
    replaced by its values at fixed pseudo-random positions (seed 0), written beside it as DIR/<name>_rows.npy."""
    os.makedirs(dirname, exist_ok=True)
    cap = (DUMP_BYTES // len(arrays) - 1024) // 16           # worst case: every array sampled, values + positions
    for name, t in arrays.items():
        if t.numel() > cap:
            rows = np.unique(np.random.default_rng(0).integers(0, t.numel(), cap))
            np.save(os.path.join(dirname, f"{name}_rows.npy"), rows.astype(np.float64))
            t = t[torch.from_numpy(rows).to(t.device)]
        np.save(os.path.join(dirname, f"{name}.npy"), t.cpu().numpy().astype(np.float64))


def run_b200(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (datatable_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    numa_node = bind_to_gpu_numa_node(torch, local_rank) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import datatable_b200 as dtb
    from datatable_b200 import engine, _lib, dist as ddist
    from datatable_b200 import f, by

    n, G = args.rows, args.groups
    gen = torch.Generator(device="cuda"); gen.manual_seed(42 + rank)
    k = torch.randint(0, G, (n,), generator=gen, device="cuda", dtype=torch.int32)
    v = torch.rand(n, generator=gen, device="cuda", dtype=torch.float64)
    torch.cuda.synchronize()

    launches = [0]
    main_prof = []            # profile records of the rank's own group()+reduce call (not of the merge)
    profiling = [False]

    local_ev = []             # N > 1: CUDA events around every rank's own group()+reduce (the part before the merge)

    def step(keep=False):
        # group(): RowIndex int32[n] + Groupby offsets int32[ng+1], both left in HBM behind the handle,
        # and the SUM reducer, evaluated inside the same engine call.  keep: return the handle open
        # (--dump-outputs reads it after the timed window)
        if world > 1 and profiling[0]:
            le0 = torch.cuda.Event(enable_timing=True); le0.record()
        gb = engine.Groupby([k], [0], _lib.NA_FIRST, reducers=[(_lib.OP_SUM, v)])
        if world > 1 and profiling[0]:
            le1 = torch.cuda.Event(enable_timing=True); le1.record()
            local_ev.append((le0, le1))
        launches[0] += _lib.last_call_stats()["kernels_launched"]
        sums = gb.reduced(0)
        ng = gb.ngroups
        if world > 1:
            gkeys = engine.gather(k, gb.first_rows())
            launches[0] += 2
            gkeys, sums = ddist.merge_partials_dense(gkeys, sums, _lib.OP_SUM, key_range=(0, G - 1))   # dictionary-coded keys
            launches[0] += ddist.LAST_MERGE_LAUNCHES
        if keep:
            return gb, gkeys if world > 1 else None, ng, sums
        gb.close()
        return None, None, ng, sums

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()

    engine.set_option("profile", 1)
    profiling[0] = True
    _lib.profile_records(reset=True)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches[0] = 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps):
        out = step(keep=args.dump_outputs is not None and i == args.steps - 1)
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    engine.set_option("profile", 0)
    profiling[0] = False
    # the engine recorded CUDA events around its kernels during the timed steps; they are read only now, so
    # that no step waited for them (the dense merge at N > 1 launches none of these families)
    own = ("col_stats", "radix_count", "radix_scatter", "group_offsets_from_counts", "group_offsets", "reduce_direct", "reduce")
    main_prof.extend(r for r in _lib.profile_records(reset=True) if r[0] in own)
    if out[0] is not None:
        if rank == 0:
            arrays = {"row_index": out[0].order(), "group_offsets": out[0].offsets(), "group_sums": out[3]}
            if world > 1:
                arrays["group_keys"] = out[1]
            dump_outputs(torch, args.dump_outputs, arrays)
            del arrays
        out[0].close()
    per_rank = None
    if world > 1:
        # every rank's own time in group()+reduce, so that the line shows how much of a step is the merge and
        # the wait for the slowest rank (the driver computes the scaling efficiency from `value` alone)
        mine = torch.tensor([sum(a.elapsed_time(b) for a, b in local_ev) / max(1, len(local_ev)), ms_total / args.steps],
                            dtype=torch.float64, device="cuda")
        allr = torch.empty(2 * world, dtype=torch.float64, device="cuda")
        dist.all_gather_into_tensor(allr, mine)
        allr = allr.cpu().numpy().reshape(world, 2)
        per_rank = {"local_group_reduce_ms": [round(float(x), 3) for x in allr[:, 0]],
                    "step_ms": [round(float(x), 3) for x in allr[:, 1]]}
        t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = world * n / (ms_step / 1e3)
    ngroups = out[2]
    launches_per_step = launches[0] / args.steps

    # ---- sanity: the sums are the column total (cheap size-independent check, not timed) ----
    tot = float(out[3].sum().item())
    vsum = v.sum()
    if world > 1:
        dist.all_reduce(vsum)                   # the merged sums cover every rank's partition
    ref_tot = float(vsum.item())
    if abs(tot - ref_tot) > 1e-6 * abs(ref_tot):
        raise SystemExit(f"bench.py: group sums do not add up: {tot} vs {ref_tot}")

    # ---- roofline of the dominant kernel: the radix scatter passes of the rank's own call ------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    fam = {}
    for name, ms in main_prof:
        fam.setdefault(name, []).append(ms)
    passes = fam.get("radix_scatter", [])
    npass_step = len(passes) // max(1, args.steps)
    # algorithmic bytes of one scatter launch over n rows (32-bit keys, int32 row ids; DESIGN.md 4):
    #   first pass : read the raw key 4 (row id = position) + write (key 4 + idx 4)  = 12 B/row
    #   middle pass: read (key 4 + idx 4)                   + write (key 4 + idx 4)  = 16 B/row
    #   last pass  : read (key 4 + idx 4)                   + write idx 4            = 12 B/row
    #                (small key domain: group sizes go to the count table, the sorted keys are not written)
    pass_bytes = ([12.0 * n] + [16.0 * n] * max(0, npass_step - 2) + [12.0 * n]) if npass_step >= 2 else [8.0 * n]
    alg_bytes_launch = sum(pass_bytes) / max(1, npass_step)
    pass_ms = sum(passes) / max(1, len(passes))
    achieved = alg_bytes_launch / (pass_ms / 1e3) / 1e9 if passes else None
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "scatter_kernel_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"kernel": "scatter_kernel (radix pass)", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                "peak_source": peak_src, "launches_per_step": npass_step, "avg_launch_ms": pass_ms,
                "alg_bytes_per_launch": alg_bytes_launch}
    step_alg = 16.0 * n / (ms_step / 1e3) / 1e9          # SURVEY 8(d): key 4 + value 8 + RowIndex 4 B/row
    kernel_ms = {nm: sum(v_) / args.steps for nm, v_ in fam.items()}
    if rank == 0 and os.environ.get("DTB_BENCH_DEBUG"):
        print("kernel_ms_per_step", kernel_ms, "step", ms_step, file=sys.stderr)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32 keys / float64 sums", "data": "synthetic",
        "config": config_of(args, world),
        "ngroups_found": ngroups,
        "roofline": roofline,
        "roofline_step": {"alg_bytes_per_row": 16, "achieved": step_alg, "peak": peak, "unit": "GB/s", "frac": step_alg / peak},
        "kernel_ms_per_step": kernel_ms,
        "gpu_launches": launches_per_step * args.steps,
        "clocks": clocks,
    }
    if per_rank:
        line["per_rank"] = per_rank

    # ---- e2e: public Frame API on pinned host columns ---------------------------------------
    if not args.no_e2e:
        # N = 1: the pinned host columns are first-touched, and the copies issued, from the GPU's own NUMA node
        # (as every rank does at N > 1); the affinity is restored before the CPU baseline leg takes all the cores
        aff0 = os.sched_getaffinity(0)
        if world == 1:
            numa_node = bind_to_gpu_numa_node(torch, local_rank)
        kh = torch.empty(n, dtype=torch.int32, pin_memory=True); kh.copy_(k)
        vh = torch.empty(n, dtype=torch.float64, pin_memory=True); vh.copy_(v)
        torch.cuda.synchronize()
        DT = dtb.Frame(k=kh, v=vh)

        def e2e_step():
            R = DT[:, dtb.sum(f.v), by(f.k)]
            if world > 1:                                   # merge the per-rank result frames over NCCL
                gk = torch.from_numpy(R.to_numpy("k")).cuda()
                gs = torch.from_numpy(R.to_numpy("v")).cuda()
                gk, gs = ddist.merge_partials_dense(gk, gs, _lib.OP_SUM)
                gs.cpu()
            return R
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        e2e_each = []
        for _ in range(args.e2e_steps):
            ts = time.perf_counter()
            R = e2e_step()
            torch.cuda.synchronize()
            e2e_each.append(1e3 * (time.perf_counter() - ts))
        dt_e2e = time.perf_counter() - t0
        steps_t = torch.tensor(e2e_each, dtype=torch.float64, device="cuda")
        if world > 1:
            t = torch.tensor([dt_e2e], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt_e2e = float(t.item())
            dist.all_reduce(steps_t, op=dist.ReduceOp.MAX)          # a step takes as long as its slowest rank
        e2e_each = [float(x) for x in steps_t.cpu()]
        # the transfer alone (same pinned buffers, same copies into preallocated device buffers, no compute):
        # the floor of this leg
        kd_ = torch.empty(n, dtype=torch.int32, device="cuda"); vd_ = torch.empty(n, dtype=torch.float64, device="cuda")
        kd_.copy_(kh, non_blocking=True); torch.cuda.synchronize()
        h0 = time.perf_counter()
        for _ in range(2):
            kd_.copy_(kh, non_blocking=True); vd_.copy_(vh, non_blocking=True)
            torch.cuda.synchronize()
        h2d_only_ms = 1e3 * (time.perf_counter() - h0) / 2
        del kd_, vd_
        # The boxes of this pool share their host (memory, PCIe root) with other tenants: single steps take 1.5-9x
        # as long with nothing of ours running but the upload (scripts/e2e_timeline.py: the key column alone 159 ms
        # instead of 73).  The figure is the MEDIAN step; the mean and every step's time are reported beside it.
        e2e_mean_ms = 1e3 * dt_e2e / args.e2e_steps
        e2e_ms = sorted(e2e_each)[len(e2e_each) // 2]
        line["e2e"] = {"value": world * n / (e2e_ms / 1e3), "unit": UNIT, "ms_per_step": e2e_ms,
                       "estimator": "median step (max over ranks per step)", "mean_ms_per_step": e2e_mean_ms,
                       "value_from_mean": world * n / (e2e_mean_ms / 1e3),
                       "steps": args.e2e_steps,
                       "h2d_bytes_per_step": int(n * 12), "d2h_bytes_per_step": int(R.nrows * 12),
                       "h2d_only_ms": h2d_only_ms, "h2d_GBps": n * 12 / h2d_only_ms / 1e6,
                       "ms_each_step": [round(x, 1) for x in e2e_each],
                       "api": "datatable_b200.Frame[:, sum(f.v), by(f.k)] on pinned host columns",
                       "host_numa_binding": (f"bound to the GPU's NUMA node {numa_node} for this leg" if world == 1 else
                                             f"each rank bound to its GPU's NUMA node (rank 0: node {numa_node})")}
        del kh, vh, DT
        if world == 1:
            os.sched_setaffinity(0, aff0)

    # ---- CPU baseline on this box's host cores (rank 0, N = 1 only) ---------------------------
    # The reference's default sort collapses between 1e7 and 3e7 rows (SURVEY.md 3.5; on this pool's boxes
    # 0.25-0.4 s at 1e7 rows, 45-53 s at 3e7: `--impl reference` records the probes), so the bounded sample
    # is 1e7 rows -- the reference's best regime; the oracle port (no such collapse) is timed at 1e8 rows.
    if rank == 0 and world == 1 and not args.no_cpu:
        rows = min(n, args.cpu_rows if args.cpu_rows > 0 else LADDER[0])
        kc_all = k[:min(n, LADDER[2])].cpu().numpy(); vc_all = v[:min(n, LADDER[2])].cpu().numpy()
        kc, vc = kc_all[:rows], vc_all[:rows]
        cpu_groupby_sum(kc, vc)                              # warm-up (thread pool, page faults)
        secs, kind, cores, ng_cpu = cpu_groupby_sum(kc, vc)
        cb = {"value": rows / secs, "unit": UNIT, "cores": cores, "kind": kind, "seconds": secs,
              "sample": f"first {rows} rows of the same C2 input (keys uniform in [0,{G}))", "result_rows": ng_cpu}
        if kind == "reference":
            try:                                            # the reference's experimental sorter, same sample
                s2, _, _, ng2 = cpu_groupby_sum(kc, vc, sort_new=True)
                cb["sort_new"] = {"value": rows / s2, "seconds": s2, "result_rows": ng2,
                                  "note": "dt.options.sort.new=True; a valid baseline only if result_rows equals the default path's"}
            except Exception as e:                          # pragma: no cover
                cb["sort_new"] = {"error": str(e)[:100]}
            try:                                            # the CPU oracle port on all cores, 1e8 rows
                from oracle import oracle as orc
                orc.build(); orc.set_threads(host_cores())
                t0 = time.perf_counter()
                o_, f_, _ = orc.group([kc_all], [0], orc.NA_FIRST)
                orc.reduce(orc.SUM, vc_all, o_, f_)
                sp = time.perf_counter() - t0
                orc.set_threads(1)
                cb["port"] = {"value": kc_all.shape[0] / sp, "seconds": sp, "rows": int(kc_all.shape[0]), "cores": host_cores(),
                              "note": "oracle/dt_oracle.c (pthreads restatement), not the reference's own code"}
                del o_, f_
            except Exception as e:                          # pragma: no cover
                cb["port"] = {"error": str(e)[:100]}
        line["cpu_baseline"] = cb
        del kc_all, vc_all

    # ---- the other BASELINE configs (N = 1): C3 sort GB/s vs peak, C4 ---------------------------
    if rank == 0 and world == 1 and not args.no_extra:
        del k, v
        torch.cuda.empty_cache()
        engine.set_option("trim_scratch", 1)
        line["other_configs"] = other_configs(torch, engine, _lib, n, peak)
    # ---- strong-scaling line (N > 1): the SAME 1e9-row C2 frame split over the ranks ------------------------
    strong = None
    if world > 1 and not args.no_extra:
        ns = n // world
        ks, vs_ = k[:ns], v[:ns]

        def sstep():
            gb = engine.Groupby([ks], [0], _lib.NA_FIRST, reducers=[(_lib.OP_SUM, vs_)])
            sums = gb.reduced(0)
            gk = engine.gather(ks, gb.first_rows())
            gb.close()
            return ddist.merge_partials_dense(gk, sums, _lib.OP_SUM, key_range=(0, G - 1))
        sstep(); sstep()
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(3):
            sstep()
        s1.record()
        barrier()
        t = torch.tensor([s0.elapsed_time(s1) / 3], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        strong = {"workload": WORKLOAD + f" -- strong scaling: {ns * world} rows in total, {ns} per GPU",
                  "ms_per_step": float(t.item()), "rows_per_s": ns * world / float(t.item()) * 1e3, "steps": 3}
        del ks, vs_

    # ---- C5 shape (N > 1 only): 1.25e9 int64-key rows per GPU, all-to-all of the partials ---------------
    if world > 1 and not args.no_extra:
        del k, v
        torch.cuda.empty_cache()
        engine.set_option("trim_scratch", 1)
        try:
            c5 = c5_record(torch, dist, engine, _lib, ddist, rank, world)
        except Exception as e:                              # pragma: no cover
            c5 = {"error": str(e)[:300]}
        if rank == 0:
            line["other_configs"] = {"C5": c5, "C2_strong": strong}

    # ---- the drop-in number: the PATCHED reference's own query with the engine options off / on -----
    patched = os.path.join(ROOT, "integration", "_ref_patched")
    if rank == 0 and world == 1 and not args.no_extra and os.path.exists(os.path.join(patched, "datatable", "__init__.py")):
        torch.cuda.empty_cache()
        engine.set_option("trim_scratch", 1)
        try:
            env = dict(os.environ, PYTHONPATH=patched)
            r = subprocess.run([sys.executable, os.path.join(ROOT, "integration", "bench_hook.py")], env=env,
                               capture_output=True, text=True, timeout=600)
            js = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            line["patched_reference"] = json.loads(js[-1]) if js else {"error": (r.stderr or r.stdout)[-300:]}
        except Exception as e:                              # pragma: no cover
            line["patched_reference"] = {"error": str(e)[:200]}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
