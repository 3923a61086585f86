"""CPU: the parts of bench.py and integration/ that run without a GPU keep their contracts."""
import hashlib
import json
import os
import subprocess
import sys


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU leg: oracle port on all host threads) prints ONE JSON line with
    the keys the driver reads."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--cpu-rows", "300000"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"].startswith("rows/sec groupby-sum")
    assert j["unit"] == "rows/s" and j["higher_is_better"] is True and j["value"] > 0
    cb = j["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == j["value"] and cb["sample"]
    assert j["e2e"]["value"] == j["value"] and j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0
    assert j["steps"] == 1 and "workload" in j["config"]


def test_hook_script_anchors_match_the_reference():
    """integration/apply_hook.py inserts next to short anchor strings: each must occur exactly once in the
    reference revision the goldens were generated from (recorded by tests/golden/make_golden_v4.py: the anchor's
    sha256 and its count in the reference's file), and the script must refuse to modify the reference's own tree."""
    sys.path.insert(0, os.path.join(ROOT, "integration"))
    try:
        import apply_hook as ah
    finally:
        sys.path.pop(0)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "integration", "apply_hook.py"), "/root/reference"],
                       capture_output=True, text=True)
    assert r.returncode != 0 and "refusing" in (r.stdout + r.stderr)
    with open(os.path.join(ROOT, "tests", "golden", "golden_v4.json")) as fh:
        recorded = json.load(fh)["anchors"]
    for name in ("INCLUDE_ANCHOR", "OPTION_ANCHOR", "REGISTER_ANCHOR", "HOOK_ANCHOR",
                 "RED_INCLUDE_ANCHOR", "RED_HELPER_ANCHOR", "RED_LOOP_ANCHOR", "EXT_ANCHOR"):
        rec = recorded[name]
        assert hashlib.sha256(getattr(ah, name).encode()).hexdigest() == rec["sha256"], \
            f"{name} changed since it was checked against the reference (tests/golden/make_golden_v4.py)"
        assert rec["count"] == 1, f"{name} occurs {rec['count']} times in the reference's {rec['file']}"
