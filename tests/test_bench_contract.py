"""bench.py's JSON-line contract, checked on CPU through the reference arm (which needs no GPU; it
times the reference's cpu backend where oracle/_ref was built, the oracle port otherwise) and
through the pure helpers of the CUDA arm."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    sys.path.insert(0, ROOT)
    from oracle import refcpu
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                        "--steps", "1", "--warmup", "0"], cwd=ROOT, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
                "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in j, key
    assert j["impl"] == "reference" and j["unit"] == "terms/s" and j["value"] > 0
    kind = "reference" if refcpu.available() else "port"
    assert j["cpu_baseline"]["kind"] == kind and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["value"] == j["value"]
    assert "workload" in j["config"]


def test_multiplier_roofline_accounting():
    sys.path.insert(0, ROOT)
    import bench
    r = bench.imad_roofline(1 << 20, 1.63, {"sm_mhz": 1965.0})
    # 16 windows x 2^20 entries, minus one run start per non-empty bucket, x 8 muls x 72 products
    assert 9.0e9 < r["imad_wide_per_step"] < 9.7e9
    assert r["bound"] == "imad_wide" and 0.5 < r["frac"] < 1.0
    assert abs(r["peak"] - 29.2 * 148 * 1965e6) < 1e6
