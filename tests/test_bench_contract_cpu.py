"""The reference arm of bench.py runs without a GPU (CPU oracle port): check the JSON contract the driver parses."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


import pytest


@pytest.mark.parametrize("ref_kind", ["auto", "port"])
def test_reference_arm_prints_one_contract_line(ref_kind):
    """auto: the unmodified reference from oracle/_ref (kind "reference") when build() staged it, else the C port."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--batch", "64", "--ref-kind", ref_kind], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "solves/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("horizon-selection solves/sec") and d["value"] > 0 and d["steps"] == 1
    staged = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "horizon_selection.py"))
    assert d["cpu_baseline"]["kind"] == ("reference" if (staged and ref_kind == "auto") else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["cpu_baseline"]["port"]["kind"] == "port" and d["cpu_baseline"]["port"]["value"] > 0
    if d["cpu_baseline"]["kind"] == "reference":
        assert d["cpu_baseline"]["T_star_reference_equals_port_on_sample"] is True
    assert d["e2e"] == {"value": d["value"], "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["dtype"] == "f64" and d["data"] == "synthetic"


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(extra, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=600,
                         cwd=tmp_path)
    assert out.returncode == 2 and "error:" in out.stderr and not os.listdir(tmp_path)


def test_hop_arm_refuses_to_run_without_a_device():
    """No CPU fallback: on a box without CUDA the product arm must fail loudly (skipped where a GPU is present)."""
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--batch", "64"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "no CUDA device" in (out.stderr + out.stdout)
