"""GPU: bench.py --dump-outputs writes what the timed kernel step returned, identically from run to run, and --steps sets
the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from _common import s1_x0
from hop import api, cases

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["J", "J_rows", "J_star", "T_star", "instances", "status"]


def _bench(out_dir, steps, batch):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                          "--batch", str(batch), "--no-cpu-legs", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_dump_outputs_hold_the_timed_selection_and_do_not_change_between_runs(tmp_path):
    B = 20000                                    # more instances than J(T) rows are kept: the row sample is exercised
    d1 = _bench(tmp_path / "a", 2, B)
    d2 = _bench(tmp_path / "b", 3, B)
    assert d1["steps"] == d1["gpu_launches"] == 2 and d2["steps"] == d2["gpu_launches"] == 3
    a = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in NAMES}
    b = {n: np.load(tmp_path / "b" / (n + ".npy")) for n in NAMES}
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in NAMES)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    for n in NAMES:
        assert a[n].dtype == np.float64 and np.array_equal(a[n], b[n], equal_nan=True), n
    rows = a["J_rows"].astype(np.int64)
    assert len(rows) == 16384 and np.all(np.diff(rows) > 0) and rows[-1] < B
    assert np.array_equal(a["instances"], np.arange(B))
    # the public API on the same initial states (rank 0's batch) runs the same kernels: the same bits
    sel = api.select_horizon_batched(cases.make_case("Quadrotor", N=128), torch.as_tensor(s1_x0(B, seed=0), device="cuda:0"),
                                     mode=api.MODE_FAST)
    assert np.array_equal(a["T_star"], sel.T_star.cpu().numpy()) and np.array_equal(a["status"], sel.status.cpu().numpy())
    assert np.array_equal(a["J_star"], sel.J_star.cpu().numpy())
    assert np.array_equal(a["J"], sel.J.cpu().numpy()[rows], equal_nan=True)
