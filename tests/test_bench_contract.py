"""The bench.py contract: one JSON line with the keys the driver reads, for both arms."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def run_bench(*args, timeout=900):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    """`bench.py --impl reference`: the reference's CPU matchNNR on the host cores (no GPU needed)."""
    d = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-seconds", "2")
    assert BASE_KEYS <= set(d), sorted(BASE_KEYS - set(d))
    assert d["impl"] == "reference" and d["metric"] == "descriptor_pairs_per_s" and d["unit"] == "pairs/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


@pytest.mark.gpu
def test_b200_arm_line(tmp_path):
    """`bench.py` on the GPU (short: no side metrics, no CPU baseline): roofline, e2e, clocks and launch count, and the
    outputs of the last timed step written by --dump-outputs."""
    import numpy as np
    d = run_bench("--steps", "3", "--warmup", "3", "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path))
    m12, count = np.load(tmp_path / "m12.npy"), np.load(tmp_path / "count.npy")
    assert m12.dtype == np.float64 and m12.shape == (6400,) and count.dtype == np.float64 and count.shape == (1,)
    assert int(count[0]) == d["matches_last_step"] == int((m12 >= 0).sum()) > 0
    assert (m12 < d["config"]["db_rows"]).all() and (m12 == np.round(m12)).all()
    assert (BASE_KEYS - {"cpu_baseline"}) <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 3 and d["value"] > 1e11
    assert d["gpu_launches"] > 0
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["frac"] > 0
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 6400 * 32 and e["d2h_bytes_per_step"] == 6400 * 4 + 4
    assert abs(e["value"] - d["value"]) / d["value"] < 0.2      # measured separately, host copies included
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert "workload" in d["config"] and "model" not in d["config"]
