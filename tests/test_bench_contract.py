"""bench.py contract: the reference arm prints exactly one JSON line on stdout with the keys its readers
expect; the product arm refuses to run without a GPU instead of falling back to the oracle; on the GPU, --steps sets
the number of timed steps and --dump-outputs writes the same outputs from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-batch", "2"], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("dual-view SSP pairs/sec") and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["steps"] == 1 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--no-cpu-baseline"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode != 0 and r.stdout.strip() == ""          # no line, no CPU fallback


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       cwd=ROOT, timeout=600)
    assert r.returncode == 2 and "--steps" in r.stderr and r.stdout == ""


@pytest.mark.gpu
def test_steps_and_dump_outputs(tmp_path):
    """Two runs of the same six steps, split 4 warm-up + 2 timed and 3 + 3: the timed launches scale with --steps, and
    the dumps after the sixth step agree up to the order of floating-point sums."""
    runs = []
    for steps, warmup in ((2, 4), (3, 3)):
        d = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                            "--no-e2e", "--no-cpu-baseline", "--no-eager-baseline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, cwd=ROOT, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout)
        assert line["steps"] == steps
        files = sorted(os.listdir(d))
        assert files == ["result.npy", "state_norms.npy", "state_sample.npy"]
        assert sum(os.path.getsize(d / f) for f in files) <= 64 << 20
        runs.append((line, {f[:-4]: np.load(d / f) for f in files}))
    (l2, a), (l3, b) = runs
    assert l2["gpu_launches"] > 0 and l2["gpu_launches"] * 3 == l3["gpu_launches"] * 2
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and a[k].shape == b[k].shape, k
    assert a["state_sample"].size == 1 << 23
    np.testing.assert_allclose(a["result"], b["result"], rtol=1e-3)
    # the backward reductions use atomics, so runs differ: Adam moves an element whose gradient is rounding noise by up
    # to 2 lr (2e-4) a step, in either direction.  A step more or less would move most elements by about lr (1e-4).
    d = np.abs(a["state_sample"] - b["state_sample"])
    assert d.max() <= 6 * 2e-4 and d.mean() <= 1e-5, (d.max(), d.mean())
    assert np.abs(a["state_norms"] - b["state_norms"]).max() <= 6 * 2e-4
