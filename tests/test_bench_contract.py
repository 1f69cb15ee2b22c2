"""bench.py contract: the reference arm runs without a GPU and prints ONE JSON line with the keys a caller
reads; the GPU arm refuses to run without a device instead of falling back; on the GPU, --dump-outputs
writes the same outputs on every run."""
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in j, key
    assert j["impl"] == "reference" and j["dtype"] == "u8" and j["scaling"] == "weak" and j["vs_baseline"] is None
    assert j["unit"] == "GiB/s" and j["value"] > 0 and j["higher_is_better"] is True
    assert "workload" in j["config"] and "model" not in j["config"]
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == j["value"] and cb["sample"]
    assert j["e2e"] == {"value": j["value"], "unit": j["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_gpu_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--no-cpu"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0                      # no device: an error, never a CPU fallback
    assert not [l for l in out.stdout.splitlines() if l.startswith("{")]


@pytest.mark.gpu
def test_dump_outputs_repeat_and_carry_their_crcs(tmp_path):
    """--dump-outputs: two runs with the same arguments write identical float arrays within 64 MB, --steps is the timed
    step count, and the dumped parity bytes are the ones the fused kernel checksummed."""
    k, m, steps = 12, 4, 2
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--stripes", "16", "--steps", str(steps),
                              "--warmup", "1", "--no-cpu", "--no-e2e", "--no-extra", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        j = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert j["steps"] == steps and j["gpu_launches"] % steps == 0 and j["gpu_launches"] > 0
        dumps.append({p.stem: np.load(p) for p in (tmp_path / run).glob("*.npy")})
    a, b = dumps
    assert sorted(a) == sorted(b) == ["crc32", "parity", "stripe_ids"]
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for name in a:
        assert a[name].dtype in (np.float32, np.float64) and np.array_equal(a[name], b[name]), name
    ids = a["stripe_ids"].astype(int)
    assert a["parity"].shape[:2] == (len(ids), m) and a["crc32"].shape == (16, k + m)
    for row, s in enumerate(ids):
        for r in range(m):
            assert zlib.crc32(a["parity"][row, r].astype(np.uint8).tobytes()) == int(a["crc32"][s, k + r])
