"""Checks of the bench.py contract.  Without a GPU: the reference arm (``--impl reference``: the C port of the reference
sampler on the host cores) prints exactly one JSON line with the agreed keys, and the GPU arm refuses to run without CUDA
instead of falling back to the CPU.  On the GPU: ``--dump-outputs`` writes the same outputs from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample", "32"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "stn_glimpses_per_sec_fwd_bwd" and d["unit"] == "glimpses/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == dict(value=d["value"], unit="glimpses/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    assert "workload" in d["config"]


def test_gpu_arm_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        return                                   # on the GPU box this arm is exercised for real
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-e2e", "--no-cpu", "--no-train"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode != 0
    assert not [l for l in p.stdout.splitlines() if l.startswith("{")]       # no number without a GPU


def test_dump_outputs_is_refused_outside_the_gpu_arm(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode != 0 and "--dump-outputs" in p.stderr
    assert not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_are_the_same_from_run_to_run(cuda_device, tmp_path):
    """``--dump-outputs DIR``: the six arrays the timed step returns (read glimpse, dU, dtheta; written canvas, dW, dtheta) for
    every image of a small batch, float32, identical over two runs with the same arguments; ``--steps`` sets the timed steps."""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--canvas", "50", "--glimpse", "28",
           "--batch", "300", "--no-e2e", "--no-cpu", "--no-train"]
    shapes = dict(read_out=(300, 28, 28, 1), read_dU=(300, 50, 50, 1), read_dtheta=(300, 6),
                  write_out=(300, 50, 50, 1), write_dU=(300, 28, 28, 1), write_dtheta=(300, 6))
    runs = []
    for k in range(2):
        out = tmp_path / str(k)
        p = subprocess.run(cmd + ["--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-2000:]
        d = json.loads(p.stdout.strip().splitlines()[-1])
        assert d["steps"] == 2 and d["gpu_launches"] == 4 * 8 * 2
        assert sorted(os.listdir(out)) == sorted(n + ".npy" for n in shapes)
        runs.append({n: np.load(out / (n + ".npy")) for n in shapes})
    for n, shape in shapes.items():
        a, b = runs[0][n], runs[1][n]
        assert a.dtype == np.float32 and a.shape == shape and np.all(np.isfinite(a)), n
        assert np.array_equal(a, b), n
    assert np.abs(runs[0]["read_dtheta"]).max() > 0 and not np.array_equal(runs[0]["read_dtheta"], runs[0]["write_dtheta"])
