"""bench.py --dump-outputs: what the last timed step computed, as .npy files, so that two builds run with the same
arguments can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_outputs_fit_the_budget_and_large_ones_are_a_fixed_sample():
    import bench
    big = torch.arange(5 << 20, dtype=torch.float64)           # 40 MB: more than its half of the budget
    small = torch.arange(10, dtype=torch.bfloat16).view(2, 5)
    a = bench.host_outputs({"big": big, "small": small})
    b = bench.host_outputs({"big": big.clone(), "small": small})
    assert a["small"].dtype == torch.float32 and torch.equal(a["small"], small.float())
    assert a["big"].dtype == torch.float64 and a["big"].numel() == bench.DUMP_BYTES // 2 // 8
    assert torch.equal(a["big"], b["big"])
    assert (a["big"][1:] > a["big"][:-1]).all()                 # distinct elements, in their original order
    assert sum(v.numel() * v.element_size() for v in a.values()) <= bench.DUMP_BYTES


def run_bench(workload, out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", "2",
                        "--warmup", "1", "--batch", "64", "--no-cpu-baseline", "--no-kernel-table",
                        "--dump-outputs", str(out)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
@pytest.mark.parametrize("workload,names", [("glow_cifar_kd_t32_s8", ["losses", "student_grads"]),
                                            ("glow_cifar_fwd_inv_k32", ["bpd", "x", "z"])])
def test_bench_writes_what_its_last_timed_step_computed(tmp_path, workload, names):
    out = tmp_path / "outputs"
    line = run_bench(workload, out)
    assert line["steps"] == 2
    assert sorted(os.listdir(out)) == [n + ".npy" for n in names]
    assert sum(os.path.getsize(out / (n + ".npy")) for n in names) <= 64 << 20
    arrays = {n: np.load(out / (n + ".npy")) for n in names}
    assert all(a.dtype == np.float32 and a.size > 0 and np.isfinite(a).all() for a in arrays.values())
    # a second run with the same arguments computes the same outputs, up to the order of the kernels' float atomics
    run_bench(workload, tmp_path / "again")
    for n, a in arrays.items():
        b = np.load(tmp_path / "again" / (n + ".npy"))
        err, scale = float(np.abs(a - b).max()), float(np.abs(a).max())
        assert err <= 1e-5 * scale, (n, err, scale)
    if "losses" in arrays:
        last = line["losses_last_step"]
        assert arrays["losses"].tolist() == [last[k] for k in ("nll", "kd", "perceptual", "loss")]
    else:
        assert arrays["bpd"].shape == (64,) and arrays["x"].shape == (64, 3, 32, 32)
        assert abs(float(arrays["bpd"].mean()) - line["last"]["bpd_mean"]) <= 1e-5 * abs(line["last"]["bpd_mean"])
