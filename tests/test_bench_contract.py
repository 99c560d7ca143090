"""bench.py's reference arm (the CPU restatement of the reference, the one place outside tests/ and smoke() that may
execute oracle/) prints the contract's JSON line; the product arm refuses to run without a GPU instead of falling back."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _run(args, timeout=300, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT, env=env)


def test_reference_arm_prints_the_contract_line():
    res = _run(["--impl", "reference", "--steps", "1", "--warmup", "1"])
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "frames/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("keypoint-voting frames/s") and line["value"] > 0
    assert line["steps"] == 1 and line["n_gpus"] == 1 and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] == line["e2e"]["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["gpu_launches"] == 0 and "workload" in line["config"]


def test_product_arm_needs_a_gpu():
    # the benchmark runs with every device hidden, so that this holds on a machine with GPUs too
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = _run(["--steps", "1", "--warmup", "1", "--no-cpu-baseline", "--no-e2e"], timeout=120, env=env)
    assert res.returncode != 0  # no CPU or PyTorch fallback of the product path
    assert not any(ln.startswith("{") for ln in res.stdout.splitlines())


@pytest.mark.gpu
def test_dumped_outputs_are_the_keypoints_of_the_last_timed_step(cuda_lib, tmp_path):
    """--dump-outputs writes what the timed path computed in its last step: the same call, made directly on the same
    seeded frames, gives those keypoints bit for bit."""
    import torch

    from casapose_b200 import synthetic
    from casapose_b200.pose_estimation import ransac_voting_layer_all_masks

    steps = 3
    res = _run(["--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(tmp_path)])
    assert res.returncode == 0, res.stderr[-2000:]
    assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == steps
    got = np.load(tmp_path / "keypoints.npy")
    d = synthetic.make_frames(16, 480, 640, synthetic.CONFIG_8_IDS, seed=synthetic.SEED_BASE)
    want = ransac_voting_layer_all_masks(torch.from_numpy(d["mask"]).cuda(), torch.from_numpy(d["vertex"]).cuda(), 512,
                                         seed=1000 + steps - 1).cpu().numpy()
    assert got.dtype == np.float32 and got.shape == (16, 8, 9, 2)
    assert np.array_equal(got, want, equal_nan=True)
