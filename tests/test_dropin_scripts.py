"""The reference's own scripts, unchanged, must reach mickey_b200 through their own import lines
(`from lib.models.builder import build_model`, `from config.default import cfg`).  The script test needs a checkout
of the reference and skips without one; without a GPU the script is expected to get as far as model(data) and stop at
mickey_b200's "CUDA only" error, which proves whose model class it instantiated.  The same call sequence, restated,
runs on the GPU in tests/test_gpu_dropin.py."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from mickey_b200.config import mickey_cfg
from mickey_b200.weights import synthetic_checkpoint
from oracle.ref_harness import REF_ROOT as REF
from tests.common import ROOT


def test_transforms3d_shim_roundtrip():
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    try:
        from transforms3d.quaternions import mat2quat, quat2mat, qmult, qinverse, rotate_vector
    finally:
        sys.path.pop(0)
    rng = np.random.default_rng(0)
    for _ in range(20):
        q = rng.normal(size=4); q /= np.linalg.norm(q); q = q if q[0] > 0 else -q
        R = quat2mat(q)
        assert np.allclose(R @ R.T, np.eye(3), atol=1e-12) and abs(np.linalg.det(R) - 1) < 1e-12
        assert np.allclose(mat2quat(R), q, atol=1e-10)
        v = rng.normal(size=3)
        assert np.allclose(rotate_vector(v, q), R @ v, atol=1e-12)
        assert np.allclose(qmult(q, qinverse(q)), [1, 0, 0, 0], atol=1e-12)


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "demo_inference.py")),
                    reason="needs a checkout of the reference (MICKEY_REFERENCE_ROOT): it runs the reference's own script")
def test_demo_inference_script_runs_unchanged_up_to_the_cuda_requirement(tmp_path):
    cfg = mickey_cfg("vits", 2, 4)
    (tmp_path / "config.yaml").write_text(cfg.dump())
    torch.save(synthetic_checkpoint(cfg, seed=0), tmp_path / "mickey.ckpt")
    toy = os.path.join(REF, "data", "toy_example")
    cmd = [sys.executable, "-m", "mickey_b200.run_script", os.path.join(REF, "demo_inference.py"),
           "--im_path_ref", os.path.join(toy, "im0.jpg"), "--im_path_dst", os.path.join(toy, "im1.jpg"),
           "--intrinsics", os.path.join(toy, "intrinsics.txt"), "--config", str(tmp_path / "config.yaml"),
           "--checkpoint", str(tmp_path / "mickey.ckpt")]
    env = dict(os.environ, PYTHONPATH=ROOT, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=str(tmp_path), env=env, timeout=600)
    out = r.stdout + r.stderr
    assert "Running MicKey relative pose estimation" in out, out[-2000:]          # demo_inference.py:112
    if torch.cuda.is_available():
        assert r.returncode == 0, out[-2000:]
    else:
        assert "mickey_b200 runs on CUDA only" in out, out[-2000:]
        assert "mickey_b200/model.py" in out
