"""Record what the unmodified reference (nianticlabs/mickey) computes for the host-side comparison tests, so that
they run without a reference checkout:

    MICKEY_REFERENCE_ROOT=<reference checkout> python tests/golden/make_reference_fixtures.py

Writes, next to this script:
  reference_configs.json           the reference's config/MicKey/{curriculum_learning,overlap_score}.yaml as parsed
                                   by yaml.safe_load (tests/test_host.py)
  reference_pose_lines.json        submission.py's Pose.__str__ on seeded poses (tests/test_submission_host.py)
  reference_mapfree_items.json     lib/datasets/mapfree.py's items on the seeded synthetic tree of tests/test_datasets.py:
                                   every field, images as a SHA-256 of their float32 bytes plus a fixed sample of values
  reference_stagewise_vits.npz     compute_matches() of the reference ViT-S model on a seeded 154x140 pair
                                   (tests/test_oracle_golden.py)
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np
import torch
import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_harness  # noqa: E402

IMAGE_SAMPLE = 64           # image values stored per image next to the digest


def configs():
    out = {}
    for name in ("curriculum_learning.yaml", "overlap_score.yaml"):
        with open(os.path.join(ref_harness.REF_ROOT, "config", "MicKey", name)) as f:
            out[name] = yaml.safe_load(f)
    return out


def pose_lines():
    src = open(os.path.join(ref_harness.REF_ROOT, "submission.py")).read()
    ns = {}
    exec("from dataclasses import dataclass\nimport numpy as np\n" + src[src.index("@dataclass"):src.index("def predict")], ns)
    rng = np.random.default_rng(0)
    cases = [("seq1/frame_00010.jpg", [0.5, -0.5, 0.5, 0.5], [1.25, -0.125, 3.0], 12.5),
             ("seq1/frame_00000.jpg", [1.0, 0.0, 0.0, 0.0], [0.0, -0.0, 0.0], 0.0)]
    for i in range(30):
        q = rng.normal(size=4)
        q = q / np.linalg.norm(q) * (1 if q[0] > 0 else -1)
        t = rng.normal(size=3) * 10.0 ** rng.integers(-7, 4)
        inl = float(rng.integers(0, 2049)) if i % 2 else float(np.float32(rng.uniform(0, 2048)))
        cases.append((f"seq1/frame_{5 * i:05d}.jpg", q.tolist(), np.float32(t).tolist(), inl))
    out = []
    for name, q, t, inl in cases:
        line = str(ns["Pose"](image_name=name, q=np.array(q), t=np.array(t, dtype=np.float32), inliers=inl))
        out.append({"image_name": name, "q": q, "t": t, "inliers": inl, "line": line})
    return out


def image_record(img, idx):
    a = np.ascontiguousarray(np.asarray(img, dtype=np.float32))
    return {"shape": list(a.shape), "sha256": hashlib.sha256(a.tobytes()).hexdigest(),
            "sample_idx": idx.tolist(), "sample": a.reshape(-1)[idx].tolist()}


def mapfree_items():
    from tests.test_datasets import _cfg_for
    from tools.make_synthetic_mapfree import make_tree
    tree = tempfile.mkdtemp()
    make_tree(tree, "val", scenes=3, queries=11, seed=2, width=200, height=260, frame_step=2)
    cfg = _cfg_for(tree)
    for k in [k for k in sys.modules if k == "lib" or k.startswith("lib.")]:
        del sys.modules[k]
    sys.path.insert(0, ref_harness.REF_ROOT)
    import lib.datasets.mapfree as ref_mapfree
    assert ref_mapfree.__file__.startswith(ref_harness.REF_ROOT)
    ds = ref_mapfree.MapFreeDataset(cfg, "val")
    idx = np.sort(np.random.default_rng(0).choice(3 * 720 * 540, IMAGE_SAMPLE, replace=False))
    items = []
    for i in range(len(ds)):
        rec = {}
        for k, v in ds[i].items():
            if k in ("image0", "image1"):
                rec[k] = {"image": image_record(v, idx)}
            elif torch.is_tensor(v) or isinstance(v, np.ndarray):
                a = np.asarray(v)
                rec[k] = {"array": a.tolist(), "dtype": str(a.dtype), "tensor": torch.is_tensor(v)}
            elif k == "scene_root":
                rec[k] = {"relpath": os.path.relpath(v, tree)}
            else:
                rec[k] = {"value": list(v) if isinstance(v, tuple) else v, "tuple": isinstance(v, tuple)}
        items.append(rec)
    return items


def stagewise():
    from mickey_b200.config import mickey_cfg
    from mickey_b200.weights import synthetic_state_dict
    from tests.common import synthetic_pair
    cfg = mickey_cfg("vits", 2, 8, float16=False)
    sd = synthetic_state_dict(cfg, seed=2)
    model = ref_harness.build_reference_model(cfg, sd, variant="vits")
    ref = synthetic_pair(1, 154, 140, seed=9)
    torch.set_num_threads(1)             # the test runs the oracle on one thread too: fp32 sums then split the same way
    with torch.no_grad():
        model.compute_matches(ref)
    return {k: ref[k].numpy() for k in ("kps0", "depth_kp0", "scr0", "dsc0", "scores", "kp_scores")}


def _write_json(name, obj):
    """One line per list element, or per key of a dict."""
    path = os.path.join(HERE, name)
    if isinstance(obj, list):
        text = "[\n" + ",\n".join(json.dumps(v) for v in obj) + "\n]\n"
    else:
        text = "{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v)}" for k, v in obj.items()) + "\n}\n"
    with open(path, "w") as f:
        f.write(text)
    print(name, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    assert ref_harness.available(), f"reference tree not found at {ref_harness.REF_ROOT} (set MICKEY_REFERENCE_ROOT)"
    _write_json("reference_configs.json", configs())
    _write_json("reference_pose_lines.json", pose_lines())
    np.savez_compressed(os.path.join(HERE, "reference_stagewise_vits.npz"), **stagewise())
    print("reference_stagewise_vits.npz", os.path.getsize(os.path.join(HERE, "reference_stagewise_vits.npz")), "bytes")
    _write_json("reference_mapfree_items.json", mapfree_items())      # last: it swaps the `lib` package for the reference's
