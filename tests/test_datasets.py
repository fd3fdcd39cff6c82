"""CPU tests of the Map-free loader side (SURVEY.md §8 f3): scene parsing, pair enumeration, rank sharding, the uint8
batch variant, and item-by-item equality with the reference's own dataset on a generated tree."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest
import torch

from tests.common import ROOT

sys.path.insert(0, os.path.join(ROOT, "compat")) if __import__("importlib").util.find_spec("transforms3d") is None else None

from config.default import cfg as _cfg                              # noqa: E402
from lib.datasets.datamodules import DataModule                      # noqa: E402
from lib.datasets.mapfree import MapFreeDataset                      # noqa: E402
from lib.datasets.sampler import ShardedSequentialSampler            # noqa: E402
from lib.datasets.utils import correct_intrinsic_scale               # noqa: E402
from mickey_b200.io import to_float_chw, from_float_chw              # noqa: E402
from tools.make_synthetic_mapfree import make_tree                   # noqa: E402


@pytest.fixture(scope="module")
def tree(tmp_path_factory):
    d = tmp_path_factory.mktemp("mapfree")
    make_tree(str(d), "val", scenes=3, queries=11, seed=2, width=200, height=260, frame_step=2)
    return str(d)


def _cfg_for(tree, bs=4):
    cfg = _cfg.clone()
    cfg.merge_from_file(os.path.join(ROOT, "config", "datasets", "mapfree.yaml"))
    assert cfg.DATASET.SCENES is None                                # yacs decoding of the literal 'None'
    cfg.DATASET.DATA_ROOT = tree
    cfg.TRAINING.BATCH_SIZE, cfg.TRAINING.NUM_WORKERS = bs, 0
    return cfg


def test_pairs_format_and_uint8_variant(tree):
    cfg = _cfg_for(tree)
    ds = MapFreeDataset(cfg, "val")
    assert len(ds) == 3 * 3                                          # 11 queries, every 5th: frames 0, 10, 20
    item = ds[4]
    assert item["pair_names"] == ("seq0/frame_00000.jpg", "seq1/frame_00010.jpg") and item["scene_id"] == "s00001"
    assert item["image0"].shape == (3, 720, 540) and item["image0"].dtype == torch.float32
    assert item["pair_id"] == 5 and item["T_0to1"].shape == (4, 4)
    # K is rescaled from the native 200x260 to 540x720 (lib/datasets/utils.py:86-99)
    sx, sy = 540 / 200, 720 / 260
    assert np.allclose(item["K_color0"].numpy(), [[590 * sx, 0, 269.2 * sx + sx / 2 - 0.5], [0, 590 * sy, 352.2 * sy + sy / 2 - 0.5], [0, 0, 1]], rtol=1e-6)
    assert np.allclose(item["Kori_color0"], [[590, 0, 269.2], [0, 590, 352.2], [0, 0, 1]])
    R = item["T_0to1"][:3, :3].double()
    assert torch.allclose(R @ R.T, torch.eye(3, dtype=torch.float64), atol=1e-5)
    u8 = MapFreeDataset(cfg, "val", uint8_images=True)[4]
    assert u8["image1"].shape == (720, 540, 3) and u8["image1"].dtype == torch.uint8
    assert torch.equal(to_float_chw(u8["image1"]), item["image1"]) and torch.equal(from_float_chw(item["image1"]), u8["image1"])
    K = correct_intrinsic_scale(np.eye(3, dtype=np.float32), 2.0, 3.0)
    assert torch.allclose(K, torch.tensor([[2.0, 0, 0.5], [0, 3.0, 1.0], [0, 0, 1.0]]))


def test_rank_sharding_covers_every_pair_once(tree):
    cfg = _cfg_for(tree, bs=2)
    ds = MapFreeDataset(cfg, "val")
    for world in (1, 2, 4, 8, 16):
        seen = []
        for r in range(world):
            seen += list(ShardedSequentialSampler(ds, r, world))
        assert seen == list(range(len(ds)))
    dl = DataModule(cfg, drop_last_val=False).val_dataloader()
    names = [n for b in dl for n in zip(b["scene_id"], b["pair_names"][1])]
    assert len(names) == len(ds) and len(set(names)) == len(ds)
    with pytest.raises(NotImplementedError):
        DataModule(cfg).train_dataloader()


def test_items_equal_the_reference_dataset(tree):
    """Item-by-item equality with the reference's own dataset (lib/datasets/mapfree.py) on the same generated tree, as
    recorded by tests/golden/make_reference_fixtures.py: images by the SHA-256 of their float32 bytes (and a fixed
    sample of values), every other field in full."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_mapfree_items.json")) as f:
        theirs = json.load(f)
    ours = MapFreeDataset(_cfg_for(tree), "val")
    assert len(theirs) == len(ours)
    # the reference lists the scenes in directory order (mapfree.py:178), ours are sorted (every rank must build
    # the same pair list): match the items by (scene, pair)
    ref_items = {(b["scene_id"]["value"], b["pair_id"]["value"]): b for b in theirs}
    for i in range(len(ours)):
        a = ours[i]
        b = ref_items[(a["scene_id"], a["pair_id"])]
        assert set(a) == set(b)
        for k in a:
            if "image" in b[k]:
                img, rec = a[k].numpy(), b[k]["image"]
                assert list(img.shape) == rec["shape"] and img.dtype == np.float32, k
                assert img.reshape(-1)[rec["sample_idx"]].tolist() == rec["sample"], k
                assert hashlib.sha256(np.ascontiguousarray(img).tobytes()).hexdigest() == rec["sha256"], k
            elif "array" in b[k]:
                ref = np.array(b[k]["array"], dtype=b[k]["dtype"])
                if torch.is_tensor(a[k]):
                    assert torch.equal(a[k], torch.as_tensor(ref)), k
                else:
                    assert isinstance(a[k], np.ndarray) and np.array_equal(a[k], ref), k
            elif "relpath" in b[k]:
                assert os.path.relpath(a[k], tree) == b[k]["relpath"], k
            else:
                ref = tuple(b[k]["value"]) if b[k]["tuple"] else b[k]["value"]
                assert a[k] == ref, k
