"""Host half of the submission writer (SURVEY.md §8 f2; reference submission.py:17-68): record filtering, the text of a
line and the zip layout.  The device half (R -> quaternion, NaN filter) is tested on the GPU in tests/test_gpu_io.py."""
import json
import os
import zipfile

import numpy as np
import pytest
import torch

from mickey_b200 import submission as sub
from tests.common import ROOT


def test_pose_line_is_the_reference_format():
    """submission.py:24-29: `<query> qw qx qy qz tx ty tz inliers`, six decimals, numpy's array2string spacing."""
    p = sub.Pose("seq1/frame_00010.jpg", np.array([0.5, -0.5, 0.5, 0.5]), np.array([1.25, -0.125, 3.0], dtype=np.float32), 12.5)
    assert str(p) == "seq1/frame_00010.jpg 0.500000 -0.500000 0.500000 0.500000 1.250000 -0.125000 3.000000 12.5"
    # the lines the reference's own dataclass writes for seeded poses (tests/golden/make_reference_fixtures.py)
    with open(os.path.join(ROOT, "tests", "golden", "reference_pose_lines.json")) as f:
        cases = json.load(f)
    assert len(cases) > 30 and cases[0]["line"] == str(p)
    for c in cases:
        ours = sub.Pose(c["image_name"], np.array(c["q"]), np.array(c["t"], dtype=np.float32), c["inliers"])
        assert str(ours) == c["line"]


def test_records_filter_and_types():
    recs = np.array([[1, 0, 0, 0, 0.1, 0.2, 0.3, 7.0, 1.0],
                     [np.nan, 0, 0, 0, 0, 0, 0, 0, 0.0],          # flagged invalid by the device filter
                     [0.5, 0.5, 0.5, 0.5, 1, 2, 3, 9.25, 1.0]])
    poses = sub.records_to_poses(recs, ["a.jpg", "b.jpg", "c.jpg"])
    assert [p.image_name for p in poses] == ["a.jpg", "c.jpg"]
    assert poses[1].t.dtype == np.float32 and poses[1].inliers == 9.25
    assert str(poses[0]).split()[-1] == "7.0"


def test_pack_poses_layout():
    R = torch.arange(18, dtype=torch.float64).reshape(2, 3, 3)
    t = torch.tensor([[[1.0, 2.0, 3.0]], [[4.0, 5.0, 6.0]]])
    inl = torch.tensor([3.5, 4.5])
    packed = sub.pack_poses(R, t, inl)
    assert packed.dtype == torch.float32 and packed.shape == (2, 13)
    assert packed[1].tolist() == [9, 10, 11, 12, 13, 14, 15, 16, 17, 4, 5, 6, 4.5]


def test_records_need_the_gpu():
    from mickey_b200 import _lib
    with pytest.raises(_lib.MickeyB200Error):
        sub.poses_to_records(torch.zeros(1, 13))


def test_save_submission_zip_layout(tmp_path):
    res = {"s00001": [sub.Pose("seq1/frame_00005.jpg", np.array([1.0, 0, 0, 0]), np.array([0, 0, 1.0], dtype=np.float32), 3.0),
                      sub.Pose("seq1/frame_00010.jpg", np.array([1.0, 0, 0, 0]), np.array([0, 0, 2.0], dtype=np.float32), 4.0)],
           "s00002": []}
    out = tmp_path / "submission.zip"
    sub.save_submission(res, out)
    with zipfile.ZipFile(out) as z:
        assert sorted(z.namelist()) == ["pose_s00001.txt", "pose_s00002.txt"]
        lines = z.read("pose_s00001.txt").decode().split("\n")
        assert len(lines) == 2 and lines[1].startswith("seq1/frame_00010.jpg 1.000000 0.000000")
        assert z.read("pose_s00002.txt") == b""


def test_uint8_float_round_trip_is_exact():
    """f1: the uint8 HWC image and the reference's float CHW tensor (lib/datasets/utils.py:74) carry the same information:
    v / 255 * 255 rounds back to v for every byte, so `from_float_chw(to_float_chw(x)) == x` bit for bit."""
    from mickey_b200 import io
    x = torch.arange(256, dtype=torch.uint8).repeat(3 * 4).reshape(4, 256, 3)
    f = io.to_float_chw(x)
    assert f.shape == (3, 4, 256) and f.dtype == torch.float32 and float(f.max()) == 1.0
    assert torch.equal(io.from_float_chw(f), x)
