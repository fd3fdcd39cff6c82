"""Pins the CPU oracle (oracle/mickey_oracle.py) to outputs of the unmodified reference.

The committed fixtures were produced by tests/golden/make_golden.py and make_reference_fixtures.py from the
reference; these tests re-create the seeded inputs/weights, run the oracle and compare.
"""
import contextlib

import pytest
import torch

from mickey_b200.config import mickey_cfg
from mickey_b200.weights import synthetic_state_dict
from oracle import mickey_oracle as mo
from tests.common import GOLDEN_CASES, load_golden, synthetic_pair, rel_err, rotation_angle_deg


@contextlib.contextmanager
def _threads(n):
    """Run torch CPU ops on n threads: how many threads split a reduction moves fp32 results by a few 1e-6, and with
    them the draws of torch.multinomial."""
    old = torch.get_num_threads()
    torch.set_num_threads(n)
    try:
        yield
    finally:
        torch.set_num_threads(old)


def _run_oracle(name, inject=True):
    spec = GOLDEN_CASES[name]
    gold = load_golden(name)
    cfg = mickey_cfg(spec["variant"], spec["it_matches"], spec["it_ransac"], float16=False)
    sd = synthetic_state_dict(cfg, seed=spec["weight_seed"])
    data = synthetic_pair(spec["batch"], spec["height"], spec["width"], seed=spec["data_seed"])
    kw = {}
    if inject:
        kw = dict(outer_idx=gold["outer_idx"].long(), inner_idx=gold["inner_idx"].long())
    trace = {}
    with torch.no_grad():
        mo.model_forward(sd, data, cfg, return_inliers=True, trace=trace, **kw)
    return spec, gold, data, trace


@pytest.mark.parametrize("name", ["vits_small", "vitb_small", "vitl_small", "vits_720x540", "vitb_720x540", "vitl_720x540"])
def test_oracle_matches_reference_golden(name):
    spec, gold, data, _ = _run_oracle(name)
    st = spec["stride"]
    for k in ("kps0", "kps1", "depth_kp0", "depth_kp1", "scr0", "scr1"):
        assert rel_err(data[k], gold[k]) < 1e-5, k
    for k in ("dsc0", "dsc1"):
        assert rel_err(data[k][:, :, ::st], gold[k]) < 1e-5, k
    for k in ("scores", "kp_scores", "final_scores"):
        assert rel_err(data[k][:, ::st, ::st], gold[k]) < 1e-4, k
    assert rel_err(data["scores"].sum(-1), gold["scores_rowsum"]) < 1e-5
    # solver with the reference's own multinomial draws injected
    assert float(rotation_angle_deg(data["R"], gold["R"]).max()) < 1e-2
    assert float((data["t"] - gold["t"]).abs().max()) < 1e-3
    assert rel_err(data["inliers"], gold["inliers"]) < 1e-3
    assert [len(x) for x in data["inliers_list"]] == gold["n_inliers_list"].tolist()
    assert rel_err(data["inliers_list"][0], gold["inliers_list0"]) < 1e-4


def test_oracle_same_rng_stream_as_reference():
    """Without injection the oracle draws from torch.multinomial in the reference's order, so the
    same torch seed reproduces the reference's samples exactly."""
    name = "vits_small"
    spec, gold, _, _ = _run_oracle(name, inject=True)
    cfg = mickey_cfg(spec["variant"], spec["it_matches"], spec["it_ransac"], float16=False)
    sd = synthetic_state_dict(cfg, seed=spec["weight_seed"])
    data = synthetic_pair(spec["batch"], spec["height"], spec["width"], seed=spec["data_seed"])
    trace = {}
    torch.manual_seed(spec["rng_seed"])
    # the recorded draws are reproduced with 2 to 8 threads; 1 or 16 threads move a few of the 16384 outer draws
    with torch.no_grad(), _threads(8):
        mo.model_forward(sd, data, cfg, trace=trace)
    assert torch.equal(trace["outer_idx"].int(), gold["outer_idx"])
    assert torch.equal(trace["inner_idx"].to(torch.int16), gold["inner_idx"])


def test_oracle_matches_live_reference_stagewise():
    """compute_matches() of the reference, recorded by tests/golden/make_reference_fixtures.py, next to the oracle."""
    cfg = mickey_cfg("vits", 2, 8, float16=False)
    sd = synthetic_state_dict(cfg, seed=2)
    data = synthetic_pair(1, 154, 140, seed=9)
    ref = load_golden("reference_stagewise_vits")
    with torch.no_grad(), _threads(1):           # recorded on one thread
        ours = mo.compute_correspondences(sd, data, cfg)
    for k in ("kps0", "depth_kp0", "scr0", "dsc0", "scores", "kp_scores"):
        assert rel_err(ours[k], ref[k]) < 1e-6, k


def test_planted_pose_recovery():
    """Planted-pose KAT (SURVEY.md §8c-iii): correspondences generated from a known (R, t) with 40 %
    corrupted depths; the oracle solver must recover the pose."""
    from tests.planted import planted_problem
    cfg = mickey_cfg("vits", 8, 64)
    prob = planted_problem(n_side=(20, 16), outlier_frac=0.4, seed=0)
    torch.manual_seed(0)
    R, t, inl = mo.solve_pose(prob["final_scores"], prob["kps0"], prob["depth0"], prob["kps1"],
                              prob["depth1"], prob["K"], prob["K"], cfg)
    assert float(rotation_angle_deg(R, prob["R"]).max()) < 0.2
    assert float((t - prob["t"]).abs().max()) < 0.02
    assert float(inl.min()) > 150      # ~0.6 * 320 diagonal cells are inliers
