"""CPU tests of the host-side logic: config tree, state-dict naming, weight packing, C-ABI exports."""
import ctypes
import json
import os
import re

import pytest
import torch
import yaml

from mickey_b200 import _lib
from mickey_b200.config import default_cfg, mickey_cfg, backbone_variant, CfgNode
from mickey_b200.engine import pack_weights, interpolate_pos_embed, sine_table_padded, make_mk_config
from mickey_b200.weights import synthetic_state_dict, synthetic_checkpoint
from tests.common import ROOT


def test_cfg_tree_access_and_merge(tmp_path):
    cfg = default_cfg()
    assert cfg.MODEL is None and cfg["MICKEY"]["DINOV2"]["FLOAT16"] is None
    y = tmp_path / "c.yaml"
    y.write_text("MODEL: 'MicKey'\nMICKEY:\n  DINOV2:\n    CHANNEL_DIM: 384\nPROCRUSTES:\n  IT_MATCHES: 8\n")
    cfg.merge_from_file(str(y))
    assert cfg.MODEL == "MicKey" and cfg.MICKEY.DINOV2.CHANNEL_DIM == 384 and cfg.PROCRUSTES.IT_MATCHES == 8
    assert backbone_variant(cfg) == "vits"
    with pytest.raises(KeyError):
        cfg.merge_from_other_cfg({"NOPE": 1})
    assert isinstance(cfg.clone(), CfgNode)


def test_reference_yaml_merges(tmp_path):
    """The reference's released configs (config/MicKey/*.yaml, stored as parsed in tests/golden) merge into ours."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_configs.json")) as fh:
        configs = json.load(fh)
    assert sorted(configs) == ["curriculum_learning.yaml", "overlap_score.yaml"]
    for f, content in configs.items():
        (tmp_path / f).write_text(yaml.safe_dump(content))
        cfg = default_cfg()
        cfg.merge_from_file(str(tmp_path / f))
        assert cfg.PROCRUSTES.NUM_SAMPLED_MATCHES == 2048
        assert backbone_variant(cfg) == "vitl"
        make_mk_config(cfg)


def test_state_dict_names_roundtrip():
    from mickey_b200.model import MickeyRelativePose
    cfg = mickey_cfg("vits", 2, 4)
    model = MickeyRelativePose(cfg)
    sd = synthetic_state_dict(cfg, seed=3)
    assert set(model.state_dict().keys()) == set(sd.keys())
    model.load_state_dict(sd, strict=True)
    k = "compute_matches.extractor.dsc_head.resblock2.bn1.running_var"
    assert torch.equal(model.state_dict()[k], sd[k])
    # a MicKey checkpoint omits the DINOv2 tensors (reference model.py:291-298); on_load_checkpoint restores them
    ck = synthetic_checkpoint(cfg, seed=4, with_backbone=False)
    assert not any("dinov2" in k for k in ck["state_dict"])
    model.on_load_checkpoint(ck)
    model.load_state_dict(ck["state_dict"], strict=True)
    assert model.e2e_Procrustes.num_samples_matches == 2048
    with pytest.raises(RuntimeError):          # no CPU fallback
        model({"image0": torch.rand(1, 3, 140, 140), "image1": torch.rand(1, 3, 140, 140),
               "K_color0": torch.eye(3)[None], "K_color1": torch.eye(3)[None]})


def test_real_checkpoint_without_dinov2_weights_is_an_error(monkeypatch):
    """A real mickey.ckpt omits the frozen DINOv2 tensors; the reference fills them from its downloaded backbone.  Without
    supplied DINOv2 weights our module only holds seeded random values, which must not be used silently."""
    from mickey_b200.model import MickeyRelativePose
    cfg = mickey_cfg("vits", 2, 4)
    ck = synthetic_checkpoint(cfg, seed=4, with_backbone=False)
    monkeypatch.setenv("MICKEY_SYNTHETIC_BACKBONE", "0")
    with pytest.raises(RuntimeError, match="RANDOM DINOv2"):
        MickeyRelativePose(cfg).on_load_checkpoint(ck)
    # supplying DINOv2 weights (native names, as in dinov2_vit*14_pretrain.pth) is the supported way
    pre = "compute_matches.extractor.dinov2_vitl14."
    dino = {k[len(pre):]: v for k, v in synthetic_state_dict(cfg, seed=9).items() if k.startswith(pre)}
    model = MickeyRelativePose(cfg, dinov2_weights=dino)
    model.on_load_checkpoint(ck)
    model.load_state_dict(ck["state_dict"], strict=True)
    assert torch.equal(model.state_dict()[pre + "blocks.3.attn.qkv.weight"], dino["blocks.3.attn.qkv.weight"])
    monkeypatch.setenv("MICKEY_SYNTHETIC_BACKBONE", "1")
    MickeyRelativePose(cfg).on_load_checkpoint(synthetic_checkpoint(cfg, seed=4, with_backbone=False))


def test_pack_weights_shapes_and_bn_fold():
    cfg = mickey_cfg("vits", 2, 4)
    sd = synthetic_state_dict(cfg, seed=0)
    pk = pack_weights(sd, cfg, "cpu")
    assert pk["patch.w"].shape == (384, 640) and pk["patch.w"].dtype == torch.float16
    assert pk["rb1.c1.w"].shape == (4 * 512, 9 * 384) and pk["rb1.sc.w"].shape == (4 * 512, 384)
    assert pk["rb3.c2.w"].shape == (4 * 128, 9 * 128) and pk["rb4k.c2.w"].shape == (3 * 64, 9 * 64)
    assert pk["att1.qkv.w"].shape == (4 * 384, 128) and pk["att2.mlp2.w"].shape == (4 * 128, 256)
    # folded conv == conv followed by eval BatchNorm, on one head
    import torch.nn.functional as F
    p = "compute_matches.extractor.det_offset.resblock2."
    x = torch.randn(1, 512, 6, 5)
    ref = F.batch_norm(F.conv2d(x, sd[p + "conv1.weight"], padding=1), sd[p + "bn1.running_mean"],
                       sd[p + "bn1.running_var"], sd[p + "bn1.weight"], sd[p + "bn1.bias"], False, eps=1e-5)
    g = 1                                            # det_offset is group 1
    w = pk["rb2.c1.w"][g * 256:(g + 1) * 256].float().reshape(256, 3, 3, 512).permute(0, 3, 1, 2)
    got = F.conv2d(x, w, padding=1) + pk["rb2.c1.b"][g * 256:(g + 1) * 256].view(1, -1, 1, 1)
    assert (got - ref).abs().max() < 2e-2 * ref.abs().max()      # fp16 weight rounding only


def test_geometry_tables():
    pos = torch.randn(1, 1 + 37 * 37, 8)
    out = interpolate_pos_embed(pos, 51, 38)
    assert out.shape == (1 + 51 * 38, 8) and torch.equal(out[0], pos[0, 0])
    pe = sine_table_padded(5, 4)
    assert pe.shape == (7 * 6, 128) and float(pe.reshape(7, 6, 128)[0].abs().max()) == 0.0


def test_abi_library_loads_and_exports_every_declared_symbol():
    """The shared library must load (no GPU needed) and export every function include/*.h declares."""
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "mickey_b200.h")).read()
    declared = set(re.findall(r"\b(mk_[a-z_0-9]+)\s*\(", header))
    declared -= {"mk_handle", "mk_config", "mk_gemm_args"}
    assert declared, "no declarations parsed"
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert b"sm_100a" in lib.mk_version()
    assert ctypes.sizeof(_lib.MkConfig) == lib.mk_sizeof_config()
    assert ctypes.sizeof(_lib.MkGemmArgs) == lib.mk_sizeof_gemm_args()


def test_hot_kernels_are_tcgen05_tma_tmem_in_sass():
    """Static evidence that the hot path is what DESIGN.md says it is: the GEMM family and the attention kernel of the
    built library issue UTCHMMA (tcgen05.mma), UTMALDG (TMA tensor loads) and LDTM (tcgen05.ld from TMEM); the SASS
    mnemonics are the ones B200_PROFILING.md lists.  Needs cuobjdump (part of the CUDA toolkit of this image)."""
    import shutil
    import subprocess
    from mickey_b200 import _lib
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    so = _lib.library_path() if hasattr(_lib, "library_path") else os.path.join(os.path.dirname(_lib.__file__), "_C", "libmickey_b200.so")
    sass = subprocess.run([exe, "-sass", so], capture_output=True, text=True, timeout=300).stdout
    per, cur = {}, None
    for line in sass.splitlines():
        if "Function :" in line:
            cur = line.split("Function :")[1].strip()
            per[cur] = {"UTCHMMA": 0, "UTCHMMA.2CTA": 0, "UTMALDG": 0, "UTMASTG": 0, "LDTM": 0, "MEMBAR.ALL.GPU": 0}
        elif cur:
            for k in per[cur]:
                if k in line:
                    per[cur][k] += 1
    hot = {n: c for n, c in per.items() if any(t in n for t in ("gemm_tc_kernel", "gemm_tc_persistent_kernel", "gemm_tc_2sm_kernel", "attention_tc_kernel"))}
    assert len(hot) >= 40
    for name, c in hot.items():
        assert c["UTCHMMA"] > 0 and c["UTMALDG"] > 0 and c["LDTM"] > 0, (name, c)
    # the cta_group::2 kernels issue the pair-wide MMA, and carry no GPU-scope fence beyond the two of the cluster set-up /
    # tear-down (a third one used to sit in the accumulator hand-back of every tile)
    two_sm = {n: c for n, c in hot.items() if "gemm_tc_2sm_kernel" in n}
    assert len(two_sm) >= 8
    for name, c in two_sm.items():
        assert c["UTCHMMA.2CTA"] > 0 and c["MEMBAR.ALL.GPU"] <= 2, (name, c)
    # matcher pass 2 (EPI_DUAL = 7) leaves through TMA tensor stores
    dual = {n: c for n, c in hot.items() if "ELi7E" in n and "gemm_tc" in n}
    assert dual and all(c["UTMASTG"] > 0 for c in dual.values()), dual
