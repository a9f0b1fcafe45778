"""Registry / builder / Config semantics (det3d/utils/registry.py, det3d/torchie/utils/config.py)
and: the stock reference config loads UNCHANGED and builds the same model as the shipped one."""
import os

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden, reference_config


def test_registry_semantics():
    from det3d.utils import Registry, build_from_cfg

    reg = Registry("thing")

    @reg.register_module
    class A:
        def __init__(self, x, y=2):
            self.x, self.y = x, y

    assert reg.get("A") is A and reg.get("nope") is None and reg.name == "thing"
    with pytest.raises(KeyError):
        reg.register_module(A)
    with pytest.raises(TypeError):
        reg.register_module(lambda: None)
    a = build_from_cfg(dict(type="A", x=1), reg, dict(y=5, x=7))
    assert (a.x, a.y) == (1, 5)
    assert build_from_cfg(dict(type=A, x=3), reg).y == 2
    with pytest.raises(KeyError):
        build_from_cfg(dict(type="B"), reg)
    with pytest.raises(TypeError):
        build_from_cfg(dict(type=3), reg)


def test_det3d_alias_shares_modules():
    import det3d.models.backbones.scn as a
    import det3d_b200.models.backbones.scn as b
    from det3d.models.registry import BACKBONES

    assert a is b
    assert BACKBONES.get("SpMiddleFHD") is b.SpMiddleFHD and BACKBONES.get("SpMiddleResNetFHD") is b.SpMiddleResNetFHD


def test_shipped_config_builds_second():
    from det3d.models import build_detector
    from det3d.torchie import Config

    cfg = Config.fromfile(os.path.join(ROOT, "configs", "second_kitti_car.py"))
    assert cfg.assigner.out_size_factor == 8 and cfg.test_cfg.nms.nms_pre_max_size == 1000
    with pytest.raises(AttributeError):
        cfg.model.nonexistent
    model = build_detector(cfg.model, train_cfg=None, test_cfg=cfg.test_cfg)
    sd = model.state_dict()
    # SURVEY App. A.3 index map
    assert tuple(sd["backbone.middle_conv.0.weight"].shape) == (3, 3, 3, 4, 16)
    assert tuple(sd["backbone.middle_conv.27.weight"].shape) == (3, 3, 3, 64, 64)
    assert tuple(sd["backbone.middle_conv.39.weight"].shape) == (3, 1, 1, 64, 64)
    assert "backbone.middle_conv.40.running_var" in sd and "backbone.middle_conv.0.bias" not in sd
    assert tuple(sd["bbox_head.tasks.0.conv_box.weight"].shape) == (14, 128, 1, 1)
    assert tuple(sd["neck.blocks.0.1.weight"].shape) == (128, 128, 3, 3)


@pytest.mark.parametrize("rel", [
    "examples/second/configs/kitti_car_vfev3_spmiddlefhd_rpn1_mghead_syncbn.py",
    "examples/cbgs/configs/nusc_all_vfev3_spmiddleresnetfhd_rpn2_mghead_syncbn.py",
    "examples/point_pillars/configs/kitti_point_pillars_mghead_syncbn.py",
])
def test_reference_config_loads_unchanged(rel):
    from det3d.models import build_detector
    from det3d.torchie import Config

    cfg = reference_config(rel)
    model = build_detector(cfg.model, train_cfg=None, test_cfg=cfg.test_cfg)
    if "point_pillars" in rel:
        assert type(model).__name__ == "PointPillars"
        mine = Config.fromfile(os.path.join(ROOT, "configs", "pointpillars_kitti_car.py"))
        m2 = build_detector(mine.model, train_cfg=None, test_cfg=mine.test_cfg)
        a, b = model.state_dict(), m2.state_dict()
        assert list(a) == list(b) and all(a[k].shape == b[k].shape for k in a)
        assert tuple(a["reader.pfn_layers.0.linear.weight"].shape) == (64, 9)
        assert tuple(a["neck.deblocks.2.0.weight"].shape) == (256, 128, 4, 4)
        for key in ("test_cfg", "voxel_generator", "target_assigner"):
            assert cfg[key].to_dict() == mine[key].to_dict()
        assert cfg.assigner.out_size_factor == 2
        return
    assert type(model).__name__ == "VoxelNet"
    if "kitti_car" in rel:
        mine = Config.fromfile(os.path.join(ROOT, "configs", "second_kitti_car.py"))
        m2 = build_detector(mine.model, train_cfg=None, test_cfg=mine.test_cfg)
        a, b = model.state_dict(), m2.state_dict()
        assert list(a) == list(b) and all(a[k].shape == b[k].shape for k in a)
        for key in ("test_cfg", "voxel_generator", "target_assigner"):
            assert cfg[key].to_dict() == mine[key].to_dict()
    else:
        sd = model.state_dict()
        assert tuple(sd["backbone.middle_conv.3.conv1.bias"].shape) == (16,)   # block convs carry a bias (scn.py:60-65)
        assert tuple(sd["backbone.middle_conv.20.weight"].shape) == (3, 1, 1, 128, 128)
        assert len(model.bbox_head.tasks) == 6


def test_anchors_match_reference_golden():
    from det3d.torchie import Config
    from det3d_b200.core.anchor.anchor_generator import anchors_for_tasks

    g = load_golden("anchors_kitti_car")
    cfg = Config.fromfile(os.path.join(ROOT, "configs", "second_kitti_car.py"))
    (a,) = anchors_for_tasks(cfg.target_assigner, [1408, 1600, 40], 8)
    assert a.shape == (70400, 7) and a.dtype == np.float32
    assert np.array_equal(a[g["sample_idx"]], g["sample"])
    assert np.allclose([a.astype(np.float64).sum(), (a.astype(np.float64) ** 2).sum()], g["checksum"], rtol=1e-12, atol=0)


def test_voxel_generator_properties():
    from det3d.core.input.voxel_generator import VoxelGenerator

    vg = VoxelGenerator([0.05, 0.05, 0.1], [0, -40, -3, 70.4, 40, 1], 5, max_voxels=20000)
    assert vg.grid_size.tolist() == [1408, 1600, 40] and vg.grid_size.dtype == np.int64
    assert vg.voxel_size.dtype == np.float32 and vg.point_cloud_range.dtype == np.float32
    assert vg.max_num_points_per_voxel == 5
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):   # the product path fails loudly without a GPU: no CPU fallback
            vg.generate(np.zeros((10, 4), np.float32))


def test_bn_fold_and_plan():
    from det3d_b200.models.backbones.scn import SpMiddleFHD, SpMiddleResNetFHD
    from det3d_b200.ops.spconv.fused import compile_plan

    p = compile_plan(SpMiddleFHD(num_input_features=4).middle_conv)
    assert len(p) == 14 and all(L.bn is not None and L.relu for L in p)
    p = compile_plan(SpMiddleResNetFHD(num_input_features=5).middle_conv)
    assert len(p) == 21 and sum(L.residual for L in p) == 8 and sum(L.save_identity for L in p) == 8


def test_box_coder_decode_matches_reference_golden_including_its_quirk():
    """GroundBox3dCoderTorch.decode_torch against the reference function run through the reference coder's own call
    (tests/golden/make_golden_decode.py): `linear_dim` lands in the ignored `bin_loss` slot and `norm_velo` is never
    forwarded (box_coders.py:106-109), so sizes always decode with exp() and velocities without the diagonal -- whatever the
    coder was built with.  The device predict path sets smooth_dim = norm_velo = 0 for the same reason (mg_head.py)."""
    import os
    import numpy as np
    import torch
    from det3d_b200.core.bbox.box_coders import GroundBox3dCoderTorch
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "decode_coder.npz"))
    for nd in (7, 9):
        for vec in (False, True):
            for lin in (False, True):
                key = "nd%d_vec%d_lin%d" % (nd, int(vec), int(lin))
                coder = GroundBox3dCoderTorch(linear_dim=lin, vec_encode=vec, n_dim=nd, norm_velo=True)
                assert coder.code_size == nd + (1 if vec else 0)
                got = coder.decode_torch(torch.from_numpy(g[key + "_enc"]), torch.from_numpy(g[key + "_anchors"])).numpy()
                assert got.shape == g[key + "_out"].shape
                assert np.allclose(got, g[key + "_out"], rtol=0, atol=1e-6), key
            # the flag changes nothing in the reference either
            assert np.array_equal(g["nd%d_vec%d_lin0_out" % (nd, int(vec))][:, 3:6] > 0, np.ones((257, 3), bool))
