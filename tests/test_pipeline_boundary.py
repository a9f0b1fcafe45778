"""The reference's dataset-side boundary (SURVEY 2.1 #16, 8a4): `Voxelization`, `AssignTarget`, `Reformat`, `Compose`
(det3d/datasets/pipelines/) and `collate_kitti` (det3d/torchie/parallel/collate.py:90-150) under their own names."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden, reference_config

STOCK = [
    "examples/second/configs/kitti_car_vfev3_spmiddlefhd_rpn1_mghead_syncbn.py",
    "examples/cbgs/configs/nusc_all_vfev3_spmiddleresnetfhd_rpn2_mghead_syncbn.py",
    "examples/point_pillars/configs/kitti_point_pillars_mghead_syncbn.py",
]


@pytest.mark.parametrize("rel", STOCK)
def test_stock_test_pipeline_builds(rel):
    """cfg.test_pipeline of an UNMODIFIED reference config builds through PIPELINES (every step is registered)."""
    from det3d.datasets.pipelines import Compose

    cfg = reference_config(rel)
    pipe = Compose(cfg.test_pipeline)
    names = [type(t).__name__ for t in pipe.transforms]
    assert names == ["LoadPointCloudFromFile", "LoadPointCloudAnnotations", "Preprocess", "Voxelization", "AssignTarget",
                     "Reformat"]
    vox = pipe.transforms[3]
    assert list(vox.voxel_generator.grid_size) == [int(round((cfg.voxel_generator.range[3 + j] - cfg.voxel_generator.range[j])
                                                             / cfg.voxel_generator.voxel_size[j])) for j in range(3)]
    with pytest.raises(NotImplementedError):        # training pipelines are out of scope, and say so
        Compose(cfg.train_pipeline)


def test_shipped_test_pipeline_builds_and_assigns_anchors():
    from det3d.datasets.pipelines import Compose
    from det3d.torchie import Config
    from conftest import load_golden

    cfg = Config.fromfile(os.path.join(ROOT, "configs", "second_kitti_car.py"))
    steps = [dict(type="Voxelization", cfg=cfg.voxel_generator), dict(type="AssignTarget", cfg=cfg.assigner)]
    pipe = Compose(steps)
    assign = pipe.transforms[1]
    (a,) = assign.anchors(pipe.transforms[0].voxel_generator.grid_size)
    g = load_golden("anchors_kitti_car")                 # reference-generated (tests/golden/make_golden.py)
    assert a.shape == (70400, 7) and np.array_equal(a[g["sample_idx"]], g["sample"])
    assert assign.anchors([1408, 1600, 40])[0] is a      # cached: generated once, not per sample


def _sample(i, n_vox, max_pts=5, ndim=4, n_anchor=12):
    rng = np.random.default_rng(i)
    return dict(
        metadata=dict(token=i), points=rng.random((50 + i, ndim), dtype=np.float32),
        voxels=rng.random((n_vox, max_pts, ndim), dtype=np.float32), shape=np.array([1408, 1600, 40]),
        num_points=rng.integers(1, max_pts + 1, n_vox).astype(np.int32), num_voxels=np.array([n_vox], np.int64),
        coordinates=rng.integers(0, 40, (n_vox, 3)).astype(np.int32),
        anchors=[rng.random((n_anchor, 7), dtype=np.float32), rng.random((n_anchor // 2, 7), dtype=np.float32)],
        calib=dict(rect=np.eye(4, dtype=np.float32) * (i + 1), P2=np.ones((4, 4), np.float32) * i),
    )


def _reference_collate_result():
    """The reference `collate_kitti` on the batch of test_collate_kitti_equals_reference_function, stored by
    tests/golden/make_golden_reference.py: a JSON skeleton whose tensors and arrays are the other entries."""
    g = load_golden("ref_collate_kitti")

    def build(node):
        kind, v = next(iter(node.items()))
        if kind == "dict":
            return {k: build(x) for k, x in v.items()}
        if kind == "list":
            return [build(x) for x in v]
        if kind == "tensor":
            return torch.from_numpy(g[v])
        return g[v] if kind == "ndarray" else v

    return build(json.loads(str(g["skeleton"])))


def _same(a, b):
    if isinstance(a, dict):
        return set(a) == set(b) and all(_same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    if torch.is_tensor(a):
        return torch.is_tensor(b) and a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b)
    if isinstance(a, np.ndarray):
        return isinstance(b, np.ndarray) and a.dtype == b.dtype and np.array_equal(a, b)
    return a == b


def test_collate_kitti_equals_reference_function():
    from det3d.torchie.parallel import collate_kitti

    batch = [_sample(i, n) for i, n in enumerate((7, 0, 13))]
    want = _reference_collate_result()
    got = collate_kitti(batch)
    assert set(got) == set(want)
    for k in want:
        assert _same(got[k], want[k]), k
    assert got["coordinates"][:, 0].tolist() == [0] * 7 + [2] * 13
    with pytest.raises(NotImplementedError):
        collate_kitti([dict(labels=[np.zeros(3)])])


def test_collate_kitti_batch_index_and_shapes():
    from det3d.torchie.parallel import collate_kitti

    got = collate_kitti([_sample(i, n) for i, n in enumerate((4, 6))])
    assert got["voxels"].shape == (10, 5, 4) and got["coordinates"].shape == (10, 4) and got["points"].shape[1] == 5
    assert got["coordinates"][:, 0].tolist() == [0] * 4 + [1] * 6
    assert got["num_voxels"].tolist() == [4, 6] and got["num_voxels"].dtype == torch.int64
    assert [tuple(a.shape) for a in got["anchors"]] == [(2, 12, 7), (2, 6, 7)]
    assert got["calib"]["rect"].shape == (2, 4, 4) and len(got["metadata"]) == 2 and got["shape"].shape == (2, 3)


@pytest.mark.gpu
def test_pipeline_steps_to_detections():
    """KITTI .bin on disk -> stock-style test pipeline -> collate_kitti -> VoxelNet forward; equals the fused serving
    path (InferencePipeline.infer_host), and collate_kitti_device equals collate_kitti of the per-sample outputs."""
    import tempfile

    from det3d.datasets.pipelines import Compose
    from det3d.models import build_detector
    from det3d.torchie import Config
    from det3d.torchie.parallel import collate_kitti, collate_kitti_device
    from det3d_b200.apis import InferencePipeline
    from det3d_b200.utils.synthetic import demo_weights_, lidar_like_cloud

    cfg = Config.fromfile(os.path.join(ROOT, "configs", "second_kitti_car.py"))
    torch.manual_seed(0)
    model = demo_weights_(build_detector(cfg.model, train_cfg=None, test_cfg=cfg.test_cfg).eval(), 0)
    serve = InferencePipeline(cfg, model=model, device="cuda")
    val_pre = dict(mode="val", shuffle_points=False, remove_environment=False, remove_unknown_examples=False)
    steps = [dict(type="LoadPointCloudFromFile"), dict(type="LoadPointCloudAnnotations", with_bbox=True),
             dict(type="Preprocess", cfg=val_pre), dict(type="Voxelization", cfg=cfg.voxel_generator),
             dict(type="AssignTarget", cfg=cfg.assigner), dict(type="Reformat")]
    pipe = Compose(steps)
    clouds = [lidar_like_cloud(6000 + 700 * i, cfg.voxel_generator.range, 4, 20 + i) for i in range(3)]
    examples = []
    with tempfile.TemporaryDirectory() as tmp:
        for i, c in enumerate(clouds):
            path = os.path.join(tmp, "%06d.bin" % i)
            c.tofile(path)
            info = dict(point_cloud=dict(velodyne_path=path, num_features=4),
                        calib=dict(R0_rect=np.eye(4, dtype=np.float32), Tr_velo_to_cam=np.eye(4, dtype=np.float32),
                                   P2=np.eye(4, dtype=np.float32)))
            res = dict(lidar=dict(type="lidar", points=None), metadata=dict(image_prefix=tmp, num_point_features=4, token=i),
                       calib=None, cam={}, mode="val")
            ex, _ = pipe(res, info)
            examples.append(ex)
    assert examples[0]["voxels"].shape[1:] == (5, 4) and examples[0]["num_voxels"].dtype == np.int64
    batch = collate_kitti(examples)
    dev_batch = collate_kitti_device(clouds, pipe.transforms[3], anchors=pipe.transforms[4].anchors([1408, 1600, 40]))
    for k in ("voxels", "coordinates", "num_points", "num_voxels"):
        assert torch.equal(dev_batch[k].cpu(), batch[k]), k               # fused collate == reference-style collate
    example = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in batch.items()}
    example["anchors"] = [a.cuda() for a in batch["anchors"]]
    example["shape"] = batch["shape"]
    with torch.no_grad():
        out = model.cuda()(example, return_loss=False)
    ref = serve.unpack(serve.infer_host([torch.from_numpy(c) for c in clouds]))
    assert len(out) == 3
    for o, r in zip(out, ref):
        assert o["box3d_lidar"].shape[0] == r["box3d_lidar"].shape[0] >= 5
        assert torch.allclose(o["box3d_lidar"].cpu(), r["box3d_lidar"], atol=1e-4)
        assert torch.allclose(o["scores"].cpu(), r["scores"], atol=1e-5)
