"""Rotated IoU / NMS on the GPU.
 * XYXYR path: BIT-EXACT against the reference CUDA kernel itself -- IoU matrices and keep lists, through the
   committed fixtures it produced (tests/golden/iou3d_*.npz, ref_iou3d_kernel.npz; make_golden_gpu.py, make_golden_iou3d_ref.py).
 * XYWLR path (rotate_nms_cc semantics): vs the C oracle (IoU within 1e-4, keep list equal).
 * 100k-box stress (BASELINE config 5): keep list equal to the reference kernel's + invariants.
"""
import glob
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, array_digest, load_golden
from det3d_b200.utils.synthetic import nms_boxes_xyxyr, xyxyr_to_xywlr

pytestmark = pytest.mark.gpu


def _sorted_boxes(n, seed, clustered):
    boxes, scores = nms_boxes_xyxyr(n, seed, clustered)
    order = np.argsort(-scores, kind="stable")
    return boxes[order], scores[order]


def _ref_golden():
    """Outputs of the reference iou3d kernel (det3d/ops/iou3d/src/iou3d_kernel.cu) on the inputs built below."""
    return load_golden("ref_iou3d_kernel")


def _iou_inputs(seed, clustered, n):
    boxes, _ = nms_boxes_xyxyr(n, seed, clustered, extent=30.0)
    return (np.concatenate([boxes[: n // 2], _degenerate_boxes()]), np.concatenate([boxes[n // 2:], _degenerate_boxes()]))


def _iou_bits(iou):
    """int32 view of an IoU matrix with every NaN as one bit pattern (NaN payloads are not part of the result)."""
    x = iou.cpu().numpy()
    bits = x.view(np.int32).copy()
    bits[np.isnan(x)] = 0x7FC00000
    return bits


def _keep_key(n, clustered, thr):
    return "n%d_c%d_t%02d" % (n, int(clustered), round(thr * 100))


def _stress_boxes():
    boxes, _ = _sorted_boxes(100_000, 0, clustered=False)
    boxes[:, :4] = boxes[:, :4] * np.float32(3.16)     # 1 km x 1 km would be trivial; keep it dense: 316 m x 316 m
    return boxes


def _degenerate_boxes():
    b = np.array([[0, 0, 2, 4, 0.3], [0, 0, 2, 4, 0.3], [0, 0, 2, 4, -0.3], [1, 1, 1, 1, 0.0], [0, 0, 2, 0, 0.5],
                  [0, 0, 1, 1, 0.0], [0, 0, 1, 1, np.pi / 4], [1, 0, 2, 1, 0.0], [0.5, 0.5, 1.5, 1.5, np.pi / 2],
                  [0, 0, 1e-4, 1e-4, 1.0], [-5, -5, 5, 5, 3.0], [100, 100, 101, 102, -2.0],
                  [0, 0, 2, 4, 1e-7], [0, 0, 2, 4, np.pi], [0, 0, 2, 4, 100.0], [0, 0, 2, 4, 1e5]], np.float32)
    return b


@pytest.mark.parametrize("overlap", [False, True])
def test_iou_matrix_bit_exact_vs_reference_kernel(overlap):
    g = _ref_golden()
    from det3d.ops.iou3d import iou3d_utils
    for seed, clustered, n in ((0, True, 1500), (1, False, 1000)):
        a, b = _iou_inputs(seed, clustered, n)
        key = "iou%d_s%d" % (int(overlap), seed)
        assert array_digest(a) + array_digest(b) == str(g[key + "_inputs"]), "inputs changed: regenerate the golden"
        a, b = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        got = _iou_bits(iou3d_utils.boxes_overlap_bev(a, b) if overlap else iou3d_utils.boxes_iou_bev(a, b))
        assert got.shape == tuple(g[key + "_shape"])
        idx = g[key + "_sample"]                   # a fixed sample of the reference's positive entries, readable on failure
        diff = got.ravel()[idx] != g[key + "_sample_bits"]
        assert not diff.any(), "%d of %d sampled values differ from the reference kernel" % (int(diff.sum()), idx.size)
        assert array_digest(got) == str(g[key]), "values differ from the reference kernel"
        assert int(g[key + "_positive"]) > 1000    # the comparison is not vacuous


@pytest.mark.parametrize("n,clustered,thr", [(1000, True, 0.01), (1000, True, 0.5), (4097, True, 0.2),
                                             (3000, False, 0.01), (64, True, 0.1), (65, True, 0.1), (1, False, 0.5)])
def test_nms_keep_bit_exact_vs_reference_kernel(n, clustered, thr):
    g = _ref_golden()
    from det3d_b200 import _lib
    from det3d_b200.ops.nms import nms_ops
    boxes, _ = _sorted_boxes(n, 3, clustered)
    key = _keep_key(n, clustered, thr)
    assert array_digest(boxes) == str(g["boxes_" + key]), "inputs changed: regenerate the golden"
    dev = torch.from_numpy(boxes).cuda()
    want = g["keep_" + key]
    keep_idx, keep_count = nms_ops.nms_sorted(dev, _lib.BOX_XYXYR, thr)
    got = keep_idx[: int(keep_count)].cpu().numpy()
    assert np.array_equal(got, want)
    want_n = g["keep_normal_" + key]
    keep_idx, keep_count = nms_ops.nms_sorted(dev, _lib.BOX_XYXYR, thr, axis_aligned=True)
    assert np.array_equal(keep_idx[: int(keep_count)].cpu().numpy(), want_n)


def test_iou3d_utils_api():
    g = _ref_golden()
    from det3d.ops.iou3d import iou3d_utils
    boxes, scores = nms_boxes_xyxyr(2000, 7, True)
    assert array_digest(boxes) + array_digest(scores) == str(g["api_inputs"]), "inputs changed: regenerate the golden"
    b, s = torch.from_numpy(boxes).cuda(), torch.from_numpy(scores).cuda()
    got = iou3d_utils.nms_gpu(b, s, 0.3)
    want = torch.from_numpy(g["api_keep"]).cuda()         # reference keep list, mapped back through the score order
    assert got.dtype == torch.int64 and got.is_cuda and torch.equal(got, want)
    assert torch.equal(iou3d_utils.nms_normal_gpu(b, s, 0.3), torch.from_numpy(g["api_keep_normal"]).cuda())


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "iou3d_*.npz"))))
def test_golden_fixtures_from_reference_kernel(path):
    from det3d_b200 import _lib
    from det3d_b200.ops.nms import nms_ops
    g = np.load(path)
    boxes = torch.from_numpy(g["boxes_sorted"]).cuda()
    keep_idx, keep_count = nms_ops.nms_sorted(boxes, _lib.BOX_XYXYR, float(g["thresh"]))
    assert np.array_equal(keep_idx[: int(keep_count)].cpu().numpy(), g["keep"])
    if "iou" in g:
        m = g["iou"].shape[0]
        got = nms_ops.boxes_iou_bev(boxes[:m], boxes[:m]).cpu().numpy()
        assert np.array_equal(got.view(np.int32), g["iou"].view(np.int32))


def test_stress_100k_boxes_vs_reference_kernel():
    g = _ref_golden()
    from det3d_b200 import _lib
    from det3d_b200.ops.nms import nms_ops
    boxes = _stress_boxes()
    n = boxes.shape[0]
    assert array_digest(boxes) == str(g["stress_boxes"]), "inputs changed: regenerate the golden"
    dev = torch.from_numpy(boxes).cuda()
    for thr in (0.01, 0.5):
        keep_idx, keep_count = nms_ops.nms_sorted(dev, _lib.BOX_XYXYR, thr)
        got = keep_idx[: int(keep_count)].cpu().numpy()
        want = np.flatnonzero(np.unpackbits(g["stress_keep_t%02d" % round(thr * 100)], count=n))   # kept-box bitmap
        assert np.array_equal(got, want)
        # invariants: ascending, first box kept, kept boxes are mutually compatible
        assert got[0] == 0 and (np.diff(got) > 0).all()
        sub = dev[torch.from_numpy(got[:3000]).cuda()]
        iou = nms_ops.boxes_iou_bev(sub, sub)
        iou.fill_diagonal_(0)
        assert float(iou.max()) <= thr
        # idempotence: NMS of the kept set keeps everything
        k2, c2 = nms_ops.nms_sorted(dev[torch.from_numpy(got).cuda()].contiguous(), _lib.BOX_XYXYR, thr)
        assert int(c2) == got.shape[0]


def _cc_oracle(dets, thr):
    from oracle.second_cpu import rotate_nms_cc
    return rotate_nms_cc(dets, thr)


@pytest.mark.parametrize("n,clustered,thr", [(1000, True, 0.01), (1000, True, 0.5), (1000, False, 0.2), (300, True, 0.0)])
def test_rotate_nms_xywlr_vs_oracle(n, clustered, thr):
    from det3d.core.bbox import box_torch_ops
    boxes, scores = nms_boxes_xyxyr(n, 5, clustered, extent=40.0)
    r = xyxyr_to_xywlr(boxes)
    dets = np.concatenate([r, scores[:, None]], 1).astype(np.float32)
    want = _cc_oracle(dets, thr)
    got = box_torch_ops.rotate_nms(torch.from_numpy(r).cuda(), torch.from_numpy(scores).cuda(), None, None, thr)
    assert got.dtype == torch.int64 and got.is_cuda
    assert np.array_equal(got.cpu().numpy(), want)
    # pre/post max sizes (box_torch_ops.py:534,542)
    got = box_torch_ops.rotate_nms(torch.from_numpy(r).cuda(), torch.from_numpy(scores).cuda(), 200, 17, thr)
    top = np.argsort(-scores, kind="stable")[:200]
    want = top[_cc_oracle(dets[top], thr)][:17]
    assert np.array_equal(got.cpu().numpy(), want)


def test_rotate_nms_empty_and_single():
    from det3d.core.bbox import box_torch_ops
    e = box_torch_ops.rotate_nms(torch.zeros((0, 5), device="cuda"), torch.zeros(0, device="cuda"), 1000, 100, 0.1)
    assert e.shape == (0,) and e.dtype == torch.int64 and e.is_cuda
    one = box_torch_ops.rotate_nms(torch.tensor([[1.0, 2, 3, 4, 0.5]], device="cuda"), torch.tensor([0.9], device="cuda"))
    assert one.tolist() == [0]


def test_axis_aligned_nms_api():
    from det3d.core.bbox import box_torch_ops
    b = torch.tensor([[0, 0, 2, 2], [0.1, 0, 2.1, 2], [5, 5, 7, 7.0]], device="cuda")
    s = torch.tensor([0.5, 0.9, 0.7], device="cuda")
    assert box_torch_ops.nms(b, s, None, None, 0.5).tolist() == [1, 2]


@pytest.mark.parametrize("thr", [0.3, 0.5, 0.7])
def test_box_torch_ops_nms_pixel_matches_reference_golden(thr):
    """a14: box_torch_ops.nms = numba nms_gpu semantics ("+1" extents, float64 after the fp32 differences)."""
    from conftest import load_golden
    from det3d.core.bbox import box_torch_ops
    g = load_golden("aa_nms_pixel_700")
    dets = torch.from_numpy(g["dets"]).cuda()
    keep = box_torch_ops.nms(dets[:, :4], dets[:, 4], iou_threshold=thr)
    assert keep.dtype == torch.int64 and keep.is_cuda
    assert np.array_equal(keep.cpu().numpy(), g["keep_t%02d" % int(thr * 100)])                # bit-exact keep list
    k2 = box_torch_ops.nms(dets[:, :4], dets[:, 4], pre_max_size=300, post_max_size=50, iou_threshold=thr)
    from oracle.aa_nms import nms_pixel
    top = np.argsort(-g["dets"][:, 4], kind="stable")[:300]
    want = top[nms_pixel(g["dets"][top], thr)][:50]
    assert np.array_equal(k2.cpu().numpy(), want)
    assert box_torch_ops.nms(dets[:0, :4], dets[:0, 4]).shape == (0,)


def test_rrpn_rotate_iou_and_nms_match_reference_golden():
    """a13: det3d.ops.nms.{rotate_iou_gpu, rotate_iou_gpu_eval, rotate_nms_gpu, nms_gpu} (numpy in/out)."""
    from conftest import load_golden
    from det3d.ops.nms import nms_gpu, rotate_iou_gpu, rotate_iou_gpu_eval, rotate_nms_gpu
    from oracle import rrpn
    g = load_golden("rrpn_600")
    a = g["mat_boxes"]
    for crit in (-1, 0, 1, 2):
        got = rotate_iou_gpu_eval(a, a[:37], crit)
        want = g["mat_c%d" % (crit + 1)][:, :37]
        assert got.shape == want.shape and got.dtype == np.float32
        # a rotated box against an exact copy of itself is a knife edge of the RRPN routine (coincident corners pass
        # or fail `abap >= 0` on the sign of a rounding residual, which FMA contraction changes): the reference's own
        # result is implementation-defined there, so those entries are compared only for unrotated boxes
        both = np.isfinite(want)
        knife = np.zeros_like(both)
        for i in range(37):
            knife[i, i] = a[i, 4] != 0.0
        both &= ~knife
        assert np.array_equal(np.isfinite(got) & ~knife, both)
        assert float((np.abs(got[both] - want[both]) / np.maximum(1.0, np.abs(want[both]))).max()) <= 1e-4   # north_star IoU tolerance; criterion 2 is an area
    assert np.array_equal(rotate_iou_gpu(a, a[:5]), rotate_iou_gpu_eval(a, a[:5], -1))
    assert rotate_iou_gpu(a[:0], a).shape == (0, a.shape[0])
    for thr in (0.1, 0.3, 0.5):
        keep = np.asarray(rotate_nms_gpu(g["dets"], thr), np.int64)
        want = g["keep_t%02d" % int(thr * 100)]
        _, near = rrpn.rotate_nms(g["dets"], thr)
        if near == 0:
            assert np.array_equal(keep, want)
        else:
            assert len(set(keep.tolist()) ^ set(want.tolist())) <= 2 * near
    ga = load_golden("aa_nms_pixel_700")
    assert np.array_equal(np.asarray(nms_gpu(ga["dets"], 0.5), np.int64), ga["keep_t50"])
    assert rotate_nms_gpu(np.zeros((0, 6), np.float32), 0.5) == []
