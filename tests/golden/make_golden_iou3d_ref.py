"""Outputs of the REFERENCE iou3d CUDA kernel (oracle/_ref/libiou3d_ref.so, compiled from
det3d/ops/iou3d/src/iou3d_kernel.cu by oracle/build.py) on the inputs of tests/test_nms_gpu.py, for
tests/golden/ref_iou3d_kernel.npz.  Needs a GPU and the reference library built:

    python tests/golden/make_golden_iou3d_ref.py OUT_DIR

IoU matrices are stored as digests plus a fixed sample of their positive entries, keep lists whole
(the 100k-box ones as bitmaps); every input is pinned by its digest."""
import os
import sys

import numpy as np
import torch

TESTS = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, TESTS)
from conftest import array_digest  # noqa: E402
from oracle import iou3d_ref  # noqa: E402
from det3d_b200.utils.synthetic import nms_boxes_xyxyr  # noqa: E402
from test_nms_gpu import _iou_bits, _iou_inputs, _keep_key, _sorted_boxes, _stress_boxes  # noqa: E402

KEEP_CASES = [(1000, True, 0.01), (1000, True, 0.5), (4097, True, 0.2), (3000, False, 0.01), (64, True, 0.1),
              (65, True, 0.1), (1, False, 0.5)]        # test_nms_keep_bit_exact_vs_reference_kernel's parameters


def main(out_dir):
    assert iou3d_ref.available(), "oracle/_ref/libiou3d_ref.so is not built"
    g = {}
    for overlap in (False, True):
        for seed, clustered, n in ((0, True, 1500), (1, False, 1000)):
            a, b = _iou_inputs(seed, clustered, n)
            key = "iou%d_s%d" % (int(overlap), seed)
            bits = _iou_bits(iou3d_ref.iou_matrix(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda(), overlap))
            flat = bits.ravel()
            positive = np.flatnonzero(flat.view(np.float32) > 0)
            idx = np.sort(np.random.default_rng(seed).choice(positive, size=min(positive.size, 2048), replace=False))
            g.update({key + "_inputs": array_digest(a) + array_digest(b), key: array_digest(bits),
                      key + "_shape": np.array(bits.shape), key + "_positive": positive.size,
                      key + "_sample": idx, key + "_sample_bits": flat[idx]})
    for n, clustered, thr in KEEP_CASES:
        boxes, _ = _sorted_boxes(n, 3, clustered)
        key = _keep_key(n, clustered, thr)
        dev = torch.from_numpy(boxes).cuda()
        g["boxes_" + key] = array_digest(boxes)
        g["keep_" + key] = iou3d_ref.nms(dev, thr)
        g["keep_normal_" + key] = iou3d_ref.nms(dev, thr, normal=True)
    boxes, scores = nms_boxes_xyxyr(2000, 7, True)
    b, s = torch.from_numpy(boxes).cuda(), torch.from_numpy(scores).cuda()
    order = torch.argsort(s, descending=True)
    g["api_inputs"] = array_digest(boxes) + array_digest(scores)
    g["api_keep"] = order[torch.from_numpy(iou3d_ref.nms(b[order].contiguous(), 0.3)).cuda()].cpu().numpy()
    g["api_keep_normal"] = order[torch.from_numpy(iou3d_ref.nms(b[order].contiguous(), 0.3, normal=True)).cuda()].cpu().numpy()
    boxes = _stress_boxes()
    dev = torch.from_numpy(boxes).cuda()
    g["stress_boxes"] = array_digest(boxes)
    for thr in (0.01, 0.5):
        mask = np.zeros(boxes.shape[0], bool)
        mask[iou3d_ref.nms(dev, thr)] = True
        g["stress_keep_t%02d" % round(thr * 100)] = np.packbits(mask)
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "ref_iou3d_kernel.npz")
    np.savez_compressed(path, **g)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1])
