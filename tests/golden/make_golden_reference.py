"""Golden data from the REFERENCE checkout for the tests that compare with it directly:

    python tests/golden/make_golden_reference.py REFERENCE_CHECKOUT [OUT_DIR]     (OUT_DIR: tests/golden)

  ref_configs.json          the stock configs' values as `Config.fromfile` sees them (test_registry_config.py,
                            test_pipeline_boundary.py): each config is run with recording stand-ins for its det3d /
                            logging imports, so a value that came from such a call is stored as the call
                            {"__call__": "module:name", "args", "kwargs"} and replayed against det3d_b200 by the tests;
                            tuples are {"__tuple__": [...]}.
  ref_collate_kitti.npz     the reference `collate_kitti` on test_pipeline_boundary._sample's batch.
  ref_voxel_*.npz           the reference numba `points_to_voxel` on test_oracle_voxel's seeded clouds: digests of the
                            outputs plus a fixed sample of voxels.
"""
import ast
import builtins
import collections
import importlib.util
import json
import os
import sys

import numpy as np
import torch

TESTS = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, TESTS)
from conftest import array_digest  # noqa: E402
from test_oracle_voxel import _fresh_seed_clouds, _random_clouds  # noqa: E402
from test_pipeline_boundary import STOCK, _sample  # noqa: E402

CONFIG_KEYS = ("model", "test_cfg", "voxel_generator", "target_assigner", "assigner", "test_pipeline", "train_pipeline")
RECORDED = ("det3d", "logging")


class _Call:
    def __init__(self, path, args, kwargs):
        self.path, self.args, self.kwargs = path, args, kwargs


class _Module:
    def __init__(self, name):
        self.name = name

    def __getattr__(self, attr):
        if attr.startswith("__"):
            raise AttributeError(attr)
        return lambda *a, **k: _Call(self.name + ":" + attr, a, k)


def _encode(v):
    if isinstance(v, _Call):
        return {"__call__": v.path, "args": _encode(list(v.args)), "kwargs": _encode(v.kwargs)}
    if isinstance(v, dict):
        assert all(isinstance(k, str) for k in v)
        return {k: _encode(x) for k, x in v.items()}
    if isinstance(v, list):
        return [_encode(x) for x in v]
    if isinstance(v, tuple):
        return {"__tuple__": [_encode(x) for x in v]}
    assert v is None or isinstance(v, (bool, int, float, str)), type(v)
    return v


def stock_config(path):
    real_import = builtins.__import__

    def recording_import(name, globals=None, locals=None, fromlist=(), level=0):
        if name.split(".")[0] in RECORDED:
            return _Module(name) if fromlist else _Module(name.split(".")[0])
        return real_import(name, globals, locals, fromlist, level)

    ns = {"__builtins__": dict(vars(builtins), __import__=recording_import), "__name__": "config", "__file__": path}
    exec(compile(open(path).read(), path, "exec"), ns)
    return {k: _encode(ns[k]) for k in CONFIG_KEYS}


def reference_collate(ref):
    """The reference function itself, lifted out of its module (whose package imports do not resolve here)."""
    src = open(os.path.join(ref, "det3d/torchie/parallel/collate.py")).read()
    fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "collate_kitti")
    ns = dict(np=np, torch=torch, collections=collections, defaultdict=collections.defaultdict)
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "collate.py", "exec"), ns)
    return ns["collate_kitti"]


def _flatten(v, path, arrays):
    """Nested result -> JSON skeleton; tensors and arrays go to `arrays` under their path."""
    if isinstance(v, dict):
        return {"dict": {k: _flatten(x, "%s.%s" % (path, k) if path else k, arrays) for k, x in v.items()}}
    if isinstance(v, (list, tuple)):
        return {"list": [_flatten(x, "%s.%d" % (path, i), arrays) for i, x in enumerate(v)]}
    if torch.is_tensor(v):
        arrays[path] = v.numpy()
        return {"tensor": path}
    if isinstance(v, np.ndarray):
        arrays[path] = v
        return {"ndarray": path}
    return {"value": v}


def voxel_golden(points_to_voxel, cases, prefix):
    g = {}
    for i, (pts, vs, pcr, max_pts, max_vox) in enumerate(cases):
        key = "%s%d" % (prefix, i)
        out = points_to_voxel(pts, vs, pcr, max_pts, True, max_vox)
        m = out[0].shape[0]
        idx = np.sort(np.random.default_rng(i).choice(m, size=min(m, 64), replace=False))
        g.update({key + "_points": array_digest(pts), key + "_count": m, key + "_sample": idx})
        for name, a in zip(("voxels", "coors", "num_points"), out):
            g[key + "_" + name] = array_digest(a)
            g[key + "_" + name + "_sample"] = a[idx]
    return g


def main(ref, out):
    os.makedirs(out, exist_ok=True)
    cfgs = {rel: stock_config(os.path.join(ref, rel)) for rel in STOCK}
    with open(os.path.join(out, "ref_configs.json"), "w") as fh:
        json.dump(cfgs, fh, indent=1)
        fh.write("\n")

    batch = [_sample(i, n) for i, n in enumerate((7, 0, 13))]      # test_collate_kitti_equals_reference_function's batch
    arrays = {}
    skeleton = _flatten(reference_collate(ref)(batch), "", arrays)
    np.savez_compressed(os.path.join(out, "ref_collate_kitti.npz"), skeleton=json.dumps(skeleton), **arrays)

    spec = importlib.util.spec_from_file_location("ref_pc_ops", os.path.join(ref, "det3d/ops/point_cloud/point_cloud_ops.py"))
    ops = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ops)
    np.savez_compressed(os.path.join(out, "ref_voxel_fresh_seeds.npz"), **voxel_golden(ops.points_to_voxel, _fresh_seed_clouds(), "s"))
    np.savez_compressed(os.path.join(out, "ref_voxel_random.npz"), **voxel_golden(ops.points_to_voxel, _random_clouds(), "c"))
    for f in sorted(os.listdir(out)):
        if f.startswith("ref_"):
            print(f, os.path.getsize(os.path.join(out, f)))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else os.path.join(TESTS, "golden"))
