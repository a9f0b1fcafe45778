import glob
import hashlib
import importlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch

    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session", autouse=True)
def _built():
    """CPU-side build products every test may rely on: the product library (cross-compiled)
    and the oracle."""
    from det3d_b200 import build as d3b_build
    from oracle import build as oracle_build

    d3b_build.build()
    oracle_build.build()


def golden_voxel_cases():
    return sorted(os.path.basename(p)[len("voxel_"):-len(".npz")] for p in glob.glob(os.path.join(GOLDEN, "voxel_*.npz")))


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz")))


def array_digest(a):
    """sha256 of an array's dtype, shape and bytes: pins outputs too large to store in tests/golden/ bit for bit."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s %s " % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def reference_config(rel):
    """Stock reference config `rel` as `Config.fromfile` returns it, from tests/golden/ref_configs.json: the calls the
    config makes into det3d and logging while it loads are made here, into det3d_b200 through the `det3d` alias."""
    from det3d.torchie import Config

    def decode(v):
        if isinstance(v, list):
            return [decode(x) for x in v]
        if not isinstance(v, dict):
            return v
        if "__call__" in v:
            module, name = v["__call__"].split(":")
            return getattr(importlib.import_module(module), name)(*decode(v["args"]), **decode(v["kwargs"]))
        if "__tuple__" in v:
            return tuple(decode(x) for x in v["__tuple__"])
        return {k: decode(x) for k, x in v.items()}

    with open(os.path.join(GOLDEN, "ref_configs.json")) as fh:
        return Config({k: decode(v) for k, v in json.load(fh)[rel].items()})
