"""BASELINE configs[3] at its stated size: CBGS (nuScenes grid, 35k-point clouds), 32 clouds sharded over all GPUs of
the box with NCCL, all-gathered detections == the single-rank result, bit for bit (tools/dist_infer.py; the reference
counterpart is tools/dist_test.py:180-215).  Needs >= 2 GPUs; the 1-GPU variant checks the same harness end to end."""
import json
import os
import subprocess
import sys

import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _run(world, config, clouds, port):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "dist_infer.py"), "--config", config,
           "--clouds", str(clouds), "--check"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, cwd=ROOT)
    assert p.returncode == 0, (p.stdout[-1500:], p.stderr[-3000:])
    line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1]
    return json.loads(line)


def test_cbgs_32_clouds_sharded_over_all_gpus():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = max(w for w in (2, 4, 8) if w <= n)
    r = _run(world, "cbgs", 32, 29671)
    assert r["world"] == world and r["clouds"] == 32 and r["gathered_equals_single_rank"] is True
    assert r["total_detections"] > 100


def test_harness_single_rank_second():
    r = _run(1, "second", 4, 29672)
    assert r["gathered_equals_single_rank"] is True and r["total_detections"] > 10
