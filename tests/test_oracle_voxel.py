"""Pins the voxelizer oracle (C restatement + numpy restatement) to the reference numba
function through the committed golden fixtures (tests/golden/make_golden.py, make_golden_reference.py)."""
import numpy as np
import pytest

from conftest import array_digest, golden_voxel_cases, load_golden
from oracle import voxel as ovoxel


@pytest.mark.parametrize("case", golden_voxel_cases())
def test_c_oracle_matches_reference_golden(case):
    g = load_golden("voxel_" + case)
    v, c, n = ovoxel.points_to_voxel(g["points"], g["voxel_size"], g["pcr"], int(g["max_points"]), True,
                                     int(g["max_voxels"]))
    assert np.array_equal(c, g["coors"])
    assert np.array_equal(n, g["num_points"])
    assert np.array_equal(v, g["voxels"])


@pytest.mark.parametrize("case", [c for c in golden_voxel_cases() if c not in ("kitti_empty", "kitti_all_outside")])
def test_numpy_restatement_matches_reference_golden(case):
    g = load_golden("voxel_" + case)
    v, c, n = ovoxel.points_to_voxel_numpy(g["points"], g["voxel_size"], g["pcr"], int(g["max_points"]),
                                           int(g["max_voxels"]))
    assert np.array_equal(c, g["coors"]) and np.array_equal(n, g["num_points"]) and np.array_equal(v, g["voxels"])


def test_overflow_break_drops_late_points_of_open_voxels():
    # 3 voxels allowed; the 4th new voxel appears at point 3 -> points 4.. are dropped even
    # though point 4 belongs to voxel 0 (point_cloud_ops.py:46-47 is a `break`).
    vs, pcr = [1.0, 1.0, 1.0], [0, 0, 0, 10, 10, 1]
    pts = np.array([[0.5, 0.5, 0.5], [1.5, 0.5, 0.5], [2.5, 0.5, 0.5], [3.5, 0.5, 0.5], [0.6, 0.5, 0.5]], np.float32)
    v, c, n = ovoxel.points_to_voxel(pts, vs, pcr, 5, True, 3)
    assert n.tolist() == [1, 1, 1] and c[:, 2].tolist() == [0, 1, 2]


def test_dense_map_scratch_is_restored():
    vs, pcr = np.float32([0.5, 0.5, 0.5]), np.float32([0, 0, 0, 4, 4, 2])
    grid = ovoxel.grid_size(vs, pcr)
    scratch = -np.ones(int(np.prod(grid)), np.int32)
    pts = np.random.default_rng(0).uniform(0, 2, (100, 3)).astype(np.float32)
    a = ovoxel.points_to_voxel(pts, vs, pcr, 4, True, 50, dense_map=scratch)
    b = ovoxel.points_to_voxel(pts, vs, pcr, 4, True, 50)
    assert (scratch == -1).all()
    assert all(np.array_equal(x, y) for x, y in zip(a, b))


def _fresh_seed_clouds():
    """(points, voxel_size, range, max_points, max_voxels): three seeded KITTI-grid clouds, ~1 m beyond the range."""
    rng = np.random.default_rng(123)
    vs, pcr = np.float32([0.05, 0.05, 0.1]), np.float32([0, -40, -3, 70.4, 40, 1])
    cases = []
    for seed in range(3):
        n = int(rng.integers(100, 5000))
        pts = np.stack([rng.uniform(-1, 71, n), rng.uniform(-41, 41, n), rng.uniform(-3.2, 1.2, n), rng.uniform(0, 1, n)], 1).astype(np.float32)
        cases.append((pts, vs, pcr, 5, 600 + 700 * seed))
    return cases


def _random_clouds():
    """(points, voxel_size, range, max_points, max_voxels): boundary-snapped points, the max_voxels `break`, ndim 3/4/5,
    an empty cloud."""
    rng = np.random.default_rng(123)
    cases = [([0.05, 0.05, 0.1], [0, -40.0, -3.0, 70.4, 40.0, 1.0], 5, 20000, 4, 30000),
             ([0.16, 0.16, 4.0], [0, -39.68, -3, 69.12, 39.68, 1], 100, 1200, 4, 9000),      # hits the max_voxels break
             ([0.1, 0.1, 0.2], [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0], 10, 60000, 5, 20000),
             ([0.05, 0.05, 0.1], [0, -40.0, -3.0, 70.4, 40.0, 1.0], 5, 20000, 3, 0)]
    out = []
    for vs, pcr, max_pts, max_vox, ndim, n in cases:
        lo, hi = np.asarray(pcr[:3], np.float32), np.asarray(pcr[3:], np.float32)
        span = (hi - lo + 2.0)[[0, 1, 2] + [0] * (ndim - 3)]
        base = (lo - 1.0)[[0, 1, 2] + [0] * (ndim - 3)]
        pts = (base + rng.random((n, ndim)).astype(np.float32) * span).astype(np.float32)      # ~ +-1 m beyond the range
        if n:
            snap = rng.random(n) < 0.3            # exact multiples of the voxel size: fp32 division edge cases
            cell = np.floor((pts[snap, :3] - lo) / np.asarray(vs, np.float32))
            pts[snap, :3] = lo + cell * np.asarray(vs, np.float32)
        out.append((pts, vs, pcr, max_pts, max_vox))
    return out


def _assert_reference_output(g, key, pts, got):
    """`got` (voxels, coors, num_points) against the reference's output stored under `key`: the voxel count, a fixed
    sample of voxels (readable on failure), then every array bit for bit through its digest."""
    assert array_digest(pts) == str(g[key + "_points"]), "input cloud changed: regenerate the golden"
    idx = g[key + "_sample"]
    for name, a in zip(("voxels", "coors", "num_points"), got):
        assert a.shape[0] == int(g[key + "_count"]), (key, name)
        assert np.array_equal(a[idx], g[key + "_" + name + "_sample"]), (key, name)
        assert array_digest(a) == str(g[key + "_" + name]), (key, name)


def test_c_oracle_matches_live_reference_on_fresh_seeds():
    """The reference's numba `points_to_voxel` (point_cloud_ops.py:112-184) on three seeded clouds; its outputs are
    stored in tests/golden/ref_voxel_fresh_seeds.npz (tests/golden/make_golden_reference.py)."""
    g = load_golden("ref_voxel_fresh_seeds")
    for i, (pts, vs, pcr, max_pts, max_vox) in enumerate(_fresh_seed_clouds()):
        _assert_reference_output(g, "s%d" % i, pts, ovoxel.points_to_voxel(pts, vs, pcr, max_pts, True, max_vox))


def test_c_oracle_equals_aot_reference_kernel_on_random_inputs():
    """Beyond the committed goldens: the C restatement must reproduce the reference's own numba kernel bit for bit on
    seeded clouds -- boundary-snapped points, overflow `break`, ndim 3/4/5, an empty cloud.  The reference outputs are
    stored in tests/golden/ref_voxel_random.npz (tests/golden/make_golden_reference.py)."""
    g = load_golden("ref_voxel_random")
    for i, (pts, vs, pcr, max_pts, max_vox) in enumerate(_random_clouds()):
        _assert_reference_output(g, "c%d" % i, pts, ovoxel.points_to_voxel(pts, vs, pcr, max_pts, True, max_vox))
