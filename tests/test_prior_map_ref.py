"""The restatement of vloam_b200_load_map (tests/prior_map_ref.py) pinned against an independent fold: cube by the f64 formula,
voxel by float32 floor(p * (1 / leaf)), points of a voxel summed one by one in float32 in input order, one division, voxels in
ascending (iz, iy, ix) order inside each cube.  The clouds put many points in one voxel, points exactly on voxel and cube faces
(+-25 m and the t < 0 branch at -75 m), NaN, points outside the grid, and a 0.05 m leaf (one cube stays below PCL's voxel-count
overflow guard)."""
import numpy as np
import pytest

from prior_map_ref import CUBE_NUM, CUBE_W, CUBE_H, CUBE_D, load_blob


def _fold(points, leaf, cen):
    pts = np.ascontiguousarray(points, np.float32).reshape(-1, 4)
    inv = np.float32(1.0) / np.float32(leaf)
    groups = {}
    dropped = 0
    for i, p in enumerate(pts):
        if not np.isfinite(p[:3]).all():
            dropped += 1
            continue
        c = []
        for a in range(3):
            t = float(p[a]) + 25.0
            ci = int(t / 50.0) + cen[a]
            if t < 0:
                ci -= 1
            c.append(ci)
        if not (0 <= c[0] < CUBE_W and 0 <= c[1] < CUBE_H and 0 <= c[2] < CUBE_D):
            dropped += 1
            continue
        cube = c[0] + CUBE_W * c[1] + CUBE_W * CUBE_H * c[2]
        v = tuple(int(np.floor(np.float32(p[a]) * inv)) for a in (2, 1, 0))
        groups.setdefault((cube, v), []).append(i)
    counts = np.zeros(CUBE_NUM, np.int32)
    out = []
    for (cube, _), idx in sorted(groups.items()):
        acc = np.zeros(4, np.float32)
        for i in idx:
            acc = (acc + pts[i]).astype(np.float32)
        out.append((acc / np.float32(len(idx))).astype(np.float32))
        counts[cube] += 1
    body = np.array(out, np.float32).reshape(-1, 4)
    return counts.tobytes() + body.tobytes(), dropped


def _cloud(seed, leaf):
    rng = np.random.RandomState(seed)
    parts = []
    # many points per voxel: a dense blob of a few voxels
    parts.append(np.c_[rng.uniform(3.0, 3.0 + 3 * leaf, (300, 3)), rng.uniform(0, 100, 300)])
    # spread points across several cubes, around the centre cube and its neighbours
    parts.append(np.c_[rng.uniform(-120, 120, (400, 2)), rng.uniform(-60, 60, 400), rng.uniform(0, 100, 400)])
    # exactly on voxel faces and on cube faces (+-25 m, -75 m: t = -50 takes the t < 0 branch twice over), and just beside them
    faces = []
    for x in (-75.0, -25.0, 25.0, 75.0, np.nextafter(np.float32(-25.0), np.float32(0)), np.nextafter(np.float32(25.0), np.float32(0))):
        for y in (0.0, leaf, 2 * leaf, -25.0, 25.0):
            for z in (0.0, -leaf, 25.0, -25.0):
                faces.append((x, y, z, float(len(faces))))
    parts.append(np.array(faces * 2, np.float64))
    # NaN and infinite coordinates, points outside the grid (beyond 525 m along x, below -275 m along z)
    parts.append(np.array([[np.nan, 1, 1, 5], [1, np.nan, 1, 5], [1, 1, np.inf, 5], [600.0, 0, 0, 1], [-600.0, 0, 0, 1],
                           [0, 0, -300.0, 1], [0, 0, 300.0, 1], [1e12, 0, 0, 1]]))
    pts = np.concatenate(parts).astype(np.float32)
    return pts[rng.permutation(len(pts))]


@pytest.mark.parametrize("leaf", [0.4, 0.8, 0.05])
@pytest.mark.parametrize("cen", [(10, 10, 5), (8, 12, 6)])
def test_load_restatement_matches_independent_fold(op, leaf, cen):
    pts = _cloud(int(leaf * 100) + cen[0], leaf)
    blob, dropped = load_blob(op, pts, leaf, cen)
    ref, ref_dropped = _fold(pts, leaf, cen)
    assert dropped == ref_dropped and dropped >= 6
    assert blob == ref
    counts = np.frombuffer(blob[:CUBE_NUM * 4], np.int32)
    assert (counts > 0).sum() > 5, "the cloud must span several cubes"
    assert counts.sum() < len(pts) - dropped, "several points per voxel must have been folded"


def test_single_dense_cube_at_the_finest_leaf(op):
    """A whole 50 m cube at 0.05 m: 1001^3 voxels fit pcl::VoxelGrid's int32 index (no overflow guard), so the cube is filtered."""
    rng = np.random.RandomState(3)
    pts = np.c_[rng.uniform(-24.99, 24.99, (3000, 3)), rng.uniform(0, 1, 3000)].astype(np.float32)
    pts = np.concatenate([pts, pts[:500] + np.float32(0.001)])
    blob, dropped = load_blob(op, pts, 0.05)
    ref, _ = _fold(pts, 0.05, (10, 10, 5))
    assert dropped == 0 and blob == ref
    assert np.frombuffer(blob[:CUBE_NUM * 4], np.int32).sum() < len(pts)


def test_empty_and_all_dropped(op):
    blob, dropped = load_blob(op, np.zeros((0, 4), np.float32), 0.4)
    assert blob == np.zeros(CUBE_NUM, np.int32).tobytes() and dropped == 0
    blob, dropped = load_blob(op, np.array([[np.nan, 0, 0, 0], [1e4, 0, 0, 0]], np.float32), 0.4)
    assert blob == np.zeros(CUBE_NUM, np.int32).tobytes() and dropped == 2
