"""pcl::VoxelGrid at the sizes and values where vl_voxel_grid_device changes regime (voxel_grid.cu):

  * the bitonic sort: one cluster launch up to 16 tiles (4096 keys x 16 CTAs at P = 65536, 8192 x 16 at P = 131072), the
    multi-launch network (bt_tile_sort / bt_global_step / bt_tile_merge) above 2^17 keys;
  * vg_centroid: runs longer than its staged VG_TILE + VG_HALO = 320 keys (the global tail loop), run heads at tile positions
    255 / 256 / 319 / 320 and at the start of a tile;
  * the overflow guard at its boundary (1290^3 voxels are filtered, 1291^3 come back unchanged);
  * points exactly on voxel faces with leaves that are not binary fractions (p * (1 / leaf) rounded, not p / leaf, no FMA);
  * the smallest leaf the library accepts (0.05) and a coarse one (2.5).

The CUDA filter is compared bit for bit with the oracle's op.voxel_grid; the CPU test pins op.voxel_grid itself against the
independent numpy restatement on the same clouds (sub-sampled where the numpy loop would be slow)."""
import numpy as np
import pytest

from test_oracle_math import np_voxel_grid


def _runs(lengths, leaf, seed):
    """Voxels along +x, voxel i holding lengths[i] points strictly inside it, in shuffled input order: the sorted key array
    then has a run head at every prefix sum of `lengths`."""
    rng = np.random.RandomState(seed)
    pts = []
    for i, m in enumerate(lengths):
        lo = np.array([i, 0, 0], np.float64) * leaf
        p = lo + rng.uniform(0.1, 0.9, (m, 3)) * leaf
        pts.append(np.concatenate([p, rng.uniform(0, 100, (m, 1))], 1))
    c = np.concatenate(pts).astype(np.float32)
    return c[rng.permutation(len(c))]


def _heads_at_tile_edges():
    # heads at 0..254, 255, 256, 319 (last staged key of tile 0), 320 (first key past the halo) and 1024 (a tile start);
    # the run at 320 (700 keys) and the one at 1024 (1000 keys) run past the staged window of their tile
    lengths = [1] * 255 + [1, 63, 1, 700, 4, 1000] + [3, 250, 2, 1, 1, 66, 1, 2] * 20
    return _runs(lengths, 0.2, 11), 0.2


def _one_long_run():
    # 5000 points in one voxel (the whole array is one run) next to 3000 singletons
    return _runs([5000] + [1] * 3000, 0.3, 12), 0.3


def _random(n, scale, leaf, seed):
    rng = np.random.RandomState(seed)
    return (rng.randn(n, 4) * scale).astype(np.float32), leaf


def _faces(leaf, seed):
    """Coordinates k * leaf exactly (as f32 products) and their f32 neighbours: the points sit on voxel faces, where
    floor(p * inv) with inv = 1 / leaf rounded differs from floor(p / leaf) or an FMA-contracted product."""
    rng = np.random.RandomState(seed)
    k = rng.randint(-60, 61, (20000, 3)).astype(np.float32)
    p = k * np.float32(leaf)
    nudge = rng.randint(-1, 2, p.shape)
    p = np.where(nudge > 0, np.nextafter(p, np.float32(np.inf)), np.where(nudge < 0, np.nextafter(p, np.float32(-np.inf)), p))
    return np.concatenate([p, rng.uniform(0, 100, (len(p), 1))], 1).astype(np.float32), leaf


def _guard_boundary(extent, leaf, seed):
    """Bounding box of exactly floor(extent / leaf) + 1 voxels per axis (two corner points), 3000 points inside."""
    rng = np.random.RandomState(seed)
    inner = rng.uniform(0, extent, (3000, 3))
    inner[:200] = np.round(inner[:200] / leaf) * leaf   # on voxel faces
    inner[200:300] = inner[:100]                        # and shared voxels: a filtered cloud is shorter than its input
    c = np.concatenate([[[0, 0, 0], [extent, extent, extent]], inner])
    return np.concatenate([c, rng.uniform(0, 100, (len(c), 1))], 1).astype(np.float32), leaf


CASES = {
    "cluster-4096x16": lambda: _random(65536, 30.0, 0.2, 1),        # P = 65536: 16 CTAs of 4096 keys
    "cluster-8192x16": lambda: _random(131072, 30.0, 0.2, 2),       # P = 131072: 16 CTAs of 8192 keys
    "multi-launch": lambda: _random(131073, 30.0, 0.2, 3),          # P = 262144: bt_tile_sort / bt_global_step / bt_tile_merge
    "multi-launch-600k": lambda: _random(600000, 20.0, 0.4, 4),     # P = 1048576
    "heads-at-tile-edges": _heads_at_tile_edges,
    "one-long-run": _one_long_run,
    "faces-0.2": lambda: _faces(0.2, 5),
    "faces-0.3": lambda: _faces(0.3, 6),
    "guard-1290-cubed": lambda: _guard_boundary(1289.5, 1.0, 7),    # 1290^3 < 2^31 - 1: filtered
    "guard-1291-cubed": lambda: _guard_boundary(1290.5, 1.0, 8),    # 1291^3 > 2^31 - 1: output = input
    "leaf-0.05": lambda: _random(50000, 3.0, 0.05, 9),
    "leaf-2.5": lambda: _random(50000, 4.0, 2.5, 10),               # runs of hundreds of points in the central voxels
}
NUMPY_CAP = 40000   # the numpy restatement folds point by point in Python


def _check_regime(name, c, leaf, out):
    """What makes the case the regime it is named after."""
    if name.startswith("guard-"):
        assert (out.tobytes() == c.tobytes()) == (name == "guard-1291-cubed"), name
    if name in ("heads-at-tile-edges", "one-long-run", "leaf-2.5"):
        inv = np.float32(1.0) / np.float32(leaf)
        _, cnt = np.unique(np.floor(c[:, :3] * inv), axis=0, return_counts=True)
        assert cnt.max() > 320, (name, cnt.max())


def _bits_equal(a, b, what):
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, a.shape, b.shape)
    bad = np.flatnonzero(a.view(np.uint32) != b.view(np.uint32))
    assert len(bad) == 0, "%s: %d floats differ, first at %s" % (what, len(bad), bad[:5].tolist())


@pytest.mark.parametrize("name", sorted(CASES))
def test_voxel_grid_regimes_oracle_matches_numpy(op, name):
    c, leaf = CASES[name]()
    if len(c) > NUMPY_CAP and not name.startswith("guard-"):
        c = c[:NUMPY_CAP]
    out = op.voxel_grid(c, leaf)
    _bits_equal(out, np_voxel_grid(c, leaf), name)
    _check_regime(name, c, leaf, out)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_voxel_grid_regimes_bit_exact(pkg, op, name):
    c, leaf = CASES[name]()
    g = pkg.Context()
    out = g.voxel_grid(c, leaf)
    g.close()
    ref = op.voxel_grid(c, leaf)
    _bits_equal(out, ref, name)
    _check_regime(name, c, leaf, ref)
