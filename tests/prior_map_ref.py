"""vloam_b200_load_map restated from the cited lines, for tests of the prior-map load: world-frame points -> the `lm.cornerMap` /
`lm.surfMap` blob (int32 counts[4851], then the points of every cube in cube order).

- Cube of a point (LM.cpp:747-756): t = double(v) + 25.0; c = int(t / 50.0) + cen; if (t < 0) c--; per axis, at the window centre
  `cen` (laserCloudCen{Width,Height,Depth}).
- Points outside the 21 x 21 x 11 grid are dropped (LM.cpp:758-761); points with a non-finite x, y or z are dropped as well.
- Every non-empty cube is then pcl::VoxelGrid-filtered over its points in input order (LM.cpp:795-808; SURVEY A.1, the tie order of
  Appendix B): the oracle's own voxel_grid, one cube at a time."""
import numpy as np

CUBE_W, CUBE_H, CUBE_D = 21, 21, 11
CUBE_NUM = CUBE_W * CUBE_H * CUBE_D


def cube_of(v, cen):
    """LM.cpp:747-756 on a float32 column: int64 cube coordinates (exact; out-of-grid values are simply out of range)."""
    t = v.astype(np.float64) + 25.0
    c = np.trunc(t / 50.0).astype(np.int64) + cen
    c[t < 0] -= 1
    return c


def bin_points(points, cen):
    """(cube index int64[n] or -1 for a dropped point) for float32[n, 4] world-frame points."""
    pts = np.ascontiguousarray(points, np.float32).reshape(-1, 4)
    finite = np.isfinite(pts[:, :3]).all(axis=1)
    safe = np.where(finite[:, None], pts[:, :3], np.float32(0))
    c = [cube_of(safe[:, a], cen[a]) for a in range(3)]
    ok = finite & (c[0] >= 0) & (c[0] < CUBE_W) & (c[1] >= 0) & (c[1] < CUBE_H) & (c[2] >= 0) & (c[2] < CUBE_D)
    return np.where(ok, c[0] + CUBE_W * c[1] + CUBE_W * CUBE_H * c[2], -1)


def load_blob(op, points, leaf, cen=(10, 10, 5)):
    """The blob load_map leaves for one kind, and the number of points it drops."""
    pts = np.ascontiguousarray(points, np.float32).reshape(-1, 4)
    cube = bin_points(pts, cen)
    kept = cube >= 0
    order = np.argsort(cube[kept], kind="stable")  # by cube, input order inside a cube
    kp, kc = pts[kept][order], cube[kept][order]
    counts = np.zeros(CUBE_NUM, np.int32)
    parts = []
    if len(kc):
        starts = np.flatnonzero(np.r_[True, kc[1:] != kc[:-1]])
        ends = np.r_[starts[1:], len(kc)]
        for s, e in zip(starts, ends):
            out = op.voxel_grid(kp[s:e], leaf)
            counts[kc[s]] = len(out)
            parts.append(out)
    body = np.concatenate(parts) if parts else np.zeros((0, 4), np.float32)
    return counts.tobytes() + np.ascontiguousarray(body, np.float32).tobytes(), int((~kept).sum())
