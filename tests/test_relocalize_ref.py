"""tests/relocalize_ref.py (the restatement the device search is checked against) pinned on the CPU: against an independent
formulation (scipy's rotations, every candidate's transform applied to the points directly), a planted truth, ties, points on cell
faces and an empty grid."""
import math
import os
import sys

import numpy as np
from scipy.spatial.transform import Rotation

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import relocalize_ref as rr  # noqa: E402


def _cloud(rng, n, spread=25.0):
    p = rng.uniform(-spread, spread, (n, 4)).astype(np.float32)
    p[:, 2] *= 0.2
    return p


def _direct_scores(sp, u_raw, q_c, occ):
    """Every candidate on its own: R = Rz(theta) R_c from scipy, cell = floor((R p + t - o) / r)."""
    Rc = Rotation.from_quat(q_c).as_matrix()
    out = np.zeros((sp.nJ, sp.nZ, sp.S, sp.S), np.int64)
    for j in range(sp.nJ):
        R = Rotation.from_euler("z", sp.theta(j)).as_matrix() @ Rc
        w = u_raw @ R.T
        for iz in range(sp.nZ):
            for iy in range(sp.S):
                for ix in range(sp.S):
                    t = sp.t_c + sp.r * np.array([ix - sp.N, iy - sp.N, iz - sp.Nz], float)
                    c = np.floor((w + t - sp.o) / sp.r).astype(np.int64)
                    ok = np.all((c >= 0) & (c < sp.dims), axis=1)
                    out[j, iz, iy, ix] = occ[c[ok, 2], c[ok, 1], c[ok, 0]].sum()
    return out


def test_matches_independent_formulation():
    rng = np.random.RandomState(3)
    for trial in range(3):
        stack_c, stack_s, world = _cloud(rng, 60), _cloud(rng, 90), _cloud(rng, 3000)
        q_c = Rotation.from_euler("xyz", rng.uniform(-0.05, 0.05, 3) + [0, 0, rng.uniform(-3, 3)]).as_quat()
        t_c = rng.uniform(-5, 5, 3)
        kw = dict(half_xy=2.0, half_z=1.0, half_yaw_deg=30.0, resolution=1.0, yaw_step_deg=10.0, max_range=30.0)
        sp, u, occ, sc, best, runner = rr.search(stack_c, stack_s, world, q_c, t_c, max_points=100, **kw)
        p = np.concatenate([stack_c, stack_s])[:, :3].astype(np.float64)
        p = p[np.linalg.norm(p, axis=1) <= 30.0]
        p = p[::math.ceil(len(p) / 100)]
        assert np.allclose(u, p @ Rotation.from_quat(q_c).as_matrix().T, atol=1e-12)
        direct = _direct_scores(sp, p, q_c, occ)
        assert (direct == sc).all(), "trial %d: %d candidates differ" % (trial, (direct != sc).sum())
        assert best == (int(np.argmax(direct)), int(direct.max()))


def test_planted_truth():
    """The map is the query itself moved by a known yaw and cell offset: that candidate scores every point."""
    rng = np.random.RandomState(5)
    stack = _cloud(rng, 400)
    q_c = Rotation.from_euler("xyz", [0.02, -0.01, 0.7]).as_quat()
    t_c = np.array([3.0, -2.0, 0.5])
    u = rr.select(stack, stack[:0], q_c)
    sp = rr.Space(u, t_c, half_xy=6.0, half_z=1.0, half_yaw_deg=180.0, yaw_step_deg=5.0)
    j, iz, iy, ix = 40, 2, 3, 9
    c, s = math.cos(sp.theta(j)), math.sin(sp.theta(j))
    m = np.stack([(c * u[:, 0] - s * u[:, 1]) + t_c[0] + (ix - sp.N), (s * u[:, 0] + c * u[:, 1]) + t_c[1] + (iy - sp.N),
                  u[:, 2] + t_c[2] + (iz - sp.Nz)], axis=1).astype(np.float32)
    occ = sp.occupancy(m)
    sc = sp.scores(occ, sp.cells(u))
    (b, score), (rI, rs) = sp.best_and_runner(sc)
    assert b == ((j * sp.nZ + iz) * sp.S + iy) * sp.S + ix and score == len(u)
    assert rs < score and not sp.in_zone(b).reshape(sp.nJ, sp.S, sp.S)[sp.decode(rI)[0], sp.decode(rI)[2], sp.decode(rI)[3]]
    q, t = sp.pose(b, q_c)
    R = Rotation.from_quat(q).as_matrix()
    assert np.allclose(R, Rotation.from_euler("z", sp.theta(j)).as_matrix() @ Rotation.from_quat(q_c).as_matrix(), atol=1e-12)
    assert np.allclose(t, t_c + [ix - sp.N, iy - sp.N, iz - sp.Nz])


def test_ties_go_to_the_lowest_index():
    """One query point and two occupied cells: every candidate that reaches either ties, and the lowest index wins; the runner-up
    is the lowest-index tie outside the exclusion zone."""
    u = np.array([[0.25, 0.25, 0.25]])
    sp = rr.Space(u, [0.0, 0.0, 0.0], half_xy=5.0, half_z=0.0, half_yaw_deg=0.0, yaw_step_deg=1.0, exclusion_m=2.0)
    cell = sp.cells(u)[0, 0]
    occ = np.zeros(sp.dims[::-1], np.uint8)
    occ[cell[2], cell[1] - 4, cell[0] + 2] = 1
    occ[cell[2], cell[1] + 3, cell[0] - 5] = 1
    sc = sp.scores(occ, sp.cells(u))
    assert sc.sum() == 2
    (b, s), (rI, rs) = sp.best_and_runner(sc)
    assert s == rs == 1
    assert sp.decode(b) == (0, 0, sp.N - 4, sp.N + 2) and sp.decode(rI) == (0, 0, sp.N + 3, sp.N - 5)
    # inside the zone the other tie is not a runner-up
    sp2 = rr.Space(u, [0.0, 0.0, 0.0], half_xy=5.0, half_z=0.0, half_yaw_deg=0.0, yaw_step_deg=1.0, exclusion_m=20.0)
    (b2, _), (r2, s2) = sp2.best_and_runner(sp2.scores(occ, sp2.cells(u)))
    assert b2 == b and (r2, s2) == (-1, -1)


def test_points_on_cell_faces():
    """A map point exactly on a cell face falls in the cell above it; a query point on a face keeps its base cell exact."""
    u = np.array([[1.0, 2.0, 0.0], [-3.0, 0.5, 0.0]])
    sp = rr.Space(u, [0.0, 0.0, 0.0], half_xy=2.0, half_z=0.0, half_yaw_deg=0.0, resolution=0.5, yaw_step_deg=1.0, max_range=10.0)
    o = sp.o
    face = np.array([[o[0] + 0.5 * 7, o[1] + 0.5 * 9, o[2] + 0.5 * 1, 0]], np.float32)
    occ = sp.occupancy(face)
    assert occ[1, 9, 7] == 1 and occ.sum() == 1
    cells = sp.cells(u)
    assert (cells[0] == np.floor((u - o) / 0.5)).all()
    assert (cells[0, 0] == [(1.0 - o[0]) / 0.5, (2.0 - o[1]) / 0.5, (0.0 - o[2]) / 0.5]).all()


def test_empty_grid():
    rng = np.random.RandomState(7)
    u = rr.select(_cloud(rng, 50), _cloud(rng, 50), [0, 0, 0, 1])
    sp = rr.Space(u, [1.0, 2.0, 0.0], half_xy=3.0, half_z=1.0, half_yaw_deg=20.0, yaw_step_deg=5.0)
    occ = sp.occupancy(np.zeros((0, 4), np.float32))
    sc = sp.scores(occ, sp.cells(u))
    (b, s), (rI, rs) = sp.best_and_runner(sc)
    assert occ.sum() == 0 and (sc == 0).all() and (b, s) == (0, 0)
    assert rs == 0 and not sp.in_zone(0).reshape(-1)[rI % (sp.S * sp.S) + (rI // (sp.nZ * sp.S * sp.S)) * sp.S * sp.S]


def test_query_selection():
    """Range gate in order, stack C before stack S, every ceil(n / max_points)-th point."""
    c = np.array([[1, 0, 0, 0], [100, 0, 0, 0], [2, 0, 0, 0]], np.float32)
    s = np.array([[3, 0, 0, 0], [0, 4, 0, 0], [0, 0, 70, 0], [5, 0, 0, 0]], np.float32)
    u = rr.select(c, s, [0, 0, 0, 1], max_range=60.0, max_points=2)
    assert (u == [[1, 0, 0], [0, 4, 0]]).all()
    assert len(rr.select(c, s, [0, 0, 0, 1], max_range=60.0, max_points=5)) == 5
    assert len(rr.select(c, s, [0, 0, 0, 1], max_range=60.0, max_points=4)) == 3
