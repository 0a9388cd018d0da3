"""GPU parity tests proper (run on the B200 box): the CUDA path through the C ABI against the CPU
oracle on identical inputs.  Bar (BASELINE.json north_star): feature clouds / labels / association
and kNN indices bit-exact, poses within 1e-4 m and 1e-5 rad (quaternion components)."""
import os

import numpy as np
import pytest

from conftest import assert_bits_equal
from test_oracle_math import make_factors

pytestmark = pytest.mark.gpu

POS_TOL, ROT_TOL = 1e-4, 1e-5
KW = {0: dict(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4),
      1: dict(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8),
      2: dict(n_scans=128, minimum_range=0.3, line_res=0.4, plane_res=0.8),
      3: dict(n_scans=32, minimum_range=0.3, line_res=0.2, plane_res=0.4)}
SR_NAMES = ("sr.laserCloud", "sr.curvature", "sr.label", "sr.scanStartInd", "sr.scanEndInd", "sr.sharp", "sr.lessSharp", "sr.flat", "sr.lessFlat")


def check_sr(o, g):
    for nm in SR_NAMES:
        assert_bits_equal(o.get(nm), g.get(nm), nm)


def pose_close(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert np.abs(a[4:7] - b[4:7]).max() < POS_TOL, (a[4:7], b[4:7])
    assert np.abs(a[0:4] - b[0:4]).max() < ROT_TOL, (a[0:4], b[0:4])


@pytest.mark.parametrize("sensor", [0, 1, 2, 3])
@pytest.mark.parametrize("order", [0, 1])
def test_scan_registration_bit_exact(pkg, op, synth, street, sensor, order):
    """Azimuth-major (Velodyne driver) and ring-major (KITTI) emission orders, all four beam tables."""
    scan = street.scan(sensor, [3.0, 0.5, 0.02, 0.03, 0.002, -0.001], 4242 + sensor, order=order)
    o, g = op.Oracle(**KW[sensor]), pkg.Context(**KW[sensor])
    o.scan_registration(scan)
    g.begin_frame(); g.scan_registration(scan)
    check_sr(o, g)
    # packed XYZ (stride 3) gives the same result as KITTI stride 4
    g.begin_frame(); g.scan_registration(np.ascontiguousarray(scan[:, :3]))
    check_sr(o, g)
    g.close()


def test_scan_registration_adversarial_rings(pkg, op):
    """Uniform random directions: every elevation, so thousands of points sit next to a ring boundary
    (the atanf / atan2f parity trap of SURVEY section 0 item 6), with NaN / inf / near returns mixed in."""
    rng = np.random.RandomState(7)
    n = 200000
    d = rng.randn(n, 3)
    d /= np.linalg.norm(d, axis=1)[:, None]
    d[:, 2] *= 0.35
    pts = (d * rng.uniform(0.2, 90.0, (n, 1))).astype(np.float32)
    pts[rng.rand(n) < 0.02] = np.nan
    pts[rng.rand(n) < 0.001, 0] = np.inf
    for sensor in (0, 1, 2, 3):
        o, g = op.Oracle(**KW[sensor]), pkg.Context(**KW[sensor])
        o.scan_registration(pts)
        g.begin_frame(); g.scan_registration(pts)
        check_sr(o, g)
        g.close()


def test_scan_registration_edge_cases(pkg, op):
    g, o = pkg.Context(**KW[0]), op.Oracle(**KW[0])
    cases = [np.zeros((0, 3), np.float32), np.full((100, 3), np.nan, np.float32),
             (np.random.RandomState(0).randn(100, 3) * 0.05).astype(np.float32),
             np.array([[5, 0, 0.1], [5, 0.1, 0.1], [5, 0.2, 0.1]], np.float32),
             np.tile(np.array([[4.0, 1.0, 0.2]], np.float32), (300, 1))]          # 300 identical points: all-tie sort keys
    for c in cases:
        o.scan_registration(c)
        g.begin_frame(); g.scan_registration(c)
        check_sr(o, g)
    g.close()


def test_dense_ring_uses_global_sort_path(pkg, op):
    """One ring with 9000 points: sector > 1024 keys and ring > 4096 / 8192 -> the global-memory sort
    and picked-flag fallbacks of sr_pick / sr_ring_voxel."""
    rng = np.random.RandomState(3)
    az = np.sort(rng.uniform(-np.pi, np.pi, 9000))[::-1]
    r = 10 + 2 * np.sin(7 * az) + 0.05 * rng.randn(9000)
    el = np.deg2rad(1.0)
    pts = np.stack([r * np.cos(el) * np.cos(az), r * np.cos(el) * np.sin(az), r * np.sin(el) + 0 * az], 1).astype(np.float32)
    o, g = op.Oracle(**KW[0]), pkg.Context(**KW[0])
    o.scan_registration(pts)
    g.begin_frame(); g.scan_registration(pts)
    check_sr(o, g)
    assert len(o.get("sr.lessFlat")) > 500
    g.close()


@pytest.mark.parametrize("n,leaf,scale", [(0, 0.2, 1.0), (1, 0.2, 1.0), (777, 0.2, 3.0), (5000, 0.4, 20.0), (70000, 0.8, 40.0), (3, 0.2, 1e6)])
def test_voxel_grid_bit_exact(pkg, op, n, leaf, scale):
    rng = np.random.RandomState(n + 1)
    c = (rng.randn(n, 4) * scale).astype(np.float32)
    g = pkg.Context()
    assert_bits_equal(op.voxel_grid(c, leaf), g.voxel_grid(c, leaf), "voxel_grid n=%d" % n)
    g.close()


def test_normal_equations_and_solver_match_oracle(pkg, op):
    from scipy.spatial.transform import Rotation as R
    rng = np.random.RandomState(23)
    q = R.from_euler("xyz", [0.01, -0.02, 0.03]).as_quat()
    t = np.array([0.8, -0.1, 0.05])
    g = pkg.Context()
    for noise, n in ((0.0, 40), (0.03, 300), (0.2, 3000)):
        f = make_factors(rng, q, t, n, n, n, noise=noise)
        x = np.concatenate([R.from_euler("xyz", [0.02, 0.0, 0.01]).as_quat(), [0.6, 0.0, 0.0]])
        co, Ho, go = op.evaluate(f, x)
        cg, Hg, gg = g.evaluate(f, x)
        assert abs(co - cg) <= 1e-12 * max(1.0, abs(co))
        assert np.abs(Ho - Hg).max() <= 1e-10 * np.abs(Ho).max()
        assert np.abs(go - gg).max() <= 1e-10 * max(1.0, np.abs(go).max())
        xo, lo = op.ceres_solve(f, x)
        xg, lg = g.solve(f, x)
        assert np.abs(xo - xg).max() < 1e-9, (xo, xg)
        assert abs(lo[2] - lg[2]) <= 1e-12 * max(1.0, lo[2]) and abs(lo[3] - lg[3]) <= 1e-10 * max(1.0, lo[3])
    xg, _ = g.solve(np.zeros((0, 10)), x)
    assert (xg == x).all()
    g.close()


@pytest.mark.gpu
def test_solver_trust_region_paths_and_sizes(pkg, op):
    """Far starting points (rejected steps, shrinking radius), Huber-dominated problems and factor counts
    that select every register-resident variant of lm_solve_cluster (1 / 2 / 4 slots per thread, and the
    memory-streaming fallback above 16384 slots): same iterate and the same number of iterations as the
    restated Ceres trust-region loop."""
    from scipy.spatial.transform import Rotation as R
    rng = np.random.RandomState(5)
    q = R.from_euler("xyz", [0.05, -0.02, 0.1]).as_quat()
    t = np.array([1.0, 0.3, -0.2])
    g = pkg.Context()
    starts = [
        np.concatenate([R.from_euler("xyz", [0.6, -0.4, 0.9]).as_quat(), [6.0, -4.0, 3.0]]),   # far: steps get rejected
        np.concatenate([R.from_euler("xyz", [0.0, 0.0, 0.0]).as_quat(), [0.0, 0.0, 0.0]]),
        np.concatenate([q, t]),                                                                  # already at the optimum
    ]
    iters = set()
    for n_each, noise in ((30, 0.0), (1400, 0.05), (2800, 0.3), (5500, 0.05), (6000, 0.02)):
        f = make_factors(rng, q, t, n_each, n_each, n_each, noise=noise)
        for x in starts:
            xo, lo = op.ceres_solve(f, x)
            xg, lg = g.solve(f, x)
            assert int(lo[0]) == int(lg[0]), ("iterations", n_each, lo, lg)
            assert np.abs(xo - xg).max() < 1e-8, (n_each, xo, xg)
            assert abs(lo[2] - lg[2]) <= 1e-11 * max(1.0, lo[2]) and abs(lo[3] - lg[3]) <= 1e-9 * max(1.0, lo[3])
            iters.add(int(lg[0]))
    assert len(iters) > 1  # early termination and full-length runs were both exercised
    g.close()


def test_fits_against_independent_witness(pkg, op):
    """vloam_b200_fit (the mapping stage's own device fits: cyclic Jacobi, Householder) on >= 1e5 five-point sets per kind --
    noisy lines / planes / blobs and the degenerate families (collinear, coplanar, duplicates, identical) -- against
    (1) the numpy / LAPACK witness (committed fixture + the same generator at 120k sets): accept flags on every decided
    set, factors to ~1e-12; (2) the oracle's restated Eigen algorithms on ALL sets: flags equal, factors ~1e-12."""
    import fit_checks as fc
    import make_golden_fit as mg
    from test_oracle_math import _witness
    gold = dict(np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fit_sets.npz")))
    g = pkg.Context()
    ok, prm = g.fit(gold["line_sets"], 0)
    fc.check_line(ok, prm, _witness(gold, "line_"))
    ok, prm = g.fit(gold["plane_sets"], 1)
    fc.check_plane(ok, prm, _witness(gold, "plane_"))
    n = 120000
    for kind, seed in ((0, 991), (1, 992)):
        sets, fam = mg.fit_sets(n, seed)
        ok_g, prm_g = g.fit(sets, kind)
        ok_o, prm_o = op.fit(sets, kind)
        wl = mg.witness_line(sets) if kind == 0 else None
        nflag, err = fc.check_same(ok_g, prm_g, ok_o, prm_o, kind, wl["decided"] if kind == 0 else None)
        assert nflag == 0, "%d accept flags differ between the CUDA path and the oracle (kind %d)" % (nflag, kind)
        assert err < 1e-12, (kind, err)
        assert np.isfinite(prm_g).all()
        if kind == 0:
            knife = int(((ok_g != 0) != (ok_o != 0)).sum())   # lambda_2 == 3 lambda_1 to the last bit (exact lattices): either answer is legal
            assert knife <= 1e-3 * n, knife
            r = fc.check_line(ok_g, prm_g, wl)
        else:
            sub = slice(0, 20000)   # (the lstsq witness is a python loop)
            r = fc.check_plane(ok_g[sub], prm_g[sub], mg.witness_plane(sets[sub]))
        assert r["accepted"] > 0.5 * r["decided"] > 0
    assert len(g.fit(np.zeros((0, 5, 3), np.float32), 0)[0]) == 0
    g.close()


def test_solver_ill_conditioned_problems_match_oracle_qr(pkg, op):
    """The CUDA solver factors the 6x6 normal equations (L D L^T); Ceres -- and the oracle -- run Householder QR on the
    stacked Jacobian.  On corridor / single-plane factor sets with cond(J^T J) >= 1e8 the two must still give the same
    iterate within the pose tolerance, the same number of iterations and the same final cost."""
    from scipy.spatial.transform import Rotation as R
    from test_oracle_math import corridor_factors
    rng = np.random.RandomState(31)
    q = R.from_euler("xyz", [0.01, -0.02, 0.03]).as_quat()
    t = np.array([0.8, -0.1, 0.05])
    g = pkg.Context()
    worst = worst_cost = 0.0
    for kind in ("corridor", "single_plane"):
        for n in (300, 3000, 9000):
            f = corridor_factors(rng, q, t, n, kind)
            _, H, _ = op.evaluate(f, np.concatenate([q, t]))
            ev = np.linalg.eigvalsh(H)
            assert ev[-1] / max(ev[0], 1e-300) >= 1e8
            for dx in ([0.05, 0.02, -0.03], [0.5, -0.3, 0.2]):
                x0 = np.concatenate([R.from_euler("xyz", [0.012, -0.018, 0.036]).as_quat(), t + dx])
                xo, lo = op.ceres_solve(f, x0)
                xg, lg = g.solve(f, x0)
                assert int(lo[0]) == int(lg[0]), (kind, n, lo, lg)
                assert np.abs(xo[4:] - xg[4:]).max() < POS_TOL and np.abs(xo[:4] - xg[:4]).max() < ROT_TOL, (kind, n, xo, xg)
                assert abs(lo[3] - lg[3]) <= 1e-5 * max(1.0, lo[3])   # the squared condition number costs ~8 digits of the cost (measured: 3e-7 relative)
                worst = max(worst, np.abs(xo - xg).max()); worst_cost = max(worst_cost, abs(lo[3] - lg[3]) / max(1.0, lo[3]))
    print("ill-conditioned solves: worst |x_gpu - x_oracle| = %.3g, worst relative final-cost difference %.3g" % (worst, worst_cost))
    g.close()


def test_deskew_factors_and_solver_match_oracle(pkg, op):
    """DISTORTION == true: residuals and the analytic Jacobians THROUGH Eigen's slerp (lm_factor_deskew) against the oracle's
    dual numbers running the literal functors (lidarFactor.hpp:29-36, 86-93): normal equations <= 1e-10, the solve's iterate
    < 1e-9 with the same iteration count; s == 1 everywhere reproduces the plain path's numbers; all three slerp branches
    (w > 0, w < 0, |w| >= 1 - eps)."""
    from scipy.spatial.transform import Rotation as R
    rng = np.random.RandomState(41)
    q = R.from_euler("xyz", [0.01, -0.02, 0.03]).as_quat()
    t = np.array([0.8, -0.1, 0.05])
    g = pkg.Context()
    starts = [np.concatenate([R.from_euler("xyz", [0.02, 0.0, 0.01]).as_quat(), [0.6, 0.0, 0.0]]),
              np.concatenate([-R.from_euler("xyz", [0.3, -0.2, 0.4]).as_quat(), [0.5, -0.1, 0.3]]),
              np.array([0, 0, 0, 1.0, 0.4, 0.0, 0.0])]
    for noise, n in ((0.0, 40), (0.05, 700), (0.2, 3000)):
        f = make_factors(rng, q, t, n, n, 0, noise=noise)
        s = rng.uniform(-0.02, 1.02, len(f))     # relTime leaves [0, 1] slightly at the sweep seam (SR.cpp:294-296)
        for x in starts:
            co, Ho, go = op.evaluate(f, x, s)
            cg, Hg, gg = g.evaluate(f, x, s)
            assert abs(co - cg) <= 1e-12 * max(1.0, abs(co))
            assert np.abs(Ho - Hg).max() <= 1e-10 * np.abs(Ho).max()
            assert np.abs(go - gg).max() <= 1e-10 * max(1.0, np.abs(go).max())
            xo, lo = op.ceres_solve(f, x, s)
            xg, lg = g.solve(f, x, s)
            assert int(lo[0]) == int(lg[0])
            assert np.abs(xo - xg).max() < 1e-9, (xo, xg)
            # s == 1 through the slerp path == the plain path (exactly-zero scale derivatives, SURVEY A.5)
            c1, H1, g1 = g.evaluate(f, x, np.ones(len(f)))
            c0, H0, g0 = g.evaluate(f, x)
            assert abs(c1 - c0) <= 1e-13 * max(1.0, c0) and np.abs(H1 - H0).max() <= 1e-11 * np.abs(H0).max()
    g.close()


@pytest.mark.parametrize("sensor", [0, 1])
def test_deskew_pipeline_teacher_forced(pkg, op, synth, street, sensor):
    """VLOAM_FLAG_DISTORTION end to end (SURVEY 8 f3): TransformToStart with the per-point s (LO.cpp:152-173), factors with s,
    three teacher-forced frames: association indices bit-exact, every stage output as in the plain mode, poses within
    tolerance; and the flag really changes the odometry."""
    frames = 3
    traj = synth.trajectory(frames)
    o, g = op.Oracle(distortion=1, **KW[sensor]), pkg.Context(distortion=1, **KW[sensor])
    plain = op.Oracle(**KW[sensor])
    g.set_capture(True)
    for k in range(frames):
        scan = street.scan(sensor, traj[k], 1000 + k)
        if k > 0:
            teacher_force(o, g)
        o.scan_registration(scan); g.begin_frame(); g.scan_registration(scan)
        o.laser_odometry(); g.laser_odometry()
        o.laser_mapping(); g.laser_mapping()
        check_frame(o, g, k)
        plain.process(scan)
    assert np.abs(plain.get("lo.pose") - o.get("lo.pose")).max() > 1e-6
    g.close()
    # free-running with the look-ahead path
    o, g = op.Oracle(distortion=1, **KW[sensor]), pkg.Context(distortion=1, **KW[sensor])
    for k in range(frames):
        scan = street.scan(sensor, traj[k], 1000 + k)
        o.process(scan)
        pose = g.process_frame(scan)
        pose_close(o.get("lo.pose")[:7], pose[:7]); pose_close(o.get("lm.pose")[:7], pose[7:])
    g.close()


def teacher_force(o, g):
    g.set_last(o.get("lo.cornerLast"), o.get("lo.surfLast"))
    g.set("lo.pose", o.get("lo.pose"))
    g.set("lm.state", o.get("lm.state")[:4])
    g.set("lm.pose", o.get("lm.pose"))
    g.set("lm.cornerMap", o.get("lm.cornerMap"))
    g.set("lm.surfMap", o.get("lm.surfMap"))


def check_frame(o, g, k):
    check_sr(o, g)
    if k > 0:
        for nm in ("lo.assoc.corner0", "lo.assoc.surf0", "lo.assoc.corner1", "lo.assoc.surf1"):
            assert_bits_equal(o.get(nm), g.get(nm), nm)
    lo_o, lo_g = o.get("lo.pose"), g.get("lo.pose")
    pose_close(lo_o[:7], lo_g[:7]); pose_close(lo_o[7:], lo_g[7:])
    for nm in ("lm.cornerStack", "lm.surfStack", "lm.cornerFromMap", "lm.surfFromMap", "lm.validInd"):
        assert_bits_equal(o.get(nm), g.get(nm), nm)
    so, sg = o.get("lm.state"), g.get("lm.state")
    assert (so == sg).all(), (so, sg)
    if so[4]:
        for p in (0, 1):
            for kind in ("c", "s"):
                oi, gi = o.get("lm.knn.%sidx%d" % (kind, p)), g.get("lm.knn.%sidx%d" % (kind, p))
                od, gd = o.get("lm.knn.%sd2%d" % (kind, p)), g.get("lm.knn.%sd2%d" % (kind, p))
                acc = od[:, 4] < 1.0   # parity contract: inside the acceptance ball (SURVEY A.2)
                assert_bits_equal(oi[acc], gi[acc], "knn idx")
                assert_bits_equal(od[acc], gd[acc], "knn d2")
                assert_bits_equal(o.get("lm.knn.%sok%d" % (kind, p)), g.get("lm.knn.%sok%d" % (kind, p)), "fit accept flags")
    lm_o, lm_g = o.get("lm.pose"), g.get("lm.pose")
    pose_close(lm_o[:7], lm_g[:7]); pose_close(lm_o[7:], lm_g[7:])
    assert o.get("lm.cornerMap") == g.get("lm.cornerMap"), "corner map bytes"
    assert o.get("lm.surfMap") == g.get("lm.surfMap"), "surf map bytes"


@pytest.mark.parametrize("sensor,frames", [(0, 4), (1, 4), (2, 2), (3, 3)])
def test_teacher_forced_chain(pkg, op, synth, street, sensor, frames):
    """Every frame the GPU context is loaded with the oracle's state, then both run SR -> LO -> LM; every
    stage output must agree (SURVEY 7.2 item 8)."""
    traj = synth.trajectory(frames)
    o, g = op.Oracle(**KW[sensor]), pkg.Context(**KW[sensor])
    g.set_capture(True)
    for k in range(frames):
        scan = street.scan(sensor, traj[k], 1000 + k)
        if k > 0:
            teacher_force(o, g)
        o.scan_registration(scan)
        g.begin_frame(); g.scan_registration(scan)
        o.laser_odometry(); g.laser_odometry()
        o.laser_mapping(); g.laser_mapping()
        check_frame(o, g, k)
    g.close()


def test_free_running_sequence_pose_tolerance(pkg, op, synth, street):
    """No teacher forcing: 10 HDL-64 frames through process_frame; poses stay within tolerance."""
    traj = synth.trajectory(10)
    o, g = op.Oracle(**KW[1], knn_backend=1), pkg.Context(**KW[1])
    for k in range(10):
        scan = street.scan(1, traj[k], 1000 + k)
        o.process(scan)
        pose = g.process_frame(scan)
        pose_close(o.get("lo.pose")[:7], pose[:7])
        pose_close(o.get("lm.pose")[:7], pose[7:])
    assert np.linalg.norm(pose[11:14] - traj[9][:3]) < 0.05
    g.close()


def test_vo_prior_path(pkg, op, synth, street):
    """detach_VO_LO == false (LO.cpp:237-250): the prior overwrites para_q / para_t at the top of both passes."""
    from scipy.spatial.transform import Rotation as R
    traj = synth.trajectory(2)
    o, g = op.Oracle(**KW[0]), pkg.Context(**KW[0])
    pq, pt = R.from_euler("z", 0.004).as_quat(), np.array([0.95, 0.0, 0.0])
    for k in range(2):
        scan = street.scan(0, traj[k], 1000 + k)
        o.scan_registration(scan); g.begin_frame(); g.scan_registration(scan)
        o.laser_odometry(pq, pt); r = g.laser_odometry(pq, pt)
    lo = o.get("lo.pose")
    pose_close(lo[:7], np.concatenate([r["q_w_curr"], r["t_w_curr"]]))
    pose_close(lo[7:], np.concatenate([r["q_last_curr"], r["t_last_curr"]]))
    g.close()


def test_mapping_skip_frame(pkg, op, synth, street):
    """mapping_skip_frame = 2: odd frames only propagate the high-frequency pose (LM.cpp:197-201)."""
    kw = dict(KW[0], mapping_skip_frame=2)
    traj = synth.trajectory(4)
    o, g = op.Oracle(**kw), pkg.Context(**kw)
    for k in range(4):
        scan = street.scan(0, traj[k], 1000 + k)
        o.process(scan)
        pose = g.process_frame(scan)
        pose_close(o.get("lo.pose")[:7], pose[:7])
    assert o.get("lm.surfMap") == g.get("lm.surfMap")
    pose_close(o.get("lm.pose")[:7], g.get("lm.pose")[:7])
    g.close()


def test_cube_window_roll_and_outside_appends(pkg, op, synth, street):
    """Jump the mapper 200+ m: the 21x21x11 window rolls (LM.cpp:252-444), the old cubes fall outside the
    5x5x3 sub-map and fresh points land in cubes that were never filtered (raw tail path)."""
    o, g = op.Oracle(**KW[1]), pkg.Context(**KW[1])
    scan = street.scan(1, [0, 0, 0, 0, 0, 0], 1000)
    o.process(scan); g.process_frame(scan)
    for jump in ([480.0, -470.0, 0.0], [-520.0, 30.0, 20.0], [60.0, 60.0, 0.0]):
        pose = o.get("lm.pose"); pose[11:14] = jump
        o.set("lm.pose", pose); g.set("lm.pose", pose)
        o.process(scan); g.process_frame(scan)
        assert (o.get("lm.state")[:3] == g.get("lm.state")[:3]).all()
        assert_bits_equal(o.get("lm.validInd"), g.get("lm.validInd"), "validInd")
        assert o.get("lm.cornerMap") == g.get("lm.cornerMap") and o.get("lm.surfMap") == g.get("lm.surfMap")
    g.close()


def test_full_size_planted_map_frame(pkg, op, synth):
    """BASELINE config C3 at full size: ~1M-point planted sub-map, one HDL-64 sweep.  kNN / fit parity
    against the oracle (KD-tree backend, itself checked against brute force) and the size-independent
    properties: re-filtering is idempotent on the planted cubes, map grows by <= Qc + Qs."""
    world = synth.World(1234, 1, 190.0)
    cb, sb = synth.cubes_blob(world.plant(0, 0.4, seed=99), 0.4), synth.cubes_blob(world.plant(1, 0.8, seed=98), 0.8)
    assert synth.blob_counts(cb).sum() + synth.blob_counts(sb).sum() > 900_000
    o, g = op.Oracle(**KW[1], knn_backend=1), pkg.Context(**KW[1])
    g.set_capture(True)
    for x in (o, g):
        x.set("lm.cornerMap", cb); x.set("lm.surfMap", sb)
    traj = synth.trajectory(2)
    for k in range(2):
        scan = world.scan(1, traj[k], 1000 + k)
        if k > 0:
            teacher_force(o, g)
        o.scan_registration(scan); g.begin_frame(); g.scan_registration(scan)
        o.laser_odometry(); g.laser_odometry()
        o.laser_mapping(); g.laser_mapping()
        check_frame(o, g, k)
    n_before = synth.blob_counts(sb).sum()
    n_after = synth.blob_counts(g.get("lm.surfMap")).sum()
    assert n_before <= n_after <= n_before + 2 * len(g.get("lm.surfStack")) + 100000
    g.close()


def test_mirror_classes_follow_reference_call_sequence(pkg, op, synth, street):
    """LidarOdometryMapping.reset / scanRegistrationIO / laserOdometryIO / laserMappingIO (MAIN.cpp:143-190)."""
    lom = pkg.LidarOdometryMapping(**KW[0])
    o = op.Oracle(**KW[0])
    traj = synth.trajectory(2)
    for k in range(2):
        scan = street.scan(0, traj[k], 1000 + k)
        lom.reset(); lom.scanRegistrationIO(scan); lom.laserOdometryIO(); lom.laserMappingIO()
        o.process(scan)
    full, sharp, less, flat, lessflat = lom.scan_registration.output()
    assert_bits_equal(o.get("sr.sharp"), sharp, "sharp"); assert_bits_equal(o.get("sr.lessFlat"), lessflat, "lessFlat")
    q, t, cl, sl, fr, skip = lom.laser_odometry.output()
    assert not skip
    assert_bits_equal(o.get("lo.cornerLast"), cl, "cornerLast")
    pose_close(o.get("lm.pose")[:7], np.concatenate(lom.laser_mapping.pose))
    lom.ctx.close()


def test_device_exact_math_matches_glibc(pkg):
    """The DEVICE compile of exact_math.h (the fdlibm atanf / atan2f of the scan-registration kernels, SR.cpp:185-187, 217, 263)
    against this machine's glibc, bit for bit: 4M bit patterns across every exponent, lidar-like magnitudes, and the special
    values.  (tests/test_exact_math.py checks the host compile of the same header.)"""
    import ctypes
    libm = ctypes.CDLL("libm.so.6")
    rng = np.random.RandomState(5)
    n = 1 << 22
    xb = rng.randint(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    yb = rng.randint(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    x = xb.view(np.float32).copy(); y = yb.view(np.float32).copy()
    x[n // 2:] = (rng.uniform(-120, 120, n - n // 2) * rng.choice([1.0, 1e-3, 1e-6], n - n // 2)).astype(np.float32)
    y[n // 2:] = (rng.uniform(-120, 120, n - n // 2) * rng.choice([1.0, 1e-4], n - n // 2)).astype(np.float32)
    sp = np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, np.nan, 1e-40, -1e-40, 3e38], np.float32)
    x[:100] = np.repeat(sp, 10); y[:100] = np.tile(sp, 10)
    g = pkg.Context()
    a_dev, b_dev = g.exact_math(y, x)
    g.close()
    # glibc through a tiny C loop (ctypes per element would take minutes)
    import subprocess, tempfile
    src = r'''
#include <math.h>
void ref(const float* y, const float* x, int n, float* a, float* b) { for (int i = 0; i < n; ++i) { a[i] = atanf(x[i]); b[i] = atan2f(y[i], x[i]); } }
'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "r.c"), "w").write(src)
        so = os.path.join(d, "r.so")
        subprocess.run(["gcc", "-O1", "-fno-builtin", "-ffp-contract=off", "-shared", "-fPIC", os.path.join(d, "r.c"), "-o", so, "-lm"], check=True)
        L = ctypes.CDLL(so)
        a_ref, b_ref = np.zeros(n, np.float32), np.zeros(n, np.float32)
        L.ref(y.ctypes.data_as(ctypes.c_void_p), x.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(n), a_ref.ctypes.data_as(ctypes.c_void_p),
              b_ref.ctypes.data_as(ctypes.c_void_p))
    for dev, ref, what in ((a_dev, a_ref, "atanf"), (b_dev, b_ref, "atan2f")):
        same = (dev.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(dev) & np.isnan(ref))
        assert same.all(), "%s: %d of %d results differ from glibc, first at x = %r y = %r" % (what, int((~same).sum()), n, x[~same][:1], y[~same][:1])


def test_golden_fixture_on_gpu(pkg):
    """tests/golden/vlp16_pair.npz (oracle outputs, made by tests/make_golden.py) reproduced by the CUDA path."""
    gold = dict(np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vlp16_pair.npz")))
    g = pkg.Context(**KW[0])
    g.set_capture(True)
    for k in range(2):
        pose = g.process_frame(gold["scan%d" % k])
        for nm in ("sr.sharp", "sr.flat", "sr.lessSharp", "sr.lessFlat"):
            assert_bits_equal(gold["f%d.%s" % (k, nm)], g.get(nm), nm)
        assert (g.get("sr.label").astype(np.int8) == gold["f%d.label" % k]).all()
        pose_close(gold["f%d.lo.pose" % k][:7], pose[:7]); pose_close(gold["f%d.lm.pose" % k][:7], pose[7:])
    assert_bits_equal(gold["f1.assoc.corner0"], g.get("lo.assoc.corner0"), "assoc")
    assert_bits_equal(gold["f1.assoc.surf0"], g.get("lo.assoc.surf0"), "assoc")
    g.close()


def test_errors_are_reported(pkg):
    with pytest.raises(pkg.VloamError):
        pkg.Context(n_scans=48)            # SR.cpp:58-61: only 16 / 32 / 64 (128 extension)
    g = pkg.Context()
    with pytest.raises(pkg.VloamError):
        g.get("no.such.buffer")
    with pytest.raises(pkg.VloamError):
        g.set("lm.surfMap", b"123")
    g.close()


def test_cpp_adapter_classes(pkg, op, synth, street, tmp_path):
    """vloam_adapter.hpp: the reference's C++ stage classes (reference signatures: default constructors, init(), input() with
    the reference's argument lists, publish() writing VloamTF) driven stage by stage from a compiled C++14 program over the
    C ABI; counts and poses must match the oracle."""
    import subprocess
    from test_abi import build_cpp_program
    exe = build_cpp_program("adapter_smoke", tmp_path)
    traj = synth.trajectory(2)
    o = op.Oracle(**KW[0])
    files = []
    for k in range(2):
        scan = street.scan(0, traj[k], 1000 + k)
        f = str(tmp_path / ("scan%d.bin" % k))
        scan.tofile(f)
        files.append(f)
        o.process(scan)
    out = subprocess.run([exe] + files, check=True, capture_output=True, text=True).stdout
    assert "adapter ok" in out, out
    last = [l for l in out.splitlines() if l.startswith("frame 1")][0].split()
    assert int(last[3]) == len(o.get("sr.laserCloud")) and int(last[5]) == len(o.get("sr.sharp")) and int(last[11]) == len(o.get("sr.lessFlat"))
    odom = np.array([float(v) for v in last[14:17]]); mapped = np.array([float(v) for v in last[19:22]])
    assert np.abs(odom - o.get("lo.pose")[4:7]).max() < POS_TOL and np.abs(mapped - o.get("lm.pose")[4:7]).max() < POS_TOL


@pytest.mark.parametrize("sensor,skip", [(0, 1), (1, 1), (0, 2)])
def test_reference_main_node_excerpt_runs_against_oracle(pkg, op, synth, street, tmp_path, sensor, skip):
    """The reference's caller, verbatim (tests/cpp/main_node_excerpt.cpp = vloam_main_node.cpp:118-124, 144, 186-190),
    on top of the adapter: parameters from the (stand-in) ROS parameter server, three frames; the poses it leaves in VloamTF
    (world_LOT_base_last, world_MOT_base_last, base_prev_LOT_base_curr: LO.cpp:612-620, LM.cpp:834-861) against the oracle."""
    import subprocess
    from test_abi import build_cpp_program
    exe = build_cpp_program("main_node_excerpt", tmp_path)
    kw = dict(KW[sensor], mapping_skip_frame=skip)
    traj = synth.trajectory(3)
    o = op.Oracle(**kw)
    files, want = [], []
    for k in range(3):
        scan = street.scan(sensor, traj[k], 1000 + k)
        f = str(tmp_path / ("scan%d.bin" % k))
        scan.tofile(f)
        files.append(f)
        o.process(scan)
        want.append((o.get("lo.pose").copy(), o.get("lm.pose").copy(), o.get("lm.poseHighFreq").copy() if skip > 1 else None))
    args = [str(kw["n_scans"]), repr(kw["minimum_range"]), repr(kw["line_res"]), repr(kw["plane_res"]), str(skip)]
    out = subprocess.run([exe] + args + files, check=True, capture_output=True, text=True).stdout
    assert "main node excerpt ok" in out, out
    rows = [l.split() for l in out.splitlines() if l.startswith("frame ")]
    assert len(rows) == 3
    for k, r in enumerate(rows):
        lo = np.array([float(v) for v in r[3:10]]); mo = np.array([float(v) for v in r[11:18]]); f2f = np.array([float(v) for v in r[19:22]])
        pose_close(want[k][0][:7], lo)
        skipped = skip > 1 and (k + 1) % skip != 0          # LO.cpp:668-678: frameCount % mapping_skip_frame after the increment
        pose_close(want[k][2][:7] if skipped else want[k][1][:7], mo)
        assert np.abs(f2f - want[k][0][11:14]).max() < POS_TOL


def test_lo_association_non_monotone_rings(pkg, op, synth, street):
    """int(intensity) of the last clouds made non-monotone on purpose (what a negative relTime does,
    SURVEY 7.2 item 3): the scans must still stop exactly where the reference's `break`s do."""
    rng = np.random.RandomState(5)
    traj = synth.trajectory(2)
    o, g = op.Oracle(**KW[1]), pkg.Context(**KW[1])
    for k in range(2):
        scan = street.scan(1, traj[k], 1000 + k)
        o.scan_registration(scan); g.begin_frame(); g.scan_registration(scan)
        if k == 0:
            o.laser_odometry(); g.laser_odometry()
    corner, surf = o.get("lo.cornerLast").copy(), o.get("lo.surfLast").copy()
    for cl in (corner, surf):
        glitch = rng.rand(len(cl)) < 0.02
        cl[glitch, 3] -= 1.0                       # ring - 1 in the middle of ring's block
        cl[rng.rand(len(cl)) < 0.002, 3] += 3.0    # and a few early `break` triggers
        cl[:, 3] = np.maximum(cl[:, 3], 0.0)
    o.set_last(corner, surf); g.set_last(corner, surf)
    x = np.array([0.0, 0.0, 0.002, 1.0, 0.9, 0.01, 0.0])
    x[:4] /= np.linalg.norm(x[:4])
    co, so = o.lo_associate(x)
    cg_, sg = g.lo_associate(x)
    assert_bits_equal(co, cg_, "corner association"); assert_bits_equal(so, sg, "surf association")
    assert (so[:, 2] >= 0).sum() > 100
    g.close()


def test_config_c4_os1_128_against_2m_map(pkg, op, synth):
    """BASELINE config C4: OS1-128 dense sweeps (~257k points, 128-beam extension) against a ~1.9M-point
    planted map; two teacher-forced frames, every stage compared."""
    world = synth.World(1234, 2, 190.0)
    cb, sb = synth.cubes_blob(world.plant(0, 0.4, seed=99), 0.4), synth.cubes_blob(world.plant(1, 0.8, seed=98), 0.8)
    assert synth.blob_counts(cb).sum() + synth.blob_counts(sb).sum() > 1_800_000
    o, g = op.Oracle(**KW[2], knn_backend=1), pkg.Context(**KW[2])
    g.set_capture(True)
    for x in (o, g):
        x.set("lm.cornerMap", cb); x.set("lm.surfMap", sb)
    for k in range(2):
        scan = world.scan(2, [1.0 * k, 0.0, 0.0, 0.0, 0.0, 0.0], 1000 + k)
        assert len(scan) > 240_000
        if k > 0:
            teacher_force(o, g)
        o.scan_registration(scan); g.begin_frame(); g.scan_registration(scan)
        o.laser_odometry(); g.laser_odometry()
        o.laser_mapping(); g.laser_mapping()
        check_frame(o, g, k)
    g.close()


def test_process_frame_is_deterministic(pkg, synth, street):
    """Two contexts fed the same sweeps give bit-identical poses and maps (fixed reduction orders)."""
    traj = synth.trajectory(5)
    scans = [street.scan(1, traj[k], 1000 + k) for k in range(5)]
    outs = []
    for _ in range(2):
        g = pkg.Context(**KW[1])
        poses = [g.process_frame(s).copy() for s in scans]
        outs.append((np.array(poses), g.get("lm.surfMap"), g.get("lm.cornerMap")))
        g.close()
    assert (outs[0][0] == outs[1][0]).all()
    assert outs[0][1] == outs[1][1] and outs[0][2] == outs[1][2]


@pytest.mark.gpu
def test_speculative_submap_equals_inline_build(pkg, op, synth, street):
    """The sub-map of frame k+1 is gathered and cell-sorted right after frame k's map update, for the window
    frame k used; lm_prepare lets the in-line build run instead when the window moved.  A 28 m drive (the
    centre cube changes at x = 25 m), a mapping_skip_frame = 2 run and a run whose map offset is edited from
    outside so that the window moves two frames later must give bit-identical poses and maps with the
    speculation switched off (VLOAM_NO_GRID); the long drive is also checked against the oracle."""
    import os
    def run(spec, kw, sensor, poses, check_oracle, shift_after=None):
        if spec: os.environ.pop("VLOAM_NO_GRID", None)
        else: os.environ["VLOAM_NO_GRID"] = "1"
        try:
            g = pkg.Context(**kw)
        finally:
            os.environ.pop("VLOAM_NO_GRID", None)
        o = op.Oracle(**kw) if check_oracle else None
        out, centres = [], []
        for k, p in enumerate(poses):
            scan = street.scan(sensor, [p[0], p[1], 0, p[2], 0, 0], 3000 + k)
            out.append(g.process_frame(scan).copy())
            centres.append(tuple(g.get("lm.validInd")[:1]))
            if o is not None:
                o.process(scan)
            if shift_after is not None and k == shift_after:
                pose = g.get("lm.pose"); pose[11] += 23.0   # t_wmap_wodom: the mapper now sits 2 m from a cube face
                g.set("lm.pose", pose)
        maps = (g.get("lm.cornerMap"), g.get("lm.surfMap"))
        if o is not None:
            assert o.get("lm.cornerMap") == maps[0] and o.get("lm.surfMap") == maps[1]
            pose_close(o.get("lm.pose")[:7], g.get("lm.pose")[:7])
        g.close()
        return np.array(out), maps, centres
    drive = [(1.1 * k, 0.05 * k, 0.002 * k) for k in range(27)]
    cases = ((KW[0], 0, drive, True, None), (dict(KW[0], mapping_skip_frame=2), 0, drive[:8], False, None), (KW[1], 1, drive[:7], False, 2))
    for i, (kw, sensor, poses, chk, shift) in enumerate(cases):
        pa, ma, ca = run(True, kw, sensor, poses, chk, shift)
        pb, mb, cb = run(False, kw, sensor, poses, False, shift)
        assert (pa == pb).all(), "poses differ with / without the speculative sub-map"
        assert ma[0] == mb[0] and ma[1] == mb[1], "maps differ with / without the speculative sub-map"
        if i != 1:
            assert len(set(ca)) > 1, "the window never moved: the mismatch path was not exercised"


@pytest.mark.gpu
def test_full_resolution_cloud_registration(pkg, op, synth, street):
    """LaserMapping::publish's loop over laserCloudFullRes (LM.cpp:901-905): every kept point of the sweep through
    pointAssociateToMap with the mapped pose -- bit-exact against the oracle given the same pose."""
    o, g = op.Oracle(**KW[1]), pkg.Context(**KW[1])
    traj = synth.trajectory(3)
    for k in range(3):
        scan = street.scan(1, traj[k], 1000 + k)
        o.process(scan); g.process_frame(scan)
        g.set("lm.pose", o.get("lm.pose"))           # same pose on both sides: the comparison is about the transform
        reg_o, reg_g = o.get("lm.fullResRegistered"), g.register_full_cloud()
        assert len(reg_g) == len(o.get("sr.laserCloud")) > 50000
        assert_bits_equal(reg_o, reg_g, "registered full-resolution cloud")
    g.close()


@pytest.mark.gpu
def test_concurrent_sequences_match_sequential_runs(pkg, synth, street):
    """BASELINE config C5 on one GPU: independent sequences, one context and one host thread each, replayed
    concurrently (every context owns four streams and a helper thread).  Poses and final maps must be bit-identical
    to the same sequences replayed one after the other."""
    import threading
    nseq, frames = 3, 6
    seqs = []
    for q in range(nseq):
        traj = synth.trajectory(frames, seed=300 + q)
        seqs.append([street.scan(0, traj[k], 7000 + 100 * q + k) for k in range(frames)])

    def replay(q, out):
        g = pkg.Context(**KW[0])
        poses = [g.process_frame(s).copy() for s in seqs[q]]
        out[q] = (np.array(poses), g.get("lm.cornerMap"), g.get("lm.surfMap"))
        g.close()

    alone, together = [None] * nseq, [None] * nseq
    for q in range(nseq):
        replay(q, alone)
    th = [threading.Thread(target=replay, args=(q, together)) for q in range(nseq)]
    for t in th: t.start()
    for t in th: t.join()
    for q in range(nseq):
        assert together[q] is not None, "a replay thread died"
        assert (alone[q][0] == together[q][0]).all(), "poses differ when sequences share the GPU"
        assert alone[q][1] == together[q][1] and alone[q][2] == together[q][2], "maps differ when sequences share the GPU"


@pytest.mark.gpu
def test_map_pools_grow_instead_of_failing(pkg, synth, street):
    """The cube pools are bump-allocated; when one is half full it is doubled at sync point S2.  A context that
    starts with tiny pools (VLOAM_POOL_POINTS) must replay a sequence with the same poses and map bytes as one
    with the default 16M / 48M-point pools, and importing a map larger than the pool must grow it too."""
    import os
    traj = synth.trajectory(8)
    scans = [street.scan(1, traj[k], 1000 + k) for k in range(8)]

    def replay():
        g = pkg.Context(**KW[1])
        poses = [g.process_frame(s).copy() for s in scans]
        maps = (g.get("lm.cornerMap"), g.get("lm.surfMap"))
        return g, np.array(poses), maps

    g0, p0, m0 = replay()
    os.environ["VLOAM_POOL_POINTS"] = "4096"
    try:
        g1, p1, m1 = replay()
    finally:
        os.environ.pop("VLOAM_POOL_POINTS", None)
    assert (p0 == p1).all() and m0 == m1
    assert len(m0[1]) > 4851 * 4 + 3 * 4096 * 16, "the surf map never outgrew the tiny pool: growth was not exercised"
    os.environ["VLOAM_POOL_POINTS"] = "4096"
    try:
        g2 = pkg.Context(**KW[1])
    finally:
        os.environ.pop("VLOAM_POOL_POINTS", None)
    g2.set("lm.cornerMap", m0[0]); g2.set("lm.surfMap", m0[1])   # import into pools that are too small
    assert g2.get("lm.surfMap") == m0[1] and g2.get("lm.cornerMap") == m0[0]
    for g in (g0, g1, g2):
        g.close()


@pytest.mark.gpu
def test_lookahead_scan_registration_gives_identical_results(pkg, synth, street):
    """vloam_b200_prefetch_scan[_device]: the next sweep's scan registration runs on a side stream, into a spare set
    of buffers, underneath the current sweep's odometry and mapping, and is adopted by the next process_frame call with
    the same buffer.  Poses and maps must equal the plain replay bit for bit -- with device and host buffers, when a
    registered sweep is never processed, and when another sweep is processed in between."""
    import torch
    traj = synth.trajectory(8)
    scans = [street.scan(1, traj[k], 1000 + k) for k in range(8)]
    a = pkg.Context(**KW[1])
    ref = [a.process_frame(s).copy() for s in scans]
    ref_maps = (a.get("lm.cornerMap"), a.get("lm.surfMap"))
    ref_sharp = a.get("sr.sharp")
    a.close()
    pinned = [torch.from_numpy(s).pin_memory() for s in scans]
    dev = [torch.from_numpy(s).cuda() for s in scans]
    for mode in ("device", "host", "device2", "host2", "mixed2", "mixed"):
        b = pkg.Context(**KW[1])
        pose = np.zeros(14)
        for k in range(8):
            if mode == "device2":  # two sweeps registered ahead: sweep k+2 is uploaded + registered while sweep k+1's odometry runs beside sweep k's mapping
                for j in (k + 1, k + 2):
                    if j < 8: b.prefetch_device(dev[j].data_ptr(), dev[j].shape[0], 4)
                b.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, pose.ctypes.data)
            elif mode == "host2":
                for j in (k + 1, k + 2):
                    if j < 8: b.prefetch_ptr(pinned[j].data_ptr(), pinned[j].shape[0], 4)
                b.process_frame_ptr(pinned[k].data_ptr(), pinned[k].shape[0], 4, pose.ctypes.data)
            elif mode == "mixed2":  # two ahead with a sweep that never comes (k = 2 registers 3 and 7), a gap (nothing registered at k = 4) and a re-start
                if k < 2 or k > 4:
                    for j in (k + 1, k + 2):
                        if j < 8: b.prefetch_ptr(pinned[j].data_ptr(), pinned[j].shape[0], 4)
                if k == 2: b.prefetch_ptr(pinned[3].data_ptr(), pinned[3].shape[0], 4); b.prefetch_device(dev[7].data_ptr(), dev[7].shape[0], 4)
                if k == 3: b.prefetch_device(dev[0].data_ptr(), dev[0].shape[0], 4)
                if k % 2: b.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, pose.ctypes.data)
                else: b.process_frame_ptr(pinned[k].data_ptr(), pinned[k].shape[0], 4, pose.ctypes.data)
            elif mode == "device":
                if k + 1 < 8: b.prefetch_device(dev[k + 1].data_ptr(), dev[k + 1].shape[0], 4)
                b.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, pose.ctypes.data)
            elif mode == "host":
                if k + 1 < 8: b.prefetch_ptr(pinned[k + 1].data_ptr(), pinned[k + 1].shape[0], 4)
                b.process_frame_ptr(pinned[k].data_ptr(), pinned[k].shape[0], 4, pose.ctypes.data)
            else:  # registrations that are skipped, stale or for the wrong sweep
                if k in (0, 1, 4): b.prefetch_ptr(pinned[k + 1].data_ptr(), pinned[k + 1].shape[0], 4)
                if k == 2: b.prefetch_ptr(pinned[7].data_ptr(), pinned[7].shape[0], 4)   # far-ahead sweep: stale by the time it comes
                if k == 5: b.prefetch_device(dev[0].data_ptr(), dev[0].shape[0], 4)        # never processed
                if k % 2: b.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, pose.ctypes.data)
                else: b.process_frame_ptr(pinned[k].data_ptr(), pinned[k].shape[0], 4, pose.ctypes.data)
            assert (pose == ref[k]).all(), "%s: frame %d differs with the look-ahead" % (mode, k)
        assert (b.get("lm.cornerMap"), b.get("lm.surfMap")) == ref_maps, mode
        assert_bits_equal(ref_sharp, b.get("sr.sharp"), "sr.sharp of the last sweep (%s)" % mode)
        b.close()


@pytest.mark.gpu
def test_segmented_update_sort_global_fallback(pkg, synth, street):
    """The map update buckets its (segment | voxel | order) keys by cube segment and sorts every bucket in shared
    memory; buckets above the capacity are sorted in a global scratch area.  With the capacity forced down to 64
    keys (VLOAM_SEG_CAP, read once per process: run in a subprocess) nearly every bucket takes that path and the maps
    must not change."""
    import os, subprocess, sys, hashlib
    code = (
        "import importlib, sys, hashlib, numpy as np\n"
        "sys.path.insert(0, %r)\n"
        "pkg = importlib.import_module('vloam-noted_b200')\n"
        "w = pkg.synth.World(1234, 0, 160.0); traj = pkg.synth.trajectory(5)\n"
        "g = pkg.Context(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8)\n"
        "poses = [g.process_frame(w.scan(1, traj[k], 1000 + k)).copy() for k in range(5)]\n"
        "h = hashlib.sha256(np.array(poses).tobytes() + g.get('lm.cornerMap') + g.get('lm.surfMap')).hexdigest()\n"
        "print('HASH', h)\n" % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    out = {}
    for cap in ("", "64"):
        env = dict(os.environ)
        env.pop("VLOAM_SEG_CAP", None)
        if cap: env["VLOAM_SEG_CAP"] = cap
        r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        out[cap] = [l for l in r.stdout.splitlines() if l.startswith("HASH")][0]
    assert out[""] == out["64"]
