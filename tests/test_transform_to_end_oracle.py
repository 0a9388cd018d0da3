"""VLOAM_FLAG_TRANSFORM_TO_END on the CPU: the restated TransformToEnd block (tests/transform_to_end_ref.py, LO.cpp:176-193 /
537-556) against an independent rotation-matrix / scipy restatement, the moving-sensor sweeps of the synthetic generator, and
the accuracy the flag exists for: on sweeps that are not motion-compensated, de-skew carried through to the map
(DISTORTION + TRANSFORM_TO_END) drifts less than no de-skew and than DISTORTION alone."""
import math

import numpy as np
import pytest
from scipy.spatial.transform import Rotation, Slerp

import transform_to_end_ref as ref

KW16 = dict(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4)


def _matrix(q):
    """Eigen's _transformVector of a (possibly non-unit) quaternion as a matrix: I + 2 w [u]x + 2 [u]x^2."""
    x, y, z, w = q
    U = np.array([[0, -z, y], [z, 0, -x], [-y, x, 0]])
    return np.eye(3) + 2 * w * U + 2 * U @ U


def _independent_to_end(p, pose, distortion):
    q, t = np.asarray(pose[:4]), np.asarray(pose[4:7])
    v = p[:, :3].astype(np.float64)
    if distortion:
        s = (p[:, 3] - np.trunc(p[:, 3])).astype(np.float64) / 0.1
        rots = Slerp([0.0, 1.0], Rotation.from_quat([[0, 0, 0, 1], q / np.linalg.norm(q)]))(np.clip(s, 0.0, 1.0))
        # Eigen's slerp extrapolates for s outside [0, 1]; the generated intensities keep s in [0, 1)
        un = rots.apply(v) + s[:, None] * t[None, :]
    else:
        un = v @ _matrix(q).T + t[None, :]
    un = un.astype(np.float32).astype(np.float64)
    Minv = np.linalg.inv(_matrix(q))
    return (un - t[None, :]) @ Minv.T


def _random_cloud(rng, n, rings=16):
    p = np.empty((n, 4), np.float32)
    p[:, :3] = rng.uniform(-60, 60, (n, 3))
    p[:, 3] = rng.randint(0, rings, n) + 0.1 * rng.uniform(0, 0.999, n)  # ring + SCAN_PERIOD * relTime (SR.cpp:305-306)
    return p


@pytest.mark.parametrize("distortion", [0, 1])
def test_transform_to_end_matches_independent_restatement(distortion):
    rng = np.random.RandomState(11 + distortion)
    for trial in range(12):
        q = Rotation.from_rotvec(rng.randn(3) * (0.02 if trial % 2 else 0.3)).as_quat()
        if trial % 3 == 0:
            q = -q                                   # w < 0: the slerp flips its second scale (shortest arc)
        q = q * (1.0 + 1e-9 * rng.randn())           # not exactly unit, as after the solver's update
        pose = np.concatenate([q, rng.randn(3) * 1.5])
        p = _random_cloud(rng, 4000)
        got = ref.transform_to_end(p, pose, distortion)
        want = _independent_to_end(p, pose, distortion)
        assert np.abs(got[:, :3] - want).max() < 1e-6 + 2e-7 * np.abs(want).max(), trial
        assert (got[:, 3] == np.trunc(p[:, 3])).all()
    # s = 1 for every point without DISTORTION: TransformToEnd(TransformToStart^-1 ...) is the identity up to float rounding
    p = _random_cloud(rng, 1000)
    pose = np.concatenate([Rotation.from_rotvec([0.01, -0.02, 0.05]).as_quat(), [0.9, 0.1, -0.02]])
    if not distortion:
        assert np.abs(ref.transform_to_end(p, pose, 0)[:, :3] - p[:, :3]).max() < 1e-4


@pytest.mark.parametrize("distortion", [0, 1])
def test_first_frame_identity_keeps_coordinates(distortion):
    """On the first frame q_last_curr is identity and t_last_curr zero: coordinates come out unchanged, the intensity is truncated."""
    p = _random_cloud(np.random.RandomState(5), 3000)
    out = ref.transform_to_end(p, [0, 0, 0, 1, 0, 0, 0], distortion)
    assert (out[:, :3].view(np.uint32) == p[:, :3].view(np.uint32)).all()
    assert (out[:, 3] == np.trunc(p[:, 3])).all() and (out[:, 3] != p[:, 3]).any()


def test_stage_driver_without_flag_is_the_plain_oracle(op, synth, street):
    """The stage-by-stage driver with the flag off leaves the oracle exactly where Pipeline::process does."""
    traj = synth.trajectory(3)
    a, b = op.Oracle(**KW16), op.Oracle(**KW16)
    for k in range(3):
        scan = street.scan(synth.VLP16, traj[k], 1000 + k)
        a.process(scan)
        ref.oracle_step(b, scan, 0, False)
    for name in ("lo.pose", "lm.pose", "lo.cornerLast", "lo.surfLast", "lm.cornerStack", "lm.surfStack"):
        assert a.get_raw(name) == b.get_raw(name), name
    assert a.get_raw("lm.cornerMap") == b.get_raw("lm.cornerMap") and a.get_raw("lm.surfMap") == b.get_raw("lm.surfMap")


def test_flag_moves_the_last_clouds_to_the_sweep_end(op, synth, street):
    """With the flag the oracle's last clouds are TransformToEnd of the raw ones, with this frame's q/t_last_curr."""
    scans, _ = ref.moving_drive(street, synth.VLP16, 3)
    o = op.Oracle(distortion=1, **KW16)
    for k in range(3):
        ref.oracle_step(o, scans[k], 1, True)
    pose = o.get("lo.pose")[7:14]
    assert np.abs(pose[4:7]).max() > 0.5                         # ~1 m per sweep
    o2 = op.Oracle(distortion=1, **KW16)
    for k in range(2):
        ref.oracle_step(o2, scans[k], 1, True)
    o2.scan_registration(scans[2]); o2.laser_odometry()
    assert (o2.get("lo.pose") == o.get("lo.pose")).all()
    for nm in ("lo.cornerLast", "lo.surfLast"):
        want = ref.transform_to_end(o2.get(nm), pose, 1)
        assert (o.get(nm).view(np.uint32) == want.view(np.uint32)).all(), nm


def test_scan_moving_with_equal_poses_is_scan(synth, street):
    for sensor in (synth.VLP16, synth.HDL64):
        for order in (0, 1):
            pose = [4.0, 0.3, 0.01, 0.02, 0.001, -0.002]
            a = street.scan(sensor, pose, 99 + sensor, order=order)
            b = street.scan_moving(sensor, pose, list(pose), 99 + sensor, order=order)
            assert a.tobytes() == b.tobytes()


def test_scan_moving_points_lie_on_the_world(synth, street):
    """Every point mapped back with the truth pose of its azimuth column (interpolated here independently with scipy's Slerp)
    lies on the world: ground returns at the ground height.  The static pose does not explain them."""
    p0 = np.array([2.0, 0.2, 0.0, 0.0, 0.0, 0.0])
    p1 = np.array([3.2, 0.35, 0.02, math.radians(3.0), math.radians(0.4), math.radians(-0.3)])
    scan = street.scan_moving(synth.VLP16, p0, p1, 42, range_sigma=0.0, nan_frac=0.0)
    n_az, az0 = 1800, -3.1
    ori = -np.arctan2(scan[:, 1].astype(np.float64), scan[:, 0].astype(np.float64))
    col = np.round(np.mod(ori - az0, 2 * np.pi) / (2 * np.pi / n_az)).astype(int) % n_az
    f = col / n_az
    q0, t0 = synth.pose_to_qt(p0)
    q1, t1 = synth.pose_to_qt(p1)
    R = Slerp([0.0, 1.0], Rotation.from_quat([q0, q1]))(f)
    world = R.apply(scan[:, :3].astype(np.float64)) + (t0[None, :] + f[:, None] * (t1 - t0)[None, :])
    ground = np.abs(world[:, 2] + 1.8) < 2e-3
    assert ground.mean() > 0.3
    # the same points placed with the start pose: the ground no longer fits where the sensor has tilted / climbed
    still = Rotation.from_quat(q0).apply(scan[:, :3].astype(np.float64)) + t0[None, :]
    assert (np.abs(still[ground, 2] + 1.8) > 2e-3).mean() > 0.5
    # and the moving sweep really differs from a static one
    assert street.scan(synth.VLP16, p0, 42, range_sigma=0.0, nan_frac=0.0).tobytes() != scan.tobytes()


def drift_table(op, synth, world, n=30, lengths=(4.0, 8.0, 12.0)):
    """Segment drift (translation %, deg/m) of the mapped and the odometry poses against the truth sweep-end poses, for the flag
    settings none / DISTORTION / DISTORTION + TRANSFORM_TO_END on a seeded moving VLP-16 street drive.  The runner `step`
    lets the GPU measurement script produce the same table from the device."""
    scans, traj = ref.moving_drive(world, synth.VLP16, n)
    gt = [synth.pose_to_qt(traj[k + 1]) for k in range(n)]
    table = {}
    for name, d, te in (("none", 0, False), ("D", 1, False), ("D+TO_END", 1, True)):
        o = op.Oracle(distortion=d, knn_backend=1, **KW16)
        lo, lm = [], []
        for k in range(n):
            ref.oracle_step(o, scans[k], d, te)
            a, b = o.get("lo.pose"), o.get("lm.pose")
            lo.append((a[0:4], a[4:7])); lm.append((b[0:4], b[4:7]))
        table[name] = {"mapped": ref.segment_drift(lm, gt, lengths), "odometry": ref.segment_drift(lo, gt, lengths)}
    return table


def test_deskew_to_end_has_the_lowest_drift(op, synth, street):
    table = drift_table(op, synth, street)
    print("segment drift (translation %%, deg/m): %s" % table)
    for kind in ("mapped", "odometry"):
        best = table["D+TO_END"][kind]
        for other in ("none", "D"):
            assert best[0] < table[other][kind][0], (kind, other, table)
            assert best[1] < table[other][kind][1], (kind, other, table)
