"""Restatement of the reference's TransformToEnd block (laser_odometry.cpp:176-193, applied at 537-556) on top of the CPU oracle.
TEST INFRASTRUCTURE.

PARITY UNPINNED: the reference is not in this checkout, and the block sits under `if (0)` there (as in A-LOAM, whose KITTI
sweeps come motion-compensated).  Its content is restated from SURVEY a11 / section 8(f) and the A-LOAM structure VLOAM-NOTED
inherits, not from the CUDA code:

    for every point p of cornerPointsLessSharp, surfPointsLessFlat and laserCloudFullRes, after the solve and the pose
    accumulation (LO.cpp:524-525) and before the swap (LO.cpp:558-564) -- on the first frame too:
        un  = TransformToStart(p)                                  pcl::PointXYZI (float); s from the intensity under
                                                                   DISTORTION, s = 1 otherwise (LO.cpp:152-173)
        end = q_last_curr.inverse() * (Vector3d(un) - t_last_curr) double, stored as float
        end.intensity = int(p.intensity)

Eigen semantics: Quaterniond * Vector3d is _transformVector (uv = 2 u x v; v + w uv + u x uv), inverse() is the conjugate
divided by squaredNorm (q_last_curr is not exactly unit after the solver's update), Identity.slerp(s, q) as in
oracle_ceres.cpp.  Every f64 expression is written in the reference's operation order; numpy evaluates them with plain IEEE
operations, so the f32 results are the ones the reference computes (up to the last bit of the libm sin / acos, which the f32
rounding absorbs).

The oracle itself is unchanged: `oracle_step` drives it stage by stage and swaps the end clouds in with its `lo.last` import,
which is exactly the state LaserOdometry hands on (the end clouds become laserCloudCornerLast / SurfLast, the next solve's
targets and the mapping stage's input)."""
import math

import numpy as np

SCAN_PERIOD = 0.1  # LO.h:93


def qrot(q, v):
    """Eigen Quaterniond * Vector3d (_transformVector) in f64; q = (x, y, z, w) per row or one quaternion, v[n, 3]."""
    q = np.broadcast_to(np.asarray(q, np.float64), (len(v), 4)) if np.ndim(q) == 1 else np.asarray(q, np.float64)
    ux, uy, uz, w = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    vx, vy, vz = v[:, 0], v[:, 1], v[:, 2]
    uvx = uy * vz - uz * vy
    uvy = uz * vx - ux * vz
    uvz = ux * vy - uy * vx
    uvx = uvx + uvx; uvy = uvy + uvy; uvz = uvz + uvz
    cx = uy * uvz - uz * uvy
    cy = uz * uvx - ux * uvz
    cz = ux * uvy - uy * uvx
    return np.stack([(vx + w * uvx) + cx, (vy + w * uvy) + cy, (vz + w * uvz) + cz], axis=1)


def point_s(intensity):
    """(intensity - int(intensity)) as float, / SCAN_PERIOD as double (LO.cpp:156-160)."""
    i = np.asarray(intensity, np.float32)
    return (i - np.trunc(i)).astype(np.float32).astype(np.float64) / SCAN_PERIOD


def slerp_identity(s, q):
    """Eigen: Quaterniond::Identity().slerp(s, q) for an array of s."""
    d = float(q[3])
    absd = abs(d)
    if absd >= 1.0 - 2.220446049250313e-16:
        scale0, scale1 = 1.0 - s, s.copy()
    else:
        theta = math.acos(absd)
        sin_theta = math.sin(theta)
        scale0 = np.sin((1.0 - s) * theta) / sin_theta
        scale1 = np.sin(s * theta) / sin_theta
    if d < 0.0:
        scale1 = -scale1
    return np.stack([scale1 * q[0], scale1 * q[1], scale1 * q[2], scale0 + scale1 * q[3]], axis=1)


def transform_to_start(p, pose, distortion):
    """TransformToStart (LO.cpp:152-173): float32[n, 3] in the frame of the sweep's start.  pose = q_last_curr[4] + t_last_curr[3]."""
    pose = np.asarray(pose, np.float64)
    q, t = pose[:4], pose[4:7]
    v = np.asarray(p, np.float32)[:, :3].astype(np.float64)
    if distortion:
        s = point_s(p[:, 3])
        r = qrot(slerp_identity(s, q), v)
        return np.stack([r[:, k] + s * t[k] for k in range(3)], axis=1).astype(np.float32)
    r = qrot(q, v)
    return (r + t[None, :]).astype(np.float32)


def transform_to_end(p, pose, distortion):
    """TransformToEnd (LO.cpp:176-193) of float32[n, 4] points -> float32[n, 4]."""
    p = np.ascontiguousarray(p, np.float32).reshape(-1, 4)
    pose = np.asarray(pose, np.float64)
    q, t = pose[:4], pose[4:7]
    un = transform_to_start(p, pose, distortion).astype(np.float64)
    n2 = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]
    qi = np.array([-q[0] / n2, -q[1] / n2, -q[2] / n2, q[3] / n2])
    r = qrot(qi, un - t[None, :])
    out = np.empty_like(p)
    out[:, :3] = r.astype(np.float32)
    out[:, 3] = np.trunc(p[:, 3]).astype(np.int32).astype(np.float32)
    return out


def associate_to_map(p, pose):
    """pointAssociateToMap (LM.cpp:154-164), pose = q_w_curr[4] + t_w_curr[3]."""
    pose = np.asarray(pose, np.float64)
    r = qrot(pose[:4], np.asarray(p, np.float32)[:, :3].astype(np.float64))
    out = np.array(p, np.float32, copy=True)
    out[:, :3] = (r + pose[None, 4:7]).astype(np.float32)
    return out


def register_full(full, lo_pose14, lm_pose7, distortion):
    """LM.cpp:901-905 on the laserCloudFullRes LaserOdometry hands over under the flag: pointAssociateToMap(TransformToEnd(p))."""
    return associate_to_map(transform_to_end(full, lo_pose14[7:14], distortion), lm_pose7)


def oracle_step(o, scan, distortion, to_end, prior=None):
    """One frame through the oracle (MAIN.cpp:143-144, 186-190), with the TransformToEnd block between solveLO and the mapping
    stage when to_end is set.  Returns the end-frame full-resolution cloud (the raw one without the flag)."""
    o.scan_registration(scan)
    if prior is None:
        o.laser_odometry()
    else:
        o.laser_odometry(*prior)
    full = o.get("sr.laserCloud")
    if to_end:
        pose = o.get("lo.pose")[7:14]
        o.set_last(transform_to_end(o.get("lo.cornerLast"), pose, distortion), transform_to_end(o.get("lo.surfLast"), pose, distortion))
        full = transform_to_end(full, pose, distortion)
    o.laser_mapping()
    return full


# ---- KITTI-style segment drift ------------------------------------------------------------------------------------------
def _rot(q):
    x, y, z, w = np.asarray(q, np.float64) / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def _T(q, t):
    T = np.eye(4)
    T[:3, :3] = _rot(q)
    T[:3, 3] = t
    return T


def segment_drift(est, gt, lengths):
    """KITTI odometry metric: for every start frame and segment length L (m of truth path), the relative pose error of the
    segment, translation as % of L and rotation in deg/m, averaged.  est / gt: lists of (q xyzw, t).  A constant offset of
    which instant within a sweep the poses refer to cancels in the relative poses."""
    Te = [_T(q, t) for q, t in est]
    Tg = [_T(q, t) for q, t in gt]
    dist = np.concatenate([[0.0], np.cumsum([np.linalg.norm(Tg[k + 1][:3, 3] - Tg[k][:3, 3]) for k in range(len(Tg) - 1)])])
    terr, rerr = [], []
    for i in range(len(Tg)):
        for L in lengths:
            j = int(np.searchsorted(dist, dist[i] + L))
            if j >= len(Tg):
                continue
            E = np.linalg.inv(np.linalg.inv(Tg[i]) @ Tg[j]) @ (np.linalg.inv(Te[i]) @ Te[j])
            terr.append(np.linalg.norm(E[:3, 3]) / L * 100.0)
            rerr.append(math.degrees(math.acos(max(-1.0, min(1.0, (np.trace(E[:3, :3]) - 1) / 2)))) / L)
    return float(np.mean(terr)), float(np.mean(rerr))


def moving_drive(world, sensor, n, seed=314, step=1.0, yaw_amp_deg=8.0):
    """n moving sweeps of a street drive: sweep k spans truth poses traj[k] -> traj[k + 1], about `step` m and up to ~2 deg of
    yaw per sweep (the heading swings +-yaw_amp_deg with a 24-sweep period, so the drive stays in the street corridor).
    Returns (scans, traj) with len(traj) == n + 1; traj[k + 1] is sweep k's end pose."""
    rng = np.random.RandomState(seed)
    traj = np.zeros((n + 1, 6))
    for k in range(1, n + 1):
        yaw = math.radians(yaw_amp_deg) * math.sin(2 * math.pi * k / 24) + math.radians(0.05) * rng.randn()
        traj[k, 0] = traj[k - 1, 0] + step * math.cos(yaw)
        traj[k, 1] = traj[k - 1, 1] + step * math.sin(yaw)
        traj[k, 2] = 0.01 * rng.randn()
        traj[k, 3] = yaw
        traj[k, 4:6] = np.radians(0.05) * rng.randn(2)
    scans = [world.scan_moving(sensor, traj[k], traj[k + 1], 7000 + k) for k in range(n)]
    return scans, traj
