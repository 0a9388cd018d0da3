"""Seeded synthetic sweeps, trajectories and planted cube maps (SURVEY.md section 8d).

Thin ctypes wrapper over synth/synth.cpp plus the numpy code that lays planted
points out the way LaserMapping stores them (21x21x11 cubes of 50 m, each cube
voxel-filtered, laser_mapping.cpp:741-808)."""
import ctypes
import numpy as np
from . import _build

VLP16, HDL64, OS128, HDL32 = 0, 1, 2, 3
N_SCANS = {VLP16: 16, HDL64: 64, OS128: 128, HDL32: 32}
CUBE_W, CUBE_H, CUBE_D = 21, 21, 11
CUBE_NUM = CUBE_W * CUBE_H * CUBE_D

_lib = None


def lib():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(_build.build_synth())
        L.vloam_synth_world_create.restype = ctypes.c_void_p
        L.vloam_synth_world_create.argtypes = [ctypes.c_uint64, ctypes.c_int, ctypes.c_double]
        L.vloam_synth_world_destroy.argtypes = [ctypes.c_void_p]
        L.vloam_synth_scan.restype = ctypes.c_int
        L.vloam_synth_scan.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_double,
                                       ctypes.c_double, ctypes.c_double, ctypes.c_int, ctypes.c_double, ctypes.c_void_p, ctypes.c_int]
        L.vloam_synth_scan_moving.restype = ctypes.c_int
        L.vloam_synth_scan_moving.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_double,
                                              ctypes.c_double, ctypes.c_double, ctypes.c_int, ctypes.c_double, ctypes.c_void_p, ctypes.c_int]
        L.vloam_synth_plant.restype = ctypes.c_int
        L.vloam_synth_plant.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                        ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_void_p, ctypes.c_int]
        _lib = L
    return _lib


class World:
    """kind 0: open street; 1: dense towers (~1M-point sub-map, config C3); 2: taller (~2M, C4)."""

    def __init__(self, seed=1234, kind=0, extent=160.0):
        self.h = lib().vloam_synth_world_create(seed, kind, extent)
        self.kind, self.extent = kind, extent

    def __del__(self):
        if getattr(self, "h", None):
            lib().vloam_synth_world_destroy(self.h)
            self.h = None

    def scan(self, sensor, pose, seed, range_sigma=0.02, nan_frac=0.01, max_range=120.0, order=0, az0=-3.1):
        """One sweep from pose (x,y,z,yaw,pitch,roll). Returns float32[n,4] (x,y,z,0), KITTI layout."""
        cap = 300000
        out = np.empty((cap, 4), np.float32)
        p = np.ascontiguousarray(pose, np.float64)
        n = lib().vloam_synth_scan(self.h, sensor, p.ctypes.data, seed, range_sigma, nan_frac, max_range, order, az0,
                                   out.ctypes.data, cap)
        assert n >= 0
        return out[:n].copy()

    def scan_moving(self, sensor, pose_start, pose_end, seed, range_sigma=0.02, nan_frac=0.01, max_range=120.0, order=0, az0=-3.1):
        """One sweep from a sensor moving from pose_start to pose_end (x,y,z,yaw,pitch,roll) during the sweep, not motion-compensated:
        azimuth column k of n_az is cast from the pose at fraction k / n_az (translation linear, rotation slerp) -- the order in which
        ScanRegistration's relTime grows (SR.cpp:183-298) -- and its points are in the sensor frame of that instant.
        pose_start == pose_end reproduces scan(pose_start) byte for byte."""
        cap = 300000
        out = np.empty((cap, 4), np.float32)
        p0 = np.ascontiguousarray(pose_start, np.float64)
        p1 = np.ascontiguousarray(pose_end, np.float64)
        n = lib().vloam_synth_scan_moving(self.h, sensor, p0.ctypes.data, p1.ctypes.data, seed, range_sigma, nan_frac, max_range, order, az0,
                                          out.ctypes.data, cap)
        assert n >= 0
        return out[:n].copy()

    def plant(self, kind_out, leaf, center=(0.0, 0.0), half_width=125.0, zlo=-10.0, zhi=140.0, seed=99):
        cap = 6_000_000
        out = np.empty((cap, 4), np.float32)
        n = lib().vloam_synth_plant(self.h, seed, kind_out, leaf, center[0], center[1], half_width, zlo, zhi, out.ctypes.data, cap)
        return out[:n].copy()


def trajectory(n, seed=77, step=1.0, yaw_sigma_deg=0.5, tilt_sigma_deg=0.1):
    """Ego-motion: `step` m/frame forward, yaw random walk, small pitch/roll/z jitter."""
    rng = np.random.RandomState(seed)
    poses = np.zeros((n, 6))
    yaw = 0.0
    x = y = 0.0
    for k in range(1, n):
        yaw += np.deg2rad(yaw_sigma_deg) * rng.randn()
        yaw = float(np.clip(yaw, -0.05, 0.05))  # stay inside the street corridor
        x += step * np.cos(yaw)
        y += step * np.sin(yaw)
        poses[k] = (x, y, 0.02 * rng.randn(), yaw, np.deg2rad(tilt_sigma_deg) * rng.randn(), np.deg2rad(tilt_sigma_deg) * rng.randn())
    return poses


def pose_to_qt(p):
    """(x,y,z,yaw,pitch,roll) -> (q xyzw, t)."""
    cy, sy = np.cos(p[3] / 2), np.sin(p[3] / 2)
    cp, sp = np.cos(p[4] / 2), np.sin(p[4] / 2)
    cr, sr = np.cos(p[5] / 2), np.sin(p[5] / 2)
    q = np.array([sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy, cr * cp * sy - sr * sp * cy, cr * cp * cy + sr * sp * sy])
    return q, np.array(p[:3], float)


def cubes_blob(points, leaf, cen=(10, 10, 5)):
    """Lay world-frame points out as LaserMapping's cube arrays: cube index as
    laser_mapping.cpp:747-761, one point per `leaf` voxel (float32 arithmetic of
    pcl::VoxelGrid), each cube in ascending (iz, iy, ix) voxel order.  Returns the
    `lm.cornerMap` / `lm.surfMap` blob: int32 counts[4851] then float32 points."""
    pts = np.ascontiguousarray(points, np.float32)
    if len(pts) == 0:
        return np.zeros(CUBE_NUM, np.int32).tobytes()
    c = []
    for a in range(3):
        v = pts[:, a].astype(np.float64) + 25.0
        ci = np.trunc(v / 50.0).astype(np.int64) + cen[a]
        ci[v < 0] -= 1
        c.append(ci)
    ok = (c[0] >= 0) & (c[0] < CUBE_W) & (c[1] >= 0) & (c[1] < CUBE_H) & (c[2] >= 0) & (c[2] < CUBE_D)
    pts, c = pts[ok], [ci[ok] for ci in c]
    cube = c[0] + CUBE_W * c[1] + CUBE_W * CUBE_H * c[2]
    inv = np.float32(1.0) / np.float32(leaf)
    vox = [np.floor(pts[:, a] * inv).astype(np.int64) for a in range(3)]
    order = np.lexsort((vox[0], vox[1], vox[2], cube))
    pts, cube = pts[order], cube[order]
    vox = [v[order] for v in vox]
    keep = np.ones(len(pts), bool)
    keep[1:] = (cube[1:] != cube[:-1]) | (vox[0][1:] != vox[0][:-1]) | (vox[1][1:] != vox[1][:-1]) | (vox[2][1:] != vox[2][:-1])
    pts, cube = pts[keep], cube[keep]
    counts = np.bincount(cube, minlength=CUBE_NUM).astype(np.int32)
    return counts.tobytes() + np.ascontiguousarray(pts).tobytes()


def blob_counts(blob):
    return np.frombuffer(blob[:CUBE_NUM * 4], np.int32)
