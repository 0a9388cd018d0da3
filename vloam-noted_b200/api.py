"""ctypes binding of libvloam_b200.so (include/vloam_b200.h) and a host-side mirror of the
reference's stage classes (ScanRegistration / LaserOdometry / LaserMapping /
LidarOdometryMapping, src/lidar_odometry_mapping) on top of it.

There is no CPU fallback: if the CUDA library is missing or a call fails, this raises."""
import ctypes
import os
import numpy as np
from . import _build

CLOUD_FULL, CLOUD_SHARP, CLOUD_LESS_SHARP, CLOUD_FLAT, CLOUD_LESS_FLAT, CLOUD_CORNER_LAST, CLOUD_SURF_LAST, CLOUD_FULL_RES = range(8)
FLAG_DISTORTION, FLAG_TRANSFORM_TO_END = 1, 2  # vloam_b200_params.reserved

EXPORTS = [
    "vloam_b200_default_params", "vloam_b200_create", "vloam_b200_destroy", "vloam_b200_last_error", "vloam_b200_begin_frame",
    "vloam_b200_scan_registration", "vloam_b200_prefetch_scan", "vloam_b200_prefetch_scan_device", "vloam_b200_scan_registration_device", "vloam_b200_get_cloud", "vloam_b200_laser_odometry",
    "vloam_b200_laser_mapping", "vloam_b200_process_frame", "vloam_b200_process_frame_device", "vloam_b200_synchronize",
    "vloam_b200_stream", "vloam_b200_kernel_launches", "vloam_b200_set_timing", "vloam_b200_stage_ms", "vloam_b200_debug_get",
    "vloam_b200_debug_set", "vloam_b200_profile_kernel", "vloam_b200_profile_result", "vloam_b200_profile_table", "vloam_b200_profile_timeline", "vloam_b200_register_full_cloud", "vloam_b200_lo_associate", "vloam_b200_voxel_grid", "vloam_b200_evaluate", "vloam_b200_solve", "vloam_b200_fit", "vloam_b200_evaluate_deskew", "vloam_b200_solve_deskew", "vloam_b200_exact_math",
    "vloam_b200_publish_map", "vloam_b200_get_map",
]


class Params(ctypes.Structure):
    """vloam_b200_params: the ROS parameters of the three init() functions."""
    _fields_ = [("n_scans", ctypes.c_int), ("minimum_range", ctypes.c_float), ("line_res", ctypes.c_float),
                ("plane_res", ctypes.c_float), ("mapping_skip_frame", ctypes.c_int), ("reserved", ctypes.c_int)]


class VloamError(RuntimeError):
    pass


_lib = None


def load_lib(build=False):
    """Load the CUDA C-ABI library; raises if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if build:
        _build.build_cuda()
    if not os.path.exists(_build.LIB):
        raise VloamError("%s not built: run `python -c 'import __graft_entry__ as g; g.build()'`" % _build.LIB)
    L = ctypes.CDLL(_build.LIB)
    vp, ci, cd = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    L.vloam_b200_default_params.argtypes = [ctypes.POINTER(Params)]
    L.vloam_b200_create.argtypes = [ctypes.POINTER(Params), ci, ctypes.POINTER(vp)]
    L.vloam_b200_destroy.argtypes = [vp]
    L.vloam_b200_last_error.argtypes = [vp]
    L.vloam_b200_last_error.restype = ctypes.c_char_p
    L.vloam_b200_begin_frame.argtypes = [vp]
    L.vloam_b200_scan_registration.argtypes = [vp, vp, ci, ci]
    L.vloam_b200_scan_registration_device.argtypes = [vp, vp, ci, ci]
    L.vloam_b200_prefetch_scan.argtypes = [vp, vp, ci, ci]
    L.vloam_b200_prefetch_scan_device.argtypes = [vp, vp, ci, ci]
    L.vloam_b200_get_cloud.argtypes = [vp, ci, vp, ci]
    L.vloam_b200_laser_odometry.argtypes = [vp, vp, vp, ci, vp, vp, vp, vp, vp]
    L.vloam_b200_laser_mapping.argtypes = [vp, vp, vp]
    L.vloam_b200_process_frame.argtypes = [vp, vp, ci, ci, vp]
    L.vloam_b200_process_frame_device.argtypes = [vp, vp, ci, ci, vp]
    L.vloam_b200_synchronize.argtypes = [vp]
    L.vloam_b200_stream.argtypes = [vp]
    L.vloam_b200_stream.restype = vp
    L.vloam_b200_kernel_launches.argtypes = [vp]
    L.vloam_b200_kernel_launches.restype = ctypes.c_longlong
    L.vloam_b200_set_timing.argtypes = [vp, ci]
    L.vloam_b200_stage_ms.argtypes = [vp, vp]
    L.vloam_b200_debug_get.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_long]
    L.vloam_b200_debug_get.restype = ctypes.c_long
    L.vloam_b200_debug_set.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_long]
    L.vloam_b200_lo_associate.argtypes = [vp, vp, vp, vp]
    L.vloam_b200_voxel_grid.argtypes = [vp, vp, ci, ctypes.c_float, vp, ci]
    L.vloam_b200_evaluate.argtypes = [vp, vp, ci, vp, vp, vp, vp]
    L.vloam_b200_solve.argtypes = [vp, vp, ci, vp, vp]
    L.vloam_b200_evaluate_deskew.argtypes = [vp, vp, vp, ci, vp, vp, vp, vp]
    L.vloam_b200_solve_deskew.argtypes = [vp, vp, vp, ci, vp, vp]
    L.vloam_b200_register_full_cloud.argtypes = [vp, vp, ci]
    L.vloam_b200_fit.argtypes = [vp, vp, ci, ci, vp, vp]
    L.vloam_b200_exact_math.argtypes = [vp, vp, vp, ci, vp, vp]
    L.vloam_b200_publish_map.argtypes = [vp]
    L.vloam_b200_get_map.argtypes = [vp, vp, ci]
    _lib = L
    return L


def _decode(name, raw):
    if name in ("lm.cornerMap", "lm.surfMap"):
        return raw
    dt = {"sr.curvature": np.float32, "sr.label": np.int32, "sr.scanStartInd": np.int32, "sr.scanEndInd": np.int32,
          "lo.pose": np.float64, "lm.pose": np.float64, "lm.state": np.int32, "lm.validInd": np.int32,
          "lo.costs": np.float64, "lm.costs": np.float64, "alloc.count": np.int64, "lm.paths": np.int64}
    if name in dt:
        return np.frombuffer(raw, dt[name]).copy()
    if name.startswith("lo.assoc.corner"):
        return np.frombuffer(raw, np.int32).reshape(-1, 2).copy()
    if name.startswith("lo.assoc.surf"):
        return np.frombuffer(raw, np.int32).reshape(-1, 3).copy()
    if name.startswith("lm.knn."):
        kind = name[len("lm.knn."):-1]
        if kind in ("cidx", "sidx"):
            return np.frombuffer(raw, np.int32).reshape(-1, 5).copy()
        if kind in ("cd2", "sd2"):
            return np.frombuffer(raw, np.float32).reshape(-1, 5).copy()
        return np.frombuffer(raw, np.int32).copy()
    return np.frombuffer(raw, np.float32).reshape(-1, 4).copy()


class Context:
    """One vloam_b200_ctx: one sequence (several CUDA streams and a helper thread inside, include/vloam_b200.h)."""

    def __init__(self, n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8, mapping_skip_frame=1, device=0, distortion=0,
                 transform_to_end=False):
        """distortion: VLOAM_FLAG_DISTORTION (per-point de-skew in the odometry); transform_to_end: VLOAM_FLAG_TRANSFORM_TO_END (every
        sweep's less-sharp / less-flat / full-resolution clouds moved to the sweep end, LO.cpp:537-556)."""
        self.L = load_lib()
        flags = (FLAG_DISTORTION if distortion else 0) | (FLAG_TRANSFORM_TO_END if transform_to_end else 0)
        self.params = Params(n_scans, minimum_range, line_res, plane_res, mapping_skip_frame, flags)
        h = ctypes.c_void_p()
        r = self.L.vloam_b200_create(ctypes.byref(self.params), device, ctypes.byref(h))
        if r != 0:
            raise VloamError("vloam_b200_create failed with %d" % r)
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.vloam_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def _chk(self, r):
        if r < 0:
            raise VloamError("vloam_b200 error %d: %s" % (r, self.L.vloam_b200_last_error(self.h).decode()))
        return r

    @staticmethod
    def _scan(a):
        a = np.ascontiguousarray(a, np.float32)
        if a.ndim != 2 or a.shape[1] < 3:
            raise ValueError("scan must be float32[n, >=3]")
        return a

    def begin_frame(self):
        self._chk(self.L.vloam_b200_begin_frame(self.h))

    def scan_registration(self, scan):
        a = self._scan(scan)
        self._keep = a
        self._chk(self.L.vloam_b200_scan_registration(self.h, a.ctypes.data, a.shape[0], a.shape[1]))

    def scan_registration_device(self, dptr, n, stride):
        self._chk(self.L.vloam_b200_scan_registration_device(self.h, dptr, n, stride))

    def get_cloud(self, which):
        n = self._chk(self.L.vloam_b200_get_cloud(self.h, which, None, 0))
        out = np.empty((n, 4), np.float32)
        if n:
            self._chk(self.L.vloam_b200_get_cloud(self.h, which, out.ctypes.data, n))
        return out

    def register_full_cloud(self):
        """LaserMapping::publish's registration of laserCloudFullRes into the map frame (LM.cpp:901-905)."""
        n = self._chk(self.L.vloam_b200_register_full_cloud(self.h, None, 0))
        out = np.empty((n, 4), np.float32)
        if n:
            self._chk(self.L.vloam_b200_register_full_cloud(self.h, out.ctypes.data, n))
        return out

    def publish_map(self):
        """LaserMapping::publish's laserCloudMap (LM.cpp:884-899): queue its assembly from the map of the last mapped frame."""
        self._chk(self.L.vloam_b200_publish_map(self.h))

    def get_map(self):
        """The cloud of the last publish_map: float32[n, 4], for each of the 4851 cubes its corner then its surf points."""
        n = self._chk(self.L.vloam_b200_get_map(self.h, None, 0))
        out = np.empty((n, 4), np.float32)
        if n:
            n = self._chk(self.L.vloam_b200_get_map(self.h, out.ctypes.data, n))
        return out[:n]

    def laser_odometry(self, prior_q=None, prior_t=None, want_pose=True):
        qw, tw, ql, tl = np.zeros(4), np.zeros(3), np.zeros(4), np.zeros(3)
        skip = ctypes.c_int(0)
        use = prior_q is not None
        pq = np.ascontiguousarray(prior_q, np.float64) if use else None
        pt = np.ascontiguousarray(prior_t, np.float64) if use else None
        self._chk(self.L.vloam_b200_laser_odometry(
            self.h, pq.ctypes.data if use else None, pt.ctypes.data if use else None, 1 if use else 0,
            qw.ctypes.data if want_pose else None, tw.ctypes.data if want_pose else None,
            ql.ctypes.data if want_pose else None, tl.ctypes.data if want_pose else None, ctypes.byref(skip)))
        return {"q_w_curr": qw, "t_w_curr": tw, "q_last_curr": ql, "t_last_curr": tl, "skip_frame": bool(skip.value)}

    def laser_mapping(self, want_pose=True):
        q, t = np.zeros(4), np.zeros(3)
        self._chk(self.L.vloam_b200_laser_mapping(self.h, q.ctypes.data if want_pose else None, t.ctypes.data if want_pose else None))
        return q, t

    def process_frame(self, scan, want_pose=True):
        a = self._scan(scan)
        self._keep = a
        pose = np.zeros(14)
        self._chk(self.L.vloam_b200_process_frame(self.h, a.ctypes.data, a.shape[0], a.shape[1], pose.ctypes.data if want_pose else None))
        return pose

    def prefetch_ptr(self, host_ptr, n, stride):
        """Register the next sweep (pinned host pointer): its scan registration runs underneath the current sweep."""
        return self._chk(self.L.vloam_b200_prefetch_scan(self.h, host_ptr, n, stride))

    def prefetch_device(self, dptr, n, stride):
        return self._chk(self.L.vloam_b200_prefetch_scan_device(self.h, dptr, n, stride))

    def process_frame_ptr(self, host_ptr, n, stride, pose_ptr):
        return self._chk(self.L.vloam_b200_process_frame(self.h, host_ptr, n, stride, pose_ptr))

    def process_frame_device(self, dptr, n, stride, pose_ptr=None):
        return self._chk(self.L.vloam_b200_process_frame_device(self.h, dptr, n, stride, pose_ptr))

    def synchronize(self):
        self._chk(self.L.vloam_b200_synchronize(self.h))

    @property
    def stream(self):
        return self.L.vloam_b200_stream(self.h)

    @property
    def kernel_launches(self):
        return int(self.L.vloam_b200_kernel_launches(self.h))

    def set_timing(self, on=True):
        self._chk(self.L.vloam_b200_set_timing(self.h, 1 if on else 0))

    def stage_ms(self):
        ms = np.zeros(3, np.float32)
        self._chk(self.L.vloam_b200_stage_ms(self.h, ms.ctypes.data))
        return ms

    def get_raw(self, name):
        n = self._chk(self.L.vloam_b200_debug_get(self.h, name.encode(), None, 0))
        buf = ctypes.create_string_buffer(max(int(n), 1))
        self._chk(self.L.vloam_b200_debug_get(self.h, name.encode(), buf, n))
        return buf.raw[:n]

    def get(self, name):
        return _decode(name, self.get_raw(name))

    def set(self, name, data):
        raw = data if isinstance(data, (bytes, bytearray)) else np.ascontiguousarray(data).tobytes()
        self._chk(self.L.vloam_b200_debug_set(self.h, name.encode(), raw, len(raw)))

    def set_capture(self, on=True):
        self.set("debug.capture", np.array([1 if on else 0], np.int32))

    def set_last(self, corner, surf):
        c = np.ascontiguousarray(corner, np.float32)
        s = np.ascontiguousarray(surf, np.float32)
        self.set("lo.last", np.array([len(c), len(s)], np.int32).tobytes() + c.tobytes() + s.tobytes())

    def lo_associate(self, x):
        x = np.ascontiguousarray(x, np.float64)
        ns, nf = len(self.get("sr.sharp")), len(self.get("sr.flat"))
        ci = np.full((max(ns, 1), 2), -1, np.int32)
        si = np.full((max(nf, 1), 3), -1, np.int32)
        self._chk(self.L.vloam_b200_lo_associate(self.h, x.ctypes.data, ci.ctypes.data, si.ctypes.data))
        return ci[:ns], si[:nf]

    def voxel_grid(self, cloud, leaf):
        c = np.ascontiguousarray(cloud, np.float32)
        out = np.empty((max(len(c), 1), 4), np.float32)
        n = self._chk(self.L.vloam_b200_voxel_grid(self.h, c.ctypes.data, len(c), leaf, out.ctypes.data, len(out)))
        return out[:n].copy()

    def evaluate(self, factors, x, s=None):
        f = np.ascontiguousarray(factors, np.float64)
        x = np.ascontiguousarray(x, np.float64)
        cost, H, g = np.zeros(1), np.zeros((6, 6)), np.zeros(6)
        sv = None if s is None else np.ascontiguousarray(s, np.float64)
        self._chk(self.L.vloam_b200_evaluate_deskew(self.h, f.ctypes.data, None if sv is None else sv.ctypes.data, len(f), x.ctypes.data,
                                                    cost.ctypes.data, H.ctypes.data, g.ctypes.data))
        return cost[0], H, g

    def fit(self, near, kind):
        """Line (kind 0) / plane (kind 1) fit of the mapping stage on five-point sets float32[n,5,3] -> (ok[n], params[n,6])."""
        a = np.ascontiguousarray(near, np.float32).reshape(-1, 15)
        ok = np.zeros(max(len(a), 1), np.int32)
        prm = np.zeros((max(len(a), 1), 6))
        self._chk(self.L.vloam_b200_fit(self.h, a.ctypes.data, len(a), kind, ok.ctypes.data, prm.ctypes.data))
        return ok[:len(a)], prm[:len(a)]

    def exact_math(self, y, x):
        """(atanf(x), atan2f(y, x)) as the device code evaluates them (float32 arrays)."""
        y = np.ascontiguousarray(y, np.float32); x = np.ascontiguousarray(x, np.float32)
        a, b = np.zeros(len(x), np.float32), np.zeros(len(x), np.float32)
        self._chk(self.L.vloam_b200_exact_math(self.h, y.ctypes.data, x.ctypes.data, len(x), a.ctypes.data, b.ctypes.data))
        return a, b

    def solve(self, factors, x, s=None):
        f = np.ascontiguousarray(factors, np.float64)
        x = np.array(x, np.float64)
        log = np.zeros(4)
        sv = None if s is None else np.ascontiguousarray(s, np.float64)
        self._chk(self.L.vloam_b200_solve_deskew(self.h, f.ctypes.data, None if sv is None else sv.ctypes.data, len(f), x.ctypes.data, log.ctypes.data))
        return x, log


# ---- host-side mirror of the reference's stage classes ------------------------------------------
class ScanRegistration:
    """vloam::ScanRegistration (scan_registration.h:64-81): init / reset / input / output."""

    def __init__(self, ctx):
        self.ctx = ctx

    def init(self):
        pass  # parameters were bound at Context creation (scan_registration.cpp:42-92)

    def reset(self):
        pass  # buffers are overwritten by the next input(); LidarOdometryMapping.reset() calls begin_frame

    def input(self, laserCloudIn):
        self.ctx.scan_registration(laserCloudIn)

    def output(self):
        g = self.ctx.get_cloud
        return g(CLOUD_FULL), g(CLOUD_SHARP), g(CLOUD_LESS_SHARP), g(CLOUD_FLAT), g(CLOUD_LESS_FLAT)


class LaserOdometry:
    """vloam::LaserOdometry (laser_odometry.h:63-87): input is implicit (clouds stay on the device)."""

    def __init__(self, ctx):
        self.ctx, self.last = ctx, None

    def init(self):
        pass

    def solveLO(self, prior_q=None, prior_t=None):
        self.last = self.ctx.laser_odometry(prior_q, prior_t)

    def output(self):
        g = self.ctx.get_cloud
        r = self.last
        return r["q_w_curr"], r["t_w_curr"], g(CLOUD_CORNER_LAST), g(CLOUD_SURF_LAST), g(CLOUD_FULL_RES), r["skip_frame"]


class LaserMapping:
    """vloam::LaserMapping (laser_mapping.h:72-100)."""

    def __init__(self, ctx, map_pub_number=20):
        self.ctx, self.pose = ctx, None
        self.map_pub_number = map_pub_number  # ROS parameter map_pub_number (LM.cpp:44-45)
        self.frameCount = 0                   # mapped frames (incremented at the end of solveMapping)
        self.skip_frame = False               # input(): the odometry skipped mapping on this frame (LM.cpp:197-201)
        self._published_at = 0

    def init(self):
        pass

    def reset(self):
        pass

    def input(self, skip_frame):
        self.skip_frame = bool(skip_frame)

    def solveMapping(self):
        """On a skipped frame this only propagates the high-frequency pose (the reference does not call solveMapping then), so the
        mapped-frame count is left alone, as in vloam_adapter.hpp."""
        self.pose = self.ctx.laser_mapping()
        if not self.skip_frame:
            self.frameCount += 1

    def publish(self):
        """LM.cpp:884-899: every map_pub_number mapped frames the global map is published (parity unpinned: the reference is
        not in this checkout); the rule of vloam_adapter.hpp's LaserMapping::publish: nothing before the first mapped frame, and
        a map already published is not queued again on the skipped frames after it.  Returns True when a publication was queued;
        Context.get_map() reads it."""
        n = self.frameCount
        if self.map_pub_number > 0 and n > 0 and n % self.map_pub_number == 0 and n != self._published_at:
            self.ctx.publish_map()
            self._published_at = n
            return True
        return False


class LidarOdometryMapping:
    """vloam::LidarOdometryMapping (lidar_odometry_mapping.h:45-86): the per-frame call sequence."""

    def __init__(self, map_pub_number=20, **params):
        self.ctx = Context(**params)
        self.scan_registration = ScanRegistration(self.ctx)
        self.laser_odometry = LaserOdometry(self.ctx)
        self.laser_mapping = LaserMapping(self.ctx, map_pub_number)

    def init(self):
        pass

    def reset(self):  # lidar_odometry_mapping.cpp:65-71
        self.ctx.begin_frame()

    def scanRegistrationIO(self, laserCloudIn):  # lidar_odometry_mapping.cpp:77-100
        self.scan_registration.input(laserCloudIn)

    def laserOdometryIO(self):  # lidar_odometry_mapping.cpp:110-141
        self.laser_odometry.solveLO()

    def laserMappingIO(self):  # lidar_odometry_mapping.cpp:144-176
        last = self.laser_odometry.last
        self.laser_mapping.input(last["skip_frame"] if last else False)
        self.laser_mapping.solveMapping()
        self.laser_mapping.publish()
