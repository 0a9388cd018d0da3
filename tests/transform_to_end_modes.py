"""One process, one scheduling mode, VLOAM_FLAG_DISTORTION | VLOAM_FLAG_TRANSFORM_TO_END (tests/test_gpu_transform_to_end.py runs
one per mode: the VLOAM_NO_* switches are read once per process).

usage: transform_to_end_modes.py <ahead: 0 | 1 | 2> <out.npz>

Moving HDL-64 street sweeps through process_frame with 0, 1 or 2 sweeps registered ahead, in three scenarios: a drive with one
dropped registration (a registered buffer that is not the one processed), mapping_skip_frame = 2, and stage-level calls with
a VO prior (use_prior) on every other frame.  Writes every pose, the final maps and lm.paths."""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import transform_to_end_ref as ref  # noqa: E402

KW = dict(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8)


def register(g, bufs, k, ahead):
    for j in range(k + 1, min(k + ahead, len(bufs) - 1) + 1):
        g.prefetch_ptr(bufs[j].ctypes.data, bufs[j].shape[0], 4)


def main():
    ahead, out = int(sys.argv[1]), sys.argv[2]
    pkg = importlib.import_module("vloam-noted_b200")
    world = pkg.synth.World(1234, 0, 160.0)
    scans, _ = ref.moving_drive(world, pkg.synth.HDL64, 15, seed=271)
    res = {}
    for name, skip, drop in (("drive", 1, 7), ("skip2", 2, -1)):
        g = pkg.Context(distortion=1, transform_to_end=True, mapping_skip_frame=skip, **KW)
        bufs = [np.ascontiguousarray(s) for s in scans]
        poses = np.zeros((len(scans) - 1, 14))
        pose = np.zeros(14)
        for k in range(len(scans) - 1):
            register(g, bufs, k, ahead)
            if k == drop:  # the registered buffer is not the one processed: everything computed ahead is dropped
                g.process_frame_ptr(np.ascontiguousarray(scans[k].copy()).ctypes.data, len(scans[k]), 4, pose.ctypes.data)
            else:
                g.process_frame_ptr(bufs[k].ctypes.data, len(bufs[k]), 4, pose.ctypes.data)
            poses[k] = pose
        res[name + "_poses"] = poses
        res[name + "_corner"] = np.frombuffer(g.get("lm.cornerMap"), np.uint8)
        res[name + "_surf"] = np.frombuffer(g.get("lm.surfMap"), np.uint8)
        res[name + "_paths"] = g.get("lm.paths")
        res[name + "_full"] = g.register_full_cloud()
        g.close()
    # stage-level calls with a VO prior on every other frame (detach_VO_LO == false, LO.cpp:237-250)
    g = pkg.Context(distortion=1, transform_to_end=True, **KW)
    bufs = [np.ascontiguousarray(s) for s in scans]
    poses = []
    for k in range(8):
        register(g, bufs, k, ahead)
        g.begin_frame()
        g.L.vloam_b200_scan_registration(g.h, bufs[k].ctypes.data, len(bufs[k]), 4)
        prior = (np.array([0.0, 0.0, 0.01, 0.99995]), np.array([0.9, 0.02, 0.0])) if k % 2 else (None, None)
        r = g.laser_odometry(*prior)
        q, t = g.laser_mapping()
        poses.append(np.concatenate([r["q_w_curr"], r["t_w_curr"], q, t]))
    res["prior_poses"] = np.array(poses)
    res["prior_corner"] = np.frombuffer(g.get("lm.cornerMap"), np.uint8)
    res["prior_paths"] = g.get("lm.paths")
    g.close()
    np.savez(out, **res)


if __name__ == "__main__":
    main()
