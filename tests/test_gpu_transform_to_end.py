"""VLOAM_FLAG_TRANSFORM_TO_END on the device (lo_transform_to_end, LO.cpp:176-193 / 537-556) against the oracle driven with the
restated block (tests/transform_to_end_ref.py), on sweeps from a moving sensor (synth World.scan_moving).

Bar: every cloud, association index, stack and map bit-exact in teacher-forced runs, poses within 1e-4 m / 1e-5; free-running
on the benchmarked path as test_gpu_benchmarked_path.py; every scheduling mode bit-identical to the plain one."""
import ctypes
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from conftest import assert_bits_equal
from test_gpu_parity import KW, check_frame, pose_close, teacher_force
import transform_to_end_ref as ref

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.mark.parametrize("distortion", [0, 1])
@pytest.mark.parametrize("sensor", [0, 1])
def test_teacher_forced_moving_sweeps(pkg, op, synth, street, sensor, distortion):
    """Frame by frame from the first one: the end clouds (lo.cornerLast / surfLast), the association, the stacks filtered from
    the end clouds, the sub-map and the maps bit-exact; the full-resolution outputs (get_cloud(FULL_RES), register_full_cloud)
    bit-exact; the raw ScanRegistration outputs untouched."""
    frames = 4
    scans, _ = ref.moving_drive(street, sensor, frames, seed=17 + sensor)
    o = op.Oracle(distortion=distortion, **KW[sensor])
    g = pkg.Context(distortion=distortion, transform_to_end=True, **KW[sensor])
    g.set_capture(True)
    for k in range(frames):
        if k > 0:
            teacher_force(o, g)
        o.scan_registration(scans[k]); g.begin_frame(); g.scan_registration(scans[k])
        o.laser_odometry(); g.laser_odometry()
        lo = o.get("lo.pose")
        full = o.get("sr.laserCloud")
        o.set_last(ref.transform_to_end(o.get("lo.cornerLast"), lo[7:], distortion), ref.transform_to_end(o.get("lo.surfLast"), lo[7:], distortion))
        o.laser_mapping(); g.laser_mapping()
        check_frame(o, g, k)
        for nm in ("lo.cornerLast", "lo.surfLast"):
            assert_bits_equal(o.get(nm), g.get(nm), nm)
        assert_bits_equal(o.get("lo.cornerLast"), g.get_cloud(pkg.CLOUD_CORNER_LAST), "CLOUD_CORNER_LAST")
        assert_bits_equal(full, g.get_cloud(pkg.CLOUD_FULL), "CLOUD_FULL stays the raw cloud")
        assert_bits_equal(ref.transform_to_end(full, lo[7:], distortion), g.get_cloud(pkg.CLOUD_FULL_RES), "CLOUD_FULL_RES")
        assert_bits_equal(ref.register_full(full, lo, o.get("lm.pose")[:7], distortion), g.register_full_cloud(), "register_full_cloud")
        if k == 0:
            assert (lo[7:] == [0, 0, 0, 1, 0, 0, 0]).all()
            assert_bits_equal(g.get("lo.cornerLast")[:, :3], o.get("sr.lessSharp")[:, :3], "first frame: coordinates unchanged")
    g.close()


def test_flag_off_full_res_is_full_and_flags_are_checked(pkg, synth, street):
    scan = street.scan(0, [1.0, 0.1, 0.0, 0.01, 0.0, 0.0], 5)
    g = pkg.Context(**KW[0])
    for k in range(2):
        g.process_frame(scan)
        assert_bits_equal(g.get_cloud(pkg.CLOUD_FULL), g.get_cloud(pkg.CLOUD_FULL_RES), "FULL_RES == FULL without the flag")
    g.close()
    L = pkg.load_lib()
    for flags, ok in ((2, True), (3, True), (1, True), (4, False), (6, False)):
        p = pkg.Params(16, 0.3, 0.2, 0.4, 1, flags)
        h = ctypes.c_void_p()
        r = L.vloam_b200_create(ctypes.byref(p), 0, ctypes.byref(h))
        assert (r == 0) == ok, (flags, r)
        if r == 0:
            L.vloam_b200_destroy(h)


def test_flag_off_allocates_nothing_new(pkg, synth, street):
    """Only a context with the flag reserves the end buffers (three generations x two clouds)."""
    scans, _ = ref.moving_drive(street, 1, 8)
    counts = {}
    for te in (False, True):
        g = pkg.Context(distortion=1, transform_to_end=te, **KW[1])
        for s in scans:
            g.process_frame(s)
        g.synchronize()
        counts[te] = int(g.get("alloc.count")[0])
        g.close()
    assert 6 <= counts[True] - counts[False] <= 12, counts


def _oracle_replay_to_end(op, scans, cb, sb, frames):
    import bench
    o = op.Oracle(knn_backend=1, distortion=1, **bench.KW)
    o.set("lm.cornerMap", cb); o.set("lm.surfMap", sb)
    poses = np.zeros((frames, 14))
    for k in range(frames):
        ref.oracle_step(o, scans[k], 1, True)
        poses[k, :7] = o.get("lo.pose")[:7]; poses[k, 7:] = o.get("lm.pose")[:7]
    return poses, (o.get("lm.cornerMap"), o.get("lm.surfMap"))


def test_free_running_benchmarked_path(pkg, op):
    """bench.py's path (two sweeps registered ahead, helper thread, in-place grid) with D + TO_END on moving HDL-64 sweeps of the C3
    world over its planted map, three contexts at once, 32 sweeps crossing a sub-map window move: poses within tolerance of
    each context's oracle replay, final maps equal (up to the rare last-bit rounding of a free-running f64 sum, as in
    test_c3_lookahead_free_running_matches_oracle)."""
    import bench
    frames, nseq = 32, 3
    world = pkg.synth.World(1234, 1, 190.0)
    _, _, cb, sb = bench.make_sequence(pkg, 0, 1)
    seqs = [ref.moving_drive(world, pkg.synth.HDL64, frames + 1, seed=900 + q) for q in range(nseq)]
    cpu, gpu, err = [None] * nseq, [None] * nseq, []

    def run(q):
        try:
            scans = seqs[q][0]
            cpu[q] = _oracle_replay_to_end(op, scans, cb, sb, frames)
            g = pkg.Context(distortion=1, transform_to_end=True, **bench.KW)
            g.set("lm.cornerMap", cb); g.set("lm.surfMap", sb)
            bufs = [np.ascontiguousarray(s) for s in scans]
            pose, poses, centres = np.zeros(14), np.zeros((frames, 14)), set()
            for k in range(frames):
                for j in range(k + 1, min(k + 2, len(bufs) - 1) + 1):  # the next two sweeps registered, as bench.prefetch_ahead does
                    g.prefetch_ptr(bufs[j].ctypes.data, len(bufs[j]), 4)
                g.process_frame_ptr(bufs[k].ctypes.data, len(bufs[k]), 4, pose.ctypes.data)
                poses[k] = pose
                centres.add(int(g.get("lm.validInd")[0]) if k % 8 == 7 else -1)
            paths = g.get("lm.paths")
            gpu[q] = (poses, (g.get("lm.cornerMap"), g.get("lm.surfMap")), len(centres - {-1}), paths)
            g.close()
        except BaseException as e:  # noqa: BLE001 -- re-raised below
            err.append(e)
    th = [threading.Thread(target=run, args=(q,)) for q in range(nseq)]
    for t in th: t.start()
    for t in th: t.join()
    if err:
        raise err[0]
    exact = 0
    for q in range(nseq):
        gp, gm, ncen, paths = gpu[q]
        cp, cm = cpu[q]
        rep = bench.parity_report(gp, gm, cp, cm)
        assert rep["max_dt_m"] < bench.POS_TOL and rep["max_dq"] < bench.ROT_TOL, (q, rep)
        for kind in ("corner", "surf"):
            d = rep.get("map_diff", {}).get(kind, {"equal": True})
            assert d.get("equal") or (d["cubes_differing"] == 0 and d["floats_differing"] <= 64 and d["max_abs_diff"] < 1e-4), (q, kind, d)
        exact += rep["map_bytes_equal"]
        assert ncen >= 2, "sequence %d never moved its sub-map window" % q
        assert paths[0] > 0, "the in-place grid path never ran"
    print("D + TO_END on the benchmarked path: final maps byte-identical in %d / %d sequences" % (exact, nseq))


MODES = [("plain", 0, {}), ("one_ahead", 1, {}), ("two_ahead", 2, {}),
         ("no_prebuild", 2, {"VLOAM_NO_PREBUILD": "1"}), ("no_stacks_lookahead", 2, {"VLOAM_NO_STACKS_LOOKAHEAD": "1"}),
         ("no_lo_lookahead", 2, {"VLOAM_NO_LO_LOOKAHEAD": "1"}), ("no_worker", 2, {"VLOAM_NO_WORKER": "1"})]


def test_scheduling_modes_are_bit_identical(tmp_path):
    """Plain, one and two sweeps ahead, and each look-ahead stage switched off (one process each): poses, maps, lm.paths and
    the registered full cloud bit-identical, with mapping_skip_frame = 2, a dropped registration and a VO prior covered."""
    res = {}
    for name, ahead, env in MODES:
        out = str(tmp_path / (name + ".npz"))
        e = dict(os.environ)
        e.update(env)
        subprocess.run([sys.executable, os.path.join(HERE, "transform_to_end_modes.py"), str(ahead), out], check=True, env=e, cwd=ROOT)
        res[name] = np.load(out)
    base = res["plain"]
    for name, _, _ in MODES[1:]:
        for key in base.files:
            a, b = base[key], res[name][key]
            assert a.shape == b.shape and a.tobytes() == b.tobytes(), (name, key)
    assert base["drive_paths"].sum() > 0 and np.isfinite(base["drive_poses"]).all()


def test_adapter_program_hands_over_end_frame_full_res(pkg, op, street, tmp_path):
    """tests/cpp/transform_to_end_adapter.cpp: the stage classes of vloam_adapter.hpp on an Engine with DISTORTION | TRANSFORM_TO_END,
    20 moving VLP-16 frames: poses within tolerance of the oracle's, LaserOdometry::output's laserCloudFullRes bit for bit the
    oracle's end-frame cloud (and LaserMapping::input accepted it)."""
    from test_abi import build_cpp_program
    exe = build_cpp_program("transform_to_end_adapter", tmp_path)
    n = 20
    scans, _ = ref.moving_drive(street, pkg.synth.VLP16, n, seed=5)
    files = []
    for k, s in enumerate(scans):
        f = str(tmp_path / ("scan%d.bin" % k))
        s.tofile(f)
        files.append(f)
    r = subprocess.run([exe, str(tmp_path)] + files, capture_output=True, text=True)
    out = r.stdout
    assert r.returncode == 0 and "transform to end ok" in out, (r.returncode, out[-2000:], r.stderr[-2000:])
    rows = [l.split() for l in out.splitlines() if l.startswith("frame ")]
    assert len(rows) == n
    o = op.Oracle(distortion=1, **KW[0])
    exact = 0
    for k in range(n):
        want = ref.oracle_step(o, scans[k], 1, True)
        odom = np.array([float(v) for v in rows[k][3:10]]); mapped = np.array([float(v) for v in rows[k][11:18]])
        pose_close(o.get("lo.pose")[:7], odom); pose_close(o.get("lm.pose")[:7], mapped)
        got = np.fromfile(str(tmp_path / ("full_%d.bin" % k)), np.float32).reshape(-1, 4)
        assert got.shape == want.shape, k
        # free-running: the two sides' f64 sums may differ in the last bit of q / t_last_curr, which moves a float of the end cloud
        # in ~1e8 values (as in test_c3_lookahead_free_running_matches_oracle); exact equality is counted
        bad = got.view(np.uint32) != want.view(np.uint32)
        assert bad.sum() <= 64 and np.abs(got - want).max() < 1e-4, (k, int(bad.sum()))
        exact += not bad.any()
    print("adapter laserCloudFullRes bit-identical to the oracle's end-frame cloud in %d / %d frames" % (exact, n))
    assert exact >= n - 2
