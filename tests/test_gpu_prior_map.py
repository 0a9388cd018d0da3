"""Prior maps: vloam_b200_load_map / set_map_pose / set_map_update / get_map_kind.

The load is checked byte for byte against tests/prior_map_ref.py (the cube formula of LM.cpp:747-761 and the oracle's VoxelGrid
per cube); localization in a frozen map against the oracle, whose map is held fixed by re-importing that reference before every
sweep; the frozen drive across scheduling modes bit for bit; and the ABI's edges."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from map_publish_ref import laser_cloud_map, split_blob  # noqa: E402
from prior_map_ref import CUBE_NUM, load_blob  # noqa: E402

pytestmark = pytest.mark.gpu

POS_TOL, ROT_TOL = 1e-4, 1e-5
_CACHE = {}


def _world(pkg):
    if "world" not in _CACHE:
        _CACHE["world"] = pkg.synth.World(1234, 1, 190.0)
    return _CACHE["world"]


def _prior(pkg, size):
    """World-frame clouds planted at a pitch finer than the mapping leaves (0.4 / 0.8 m): several points per voxel.
    C3: ~1.3M points, C4: ~2.0M."""
    if size not in _CACHE:
        pc, ps = {"C3": (0.3, 0.7), "C4": (0.25, 0.6)}[size]
        w = _world(pkg)
        _CACHE[size] = (w.plant(0, pc, seed=99), w.plant(1, ps, seed=98))
    return _CACHE[size]


def _ref(op, corner, surf, cen):
    return load_blob(op, corner, 0.4, cen), load_blob(op, surf, 0.8, cen)


def _layout(a, stride, w):
    """float32[n, 4] -> records of `stride` floats, x y z at 0..2 and the intensity at w (other floats garbage)."""
    out = np.full((len(a), stride), -7.5, np.float32)
    out[:, :3] = a[:, :3]
    out[:, w] = a[:, 3]
    return out


def _ctx(pkg, **kw):
    import bench
    args = dict(bench.KW)
    args.update(kw)
    return pkg.Context(**args)


def _rot_err(q1, q2):
    return min(np.abs(q1 - q2).max(), np.abs(q1 + q2).max())


@pytest.mark.parametrize("size,where,layout,cen", [
    ("C3", "host", (4, 3), (10, 10, 5)), ("C3", "device", (8, 4), (10, 10, 5)), ("C3", "host", (5, 3), (9, 11, 5)),
    ("C4", "device", (4, 3), (10, 10, 5)), ("C4", "host", (8, 4), (11, 9, 6)), ("C4", "device", (5, 3), (9, 11, 5))])
def test_load_matches_reference(pkg, op, size, where, layout, cen):
    import torch
    corner, surf = _prior(pkg, size)
    # a few points the load must drop: non-finite, and outside the grid
    junk = np.array([[np.nan, 0, 0, 1], [0, np.inf, 0, 1], [5000.0, 0, 0, 1], [0, 0, -900.0, 1]], np.float32)
    corner = np.concatenate([corner[:1000], junk, corner[1000:]])
    surf = np.concatenate([junk[:2], surf])
    (cref, cdrop), (sref, sdrop) = _ref(op, corner, surf, cen)
    g = _ctx(pkg)
    if cen != (10, 10, 5):
        g.set("lm.state", np.array(list(cen) + [0], np.int32))  # a centre another than the initial one (window rolled before)
    args = [_layout(corner, *layout), _layout(surf, *layout)]
    if where == "device":
        args = [torch.from_numpy(a).cuda() for a in args]
    dropped = g.load_map(*args, w_offset=layout[1])
    assert list(dropped) == [cdrop, sdrop] and cdrop >= 4 and sdrop >= 2
    assert list(g.get("lm.state")[:3]) == list(cen), "the load moved the window"
    gc, gs = g.get("lm.cornerMap"), g.get("lm.surfMap")
    assert gc == cref, "corner map differs from the reference"
    assert gs == sref, "surf map differs from the reference"
    counts = split_blob(gs)[0]
    assert counts.sum() < len(surf) - sdrop, "no voxel held several points"
    g.close()


def _drive(pkg, n, x0=40.0, seed=91, step=1.5):
    """A C3 drive starting x0 m from the map origin: scans of the planted world and the ground-truth poses."""
    import bench
    key = ("drive", n, x0, seed, step)
    if key not in _CACHE:
        traj = pkg.synth.trajectory(n + 1, seed=seed, step=step)
        traj[:, 0] += x0
        scans = bench._gen_scans(pkg, _world(pkg), traj, [5000 + k for k in range(n + 1)])
        _CACHE[key] = (scans, traj)
    return _CACHE[key]


def _guess(pkg, traj0, dxy=(0.4, 0.3), dyaw_deg=2.0):
    """q_wmap_wodom / t_wmap_wodom about 0.5 m and 2 degrees off the truth (the odometry frame is the first sweep's)."""
    p = np.array(traj0, float)
    p[0] += dxy[0]; p[1] += dxy[1]; p[3] += np.deg2rad(dyaw_deg)
    return pkg.synth.pose_to_qt(p)


def _frozen_gpu(pkg, n, mode="two", env=None, skip=1, publish_load=False):
    """Load the C3 prior, set the guess, freeze, and run n sweeps.  mode: plain (one sweep at a time), one / two (sweeps registered
    ahead, pinned host buffers).  Returns (poses [n, 14], context)."""
    import torch
    import bench
    scans, traj = _drive(pkg, n)
    corner, surf = _prior(pkg, "C3")
    for k, v in (env or {}).items():
        os.environ[k] = v
    try:
        g = _ctx(pkg, mapping_skip_frame=skip)
    finally:
        for k in (env or {}):
            os.environ.pop(k, None)
    if publish_load:  # a publication pending across the load: it still returns the map it was queued for (empty here)
        g.publish_map()
    g.load_map(corner, surf)
    if publish_load:
        assert len(g.get_map()) == 0
    q, t = _guess(pkg, traj[0])
    g.set_map_pose(q, t)
    g.set_map_update(False)
    pinned = [torch.from_numpy(s).pin_memory() for s in scans]
    pose, poses = np.zeros(14), []
    for k in range(n):
        if mode == "two":
            bench.prefetch_ahead(g, pinned, k, False)
        elif mode == "one" and k + 1 < len(pinned):
            g.prefetch_ptr(pinned[k + 1].data_ptr(), pinned[k + 1].shape[0], 4)
        g.process_frame_ptr(pinned[k].data_ptr(), pinned[k].shape[0], 4, pose.ctypes.data)
        poses.append(pose.copy())
    return np.array(poses), g


def _frozen_oracle(pkg, op, n, first_frozen=0, last_frozen=None):
    """The oracle on the same drive, its map held fixed on sweeps [first_frozen, last_frozen) by re-importing, before each of them,
    the reference load at its current window centre (sweeps outside that range map normally; a normal prefix starts from the
    loaded map as well)."""
    import bench
    scans, traj = _drive(pkg, n)
    corner, surf = _prior(pkg, "C3")
    o = op.Oracle(knn_backend=1, **bench.KW)
    refs = {}

    def ref(cen):
        if cen not in refs:
            refs[cen] = _ref(op, corner, surf, cen)
        return refs[cen]
    (cb, _), (sb, _) = ref((10, 10, 5))
    o.set("lm.cornerMap", cb); o.set("lm.surfMap", sb)
    q, t = _guess(pkg, traj[0])
    o.set("lm.pose", np.r_[0, 0, 0, 1, 0, 0, 0, q, t].astype(np.float64))
    last_frozen = n if last_frozen is None else last_frozen
    frozen_maps = None
    poses, truth_err = [], []
    for k in range(n):
        # (up to and including the first sweep after the frozen range: the last frozen sweep's insert must not reach it)
        if first_frozen <= k <= last_frozen:
            if first_frozen == 0:
                cen = tuple(int(v) for v in o.get("lm.state")[:3])
                (cb, _), (sb, _) = ref(cen)
            else:  # frozen after mapping: the map as the mapped prefix left it
                if frozen_maps is None:
                    frozen_maps = (o.get("lm.cornerMap"), o.get("lm.surfMap"))
                cb, sb = frozen_maps
            o.set("lm.cornerMap", cb); o.set("lm.surfMap", sb)
        o.process(scans[k])
        poses.append(o.get("lm.pose")[:7].copy())
    return np.array(poses)


def _assert_close(gpu, cpu, what):
    for k in range(len(cpu)):
        dt = np.abs(gpu[k, 11:14] - cpu[k, 4:7]).max()
        dq = _rot_err(gpu[k, 7:11], cpu[k, 0:4])
        assert dt < POS_TOL and dq < ROT_TOL, "%s: sweep %d differs from the oracle by %.3g m / %.3g" % (what, k, dt, dq)


def test_frozen_localization_matches_oracle(pkg, op):
    """Free-running frozen drive on the benchmarked path (two sweeps ahead, helper thread, pinned host buffers), 40 m from the map
    origin with a guess 0.5 m / 2 degrees off, across a move of the sub-map window: every pose against the oracle; the map stays
    what was loaded; the in-place path runs; a frozen sweep allocates nothing.  Accuracy against the generator's truth: from sweep 15
    on the localized position stays within 0.05 m (the oracle's own frozen run of this drive stays within 0.026 m there, after
    converging from the guess), below the drift of the same drive mapped from scratch (~2.2 m: at 1.5 m per sweep the odometry
    lags the truth by ~2 m)."""
    n = 30
    gpu, g = _frozen_gpu(pkg, n)
    cpu = _frozen_oracle(pkg, op, n)
    _assert_close(gpu, cpu, "frozen drive")
    scans, traj = _drive(pkg, n)
    centres = {int(np.floor((p[0] + 25.0) / 50.0)) for p in traj[:n]}
    assert len(centres) >= 2, "the drive never crossed a cube boundary (no window move)"
    paths = g.get("lm.paths")
    assert paths[0] > n // 2, "the frozen drive did not stay on the in-place path: %s" % paths
    corner, surf = _prior(pkg, "C3")
    cen = tuple(int(v) for v in g.get("lm.state")[:3])
    (cb, _), (sb, _) = _ref(op, corner, surf, cen)
    assert g.get("lm.cornerMap") == cb and g.get("lm.surfMap") == sb, "the frozen map changed"
    g.publish_map(); m1 = g.get_map()  # (the first publication reserves its output buffer)
    a0 = int(g.get("alloc.count")[0])
    import torch
    pinned = [torch.from_numpy(s).pin_memory() for s in scans]
    pose = np.zeros(14)
    g.process_frame_ptr(pinned[n].data_ptr(), pinned[n].shape[0], 4, pose.ctypes.data)
    g.publish_map(); m2 = g.get_map()
    assert m1.tobytes() == m2.tobytes(), "publish_map changed between frozen sweeps"
    assert int(g.get("alloc.count")[0]) == a0, "a frozen sweep allocated"
    g.close()
    # accuracy against the generator's truth (sensor pose in the world)
    m = _ctx(pkg)
    pm = [m.process_frame(s) for s in scans[:n]]
    m.close()
    drift = [np.abs((pm[k][11:13] - pm[0][11:13]) - (traj[k, :2] - traj[0, :2])).max() for k in range(15, n)]
    loc = [np.abs(gpu[k, 11:13] - traj[k, :2]).max() for k in range(15, n)]
    print("frozen localization error (sweeps 15..%d) %.4f m, mapped-from-scratch drift %.4f .. %.4f m" % (n - 1, max(loc), min(drift), max(drift)))
    assert max(loc) < 0.05, "localization error %.3f m" % max(loc)
    assert max(loc) < min(drift), "frozen localization (%.3f m) is not better than mapping from scratch (%.3f m)" % (max(loc), min(drift))


@pytest.mark.parametrize("variant", ["plain", "one", "no_grid", "no_worker", "no_lo_lookahead", "no_stacks_lookahead", "publish_load"])
def test_frozen_drive_bit_identical_across_modes(pkg, variant):
    n = 24
    ref, g = _frozen_gpu(pkg, n, mode="two")
    ref_maps = (g.get("lm.cornerMap"), g.get("lm.surfMap"))
    g.close()
    env = {"no_grid": {"VLOAM_NO_GRID": "1"}, "no_worker": {"VLOAM_NO_WORKER": "1"}, "no_lo_lookahead": {"VLOAM_NO_LO_LOOKAHEAD": "1"},
           "no_stacks_lookahead": {"VLOAM_NO_STACKS_LOOKAHEAD": "1"}}.get(variant)
    mode = {"plain": "plain", "one": "one"}.get(variant, "two")
    out, g = _frozen_gpu(pkg, n, mode=mode, env=env, publish_load=variant == "publish_load")
    assert (out == ref).all(), "%s: poses differ from the two-ahead frozen drive" % variant
    assert (g.get("lm.cornerMap"), g.get("lm.surfMap")) == ref_maps
    g.close()


def test_frozen_drive_skip_frame_two(pkg):
    a, g = _frozen_gpu(pkg, 16, mode="plain", skip=2)
    g.close()
    b, g = _frozen_gpu(pkg, 16, mode="two", skip=2)
    g.close()
    assert (a == b).all()


def test_map_freeze_unfreeze_matches_oracle(pkg, op):
    """Map 10 sweeps, freeze 10, map 10 again -- against the oracle, whose map is held at what its first 10 sweeps left."""
    import torch
    import bench
    n = 30
    scans, traj = _drive(pkg, n)
    corner, surf = _prior(pkg, "C3")
    g = _ctx(pkg)
    g.load_map(corner, surf)
    q, t = _guess(pkg, traj[0])
    g.set_map_pose(q, t)
    pinned = [torch.from_numpy(s).pin_memory() for s in scans]
    pose, gpu = np.zeros(14), []
    for k in range(n):
        if k == 10: g.set_map_update(False)
        if k == 20: g.set_map_update(True)
        bench.prefetch_ahead(g, pinned, k, False)
        g.process_frame_ptr(pinned[k].data_ptr(), pinned[k].shape[0], 4, pose.ctypes.data)
        gpu.append(pose.copy())
    g.close()
    cpu = _frozen_oracle(pkg, op, n, first_frozen=10, last_frozen=20)
    _assert_close(np.array(gpu), cpu, "map / freeze / map")


def test_round_trip_through_get_map_kind(pkg, op):
    """Context A maps the 45-sweep drive of test_grid_update_equals_pool_update and publishes; its two get_map_kind clouds are the
    cubes of get_map, and context B, loading them at A's window centre, holds exactly the reference load of them."""
    import torch
    import bench
    n = 45
    traj = pkg.synth.trajectory(n + 1, seed=91, step=1.5)
    scans = bench._gen_scans(pkg, pkg.synth.World(1234, 1, 190.0), traj, [4000 + k for k in range(n + 1)])
    _, _, cb, sb = bench.make_sequence(pkg, 0, 1)
    dev = [torch.from_numpy(s).cuda() for s in scans]
    a = _ctx(pkg)
    a.set("lm.cornerMap", cb); a.set("lm.surfMap", sb)
    pose = np.zeros(14)
    for k in range(n):
        bench.prefetch_ahead(a, dev, k, True)
        a.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, pose.ctypes.data)
    a.publish_map()
    full, kc, ks = a.get_map(), a.get_map_kind(0), a.get_map_kind(1)
    ac, asb = a.get("lm.cornerMap"), a.get("lm.surfMap")
    cen = a.get("lm.state")[:3].copy()
    a.close()
    assert laser_cloud_map(ac, asb).tobytes() == full.tobytes()
    assert kc.tobytes() == split_blob(ac)[1].tobytes() and ks.tobytes() == split_blob(asb)[1].tobytes()
    assert len(kc) + len(ks) == len(full) and len(kc) > 0 and len(ks) > 0
    b = _ctx(pkg)
    b.set("lm.state", np.r_[cen, 0].astype(np.int32))
    dropped = b.load_map(torch.from_numpy(kc).cuda(), torch.from_numpy(ks).cuda())
    (rc, dc), (rs, ds) = _ref(op, kc, ks, tuple(int(v) for v in cen))
    assert list(dropped) == [dc, ds] == [0, 0]
    assert b.get("lm.cornerMap") == rc and b.get("lm.surfMap") == rs
    b.close()


def test_publish_then_load_returns_the_published_map(pkg):
    import bench
    scans, traj = _drive(pkg, 4)
    corner, surf = _prior(pkg, "C3")
    g = _ctx(pkg)
    g.load_map(corner, surf)
    for k in range(3):
        g.process_frame(scans[k])
    g.publish_map()
    before = laser_cloud_map(g.get("lm.cornerMap"), g.get("lm.surfMap"))
    g.publish_map()
    g.load_map(corner[: len(corner) // 2], surf[: len(surf) // 2])
    assert g.get_map().tobytes() == before.tobytes(), "the publication queued before the load must return the old map"
    g.close()


def test_load_while_sweeps_are_registered_ahead(pkg):
    """A load between sweeps with two sweeps registered ahead gives what the same calls give one sweep at a time."""
    import torch
    import bench
    n = 12
    scans, traj = _drive(pkg, n)
    corner, surf = _prior(pkg, "C3")
    pinned = [torch.from_numpy(s).pin_memory() for s in scans]
    out = []
    for ahead in (False, True):
        g = _ctx(pkg)
        g.load_map(corner, surf)
        q, t = _guess(pkg, traj[0])
        g.set_map_pose(q, t)
        pose, poses = np.zeros(14), []
        for k in range(n):
            if k == 6:
                g.load_map(corner, surf)
                g.set_map_update(False)
            if ahead: bench.prefetch_ahead(g, pinned, k, False)
            g.process_frame_ptr(pinned[k].data_ptr(), pinned[k].shape[0], 4, pose.ctypes.data)
            poses.append(pose.copy())
        out.append((np.array(poses), g.get("lm.cornerMap"), g.get("lm.surfMap")))
        g.close()
    assert (out[0][0] == out[1][0]).all() and out[0][1:] == out[1][1:]


def test_contract_edges(pkg):
    pkg_L = pkg.load_lib()
    corner, surf = _prior(pkg, "C3")
    g = _ctx(pkg)
    g.load_map(corner[:5000], surf[:5000])
    maps = (g.get("lm.cornerMap"), g.get("lm.surfMap"))
    h = g.h
    c4 = np.ascontiguousarray(corner[:10], np.float32)
    dr = np.zeros(2, np.int64)
    assert pkg_L.vloam_b200_load_map(h, c4.ctypes.data, 10, c4.ctypes.data, 10, 3, 3, dr.ctypes.data) == -1  # stride < 4
    assert pkg_L.vloam_b200_load_map(h, c4.ctypes.data, 10, c4.ctypes.data, 10, 4, 4, dr.ctypes.data) == -1  # w_offset outside
    assert pkg_L.vloam_b200_load_map(h, None, 10, c4.ctypes.data, 10, 4, 3, dr.ctypes.data) == -1          # NULL with n > 0
    assert pkg_L.vloam_b200_load_map(h, c4.ctypes.data, -1, c4.ctypes.data, 10, 4, 3, dr.ctypes.data) == -1  # n < 0
    big = np.zeros((1 << 21, 4), np.float32)
    assert pkg_L.vloam_b200_load_map(h, big.ctypes.data, len(big), c4.ctypes.data, 10, 4, 3, dr.ctypes.data) == -3
    assert (g.get("lm.cornerMap"), g.get("lm.surfMap")) == maps, "a refused load changed the map"
    with pytest.raises(pkg.VloamError):
        g.set_map_pose([0, 0, 0, np.nan], [0, 0, 0])
    with pytest.raises(pkg.VloamError):
        g.get_map_kind(0)  # nothing published yet
    assert pkg_L.vloam_b200_get_map_kind(h, 2, None, 0) == -1
    g.publish_map()
    n0 = pkg_L.vloam_b200_get_map_kind(h, 0, None, 0)
    out = np.zeros((max(n0 - 1, 1), 4), np.float32)
    assert n0 > 1 and pkg_L.vloam_b200_get_map_kind(h, 0, out.ctypes.data, n0 - 1) == -3
    assert (g.load_map(np.zeros((0, 4), np.float32), np.zeros((0, 4), np.float32)) == 0).all()
    empty = np.zeros(CUBE_NUM, np.int32).tobytes()
    assert g.get("lm.cornerMap") == empty and g.get("lm.surfMap") == empty, "an empty load must clear the map"
    g.close()


def test_eight_concurrent_contexts(pkg):
    from test_gpu_benchmarked_path import _run_threads
    n = 8
    ref, g = _frozen_gpu(pkg, n, mode="plain")
    g.close()

    def one():
        p, c = _frozen_gpu(pkg, n, mode="two")
        c.close()
        return p
    for p in _run_threads([one] * 8):
        assert (p == ref).all()



def test_adapter_localizes_in_a_prior_map(pkg, synth, street, tmp_path):
    """vloam_adapter.hpp (tests/cpp/prior_map_adapter.cpp): LaserMapping::loadMap from KITTI-style .bin files, setMapPose,
    setMapUpdate(false) and the IO calls of vloam_main_node.cpp -- its poses bit for bit those of the same calls through the C ABI."""
    import subprocess
    from test_abi import build_cpp_program
    exe = build_cpp_program("prior_map_adapter", tmp_path)
    kw = dict(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4)
    n = 12
    traj = synth.trajectory(n, seed=5)
    traj[:, 0] += 30.0
    scans = [street.scan(0, traj[k], 1000 + k) for k in range(n)]
    corner, surf = street.plant(0, 0.15, seed=9), street.plant(1, 0.3, seed=8)
    files = []
    for name, a in [("corner", corner), ("surf", surf)] + [("scan%d" % k, s) for k, s in enumerate(scans)]:
        f = str(tmp_path / (name + ".bin"))
        np.ascontiguousarray(a, np.float32).tofile(f)
        files.append(f)
    q, t = _guess(pkg, traj[0], (0.3, -0.2), 1.0)
    args = [exe, files[0], files[1]] + ["%.17g" % v for v in np.r_[q, t]] + files[2:]
    out = subprocess.run(args, check=True, capture_output=True, text=True).stdout
    assert "prior map ok" in out, out
    got = np.array([[float(v) for v in l.split()[1:]] for l in out.splitlines() if l.startswith("pose ")])
    lom = pkg.LidarOdometryMapping(**kw)
    dropped = lom.laser_mapping.load_map(corner, surf)
    assert out.splitlines()[0] == "dropped %d %d" % tuple(dropped)
    lom.laser_mapping.set_map_pose(q, t)
    lom.laser_mapping.set_map_update(False)
    ref = []
    for s in scans:
        lom.reset(); lom.scanRegistrationIO(s); lom.laserOdometryIO(); lom.laserMappingIO()
        ref.append(np.r_[lom.laser_mapping.pose[0], lom.laser_mapping.pose[1]])
    assert got.shape == (n, 7) and (got == np.array(ref)).all(), "adapter poses differ from the C ABI run"
