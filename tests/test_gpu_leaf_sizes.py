"""The mapping stage at the leaf sizes vloam_b200_create accepts (line_res / plane_res >= 0.05 m), not only the 0.2/0.4 and
0.4/0.8 of the other tests.  The in-place voxel-hash map update changes behaviour with the leaf size:

  * leaf <= 0.95 m: an entry whose centroid slid into the neighbouring 2 m cell stays where it is; above that it is tombstoned
    and re-inserted (mu_apply), and the kNN search, the grid write-back (mz_collect) and the map publication skip the tombstones;
  * leaf >~ 1.96 m: a voxel's box spans more than 2 x 2 x 2 cells and mu_lookup walks them serially;
  * leaf 0.05 m: voxel keys reach ~1000 of their 10 bits per axis, and the stack filter (LM.cpp:492-500) overflows PCL's
    index guard on the corner stack, which then passes through unfiltered.

For every pair, on a street drive whose sub-map window moves: the grid path against the pool path (VLOAM_NO_GRID=1) bit for bit,
the free-running replay against the oracle, teacher-forced bit-exact checkpoints, and the published map against the export.
The grid bookkeeping read after every sweep proves which branch ran.  (mu_apply's walk over the whole stack for a voxel with more
than MU_CAP = 16 new points is not reached: the stacks are voxel-filtered at the map's own leaf.)"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from map_publish_ref import laser_cloud_map, laser_cloud_map_of  # noqa: E402
from test_gpu_benchmarked_path import _run_threads  # noqa: E402
from test_gpu_parity import check_frame, pose_close, teacher_force  # noqa: E402

pytestmark = pytest.mark.gpu

INPLACE_MAX_LEAF = 0.95   # mu_apply keeps a drifted entry in its cell up to this leaf
# (sensor, line_res, plane_res, sweeps): VLP-16 over 27 sweeps at 1.1 m per sweep (the window moves at x = 25 m), one HDL-64 case
CASES = [(0, 0.05, 0.1, 27),    # minimum leaf: stack guard on the corner stack, long cell chains, keys near 1000
         (0, 0.15, 0.3, 27),    # not a divisor of 50 m, not representable in binary
         (0, 0.95, 0.95, 27),   # the largest leaf that keeps drifted entries in place
         (0, 0.4, 1.2, 27),     # surf above the threshold, corner below
         (0, 0.2, 2.0, 27),     # surf boxes over 2 m: unrolled and serial look-ups mixed
         (0, 1.0, 3.0, 27),     # both above the threshold, serial look-up for surf
         (1, 0.05, 0.1, 10)]
IDS = ["vlp16-%g-%g" % c[1:3] if c[0] == 0 else "hdl64-%g-%g" % c[1:3] for c in CASES]


def _kw(case):
    sensor, line, plane, _ = case
    return dict(n_scans=16 if sensor == 0 else 64, minimum_range=0.3 if sensor == 0 else 5.0, line_res=line, plane_res=plane)


def _scans(street, case):
    sensor, n = case[0], case[3]
    drive = [(1.1 * k, 0.05 * k, 0.002 * k) for k in range(n + 1)]   # (test_speculative_submap_equals_inline_build's drive)
    return [street.scan(sensor, [p[0], p[1], 0, p[2], 0, 0], 3000 + k) for k, p in enumerate(drive)]


def _guard_fires(cloud, leaf):
    """pcl::VoxelGrid's overflow guard (output = input) for this cloud and leaf: the test of test_oracle_math.np_voxel_grid."""
    if len(cloud) == 0:
        return False
    inv = np.float32(1.0) / np.float32(leaf)
    c = np.ascontiguousarray(cloud[:, :3], np.float32)
    d = ((c.max(0) - c.min(0)) * inv).astype(np.int64) + 1
    return int(d[0]) * int(d[1]) * int(d[2]) > 2**31 - 1


def _compare_maps(a, b):
    """bench.compare_maps with the bar of test_c3_lookahead_free_running_matches_oracle: -> (passes, 'byte-equal' or the numbers)."""
    import bench
    d = bench.compare_maps(a, b)
    if d["equal"]:
        return True, "byte-equal"
    ok = d["cubes_differing"] == 0 and d["floats_differing"] <= 64 and d["max_abs_diff"] < 1e-4
    return ok, "%d cubes / %s floats differ, max %s" % (d["cubes_differing"], d.get("floats_differing"), d.get("max_abs_diff"))


@pytest.fixture(scope="module")
def sweeps(street):
    return {case: _scans(street, case) for case in CASES}


@pytest.fixture(scope="module")
def oracle_runs(op, sweeps):
    """Free-running oracle replays (KD-tree kNN) of every case, in threads (ctypes releases the GIL)."""
    def replay(case):
        scans, n = sweeps[case], case[3]
        o = op.Oracle(knn_backend=1, **_kw(case))
        poses = np.zeros((n, 14))
        for k in range(n):
            o.process(scans[k])
            poses[k, :7], poses[k, 7:] = o.get("lo.pose")[:7], o.get("lm.pose")[:7]
        return poses, (o.get("lm.cornerMap"), o.get("lm.surfMap"))
    out = _run_threads([(lambda c=c: replay(c)) for c in CASES])
    return dict(zip(CASES, out))


def _gpu_replay(pkg, kw, dev, no_grid):
    """bench.py's replay order on device buffers: the next two sweeps registered ahead, then process_frame_device.  The grid
    bookkeeping {chunks, live, tombstones, dirty} is read after every sweep (host copies as of the last S2); at the end the map is
    published and read, then exported (the export forces the pool path, so it comes last)."""
    if no_grid: os.environ["VLOAM_NO_GRID"] = "1"
    try:
        g = pkg.Context(**kw)
    finally:
        os.environ.pop("VLOAM_NO_GRID", None)
    import bench
    n = len(dev) - 1
    pose, poses, grid, centres = np.zeros(14), [], [], []
    for k in range(n):
        bench.prefetch_ahead(g, dev, k, True)
        g.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, pose.ctypes.data)
        poses.append(pose.copy())
        grid.append(np.frombuffer(g.get_raw("lm.grid"), np.int32).copy())
        centres.append(int(g.get("lm.validInd")[0]))
    paths = g.get("lm.paths")
    g.publish_map()
    pub = g.get_map()
    maps = (g.get("lm.cornerMap"), g.get("lm.surfMap"))
    g.close()
    return dict(poses=np.array(poses), grid=np.array(grid), paths=paths, pub=pub, maps=maps, centres=centres)


def _checkpoints(pkg, op, kw, scans, n):
    """Oracle and GPU context in lock step, free-running (capture off) between teacher-forced, stage-by-stage, bit-exact
    checkpoints (capture on): sweep 1, and the sweep after the sub-map window moved (the last sweep when it never moves).
    Returns the checkpoint sweeps and, per checkpoint, whether the stack guard fired on the corner / surf stack."""
    o, g = op.Oracle(knn_backend=1, **kw), pkg.Context(**kw)
    g.set_capture(True)
    o.scan_registration(scans[0]); g.begin_frame(); g.scan_registration(scans[0])
    o.laser_odometry(); g.laser_odometry()
    o.laser_mapping(); g.laser_mapping()
    check_frame(o, g, 0)
    g.set_capture(False)
    centre0, moved_at, done, guards = int(o.get("lm.validInd")[0]), None, [], []
    for k in range(1, n):
        if k == 1 or (moved_at is not None and k == moved_at + 1) or (moved_at is None and k == n - 1):
            teacher_force(o, g)
            g.set_capture(True)
            o.scan_registration(scans[k]); g.begin_frame(); g.scan_registration(scans[k])
            o.laser_odometry(); g.laser_odometry()
            o.laser_mapping(); g.laser_mapping()
            check_frame(o, g, k)
            fired = []
            for last, stack, leaf in (("lo.cornerLast", "lm.cornerStack", kw["line_res"]), ("lo.surfLast", "lm.surfStack", kw["plane_res"])):
                src = o.get(last)
                fired.append(_guard_fires(src, leaf))
                if fired[-1]:   # the guard's output is its input (check_frame pinned the GPU stack to the oracle's)
                    assert o.get(stack).tobytes() == src.tobytes(), "%s: the guard fired but the stack is not the input" % stack
            guards.append(fired)
            g.set_capture(False)
            done.append(k)
        else:
            o.process(scans[k]); g.process_frame(scans[k])
        if moved_at is None and int(o.get("lm.validInd")[0]) != centre0:
            moved_at = k
    g.close()
    return done, moved_at, guards


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_leaf_sizes_grid_pool_oracle_publication(pkg, op, sweeps, oracle_runs, case):
    import torch
    kw, n = _kw(case), case[3]
    scans = sweeps[case]
    dev = [torch.from_numpy(s).cuda() for s in scans]
    grid = _gpu_replay(pkg, kw, dev, False)
    pool = _gpu_replay(pkg, kw, dev, True)
    cpu_poses, cpu_maps = oracle_runs[case]

    # a. the in-place grid update against the pool path: bit-identical poses, maps and published clouds
    assert (grid["poses"] == pool["poses"]).all(), "poses differ between the grid and the pool path"
    assert grid["maps"][0] == pool["maps"][0] and grid["maps"][1] == pool["maps"][1], "maps differ between the grid and the pool path"
    assert grid["pub"].tobytes() == pool["pub"].tobytes(), "published maps differ between the grid and the pool path"

    # branches: the in-place path really ran, and tombstones appear exactly when a leaf is above the threshold
    inplace, poolpath = int(grid["paths"][0]), int(grid["paths"][1])
    assert n - 1 <= inplace + poolpath <= n and pool["paths"][0] == 0, (grid["paths"], pool["paths"])
    assert inplace >= n / 2, "the in-place path ran on only %d of %d mapped sweeps" % (inplace, n)
    max_dead = int(grid["grid"][:, 2].max())
    if max(kw["line_res"], kw["plane_res"]) <= INPLACE_MAX_LEAF:
        assert max_dead == 0, "%d tombstones with both leaves <= %g m" % (max_dead, INPLACE_MAX_LEAF)
    else:
        assert max_dead > 0, "no tombstone with a leaf above %g m: the re-insert path never ran" % INPLACE_MAX_LEAF
    if n > 23:
        assert len(set(grid["centres"])) > 1, "the window never moved"

    # b. free-running against the oracle: poses within tolerance, maps byte-equal or within the C3 bar
    for k in range(n):
        pose_close(cpu_poses[k, :7], grid["poses"][k, :7]); pose_close(cpu_poses[k, 7:], grid["poses"][k, 7:])
    verdicts = []
    for kind, a, b in (("corner", grid["maps"][0], cpu_maps[0]), ("surf", grid["maps"][1], cpu_maps[1])):
        ok, why = _compare_maps(a, b)
        assert ok, (kind, why)
        verdicts.append("%s %s" % (kind, why))

    # d. the publication: LM.cpp:884-899 over the export of the same map, and over the oracle's
    assert grid["pub"].tobytes() == laser_cloud_map(*grid["maps"]).tobytes(), "published map differs from the interleaved export"
    pub_exact = grid["pub"].tobytes() == laser_cloud_map(*cpu_maps).tobytes()

    # c. teacher-forced checkpoints: stacks, from-map clouds, kNN, fit flags and maps bit-exact on the pool path
    done, moved_at, guards = _checkpoints(pkg, op, kw, scans, n)
    assert len(done) == 2, done
    if n > 23:
        assert moved_at is not None and done[1] == moved_at + 1, (done, moved_at)

    print("%s leaf %g/%g: in-place %d / pool %d sweeps, max tombstones %d, stack guard corner/surf %s, "
          "maps vs oracle: %s, publication vs oracle %s, checkpoints at sweeps %s"
          % ("VLP-16" if case[0] == 0 else "HDL-64", kw["line_res"], kw["plane_res"], inplace, poolpath, max_dead,
             "/".join("yes" if f else "no" for f in guards[0]), ", ".join(verdicts), "byte-equal" if pub_exact else "within the bar", done))
