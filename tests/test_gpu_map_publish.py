"""vloam_b200_publish_map / get_map: LaserMapping::publish's global map (LM.cpp:884-899) assembled on the device.

The assembly reads the map as the last mapped frame left it -- the cube pools, or the voxel-hash grid for the window's cubes after
in-place updates -- and writes nothing of it.  These tests check the published cloud against the oracle on the benchmarked path,
the grid branch against the pool branch bit for bit, that publishing changes no pose, map or map path, and the edges of the ABI."""
import os
import sys
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from map_publish_ref import laser_cloud_map, laser_cloud_map_of  # noqa: E402

pytestmark = pytest.mark.gpu

STREET_KW = dict(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8)


def _close_enough(a, b):
    """The bar of test_c3_lookahead_free_running_matches_oracle: equal length; byte-identical, or at most 64 floats differing by < 1e-4."""
    if len(a) != len(b):
        return False, "length %d vs %d" % (len(a), len(b))
    if a.tobytes() == b.tobytes():
        return True, "equal"
    d = np.abs(a.astype(np.float64) - b.astype(np.float64))
    nd = int((a.view(np.uint32) != b.view(np.uint32)).sum())
    return nd <= 64 and float(d.max()) < 1e-4, "%d floats differ, max %.3g" % (nd, float(d.max()))


def test_publish_matches_oracle_on_benchmarked_path(pkg):
    """bench.py's eight C3 sequences, 27 free-running sweeps, two sweeps registered ahead, host buffers, helper thread on,
    capture off; publish after every 5th mapped frame: every published cloud against the oracle's global map at that frame."""
    import torch
    import bench
    from test_gpu_benchmarked_path import _run_threads
    import oracle_py as op
    frames, every = 27, 5
    seqs = [bench.make_sequence(pkg, sid, frames + 1) for sid in range(8)]

    def oracle(s):
        o = op.Oracle(knn_backend=1, **bench.KW)
        o.set("lm.cornerMap", s[2]); o.set("lm.surfMap", s[3])
        maps = []
        for k in range(frames):
            o.process(s[0][k])
            if (k + 1) % every == 0:
                maps.append(laser_cloud_map_of(o))
        return maps
    cpu = _run_threads([(lambda s=s: oracle(s)) for s in seqs])
    exact, worst = 0, []
    for sid, (scans, _, cb, sb) in enumerate(seqs):
        g = pkg.Context(**bench.KW)
        g.set("lm.cornerMap", cb); g.set("lm.surfMap", sb)
        pinned = [torch.from_numpy(s).pin_memory() for s in scans[:frames + 1]]
        pose, pubs = np.zeros(14), []
        for k in range(frames):
            bench.prefetch_ahead(g, pinned, k, False)
            g.process_frame_ptr(pinned[k].data_ptr(), pinned[k].shape[0], 4, pose.ctypes.data)
            if (k + 1) % every == 0:
                g.publish_map()
                pubs.append(g.get_map())
        paths = g.get("lm.paths")
        g.close()
        assert paths[0] > 0, "sequence %d never took the in-place path: the grid branch of the assembly was not exercised" % sid
        assert len(pubs) == len(cpu[sid]) == frames // every
        for i, (a, b) in enumerate(zip(pubs, cpu[sid])):
            ok, why = _close_enough(a, b)
            assert ok, (sid, i, why)
            exact += a.tobytes() == b.tobytes()
            worst.append(why)
    print("published maps vs oracle: %d / %d byte-identical" % (exact, 8 * (frames // every)))
    assert exact >= 6 * (frames // every)


@pytest.fixture(scope="module")
def drive(pkg):
    """The 45-sweep, 1.5 m/sweep C3 drive of test_grid_update_equals_pool_update (two window moves), device-resident, two ahead:
    the grid with a publication after every sweep, the pool path (VLOAM_NO_GRID=1) with the same, and the grid without any."""
    import torch
    import bench
    n = 45
    world = pkg.synth.World(1234, 1, 190.0)
    traj = pkg.synth.trajectory(n + 1, seed=91, step=1.5)
    scans = bench._gen_scans(pkg, world, traj, [4000 + k for k in range(n + 1)])
    _, _, cb, sb = bench.make_sequence(pkg, 0, 1)
    dev = [torch.from_numpy(s).cuda() for s in scans]
    out = {}
    for mode, publish in (("grid", True), ("pool", True), ("quiet", False)):
        if mode == "pool": os.environ["VLOAM_NO_GRID"] = "1"
        try:
            g = pkg.Context(**bench.KW)
        finally:
            os.environ.pop("VLOAM_NO_GRID", None)
        g.set("lm.cornerMap", cb); g.set("lm.surfMap", sb)
        pose, poses, pubs, centres, allocs = np.zeros(14), [], [], set(), []
        for k in range(n):
            bench.prefetch_ahead(g, dev, k, True)
            g.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, pose.ctypes.data)
            poses.append(pose.copy())
            if publish:
                g.publish_map()
                pubs.append(g.get_map())
            if k % 5 == 4: centres.add(int(g.get("lm.validInd")[0]))
            allocs.append(int(g.get("alloc.count")[0]))
        out[mode] = dict(poses=np.array(poses), pubs=pubs, paths=g.get("lm.paths"), grid=g.get_raw("lm.grid"), allocs=allocs,
                         ncentres=len(centres), final=laser_cloud_map_of(g), maps=(g.get("lm.cornerMap"), g.get("lm.surfMap")))
        g.close()
    # Deferred reads: publish after sweep p (p even) and call get_map only after sweeps p+1 and p+2 have been processed, so the
    # assembly is in flight while they edit the map (in-place updates, window moves, lm_materialize): every sweep after the first
    # runs under a pending publication.  Nothing between the
    # publication and the read talks to the context except process_frame (a debug get would drain the publication stream).
    g = pkg.Context(**bench.KW)
    g.set("lm.cornerMap", cb); g.set("lm.surfMap", sb)
    pose, poses, pubs, windows, pending = np.zeros(14), [], {}, [], None
    for k in range(n):
        bench.prefetch_ahead(g, dev, k, True)
        g.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, pose.ctypes.data)
        poses.append(pose.copy())
        if pending is not None and k == pending[0] + 2:
            pubs[pending[0]] = g.get_map()
            windows.append(g.get("lm.paths") - pending[1])  # map paths the sweeps of the window took
            pending = None
        if k % 2 == 0:
            paths = g.get("lm.paths")  # (no publication pending: this drains nothing that matters)
            g.publish_map()
            pending = (k, paths)
    if pending is not None:
        pubs[pending[0]] = g.get_map()
    out["deferred"] = dict(poses=np.array(poses), pubs=pubs, windows=windows)
    g.close()
    return out


def test_grid_publication_equals_pool_publication(drive):
    """Every cloud published on the in-place path (grid + stale pools) equals the pool path's, byte for byte; the last one equals
    the interleave of the debug export taken after the last sweep."""
    g, p = drive["grid"], drive["pool"]
    assert g["ncentres"] >= 2, "the window never moved"
    assert g["paths"][0] > 0 and p["paths"][0] == 0, (g["paths"], p["paths"])
    assert (g["poses"] == p["poses"]).all()
    for k, (a, b) in enumerate(zip(g["pubs"], p["pubs"])):
        assert a.tobytes() == b.tobytes(), "sweep %d: published maps differ between the grid and the pool path (%d vs %d points)" % (k, len(a), len(b))
    assert g["pubs"][-1].tobytes() == g["final"].tobytes()
    assert len(g["pubs"][-1]) > 1000000


def test_publication_does_not_perturb(drive):
    """Publishing after every sweep against never publishing: identical poses, maps, map paths and grid bookkeeping, and no
    device allocation once the first publication has sized its buffers."""
    g, q = drive["grid"], drive["quiet"]
    assert (g["poses"] == q["poses"]).all(), "publishing changed a pose"
    assert g["maps"] == q["maps"], "publishing changed the map"
    assert (g["paths"] == q["paths"]).all(), ("publishing changed which map path the sweeps took", g["paths"], q["paths"])
    # grid bookkeeping {live points, tombstones, dirty} (not the chunk bump pointer: chunks leaked by lost CAS races vary run to run)
    assert (np.frombuffer(g["grid"], np.int32)[1:] == np.frombuffer(q["grid"], np.int32)[1:]).all(), "publishing changed the grid bookkeeping"
    # the publishing run allocates its buffers at the first publication; after that it allocates exactly what the quiet run does
    assert np.array_equal(np.diff(g["allocs"][1:]), np.diff(q["allocs"][1:])), (g["allocs"], q["allocs"])


def test_deferred_reads_equal_synchronous_reads(drive):
    """A publication read two sweeps after it was queued -- the next sweeps edited the map in place, moved the window and wrote
    the grid back to the pools while it was in flight -- equals the one read at once after the same sweep."""
    d, g = drive["deferred"], drive["grid"]
    assert (d["poses"] == g["poses"]).all()
    assert len(d["pubs"]) == 23
    for k, cloud in d["pubs"].items():
        assert cloud.tobytes() == g["pubs"][k].tobytes(), "publication after sweep %d changed while it was in flight" % k
    w = np.array(d["windows"])
    assert (w[:, 0] > 0).any() and (w[:, 1] > 0).any(), ("no in-place sweep or no pool-path sweep ran under a pending publication", w.tolist())


def _street_replay(pkg, synth, street, n, env=None, kw=STREET_KW, defer=0):
    """Street replay that publishes after every sweep and reads at once (defer = 0), or publishes after every `defer`-th sweep
    and reads only after `defer` more sweeps (every later sweep runs under a pending publication).  Returns poses, {sweep: cloud}, the final maps and the device allocations
    made while publications were pending."""
    traj = synth.trajectory(n)
    scans = [street.scan(1, traj[k], 1000 + k) for k in range(n)]
    for key, v in (env or {}).items(): os.environ[key] = v
    try:
        g = pkg.Context(**kw)
    finally:
        for key in (env or {}): os.environ.pop(key, None)
    poses, pubs, grew, pending = [], {}, 0, None
    for k in range(n):
        poses.append(g.process_frame(scans[k]).copy())
        if pending is not None and k == pending[0] + defer:
            pubs[pending[0]] = g.get_map()
            grew += int(g.get("alloc.count")[0]) - pending[1]
            pending = None
        if defer == 0:
            g.publish_map()
            pubs[k] = g.get_map()
        elif k % defer == 0:
            allocs = int(g.get("alloc.count")[0])
            g.publish_map()
            pending = (k, allocs)
    if pending is not None:
        pubs[pending[0]] = g.get_map()
    maps = (g.get("lm.cornerMap"), g.get("lm.surfMap"))
    g.close()
    return np.array(poses), pubs, maps, grew


def test_pool_regrow_under_publication(pkg, synth, street):
    """Tiny initial pools (VLOAM_POOL_POINTS=4096, as test_map_pools_grow_instead_of_failing) with every sweep after the first under a
    pending publication (queued after sweep p, read after sweep p+2): every publication equals the one a default-pool run reads at
    once after the same sweep, and so do poses and maps."""
    n = 12
    p0, m0, e0, _ = _street_replay(pkg, synth, street, n)
    p1, m1, e1, _ = _street_replay(pkg, synth, street, n, env={"VLOAM_POOL_POINTS": "4096"}, defer=2)
    p2, m2, e2, _ = _street_replay(pkg, synth, street, n, defer=2)
    assert (p0 == p1).all() and (p0 == p2).all() and e0 == e1 == e2
    assert sorted(m1) == sorted(m2) == [0, 2, 4, 6, 8, 10]
    for k in m1:
        assert m1[k].tobytes() == m0[k].tobytes(), "tiny pools, publication after sweep %d" % k
        assert m2[k].tobytes() == m0[k].tobytes(), "default pools, publication after sweep %d" % k
    assert len(e0[1]) > 4851 * 4 + 3 * 4096 * 16, "the surf map never outgrew the tiny pool: growth was not exercised"
    assert m0[n - 1].tobytes() == laser_cloud_map(*e0).tobytes()


def test_pool_regrow_behind_pending_publication(pkg):
    """The planted C3 map imported into tiny pools (VLOAM_POOL_POINTS=4096: the import sizes them to twice the map, the first
    sweep's head-room check then doubles both), published at once, and read only after three sweeps: the first sweep replaces
    both pools while that publication is queued behind nothing else.  The cloud must be the imported map, as with default pools
    (which never regrow here), and the tiny-pool run must have made more allocations in that window."""
    import bench
    scans, _, cb, sb = bench.make_sequence(pkg, 0, 3)

    def run(env):
        for key, v in env.items(): os.environ[key] = v
        try:
            g = pkg.Context(**bench.KW)
        finally:
            for key in env: os.environ.pop(key, None)
        g.set("lm.cornerMap", cb); g.set("lm.surfMap", sb)
        a0 = int(g.get("alloc.count")[0])
        g.publish_map()
        for k in range(3):
            g.process_frame(scans[k])
        cloud = g.get_map()
        grew = int(g.get("alloc.count")[0]) - a0
        g.close()
        return cloud, grew

    want = laser_cloud_map(cb, sb)
    tiny, grew_tiny = run({"VLOAM_POOL_POINTS": "4096"})
    default, grew_default = run({})
    assert tiny.tobytes() == want.tobytes() and default.tobytes() == want.tobytes()
    assert grew_tiny > grew_default, ("no pool regrow happened while the publication was pending", grew_tiny, grew_default)


def test_get_map_edges(pkg, synth, street):
    """Nothing published yet: VLOAM_E_INVALID; an empty map publishes 0 points; a too small buffer: VLOAM_E_CAPACITY."""
    g = pkg.Context(**STREET_KW)
    assert g.L.vloam_b200_get_map(g.h, None, 0) == -1
    with pytest.raises(pkg.VloamError):
        g.get_map()
    g.publish_map()
    assert g.get_map().shape == (0, 4)
    traj = synth.trajectory(3)
    for k in range(3):
        g.process_frame(street.scan(1, traj[k], 1000 + k))
    g.publish_map()
    n = g.L.vloam_b200_get_map(g.h, None, 0)
    assert n > 0
    buf = np.zeros((n, 4), np.float32)
    assert g.L.vloam_b200_get_map(g.h, buf.ctypes.data, n - 1) == -3
    assert g.L.vloam_b200_get_map(g.h, buf.ctypes.data, n) == n
    g.publish_map(); g.publish_map()  # a second publication replaces the first
    assert g.get_map().tobytes() == buf.tobytes() == laser_cloud_map_of(g).tobytes()
    g.close()


def test_publication_on_skipped_frame(pkg, synth, street):
    """mapping_skip_frame = 2: a publication after a skipped frame equals the one after the last mapped frame."""
    kw = dict(STREET_KW, mapping_skip_frame=2)
    traj = synth.trajectory(9)
    g = pkg.Context(**kw)
    last_count, last_pub, skipped = None, None, 0
    for k in range(9):
        g.process_frame(street.scan(1, traj[k], 1000 + k))
        g.publish_map()
        pub = g.get_map()
        count = int(g.get("lm.state")[3])  # mapped frames so far
        if count == last_count and count > 0:
            assert pub.tobytes() == last_pub.tobytes(), "frame %d (skipped) published another map" % k
            skipped += 1
        last_count, last_pub = count, pub
    g.close()
    assert skipped >= 3


def test_concurrent_contexts_publish(pkg, synth, street):
    """Eight contexts that publish while they replay, one host thread each, give the clouds of sequential runs."""
    nseq, n = 8, 6
    seqs = []
    for q in range(nseq):
        traj = synth.trajectory(n, seed=300 + q)
        seqs.append([street.scan(1, traj[k], 5000 + 100 * q + k) for k in range(n)])

    def replay(q, out):
        g = pkg.Context(**STREET_KW)
        pubs = []
        for k in range(n):
            g.process_frame(seqs[q][k])
            if k % 2 == 1:
                g.publish_map()
                pubs.append(g.get_map())
        g.close()
        out[q] = pubs

    alone, together = [None] * nseq, [None] * nseq
    for q in range(nseq):
        replay(q, alone)
    th = [threading.Thread(target=replay, args=(q, together)) for q in range(nseq)]
    for t in th: t.start()
    for t in th: t.join()
    for q in range(nseq):
        assert together[q] is not None, "a replay thread died"
        assert [a.tobytes() for a in alone[q]] == [b.tobytes() for b in together[q]], "sequence %d: published maps differ when contexts share the GPU" % q


def test_adapter_publishes_laser_cloud_map(pkg, op, synth, street, tmp_path):
    """vloam_adapter.hpp, LidarOdometryMapping over 41 frames with map_pub_number = 20 (tests/cpp/map_publish_adapter.cpp):
    laserCloudMap is published exactly when the mapped-frame count reaches 20 and 40 (LM.cpp:884-899), and its points equal
    Context.get_map() of a parallel Python run with the same rule and the oracle's global map at those frames."""
    import subprocess
    from test_abi import build_cpp_program
    exe = build_cpp_program("map_publish_adapter", tmp_path)
    kw = dict(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4)
    n = 41
    traj = synth.trajectory(n)
    scans = [street.scan(0, traj[k], 1000 + k) for k in range(n)]
    files = []
    for k, s in enumerate(scans):
        f = str(tmp_path / ("scan%d.bin" % k))
        s.tofile(f)
        files.append(f)
    out = subprocess.run([exe, str(tmp_path)] + files, check=True, capture_output=True, text=True).stdout
    assert "map publish ok" in out, out
    rows = [l.split() for l in out.splitlines() if l.startswith("frame ")]
    assert len(rows) == n
    published = [int(r[1]) for r in rows if r[5] == "1"]
    assert published == [19, 39], published
    assert all(int(r[7]) == 0 for r in rows[:19]), "laserCloudMap returned a cloud before the first publication"
    lom = pkg.LidarOdometryMapping(**kw)
    o = op.Oracle(**kw)
    py, cpu = {}, {}
    for k in range(n):
        lom.reset(); lom.scanRegistrationIO(scans[k]); lom.laserOdometryIO(); lom.laserMappingIO()
        o.process(scans[k])
        if lom.laser_mapping.frameCount % 20 == 0:
            py[k] = lom.ctx.get_map()
            cpu[k] = laser_cloud_map_of(o)
    lom.ctx.close()
    assert sorted(py) == [19, 39]
    for k in (19, 39):
        cpp = np.fromfile(str(tmp_path / ("map_%d.bin" % k)), np.float32).reshape(-1, 4)
        assert cpp.tobytes() == py[k].tobytes(), "frame %d: the adapter's laserCloudMap differs from Context.get_map()" % k
        ok, why = _close_enough(cpp, cpu[k])
        assert ok, (k, why)


def test_python_mirror_counts_mapped_frames(pkg, synth, street):
    """api.LidarOdometryMapping with mapping_skip_frame = 2: LaserMapping.frameCount counts mapped frames only (the device's
    count), and the map is queued once per multiple of map_pub_number, as vloam_adapter.hpp's LaserMapping::publish does."""
    lom = pkg.LidarOdometryMapping(map_pub_number=3, **dict(STREET_KW, mapping_skip_frame=2))
    traj = synth.trajectory(14)
    queued = [0]
    for k in range(14):
        lom.reset(); lom.scanRegistrationIO(street.scan(1, traj[k], 1000 + k)); lom.laserOdometryIO(); lom.laserMappingIO()
        if lom.laser_mapping._published_at != queued[-1]:
            queued.append(lom.laser_mapping._published_at)
    count = int(lom.ctx.get("lm.state")[3])
    assert 3 <= lom.laser_mapping.frameCount == count < 14
    assert queued[1:] == list(range(3, count + 1, 3))
    lom.ctx.close()
