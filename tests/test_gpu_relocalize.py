"""vloam_b200_relocalize: the device search against tests/relocalize_ref.py (query points, occupancy and yaw table byte for byte; best
and runner-up against the exhaustive search), global relocalization in the C3 prior and the street world followed by frozen
localization, bit-identical results across scheduling modes, the stale-pool path, no cost when unused and the ABI's edges."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import relocalize_ref as rr  # noqa: E402
from map_publish_ref import split_blob  # noqa: E402
from test_gpu_prior_map import _ctx, _drive, _prior  # noqa: E402

pytestmark = pytest.mark.gpu

_CACHE = {}


def _frozen_start(pkg, n_first=1, env=None, x0=40.0):
    """Load the C3 prior, freeze it, and map the first sweep(s) of the drive from the identity map pose."""
    scans, traj = _drive(pkg, 30, x0=x0)
    corner, surf = _prior(pkg, "C3")
    for k, v in (env or {}).items():
        os.environ[k] = v
    try:
        g = _ctx(pkg)
    finally:
        for k in (env or {}):
            os.environ.pop(k, None)
    g.load_map(corner, surf)
    g.set_map_update(False)
    for k in range(n_first):
        g.process_frame(scans[k])
    return g, scans, traj


def _check_against_ref(pkg, g, q_c, t_c, exhaustive=True, **kw):
    res = g.relocalize(q_c, t_c, apply=False, **kw)
    stack_c, stack_s = g.get("lm.cornerStack"), g.get("lm.surfStack")
    mp = np.concatenate([split_blob(g.get("lm.cornerMap"))[1], split_blob(g.get("lm.surfMap"))[1]])
    opts = {k: v for k, v in kw.items() if k not in ("max_range", "max_points", "min_score")}
    u = rr.select(stack_c, stack_s, q_c, kw.get("max_range", 60.0), kw.get("max_points", 2048))
    sp = rr.Space(u, t_c, max_range=kw.get("max_range", 60.0), **opts)
    assert g.get("rl.points").tobytes() == u.tobytes(), "query points differ"
    o, dims, occ = g.get("rl.occ")
    assert o.tobytes() == sp.o.tobytes() and list(dims) == list(sp.dims), "grid geometry differs"
    ref_occ = sp.occupancy(mp)
    assert occ.tobytes() == ref_occ.tobytes(), "occupancy differs in %d cells" % (occ != ref_occ).sum()
    assert g.get("rl.yaw").tobytes() == sp.yaw_table().tobytes(), "yaw table differs"
    assert res.n_points == len(u) and res.candidates == sp.candidates
    if exhaustive:
        sc = sp.scores(ref_occ, sp.cells(u))
        (b, s), (rI, rs) = sp.best_and_runner(sc)
        assert (res.index, res.score) == (b, s), "best (%d, %d) != exhaustive (%d, %d)" % (res.index, res.score, b, s)
        assert (res.runner_index, res.runner_score) == (rI, rs), "runner-up (%d, %d) != exhaustive (%d, %d)" % (
            res.runner_index, res.runner_score, rI, rs)
        q, t = sp.pose(b, q_c)
        assert np.array(res.q).tobytes() == q.tobytes() and np.array(res.t).tobytes() == t.tobytes()
        if rI >= 0:
            q, t = sp.pose(rI, q_c)
            assert np.array(res.runner_q).tobytes() == q.tobytes() and np.array(res.runner_t).tobytes() == t.tobytes()
        lv = g.get("rl.levels")
        assert lv[32] < sp.candidates and lv[33] < sp.candidates, "a search evaluated more nodes than the exhaustive one scores"
    return res


def test_grids_match_reference(pkg, street, synth):
    """rl.points / rl.occ / rl.yaw byte-equal to the restatement: C3 at the defaults and at r = 0.5, range 40; the street world."""
    from test_gpu_prior_map import _guess
    g, scans, traj = _frozen_start(pkg)
    q, t = _guess(pkg, traj[0], (3.0, -2.0), 40.0)
    _check_against_ref(pkg, g, q, t, exhaustive=False)
    _check_against_ref(pkg, g, q, t, exhaustive=False, resolution=0.5, max_range=40.0, half_xy=10.0, yaw_step_deg=4.0)
    g.close()
    s, st = _street(pkg, synth, street)
    q, t = _guess(pkg, st[0], (2.0, 1.0), -30.0)
    _check_against_ref(pkg, s, q, t, exhaustive=False, max_points=700)
    s.close()


def _street(pkg, synth, street, n=1):
    traj = synth.trajectory(16, seed=5)
    traj[:, 0] += 30.0
    scans = [street.scan(0, traj[k], 1000 + k) for k in range(16)]
    g = pkg.Context(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4)
    g.load_map(street.plant(0, 0.15, seed=9), street.plant(1, 0.3, seed=8))
    g.set_map_update(False)
    for k in range(n):
        g.process_frame(scans[k])
    _CACHE["street_scans"] = scans
    return g, traj


@pytest.mark.parametrize("start,guess", [(40.0, (3.0, -4.0, 25.0)), (52.0, (-7.0, 2.0, -100.0)), (46.0, (0.0, 6.25, 170.0))])
def test_exact_against_exhaustive_search(pkg, start, guess):
    """Best and runner-up (index, score, pose) equal the numpy exhaustive search at +-20 m x 360 deg at 3 deg, z +-1 m.  The third
    start sits half a tower pitch (12.5 m / 2) off in y, where the runner-up is a neighbouring tower row."""
    from test_gpu_prior_map import _guess
    g, scans, traj = _frozen_start(pkg, x0=start)
    q, t = _guess(pkg, traj[0], guess[:2], guess[2])
    res = _check_against_ref(pkg, g, q, t, half_xy=20.0, half_z=1.0, yaw_step_deg=3.0, max_points=1024)
    print("exhaustive match: %r" % res)
    g.close()


def _frozen_after_reloc(pkg, g, scans, n, start=1, mode="two"):
    import torch
    import bench
    pinned = [torch.from_numpy(s).pin_memory() for s in scans]
    pose, poses = np.zeros(14), []
    for k in range(start, start + n):
        if mode == "two":
            bench.prefetch_ahead(g, pinned, k, False)
        g.process_frame_ptr(pinned[k].data_ptr(), pinned[k].shape[0], 4, pose.ctypes.data)
        poses.append(pose.copy())
    return np.array(poses)


def test_global_relocalization_c3(pkg):
    """A guess 30 m and 150 deg off, searched over +-50 m x 360 deg; then frozen sweeps on the benchmarked path: within 0.05 m of the
    generator's truth from sweep 15 on, the bar of test_frozen_localization_matches_oracle on this drive.  (At 1.5 m per sweep the
    odometry lags the truth by ~2 m; from a 0.5 m / 2 deg guess the frozen drive itself is 1.6 m off at sweep 10 and converges by
    sweep 14, and after the relocalization the errors from sweep 10 on are that series: the half-cell start is not what limits it.)"""
    from test_gpu_prior_map import _guess
    g, scans, traj = _frozen_start(pkg)
    q, t = _guess(pkg, traj[0], (21.2, -21.2), 150.0)
    res = g.relocalize(q, t, half_xy=50.0)
    print("C3 relocalization: %r, truth %s" % (res, np.round(traj[0, :3], 3)))
    assert res.found and res.score > res.runner_score
    assert np.abs(np.array(res.t[:2]) - traj[0, :2]).max() <= 0.5 + 1e-9
    poses = _frozen_after_reloc(pkg, g, scans, 24)
    err = [np.abs(poses[k - 1, 11:13] - traj[k, :2]).max() for k in range(15, 25)]
    print("C3 localization error after relocalization, sweeps 15..24: %.4f m" % max(err))
    assert max(err) < 0.05
    g.close()


def test_global_relocalization_street(pkg, synth, street):
    from test_gpu_prior_map import _guess
    g, traj = _street(pkg, synth, street)
    scans = _CACHE["street_scans"]
    q, t = _guess(pkg, traj[0], (-21.2, 21.2), -150.0)
    res = g.relocalize(q, t, half_xy=50.0)
    print("street relocalization: %r, truth %s" % (res, np.round(traj[0, :3], 3)))
    assert res.found and res.score > res.runner_score
    poses = _frozen_after_reloc(pkg, g, scans, 15)
    err = [np.abs(poses[k, 11:13] - traj[1 + k, :2]).max() for k in range(9, 15)]
    print("street localization error after relocalization, sweeps 10..15: %.4f m" % max(err))
    assert max(err) < 0.05
    g.close()


def _reloc_drive(pkg, env=None, mode="two"):
    from test_gpu_prior_map import _guess
    g, scans, traj = _frozen_start(pkg, env=env)
    q, t = _guess(pkg, traj[0], (21.2, -21.2), 150.0)
    res = g.relocalize(q, t, half_xy=30.0)
    out = (res.index, res.score, res.runner_index, res.runner_score, res.nodes, bytes(res))
    poses = _frozen_after_reloc(pkg, g, scans, 6, mode=mode)
    g.close()
    return out, poses


@pytest.mark.parametrize("variant", ["plain", "no_worker", "no_grid", "no_lo_lookahead", "no_stacks_lookahead"])
def test_bit_identical_across_modes(pkg, variant):
    ref = _CACHE.get("mode_ref") or _reloc_drive(pkg)
    _CACHE["mode_ref"] = ref
    env = {"no_worker": {"VLOAM_NO_WORKER": "1"}, "no_grid": {"VLOAM_NO_GRID": "1"}, "no_lo_lookahead": {"VLOAM_NO_LO_LOOKAHEAD": "1"},
           "no_stacks_lookahead": {"VLOAM_NO_STACKS_LOOKAHEAD": "1"}}.get(variant)
    out = _reloc_drive(pkg, env=env, mode="plain" if variant == "plain" else "two")
    assert out[0] == ref[0], "%s: search result differs" % variant
    assert (out[1] == ref[1]).all(), "%s: poses after the relocalization differ" % variant


def test_stale_pools_equal_loaded_map(pkg):
    """Sweeps mapped in place leave the cube pools behind the grid: a relocalization then builds its occupancy from the map as it
    stands (the map the export, which writes the pools back, returns) and gives what it gives once the pools are current."""
    from test_gpu_prior_map import _guess
    scans, traj = _drive(pkg, 20)
    corner, surf = _prior(pkg, "C3")
    g = _ctx(pkg)
    g.load_map(corner, surf)
    q0, t0 = _guess(pkg, traj[0])
    g.set_map_pose(q0, t0)
    for k in range(8):
        g.process_frame(scans[k])
    assert g.get("lm.paths")[0] > 0, "no sweep took the in-place path"
    q, t = _guess(pkg, traj[7], (5.0, 3.0), 60.0)
    stale = g.relocalize(q, t, apply=False)
    occ_stale = g.get("rl.occ")[2]
    mp = np.concatenate([split_blob(g.get("lm.cornerMap"))[1], split_blob(g.get("lm.surfMap"))[1]])
    current = g.relocalize(q, t, apply=False)
    sp = rr.Space(g.get("rl.points"), t)
    assert occ_stale.tobytes() == sp.occupancy(mp).tobytes() == g.get("rl.occ")[2].tobytes()
    assert bytes(stale) == bytes(current)
    g.close()


def test_no_cost_when_unused(pkg):
    """Localizing in a frozen map, a relocalization adds launches and allocations of its own only: the sweeps after it launch and
    allocate what the same sweeps launch and allocate in a context that never calls it.  (After sweeps mapped in place the call first
    writes the grid back to the cube pools, and the next sweep then rebuilds its grid, as after an export.)"""
    per = []
    for reloc in (False, True):
        g, scans, traj = _frozen_start(pkg, n_first=10)
        if reloc:
            g.relocalize([0, 0, 0, 1], [40, 0, 0], apply=False)
        g.synchronize()
        l0, a0 = g.kernel_launches, int(g.get("alloc.count")[0])
        for k in range(10, 30):
            g.process_frame(scans[k])
        g.synchronize()
        per.append((g.kernel_launches - l0, int(g.get("alloc.count")[0]) - a0))
        g.close()
    assert per[0] == per[1], per


def test_adapter_relocalizes_in_a_prior_map(pkg, synth, street, tmp_path):
    """vloam_adapter.hpp (tests/cpp/relocalize_adapter.cpp): loadMap from .bin files, setMapUpdate(false), one sweep, relocalize from a
    guess 20 m / 120 deg off, then localize -- its result and poses bit for bit those of the same calls through Python."""
    import subprocess
    from test_abi import build_cpp_program
    from test_gpu_prior_map import _guess
    exe = build_cpp_program("relocalize_adapter", tmp_path)
    kw = dict(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4)
    n = 8
    traj = synth.trajectory(n, seed=5)
    traj[:, 0] += 30.0
    scans = [street.scan(0, traj[k], 1000 + k) for k in range(n)]
    corner, surf = street.plant(0, 0.15, seed=9), street.plant(1, 0.3, seed=8)
    files = []
    for name, a in [("corner", corner), ("surf", surf)] + [("scan%d" % k, s) for k, s in enumerate(scans)]:
        f = str(tmp_path / (name + ".bin"))
        np.ascontiguousarray(a, np.float32).tofile(f)
        files.append(f)
    q, t = _guess(pkg, traj[0], (14.1, -14.1), 120.0)
    out = subprocess.run([exe, files[0], files[1]] + ["%.17g" % v for v in np.r_[q, t]] + files[2:], check=True, capture_output=True,
                         text=True).stdout
    assert "relocalize ok" in out, out
    lines = out.splitlines()
    got = np.array([[float(v) for v in l.split()[1:]] for l in lines if l.startswith("pose ")])
    lom = pkg.LidarOdometryMapping(**kw)
    lom.laser_mapping.load_map(corner, surf)
    lom.laser_mapping.set_map_update(False)
    ref = []
    for k, s in enumerate(scans):
        lom.reset(); lom.scanRegistrationIO(s); lom.laserOdometryIO(); lom.laserMappingIO()
        ref.append(np.r_[lom.laser_mapping.pose[0], lom.laser_mapping.pose[1]])
        if k == 0:
            res = lom.laser_mapping.relocalize(q, t, half_xy=30.0)
            assert res.found
            assert [l for l in lines if l.startswith("reloc ")][0] == "reloc %d %d %d %d" % (res.index, res.score, res.runner_score, res.found)
    assert got.shape == (n, 7) and (got == np.array(ref)).all(), "adapter poses differ from the Python run"


def test_eight_concurrent_contexts(pkg):
    from test_gpu_benchmarked_path import _run_threads
    ref = _reloc_drive(pkg, mode="plain")

    def one():
        return _reloc_drive(pkg, mode="two")
    for out in _run_threads([one] * 8):
        assert out[0] == ref[0] and (out[1] == ref[1]).all()


def test_contract_edges(pkg):
    L = pkg.load_lib()
    g = _ctx(pkg)
    with pytest.raises(pkg.VloamError, match="no mapped sweep"):
        g.relocalize([0, 0, 0, 1], [0, 0, 0])
    g.close()
    g, scans, traj = _frozen_start(pkg)
    for bad in (dict(resolution=0.0), dict(max_range=-1.0), dict(max_points=0), dict(half_xy=float("nan")), dict(half_yaw_deg=200.0),
                dict(min_score=-0.1), dict(exclusion_m=float("inf"))):
        with pytest.raises(pkg.VloamError):
            g.relocalize([0, 0, 0, 1], [0, 0, 0], **bad)
    with pytest.raises(pkg.VloamError):
        g.relocalize([0, 0, 0, 0], [0, 0, 0])
    with pytest.raises(pkg.VloamError):
        g.relocalize([0, 0, 0, 1], [0, np.nan, 0])
    assert L.vloam_b200_relocalize(g.h, None, None) == -1
    with pytest.raises(pkg.VloamError, match="candidates"):
        g.relocalize([0, 0, 0, 1], [0, 0, 0], half_xy=2000.0, yaw_step_deg=0.5, half_z=20.0)
    # apply = 0 leaves the mapping state alone; apply = 1 changes q/t_wmap_wodom only
    before = g.get("lm.pose")
    g.relocalize([0, 0, 0, 1], [40, 0, 0], apply=False)
    assert g.get("lm.pose").tobytes() == before.tobytes()
    res = g.relocalize([0, 0, 0, 1], [40, 0, 0], min_score=0.0)
    after = g.get("lm.pose")
    assert res.found and after[:7].tobytes() == before[:7].tobytes() and after[7:].tobytes() != before[7:].tobytes()
    # an empty map
    g.load_map(np.zeros((0, 4), np.float32), np.zeros((0, 4), np.float32))
    g.process_frame(scans[1])
    with pytest.raises(pkg.VloamError, match="empty"):
        g.relocalize([0, 0, 0, 1], [0, 0, 0])
    # a load drops the query (its stacks were mapped in the old map)
    g.load_map(*_prior(pkg, "C3"))
    with pytest.raises(pkg.VloamError, match="no mapped sweep"):
        g.relocalize([0, 0, 0, 1], [0, 0, 0])
    g.close()
