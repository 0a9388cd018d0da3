"""Stage inputs from the caller: vloam_b200_laser_odometry_input[_device] and vloam_b200_laser_mapping_input[_device]
(LaserOdometry::input LO.cpp:137-148, LaserMapping::input LM.cpp:178-209 deep-copy what they are handed).

A context fed another context's stage outputs through these calls must compute exactly what that context computed; foreign
inputs (edited clouds, another odometry pose, permuted or subsampled features) are checked against the CPU oracle driven stage by
stage on the same inputs; and a context that never makes these calls does exactly what it did before."""
import ctypes
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from conftest import assert_bits_equal  # noqa: E402
from test_gpu_parity import pose_close  # noqa: E402
from transform_to_end_ref import associate_to_map  # noqa: E402

pytestmark = pytest.mark.gpu

VLP = dict(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4)
CORNER_LAST, SURF_LAST, FULL_RES = 5, 6, 7
LAYOUTS = [(4, 3), (8, 4)]  # packed xyzi; pcl::PointXYZI as PCL lays it out (x y z pad | intensity pad pad pad)
SR_CLOUDS = ("sr.laserCloud", "sr.sharp", "sr.lessSharp", "sr.flat", "sr.lessFlat")


def as_layout(cloud, layout):
    """float32[n, 4] xyzi -> float32[n, stride] with the intensity at w_offset and every other float NaN."""
    stride, w = layout
    if layout == (4, 3):
        return np.ascontiguousarray(cloud, np.float32)
    out = np.full((len(cloud), stride), np.nan, np.float32)
    out[:, :3] = cloud[:, :3]
    out[:, w] = cloud[:, 3]
    return out


def as_input(clouds, layout, device):
    arrs = [as_layout(c, layout) for c in clouds]
    if device:
        import torch
        arrs = [torch.from_numpy(a).cuda() for a in arrs]
    return arrs


def skip_of(k, m):
    """LO.cpp:668-678: after the odometry of sweep k (0-based) frameCount is k + 1."""
    return ((k + 1) % m) != 0


def street_drive(synth, street, n, step=1.5):
    traj = synth.trajectory(n, seed=91, step=step)
    return [street.scan(synth.VLP16, traj[k], 1000 + k) for k in range(n)], traj


def run_own(pkg, scans, kw, maps=None, publish_at=()):
    """Context A: the plain per-frame call; records what LaserOdometry::output hands to LaserMapping and every mapping output."""
    g = pkg.Context(**kw)
    if maps:
        g.set("lm.cornerMap", maps[0]); g.set("lm.surfMap", maps[1])
    out = dict(inputs=[], poses=[], reg=[], pubs={}, windows=set())
    for k, s in enumerate(scans):
        pose = g.process_frame(s)
        out["inputs"].append((g.get_cloud(CORNER_LAST), g.get_cloud(SURF_LAST), g.get_cloud(FULL_RES), pose[0:4].copy(), pose[4:7].copy()))
        out["poses"].append(pose[7:14].copy())
        out["reg"].append(g.register_full_cloud())
        valid = g.get("lm.validInd")
        if len(valid):  # (empty until the first mapped frame)
            out["windows"].add(int(valid[0]))
        if k in publish_at:
            g.publish_map(); out["pubs"][k] = g.get_map()
    out["maps"] = (g.get("lm.cornerMap"), g.get("lm.surfMap"))
    out["paths"] = g.get("lm.paths")
    g.close()
    return out


def run_fed(pkg, a, kw, m, layout, device, maps=None, publish_at=()):
    """Context B: begin_frame + laser_mapping_input(A's outputs) + laser_mapping, nothing else."""
    g = pkg.Context(**kw)
    if maps:
        g.set("lm.cornerMap", maps[0]); g.set("lm.surfMap", maps[1])
    out = dict(poses=[], reg=[], pubs={})
    for k, (corner, surf, full, q, t) in enumerate(a["inputs"]):
        g.begin_frame()
        c, s, f = as_input((corner, surf, full), layout, device)
        g.laser_mapping_input(c, s, f, q, t, skip_of(k, m), w_offset=layout[1])
        q_m, t_m = g.laser_mapping()
        out["poses"].append(np.concatenate([q_m, t_m]))
        out["reg"].append(g.register_full_cloud())
        if k in publish_at:
            g.publish_map(); out["pubs"][k] = g.get_map()
    out["maps"] = (g.get("lm.cornerMap"), g.get("lm.surfMap"))
    out["paths"] = g.get("lm.paths")
    g.close()
    return out


def assert_same_mapping(a, b):
    for k, (pa, pb) in enumerate(zip(a["poses"], b["poses"])):
        assert pa.tobytes() == pb.tobytes(), ("mapped pose", k, pa, pb)
    for k, (ra, rb) in enumerate(zip(a["reg"], b["reg"])):
        assert_bits_equal(ra, rb, "register_full_cloud %d" % k)
    assert sorted(a["pubs"]) == sorted(b["pubs"])
    for k in a["pubs"]:
        assert_bits_equal(a["pubs"][k], b["pubs"][k], "get_map after sweep %d" % k)
    assert a["maps"][0] == b["maps"][0], "lm.cornerMap"
    assert a["maps"][1] == b["maps"][1], "lm.surfMap"
    assert (a["paths"] == b["paths"]).all(), (a["paths"], b["paths"])


# ---- 1. mapping round trip ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("to_end", [False, True])
@pytest.mark.parametrize("skip", [1, 2])
@pytest.mark.parametrize("device", [False, True])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_mapping_round_trip_street(pkg, synth, street, to_end, skip, device, layout):
    """A VLP-16 street drive across a window move: B, fed only A's CORNER_LAST / SURF_LAST / FULL_RES, odometry pose and skip,
    maps byte for byte what A maps."""
    n = 36
    scans, _ = street_drive(synth, street, n)
    kw = dict(VLP, mapping_skip_frame=skip, distortion=1 if to_end else 0, transform_to_end=to_end)
    pubs = (11, 23, n - 1)
    a = run_own(pkg, scans, kw, publish_at=pubs)
    assert len(a["windows"]) >= 2, "the drive never moved the window"
    b = run_fed(pkg, a, kw, skip, layout, device, publish_at=pubs)
    assert_same_mapping(a, b)


@pytest.mark.parametrize("device,layout", [(False, (4, 3)), (True, (8, 4))])
def test_mapping_round_trip_c3(pkg, device, layout):
    """A few C3 sweeps (HDL-64 against the planted 1M-point map): same bar."""
    import bench
    n = 5
    scans, _, cb, sb = bench.make_sequence(pkg, 0, n)
    a = run_own(pkg, scans, bench.KW, maps=(cb, sb), publish_at=(2, n - 1))
    b = run_fed(pkg, a, bench.KW, 1, layout, device, maps=(cb, sb), publish_at=(2, n - 1))
    assert_same_mapping(a, b)


# ---- 2. mixed mode ---------------------------------------------------------------------------------------------------------
def _mixed(pkg, scans, dev, ahead, feed_every):
    import bench
    g = pkg.Context(**VLP)
    lo, lm = [], []
    for k in range(len(scans)):
        g.begin_frame()
        if ahead:
            bench.prefetch_ahead(g, dev, k, True)
            g.scan_registration_device(dev[k].data_ptr(), dev[k].shape[0], dev[k].shape[1])
        else:
            g.scan_registration(scans[k])
        r = g.laser_odometry()
        lo.append(np.concatenate([r["q_w_curr"], r["t_w_curr"]]))
        if feed_every and k % feed_every == feed_every - 1:
            g.laser_mapping_input(g.get_cloud(CORNER_LAST), g.get_cloud(SURF_LAST), g.get_cloud(FULL_RES), r["q_w_curr"], r["t_w_curr"],
                                  r["skip_frame"])
        q, t = g.laser_mapping()
        lm.append(np.concatenate([q, t]))
    out = dict(lo=np.array(lo), lm=np.array(lm), maps=(g.get("lm.cornerMap"), g.get("lm.surfMap")), paths=g.get("lm.paths"))
    g.close()
    return out


def test_mixed_mode_equals_plain(pkg, synth, street):
    """Own scan registration and odometry, and every third frame a mapping input equal to the context's own output: the stacks this
    frame's odometry queued are superseded by the same clouds filtered again, and the odometry state is untouched, so odometry
    poses, mapped poses, maps and map paths equal the plain run -- one sweep at a time and with two sweeps registered ahead."""
    import torch
    scans, _ = street_drive(synth, street, 24)
    dev = [torch.from_numpy(np.ascontiguousarray(s[:, :4])).cuda() for s in scans]
    plain = _mixed(pkg, scans, dev, False, 0)
    for ahead in (False, True):
        for feed in (0, 3):
            r = _mixed(pkg, scans, dev, ahead, feed)
            assert r["lo"].tobytes() == plain["lo"].tobytes(), ("odometry", ahead, feed)
            assert r["lm"].tobytes() == plain["lm"].tobytes(), ("mapping", ahead, feed)
            assert r["maps"] == plain["maps"], ("maps", ahead, feed)
            assert (r["paths"] == plain["paths"]).all(), ("paths", ahead, feed, r["paths"], plain["paths"])


# ---- 3. foreign mapping inputs against the oracle ---------------------------------------------------------------------------
def _perturbed(synth, p, rng):
    q, t = synth.pose_to_qt(p)
    q = q + rng.normal(0.0, 2e-3, 4)
    return q / np.linalg.norm(q), t + rng.normal(0.0, 0.05, 3)


@pytest.mark.parametrize("variant", ["box_removed", "foreign_pose"])
def test_foreign_mapping_inputs_match_oracle(pkg, op, synth, street, variant):
    """(box_removed) the oracle's own clouds with every point inside a box around the sensor removed; (foreign_pose) the perturbed
    synthetic truth as q_wodom / t_wodom.  Teacher-forced, capture on: stacks, sub-map, kNN, stored maps and the registered
    full-resolution cloud bit-exact, poses within the parity tolerance."""
    frames = 5
    scans, traj = street_drive(synth, street, frames, step=1.0)
    rng = np.random.RandomState(5)
    src = op.Oracle(**VLP)          # produces the inputs
    o = op.Oracle(**VLP)            # the mapping stage on them
    g = pkg.Context(**VLP)
    g.set_capture(True)
    for k in range(frames):
        src.process(scans[k])
        corner, surf, full = src.get("lo.cornerLast"), src.get("lo.surfLast"), src.get("sr.laserCloud")
        lo = src.get("lo.pose")
        q, t = lo[0:4], lo[4:7]
        if variant == "box_removed":
            keep = lambda c: c[~((np.abs(c[:, 0]) < 8.0) & (np.abs(c[:, 1]) < 4.0))]
            corner, surf, full = keep(corner), keep(surf), keep(full)
        else:
            q, t = _perturbed(synth, traj[k], rng)
        if k > 0:
            g.set("lm.state", o.get("lm.state")[:4]); g.set("lm.pose", o.get("lm.pose"))
            g.set("lm.cornerMap", o.get("lm.cornerMap")); g.set("lm.surfMap", o.get("lm.surfMap"))
        o.scan_registration(scans[k])  # (LaserMapping::reset, as LOM.cpp:65-71 calls it every frame)
        o.set_last(corner, surf)
        o.set("lo.pose", np.concatenate([q, t, [0, 0, 0, 1], [0, 0, 0]]))
        o.laser_mapping()
        g.begin_frame()
        g.laser_mapping_input(corner, surf, full, q, t, False)
        g.laser_mapping()
        for nm in ("lm.cornerStack", "lm.surfStack", "lm.cornerFromMap", "lm.surfFromMap", "lm.validInd"):
            assert_bits_equal(o.get(nm), g.get(nm), "%s frame %d" % (nm, k))
        so, sg = o.get("lm.state"), g.get("lm.state")
        assert (so == sg).all(), (so, sg)
        if so[4]:
            for p in (0, 1):
                for kind in ("c", "s"):
                    od = o.get("lm.knn.%sd2%d" % (kind, p))
                    acc = od[:, 4] < 1.0
                    assert_bits_equal(o.get("lm.knn.%sidx%d" % (kind, p))[acc], g.get("lm.knn.%sidx%d" % (kind, p))[acc], "knn idx")
                    assert_bits_equal(od[acc], g.get("lm.knn.%sd2%d" % (kind, p))[acc], "knn d2")
                    assert_bits_equal(o.get("lm.knn.%sok%d" % (kind, p)), g.get("lm.knn.%sok%d" % (kind, p)), "fit accept flags")
        lm_o, lm_g = o.get("lm.pose"), g.get("lm.pose")
        pose_close(lm_o[:7], lm_g[:7]); pose_close(lm_o[7:], lm_g[7:])
        assert o.get("lm.cornerMap") == g.get("lm.cornerMap"), "corner map bytes"
        assert o.get("lm.surfMap") == g.get("lm.surfMap"), "surf map bytes"
        assert_bits_equal(associate_to_map(full, lm_g[:7]), g.register_full_cloud(), "register_full_cloud")
    g.close()


# ---- 4. odometry round trip ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("device,layout", [(False, (4, 3)), (True, (8, 4)), (False, (8, 4))])
@pytest.mark.parametrize("to_end", [False, True])
def test_odometry_round_trip(pkg, synth, street, device, layout, to_end):
    """B gets A's five ScanRegistration clouds through laser_odometry_input: odometry pose, last clouds, association snapshots and
    the whole downstream chain equal A's."""
    n = 10
    scans, _ = street_drive(synth, street, n)
    kw = dict(VLP, distortion=1 if to_end else 0, transform_to_end=to_end)
    a, b = pkg.Context(**kw), pkg.Context(**kw)
    a.set_capture(True); b.set_capture(True)
    for k in range(n):
        a.begin_frame(); a.scan_registration(scans[k])
        clouds = [a.get(nm) for nm in SR_CLOUDS]
        b.begin_frame(); b.laser_odometry_input(as_input(clouds, layout, device), w_offset=layout[1])
        for nm, c in zip(SR_CLOUDS, clouds):
            assert_bits_equal(c, b.get(nm), nm)
        ra, rb = a.laser_odometry(), b.laser_odometry()
        for key in ("q_w_curr", "t_w_curr", "q_last_curr", "t_last_curr"):
            assert ra[key].tobytes() == rb[key].tobytes(), (k, key)
        assert ra["skip_frame"] == rb["skip_frame"]
        names = ["lo.cornerLast", "lo.surfLast"] + (["lo.assoc.corner0", "lo.assoc.surf0", "lo.assoc.corner1", "lo.assoc.surf1"] if k else [])
        for nm in names:
            assert_bits_equal(a.get(nm), b.get(nm), "%s frame %d" % (nm, k))
        qa, ta = a.laser_mapping(); qb, tb = b.laser_mapping()
        assert qa.tobytes() == qb.tobytes() and ta.tobytes() == tb.tobytes(), k
        assert_bits_equal(a.register_full_cloud(), b.register_full_cloud(), "register_full_cloud")
        assert_bits_equal(a.get_cloud(FULL_RES), b.get_cloud(FULL_RES), "FULL_RES")
    assert a.get("lm.cornerMap") == b.get("lm.cornerMap") and a.get("lm.surfMap") == b.get("lm.surfMap")
    a.close(); b.close()


# ---- 5. foreign odometry inputs against the oracle -----------------------------------------------------------------------
@pytest.fixture(scope="module")
def oracle_features(op, tmp_path_factory):
    """oracle_sr_features.cpp built against the oracle's header: sets the five clouds the oracle's next laser_odometry copies."""
    out = str(tmp_path_factory.mktemp("oracle_features") / "liboracle_features.so")
    here = os.path.dirname(os.path.abspath(__file__))
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-I", os.path.join(ROOT, "oracle"), "-o", out,
                    os.path.join(here, "oracle_sr_features.cpp")], check=True)
    lib = ctypes.CDLL(out)
    lib.vloam_oracle_set_sr_features.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]

    def set_features(o, clouds):
        n = np.array([len(c) for c in clouds], np.int32)
        pts = np.ascontiguousarray(np.concatenate([np.asarray(c, np.float32).reshape(-1, 4) for c in clouds]), np.float32)
        lib.vloam_oracle_set_sr_features(o.h, n.ctypes.data, pts.ctypes.data)
    return set_features


@pytest.mark.parametrize("variant", ["permuted", "subsampled"])
def test_foreign_odometry_inputs_match_oracle(pkg, op, synth, street, oracle_features, variant):
    """Scan-registration clouds permuted within each cloud (ring ids no longer monotone: the ballot association path) or
    subsampled, fed to the oracle's odometry and to the device's: association indices and last clouds bit-exact, poses within
    tolerance."""
    frames = 5
    scans, _ = street_drive(synth, street, frames, step=1.0)
    rng = np.random.RandomState(11)
    src, o, g = op.Oracle(**VLP), op.Oracle(**VLP), pkg.Context(**VLP)
    g.set_capture(True)
    for k in range(frames):
        src.scan_registration(scans[k])
        clouds = [src.get(nm) for nm in SR_CLOUDS]
        if variant == "permuted":
            clouds = [c[rng.permutation(len(c))] for c in clouds]
        else:
            clouds = [c[rng.rand(len(c)) < 0.7] for c in clouds]
        o.scan_registration(scans[k])  # (resets the stages as LOM.cpp:65-71 does; its clouds are replaced below)
        oracle_features(o, clouds)
        o.laser_odometry()
        g.begin_frame()
        g.laser_odometry_input(clouds)
        g.laser_odometry()
        names = ["lo.cornerLast", "lo.surfLast"] + (["lo.assoc.corner0", "lo.assoc.surf0", "lo.assoc.corner1", "lo.assoc.surf1"] if k else [])
        for nm in names:
            assert_bits_equal(o.get(nm), g.get(nm), "%s frame %d" % (nm, k))
        lo_o, lo_g = o.get("lo.pose"), g.get("lo.pose")
        pose_close(lo_o[:7], lo_g[:7]); pose_close(lo_o[7:], lo_g[7:])
        # teacher-force the odometry state so that the next frame's association starts from the oracle's pose
        g.set("lo.pose", lo_o)
    g.close()


# ---- 6. contract edges -----------------------------------------------------------------------------------------------------
def test_invalid_arguments(pkg):
    g = pkg.Context(**VLP)
    L, h = g.L, g.h
    pts = np.zeros((4, 8), np.float32)
    q, t = np.array([0, 0, 0, 1.0]), np.zeros(3)
    P = pts.ctypes.data

    def mi(corner=P, nc=4, surf=P, ns=4, full=P, nf=4, stride=8, w=4, qq=q.ctypes.data, tt=t.ctypes.data, skip=0):
        return L.vloam_b200_laser_mapping_input(h, corner, nc, surf, ns, full, nf, stride, w, qq, tt, skip)
    bad = [dict(nc=-1), dict(ns=-2), dict(nf=-1), dict(corner=None), dict(surf=None), dict(full=None), dict(stride=3, w=3),
           dict(w=2), dict(w=8), dict(stride=4, w=4), dict(qq=None), dict(tt=None), dict(skip=2), dict(skip=-1)]
    for kw in bad:
        assert mi(**kw) == -1, kw
        assert L.vloam_b200_last_error(h).decode(), kw
    assert mi(corner=None, nc=0) == 0  # NULL with n == 0 is an empty cloud
    ptrs = (ctypes.c_void_p * 5)(*([P] * 5))
    for n5, stride, w in ([[4, 4, 4, 4, -1], 8, 4], [[4, 4, 4, 4, 4], 3, 3], [[4, 4, 4, 4, 4], 8, 2], [[4, 4, 4, 4, 4], 8, 8]):
        assert L.vloam_b200_laser_odometry_input(h, ptrs, (ctypes.c_int * 5)(*n5), stride, w) == -1
        assert L.vloam_b200_last_error(h).decode()
    nulls = (ctypes.c_void_p * 5)(P, P, None, P, P)
    assert L.vloam_b200_laser_odometry_input(h, nulls, (ctypes.c_int * 5)(4, 4, 4, 4, 4), 4, 3) == -1
    assert L.vloam_b200_laser_odometry_input(None, ptrs, (ctypes.c_int * 5)(4, 4, 4, 4, 4), 4, 3) == -1
    assert L.vloam_b200_laser_mapping_input(None, P, 4, P, 4, P, 4, 4, 3, q.ctypes.data, t.ctypes.data, 0) == -1
    g.close()


def test_unconsumed_input_dropped_and_skipped_frame(pkg, synth, street):
    """A mapping input no laser_mapping call consumed is dropped by begin_frame: the next frame maps the context's own output.
    A mapping input on a skipped frame gives the high-frequency pose q_wmap_wodom * q_wodom (LM.cpp:197-201)."""
    scans, _ = street_drive(synth, street, 6)
    ref = pkg.Context(**VLP)
    g = pkg.Context(**VLP)
    junk = np.random.RandomState(3).rand(50, 4).astype(np.float32) * 20
    for k, s in enumerate(scans):
        pr = ref.process_frame(s)
        g.begin_frame(); g.scan_registration(s); r = g.laser_odometry()
        g.laser_mapping_input(junk, junk, junk, [0, 0, 0.3, 0.95], [5, 5, 5], False)  # never consumed ...
        g.begin_frame()  # ... dropped here
        q, t = g.laser_mapping()
        assert np.concatenate([q, t]).tobytes() == pr[7:14].tobytes(), k
    # skipped frame: the pose handed in is propagated through q_wmap_wodom / t_wmap_wodom
    lm = g.get("lm.pose")
    qo, to = np.array([0.01, -0.02, 0.1, 0.9945]), np.array([3.0, -1.0, 0.5])
    qo = qo / np.linalg.norm(qo)
    g.begin_frame()
    g.laser_mapping_input(junk, junk, junk, qo, to, True)
    q, t = g.laser_mapping()
    from transform_to_end_ref import qrot
    qm, tm = lm[7:11], lm[11:14]
    qx = np.array([qm[3] * qo[0] + qm[0] * qo[3] + qm[1] * qo[2] - qm[2] * qo[1],
                   qm[3] * qo[1] + qm[1] * qo[3] + qm[2] * qo[0] - qm[0] * qo[2],
                   qm[3] * qo[2] + qm[2] * qo[3] + qm[0] * qo[1] - qm[1] * qo[0],
                   qm[3] * qo[3] - qm[0] * qo[0] - qm[1] * qo[1] - qm[2] * qo[2]])
    assert np.abs(q - qx).max() < 1e-12
    assert np.abs(t - (qrot(qm, to[None, :])[0] + tm)).max() < 1e-9
    assert (g.get("lm.pose") == lm).all(), "a skipped frame leaves the mapped state alone"
    ref.close(); g.close()


def test_odometry_input_after_prefetch_drops_lookahead(pkg, synth, street):
    """Two sweeps registered ahead, then the next sweep arrives through laser_odometry_input instead (its own clouds): the look-ahead
    is dropped and every result equals the plain run."""
    import torch
    scans, _ = street_drive(synth, street, 8)
    dev = [torch.from_numpy(np.ascontiguousarray(s[:, :4])).cuda() for s in scans]
    ref = pkg.Context(**VLP)
    plain = [ref.process_frame(s).copy() for s in scans]
    cap = pkg.Context(**VLP)
    clouds = []
    for s in scans:
        cap.begin_frame(); cap.scan_registration(s)
        clouds.append([cap.get_cloud(w) for w in range(5)])
        cap.laser_odometry(); cap.laser_mapping()
    cap.close()
    g = pkg.Context(**VLP)
    import bench
    for k in range(len(scans)):
        g.begin_frame()
        if k % 3 == 2:
            bench.prefetch_ahead(g, dev, k, True)
            g.laser_odometry_input(clouds[k])
        else:
            bench.prefetch_ahead(g, dev, k, True)
            g.scan_registration_device(dev[k].data_ptr(), dev[k].shape[0], 4)
        r = g.laser_odometry()
        q, t = g.laser_mapping()
        got = np.concatenate([r["q_w_curr"], r["t_w_curr"], q, t])
        assert got.tobytes() == plain[k].tobytes(), k
    assert g.get("lm.cornerMap") == ref.get("lm.cornerMap")
    ref.close(); g.close()


def test_concurrent_contexts_fed_through_inputs(pkg, synth, street):
    """Eight contexts on eight threads, each fed another context's outputs through both input calls: equal to sequential runs."""
    scans, _ = street_drive(synth, street, 8)
    a = run_own(pkg, scans, VLP)
    sr = pkg.Context(**VLP)
    feats = []
    for s in scans:
        sr.begin_frame(); sr.scan_registration(s)
        feats.append([sr.get_cloud(w) for w in range(5)])
        sr.laser_odometry(); sr.laser_mapping()
    sr.close()

    def job(idx, out):
        g = pkg.Context(**VLP)
        res = []
        for k in range(len(scans)):
            g.begin_frame()
            if idx % 2:
                corner, surf, full, q, t = a["inputs"][k]
                g.laser_mapping_input(as_layout(corner, (8, 4)), as_layout(surf, (8, 4)), as_layout(full, (8, 4)), q, t, False, w_offset=4)
                res.append(np.concatenate(g.laser_mapping()))
            else:
                g.laser_odometry_input(feats[k])
                r = g.laser_odometry()
                res.append(np.concatenate([r["q_w_curr"], r["t_w_curr"], *g.laser_mapping()]))
        out[idx] = np.array(res)
        g.close()
    seq = {}
    for i in range(2):
        job(i, seq)
    par = {}
    threads = [threading.Thread(target=job, args=(i, par)) for i in range(8)]
    for th in threads: th.start()
    for th in threads: th.join()
    for i in range(8):
        assert par[i].tobytes() == seq[i % 2].tobytes(), i
    assert seq[1].tobytes() == np.array(a["poses"]).tobytes()


# ---- 7. no cost on the plain path ------------------------------------------------------------------------------------------
def test_reservations_only_on_first_input(pkg, synth, street):
    """The input buffers are reserved by the first input call, not at create: alloc.count grows at that call and not before."""
    scans, _ = street_drive(synth, street, 3)
    g = pkg.Context(**VLP)
    for s in scans[:2]:
        g.process_frame(s)
    corner, surf, full = g.get_cloud(CORNER_LAST), g.get_cloud(SURF_LAST), g.get_cloud(FULL_RES)
    pose = g.get("lo.pose")
    before = int(g.get("alloc.count")[0])
    g.begin_frame()
    g.laser_mapping_input(as_layout(corner, (8, 4)), as_layout(surf, (8, 4)), as_layout(full, (8, 4)), pose[0:4], pose[4:7], False, w_offset=4)
    after = int(g.get("alloc.count")[0])
    assert after > before, (before, after)
    g.laser_mapping()
    g.close()


# ---- 8. the adapter ----------------------------------------------------------------------------------------------------------
def test_adapter_stage_inputs(pkg, synth, street, tmp_path):
    """tests/cpp/stage_inputs_adapter.cpp, compiled against vloam_adapter.hpp: a stand-alone LaserMapping behind the pipeline's
    odometry, caller_clouds with an edit in the middle of the clouds against the C ABI, and a stand-alone ScanRegistration ->
    LaserOdometry pair on Engines of their own, all bit for bit."""
    from test_abi import build_cpp_program
    exe = build_cpp_program("stage_inputs_adapter", tmp_path)
    scans, _ = street_drive(synth, street, 8)
    files = []
    for k, s in enumerate(scans):
        f = str(tmp_path / ("scan%d.bin" % k))
        np.ascontiguousarray(s[:, :4], np.float32).tofile(f)
        files.append(f)
    r = subprocess.run([exe] + files, capture_output=True, text=True)
    assert r.returncode == 0 and "stage inputs ok" in r.stdout, (r.returncode, r.stdout[-3000:], r.stderr[-2000:])
