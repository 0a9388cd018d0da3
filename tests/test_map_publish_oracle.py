"""The restatement of LaserMapping::publish's global map (tests/map_publish_ref.py, LM.cpp:884-899) pinned on the CPU oracle's
own map state: after a few street sweeps that move the sub-map window, it must equal an independent vectorised interleave of the
oracle's `lm.cornerMap` / `lm.surfMap` blobs (corner cube i, then surf cube i, for i in table order)."""
import numpy as np

from map_publish_ref import CUBE_NUM, laser_cloud_map, split_blob


def _interleave(corner_blob, surf_blob):
    cc, cp = split_blob(corner_blob)
    sc, sp = split_blob(surf_blob)
    seg = np.concatenate([2 * np.repeat(np.arange(CUBE_NUM), cc), 2 * np.repeat(np.arange(CUBE_NUM), sc) + 1])
    order = np.argsort(seg, kind="stable")  # (cube, kind), keeping each cube's own point order
    return np.concatenate([cp, sp])[order]


def test_laser_cloud_map_restatement_matches_interleave(op, synth, street):
    o = op.Oracle(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4)
    traj = synth.trajectory(9, seed=5, step=4.0)
    centres, checked = set(), 0
    for k in range(9):
        o.process(street.scan(0, traj[k], 3000 + k))
        centres.add(int(o.get("lm.validInd")[0]))
        if k % 2 == 0 or k == 8:
            cb, sb = o.get("lm.cornerMap"), o.get("lm.surfMap")
            ref = laser_cloud_map(cb, sb)
            assert len(ref) == split_blob(cb)[0].sum() + split_blob(sb)[0].sum()
            assert ref.tobytes() == _interleave(cb, sb).tobytes(), "frame %d" % k
            checked += 1
    assert len(centres) > 1, "the sub-map window never moved"
    assert checked == 5 and len(ref) > 0
