"""LaserMapping::publish's global map (LM.cpp:884-899) restated from the per-cube map blobs ("lm.cornerMap" / "lm.surfMap":
int32 counts[4851], then the points of every cube in cube order), for tests of vloam_b200_publish_map / get_map."""
import numpy as np

CUBE_NUM = 4851


def split_blob(blob):
    """`lm.*Map` blob -> (counts int32[4851], points float32[n, 4])."""
    counts = np.frombuffer(blob[:CUBE_NUM * 4], np.int32)
    return counts, np.frombuffer(blob[CUBE_NUM * 4:], np.float32).reshape(-1, 4)


def laser_cloud_map(corner_blob, surf_blob):
    """LM.cpp:884-899 literally: laserCloudMap.clear(); for (i = 0; i < 4851; i++) { laserCloudMap += *cornerArray[i];
    laserCloudMap += *surfArray[i]; }  (parity of the loop itself unpinned: the reference is not in this checkout)."""
    cc, cp = split_blob(corner_blob)
    sc, sp = split_blob(surf_blob)
    parts, co, so = [], 0, 0
    for i in range(CUBE_NUM):
        parts.append(cp[co:co + cc[i]]); co += int(cc[i])
        parts.append(sp[so:so + sc[i]]); so += int(sc[i])
    return np.concatenate(parts) if parts else np.zeros((0, 4), np.float32)


def laser_cloud_map_of(x):
    """The global map of an oracle or a Context as of its last mapped frame (through its map export)."""
    return laser_cloud_map(x.get("lm.cornerMap"), x.get("lm.surfMap"))
