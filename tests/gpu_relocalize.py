"""Measure vloam_b200_relocalize on the GPU: wall and device time per call at +-20, +-50 and +-100 m over 360 degrees (default
resolution 1 m, yaw step r / max_range), nodes evaluated per level against the exhaustive candidate count, and the occupancy build
time, on the C3 prior 40 m from the map origin.  Prints the card and its power limit read in the same run, one JSON line per search
width, and with --out PATH writes all of it to PATH as JSON."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--out", help="write the card and the rows as JSON here")
    args = ap.parse_args()
    import importlib
    pkg = importlib.import_module("vloam-noted_b200")
    from test_gpu_prior_map import _ctx, _drive, _guess, _prior
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip()
    print("card:", card)
    scans, traj = _drive(pkg, 4)
    corner, surf = _prior(pkg, "C3")
    g = _ctx(pkg)
    g.load_map(corner, surf)
    g.set_map_update(False)
    g.process_frame(scans[0])
    q, t = _guess(pkg, traj[0], (21.2, -21.2), 150.0)
    rows = []
    for half in (20.0, 50.0, 100.0):
        g.relocalize(q, t, half_xy=half, apply=False)  # warm-up (module load, first reservations)
        wall, dev, occ = [], [], []
        for _ in range(5):
            t0 = time.perf_counter()
            res = g.relocalize(q, t, half_xy=half, apply=False)
            wall.append((time.perf_counter() - t0) * 1e3)
            ms = g.get("rl.ms")
            dev.append(float(ms[0])); occ.append(float(ms[1]))
        lv = g.get("rl.levels")
        front = lv[:16].tolist()
        row = dict(half_xy=half, wall_ms_median=float(np.median(wall)), device_ms_median=float(np.median(dev)),
                   occupancy_ms_median=float(np.median(occ)), candidates=int(res.candidates), nodes=int(res.nodes),
                   nodes_best=int(lv[32]), nodes_runner=int(lv[33]), frontier_per_level_best=front,
                   frontier_per_level_runner=lv[16:32].tolist(), score=int(res.score), runner_score=int(res.runner_score),
                   n_points=int(res.n_points), t=list(res.t))
        rows.append(row)
        print(json.dumps(row))
    g.close()
    out = dict(card=card, rows=rows)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
