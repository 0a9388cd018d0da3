"""Measurements of the prior-map calls on one GPU -> profiles/r3_prior_map.json (or the path given as argv[1]).

- load time of the C3-sized (~1.3M points) and C4-sized (~2.0M points) planted clouds: device time of the load's kernels (CUDA
  events around them, vloam_b200_profile_kernel) and wall time from pinned and from pageable host memory, against the debug blob
  import (`lm.cornerMap` / `lm.surfMap`) that tests use;
- scans/s on C3, device-resident sweeps, two sweeps ahead: mapping against frozen localization, runs alternated, 200 sweeps each;
- kernel launches and allocations of a plain replay that never calls the new functions.
The card's name and power limit are recorded with the numbers."""
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")]


def main():
    import torch
    import bench
    pkg = importlib.import_module("vloam-noted_b200")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    world = pkg.synth.World(1234, 1, 190.0)
    out = {"gpu": smi, "load": {}}
    for size, (pc, ps) in {"C3": (0.3, 0.7), "C4": (0.25, 0.6)}.items():
        corner, surf = world.plant(0, pc, seed=99), world.plant(1, ps, seed=98)
        pin = [torch.from_numpy(a).pin_memory() for a in (corner, surf)]
        g = pkg.Context(**bench.KW)
        rec = {"points": [len(corner), len(surf)]}
        g.load_map(corner, surf)  # warm-up (first-use reservations)
        for how in ("pageable", "pinned"):
            ts = []
            for _ in range(5):
                g.synchronize()
                t0 = time.perf_counter()
                if how == "pinned":
                    g.load_map(pin[0].numpy(), pin[1].numpy())
                else:
                    g.load_map(corner, surf)
                g.synchronize()
                ts.append((time.perf_counter() - t0) * 1e3)
            rec["wall_ms_" + how] = [round(min(ts), 3), round(float(np.median(ts)), 3)]
        L = g.L
        L.vloam_b200_profile_kernel(g.h, b"*")
        g.load_map(corner, surf)
        import ctypes
        cb = ctypes.create_string_buffer(1 << 16)
        L.vloam_b200_profile_table(g.h, cb, 1 << 16)
        table = [l.split() for l in cb.value.decode().splitlines()]
        rec["device_ms"] = round(sum(float(t[2]) for t in table), 4)
        rec["kernels"] = {t[0]: [int(t[1]), round(float(t[2]), 4)] for t in table}
        L.vloam_b200_profile_kernel(g.h, None)
        cblob, sblob = g.get("lm.cornerMap"), g.get("lm.surfMap")
        ts = []
        for _ in range(3):
            g.synchronize()
            t0 = time.perf_counter()
            g.set("lm.cornerMap", cblob); g.set("lm.surfMap", sblob)
            g.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        rec["debug_import_wall_ms"] = round(min(ts), 3)
        g.close()
        out["load"][size] = rec
    # scans/s: mapping vs frozen localization, alternated
    n = 200
    traj = pkg.synth.trajectory(n + 3, seed=91, step=1.0)
    traj[:, 0] += 40.0
    scans = bench._gen_scans(pkg, world, traj, [7000 + k for k in range(n + 3)])
    dev = [torch.from_numpy(s).cuda() for s in scans]
    corner, surf = world.plant(0, 0.3, seed=99), world.plant(1, 0.7, seed=98)
    q, t = pkg.synth.pose_to_qt(traj[0])
    rates = {"mapping": [], "frozen": []}
    for rep in range(3):
        for mode in ("mapping", "frozen"):
            g = pkg.Context(**bench.KW)
            g.load_map(corner, surf)
            g.set_map_pose(q, t)
            g.set_map_update(mode == "mapping")
            for k in range(3):  # warm-up sweeps are not timed
                bench.prefetch_ahead(g, dev, k, True)
                g.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, None)
            g.synchronize()
            pose = np.zeros(14)
            t0 = time.perf_counter()
            for k in range(3, n):
                bench.prefetch_ahead(g, dev, k, True)
                g.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, pose.ctypes.data)
            g.synchronize()
            rates[mode].append((n - 3) / (time.perf_counter() - t0))
            g.close()
    out["scans_per_s_C3_two_ahead_device"] = {m: {"runs": [round(r, 1) for r in v], "median": round(float(np.median(v)), 1),
                                                  "spread": round(max(v) - min(v), 1)} for m, v in rates.items()}
    # the default path: launches and allocations of a plain replay (no new call)
    _, _, cb, sb = bench.make_sequence(pkg, 0, 1)
    g = pkg.Context(**bench.KW)
    g.set("lm.cornerMap", cb); g.set("lm.surfMap", sb)
    l0, a0 = g.kernel_launches, int(g.get("alloc.count")[0])
    for s in scans[:30]:
        g.process_frame(s)
    out["plain_replay_30_sweeps"] = {"launches": g.kernel_launches - l0, "alloc_count": int(g.get("alloc.count")[0]) - a0}
    g.close()
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_prior_map.json")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
