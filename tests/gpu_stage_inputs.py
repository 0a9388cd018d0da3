"""Measurement of the stage-input calls (vloam_b200_laser_mapping_input / vloam_b200_laser_odometry_input) on the GPU.

    python tests/gpu_stage_inputs.py [--parent DIR] [--out profiles/r4_stage_inputs.json]

Reports, with the card's name and power limit read in the same run:
  - per-sweep wall time on C3 (HDL-64 sweeps against the planted 1M-point map, one sweep at a time, host clock around each call
    that ends at sync point S2): the plain path (process_frame), and the mapping stage alone fed A's outputs through
    laser_mapping_input from pageable host memory, pinned host memory and device memory;
  - the device time of the pack kernel (vl_pack_xyzi) for the (8, 4) layout, and the bytes the mapping input uploads per sweep;
  - the plain path's kernel launches and device allocations for one seeded drive, in this tree and (--parent) in another build
    of the library, which must be equal: the plain path pays nothing for the new calls;
  - bench.py at --parent and in this tree, alternated in one call.
Nothing is written in the tree except --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def plain_counts(tree):
    """Kernel launches and device allocations of a seeded 12-sweep VLP-16 drive through process_frame, in the library of `tree`."""
    code = r"""
import importlib, json, sys
sys.path.insert(0, %r)
pkg = importlib.import_module("vloam-noted_b200")
s = pkg.synth
w = s.World(1234, 0, 160.0)
tr = s.trajectory(12, seed=91, step=1.5)
g = pkg.Context(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4)
for k in range(12):
    g.process_frame(w.scan(s.VLP16, tr[k], 1000 + k))
g.synchronize()
print(json.dumps({"kernel_launches": g.kernel_launches, "alloc_count": int(g.get("alloc.count")[0])}))
""" % tree
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tree)
    if r.returncode != 0:
        raise RuntimeError(r.stderr[-2000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def bench_line(tree, args):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.steps), "--warmup", str(args.warmup), "--no-cpu-baseline", "--no-extras"]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=tree)
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError(r.stderr[-2000:])


def c3_timings(args):
    import torch
    sys.path.insert(0, ROOT)
    import importlib
    import bench
    pkg = importlib.import_module("vloam-noted_b200")
    n, warm = args.sweeps, 5
    scans, _, cb, sb = bench.make_sequence(pkg, 0, n)
    a = pkg.Context(**bench.KW)
    a.set("lm.cornerMap", cb); a.set("lm.surfMap", sb)
    plain, inputs = [], []
    for k in range(n):
        t0 = time.perf_counter()
        pose = a.process_frame(scans[k])
        plain.append(time.perf_counter() - t0)
        inputs.append((a.get_cloud(5), a.get_cloud(6), a.get_cloud(7), pose[0:4].copy(), pose[4:7].copy()))
    a.close()
    out = {"plain_process_frame_ms": 1e3 * float(np.median(plain[warm:]))}
    for mode in ("pageable", "pinned", "device"):
        b = pkg.Context(**bench.KW)
        b.set("lm.cornerMap", cb); b.set("lm.surfMap", sb)
        feed = []
        for c, s, f, q, t in inputs:
            arrs = [np.ascontiguousarray(x) for x in (c, s, f)]
            if mode == "pinned":
                arrs = [torch.from_numpy(x).pin_memory().numpy() for x in arrs]
            elif mode == "device":
                arrs = [torch.from_numpy(x).cuda() for x in arrs]
            feed.append((arrs, q, t))
        torch.cuda.synchronize()
        times = []
        for arrs, q, t in feed:
            t0 = time.perf_counter()
            b.begin_frame()
            b.laser_mapping_input(arrs[0], arrs[1], arrs[2], q, t, False)
            b.laser_mapping()
            times.append(time.perf_counter() - t0)
        out["fed_mapping_%s_ms" % mode] = 1e3 * float(np.median(times[warm:]))
        b.close()
    out["upload_bytes_per_sweep_packed"] = float(np.mean([16.0 * (len(c) + len(s) + len(f)) for c, s, f, _, _ in inputs]))
    out["points_per_sweep"] = [float(np.mean([len(x[i]) for x in inputs])) for i in range(3)]
    # pack kernel: (8, 4) layout from device memory (upload excluded), timed by the library's per-kernel events
    b = pkg.Context(**bench.KW)
    b.set("lm.cornerMap", cb); b.set("lm.surfMap", sb)
    pad = []
    for c, s, f, q, t in inputs:
        d = []
        for x in (c, s, f):
            y = np.full((len(x), 8), np.nan, np.float32); y[:, :3] = x[:, :3]; y[:, 4] = x[:, 3]
            d.append(torch.from_numpy(y).cuda())
        pad.append((d, q, t))
    torch.cuda.synchronize()
    b.L.vloam_b200_profile_kernel(b.h, b"vl_pack_xyzi")
    for d, q, t in pad:
        b.begin_frame()
        b.laser_mapping_input(d[0], d[1], d[2], q, t, False, w_offset=4)
        b.laser_mapping()
    import ctypes
    nl, ms, by = ctypes.c_int(0), ctypes.c_double(0), ctypes.c_double(0)
    b.L.vloam_b200_profile_result(b.h, ctypes.byref(nl), ctypes.byref(ms), ctypes.byref(by))
    out["pack_kernel"] = {"launches": nl.value, "mean_us": 1e3 * ms.value / max(nl.value, 1), "bytes_per_launch": by.value / max(nl.value, 1),
                          "GBps": by.value / max(ms.value * 1e-3, 1e-12) / 1e9}
    out["upload_bytes_per_sweep_8x4"] = float(np.mean([32.0 * (len(c) + len(s) + len(f)) for c, s, f, _, _ in inputs]))
    b.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", help="another checkout with its library built (the commit before this change)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_stage_inputs.json"))
    ap.add_argument("--sweeps", type=int, default=30)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--bench-rounds", type=int, default=2)
    args = ap.parse_args()
    res = {"card": card()}
    res["c3"] = c3_timings(args)
    print(json.dumps(res["c3"]), flush=True)
    res["plain_counts"] = {"this": plain_counts(ROOT)}
    if args.parent:
        res["plain_counts"]["parent"] = plain_counts(os.path.abspath(args.parent))
        runs = []
        for r in range(args.bench_rounds):
            for name, tree in (("parent", os.path.abspath(args.parent)), ("this", ROOT)):
                line = bench_line(tree, args)
                runs.append({"tree": name, "round": r, "value": line.get("value"), "unit": line.get("unit")})
                print(json.dumps(runs[-1]), flush=True)
        res["bench"] = runs
    res["card_after"] = card()
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
