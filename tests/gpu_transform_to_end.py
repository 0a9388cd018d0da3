"""Cost and accuracy of VLOAM_FLAG_TRANSFORM_TO_END on one GPU (not collected by pytest).  One command;
`python tests/gpu_transform_to_end.py OUT.json [PARENT_TREE]` also writes the results as JSON:

  * scans/s under the flag settings {0, D, D + TO_END}, runs alternated, on moving HDL-64 sweeps:
      C1  street world, one sweep at a time (process_frame, host buffer, nothing registered ahead),
      C3  the planted ~1M-point map of bench.py's C3 world, two sweeps registered ahead (device buffers);
  * device time of lo_transform_to_end per sweep (vloam_b200_profile_kernel: CUDA events around each launch);
  * the segment-drift table of tests/test_transform_to_end_oracle.py, produced by the device;
  * with PARENT_TREE (a checkout of the parent commit, built): bench.py there and here, alternated, and alloc.count of a
    flag-off replay in both trees."""
import ctypes, importlib, json, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
pkg = importlib.import_module("vloam-noted_b200")
import bench
import torch
import transform_to_end_ref as ref

SETTINGS = (("0", 0, False), ("D", 1, False), ("D+TO_END", 1, True))
N, WARM = int(os.environ.get("SWEEPS", "90")), 10


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q.splitlines()[0] if q else torch.cuda.get_device_name(0)


street = pkg.synth.World(1234, 0, 160.0)
c1_scans, _ = ref.moving_drive(street, pkg.synth.HDL64, N + 1, seed=61)
c3_world = pkg.synth.World(1234, 1, 190.0)
c3_scans, _ = ref.moving_drive(c3_world, pkg.synth.HDL64, N + 1, seed=62)
_, _, cb, sb = bench.make_sequence(pkg, 0, 1)
c3_dev = [torch.from_numpy(s).cuda() for s in c3_scans]
c1_host = [np.ascontiguousarray(s) for s in c1_scans]


def replay(config, d, te):
    g = pkg.Context(distortion=d, transform_to_end=te, **bench.KW)
    if config == "C3":
        g.set("lm.cornerMap", cb); g.set("lm.surfMap", sb)
    pose = np.zeros(14)
    for k in range(N):
        if k == WARM:
            g.synchronize(); t0 = time.perf_counter()
        if config == "C3":
            bench.prefetch_ahead(g, c3_dev, k, True)
            g.process_frame_device(c3_dev[k].data_ptr(), c3_dev[k].shape[0], 4, pose.ctypes.data)
        else:
            g.process_frame_ptr(c1_host[k].ctypes.data, len(c1_host[k]), 4, pose.ctypes.data)
    g.synchronize()
    sps = (N - WARM) / (time.perf_counter() - t0)
    g.close()
    return sps


def kernel_time(scans, n=30):
    g = pkg.Context(distortion=1, transform_to_end=True, **bench.KW)
    pose = np.zeros(14)
    for k in range(5):
        g.process_frame(scans[k])
    g._chk(g.L.vloam_b200_profile_kernel(g.h, b"lo_transform_to_end"))
    pts = 0
    for k in range(5, 5 + n):
        g.process_frame_ptr(c1_host[k].ctypes.data, len(c1_host[k]), 4, pose.ctypes.data)
        pts += len(g.get_cloud(pkg.CLOUD_LESS_SHARP)) + len(g.get_cloud(pkg.CLOUD_LESS_FLAT))
    launches, ms, by = ctypes.c_int(), ctypes.c_double(), ctypes.c_double()
    g._chk(g.L.vloam_b200_profile_result(g.h, ctypes.byref(launches), ctypes.byref(ms), ctypes.byref(by)))
    g.close()
    return {"launches": launches.value, "sweeps": n, "device_us_per_sweep": ms.value * 1e3 / n, "points_per_sweep": pts / n}


def drift_table(n=30, lengths=(4.0, 8.0, 12.0)):
    scans, traj = ref.moving_drive(street, pkg.synth.VLP16, n)
    gt = [pkg.synth.pose_to_qt(traj[k + 1]) for k in range(n)]
    kw = dict(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4)
    out = {}
    for name, d, te in SETTINGS:
        g = pkg.Context(distortion=d, transform_to_end=te, **kw)
        lo, lm = [], []
        for s in scans:
            p = g.process_frame(s)
            lo.append((p[0:4], p[4:7])); lm.append((p[7:11], p[11:14]))
        g.close()
        out[name] = {"mapped": ref.segment_drift(lm, gt, lengths), "odometry": ref.segment_drift(lo, gt, lengths)}
    return out


def alloc_count(tree):
    code = ("import importlib, sys, numpy as np; sys.path.insert(0, %r); p = importlib.import_module('vloam-noted_b200'); "
            "w = p.synth.World(1234, 0, 160.0); t = p.synth.trajectory(9); g = p.Context(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8); "
            "[g.process_frame(w.scan(1, t[k], 1000 + k)) for k in range(9)]; g.synchronize(); print(int(g.get('alloc.count')[0]))" % tree)
    return int(subprocess.run([sys.executable, "-c", code], cwd=tree, capture_output=True, text=True, check=True).stdout.split()[-1])


def bench_line(tree):
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "20", "--warmup", "5", "--no-cpu-baseline", "--no-extras", "--no-c5"],
                       cwd=tree, capture_output=True, text=True, check=True)
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    return {k: line[k] for k in line if isinstance(line[k], (int, float))}


res = {"card": card(), "sweeps": N, "warmup": WARM, "scans_per_s": {"C1": {}, "C3": {}}}
for rep in range(2):
    for config in ("C1", "C3"):
        for name, d, te in (SETTINGS if rep == 0 else SETTINGS[::-1]):
            res["scans_per_s"][config].setdefault(name, []).append(replay(config, d, te))
print(json.dumps(res["scans_per_s"]), flush=True)
res["lo_transform_to_end"] = kernel_time(c1_scans)
print(json.dumps(res["lo_transform_to_end"]), flush=True)
res["drift"] = drift_table()
print(json.dumps(res["drift"]), flush=True)
if len(sys.argv) > 2:
    parent = os.path.abspath(sys.argv[2])
    res["alloc_count_flag_off"] = {"parent": alloc_count(parent), "branch": alloc_count(ROOT)}
    runs = []
    for tree in (parent, ROOT, parent, ROOT):
        runs.append({"tree": "parent" if tree == parent else "branch", **bench_line(tree)})
        print(json.dumps(runs[-1]), flush=True)
    res["bench"] = runs
if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        json.dump(res, f, indent=1)
print("card:", res["card"])
