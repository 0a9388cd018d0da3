"""Cost of publishing the global map (vloam_b200_publish_map / get_map) on config C3 (planted ~1.03M-point map), in bench.py's
device-resident two-ahead replay mode (not collected by pytest).  One command; `python tests/gpu_map_publish.py OUT.json` also
writes the results as JSON:

  * sweeps/s and p50 / p99 / max ms per sweep, publishing every 20 mapped sweeps against not publishing (alternated twice);
  * the p99 of the sweeps that directly follow a publication;
  * device time of the assembly's kernels (CUDA events on the publication stream, vloam_b200_profile_table), grid and pool branch;
  * get_map's device -> host copy: time and bytes;
  * for contrast: one debug_get("lm.cornerMap") and the pool-path sweep it forces afterwards."""
import ctypes, importlib, json, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("vloam-noted_b200")
import bench
import torch

N, WARM, EVERY = int(os.environ.get("SWEEPS", "220")), 20, 20
scans, _, cb, sb = bench.make_sequence(pkg, 0, N + 1)
dev = [torch.from_numpy(s).cuda() for s in scans]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q.splitlines()[0] if q else torch.cuda.get_device_name(0)


def context():
    g = pkg.Context(**bench.KW)
    g.set("lm.cornerMap", cb); g.set("lm.surfMap", sb)
    return g


def replay(publish):
    g = context()
    pose = np.zeros(14)
    per, after = [], []
    published_before = False
    t0 = None
    for k in range(N):
        if k == WARM:
            g.synchronize(); t0 = time.perf_counter()
        bench.prefetch_ahead(g, dev, k, True)
        t1 = time.perf_counter()
        g.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, pose.ctypes.data)
        dt = (time.perf_counter() - t1) * 1e3
        if k >= WARM:
            per.append(dt)
            if published_before: after.append(dt)
        published_before = False
        if publish and (k + 1) % EVERY == 0:
            g.publish_map()
            published_before = True
    g.synchronize()
    total = time.perf_counter() - t0
    paths = g.get("lm.paths").tolist()
    g.close()
    per = np.array(per)
    return {"sweeps_per_s": (N - WARM) / total, "p50_ms": float(np.percentile(per, 50)), "p99_ms": float(np.percentile(per, 99)),
            "max_ms": float(per.max()), "after_publication_ms": [round(x, 4) for x in after], "paths": paths}


def assembly_and_copy():
    """Per-kernel device time of single publications (grid branch after in-place sweeps, pool branch right after a pool-path sweep)."""
    g = context()
    pose = np.zeros(14)
    out = {}
    for k in range(60):
        bench.prefetch_ahead(g, dev, k, True)
        g.process_frame_device(dev[k].data_ptr(), dev[k].shape[0], 4, pose.ctypes.data)
        if k in (30, 40, 50):
            g.synchronize()
            g._chk(g.L.vloam_b200_profile_kernel(g.h, b"*"))
            g.publish_map()
            n = g.get_map().shape[0]
            tb = ctypes.create_string_buffer(1 << 16)
            g._chk(g.L.vloam_b200_profile_table(g.h, tb, 1 << 16))
            g._chk(g.L.vloam_b200_profile_kernel(g.h, None))
            rows = [l.split() for l in tb.value.decode().splitlines() if l.strip()]
            ms = sum(float(r[2]) for r in rows)
            # get_map's copy alone: the assembly is complete, the size query returned
            host = np.empty((n, 4), np.float32)
            reps = []
            for _ in range(5):
                t1 = time.perf_counter()
                g._chk(g.L.vloam_b200_get_map(g.h, host.ctypes.data, n))
                reps.append((time.perf_counter() - t1) * 1e3)
            out["sweep%d" % k] = {"points": n, "assembly_device_ms": ms, "kernels": {r[0]: float(r[2]) for r in rows},
                                  "get_map_ms_median": float(np.median(reps)), "get_map_bytes": n * 16, "paths_so_far": g.get("lm.paths").tolist()}
    # contrast: the debug export, and the sweep after it (the export invalidates the grid: pool path)
    g.synchronize()
    t1 = time.perf_counter(); raw = g.get_raw("lm.cornerMap"); t_exp = (time.perf_counter() - t1) * 1e3
    p0 = g.get("lm.paths").tolist()
    bench.prefetch_ahead(g, dev, 60, True)
    t1 = time.perf_counter(); g.process_frame_device(dev[60].data_ptr(), dev[60].shape[0], 4, pose.ctypes.data); t_next = (time.perf_counter() - t1) * 1e3
    out["debug_export"] = {"lm.cornerMap_ms": t_exp, "bytes": len(raw), "next_sweep_ms": t_next, "paths_before_after": [p0, g.get("lm.paths").tolist()]}
    g.close()
    return out


res = {"card": card(), "sweeps": N, "warmup": WARM, "publish_every": EVERY, "runs": []}
for publish in (False, True, False, True):
    r = replay(publish); r["publish"] = publish
    res["runs"].append(r)
    print(json.dumps({k: v for k, v in r.items() if k != "after_publication_ms"}), flush=True)
res["assembly"] = assembly_and_copy()
print(json.dumps(res["assembly"], indent=1))
if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        json.dump(res, f, indent=1)
print("card:", res["card"])
