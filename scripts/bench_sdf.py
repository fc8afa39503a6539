"""Triangle-mesh signed distance (ds_mesh_sdf, csrc/sdf.cu): BVH build, BVH query and the brute-force reference, timed on
the device after a warm-up.

Workloads: the 64 background grid x 1.5 (tests/golden/grid64_tets.npz, 36 562 vertices, BASELINE config 4), and 2 M seeded
random points in the same box as a stand-in for the finer Quartet grids (the vertex count a 128 grid reaches is not in
this checkout); against radius-0.6 icospheres of 20 480, 81 920, 327 680 and 1 310 720 triangles generated here.  Build
and query times come from the library's per-class device timing (CUDA events around each stage, classes sdf_build /
sdf_query); call_ms is the whole call between two CUDA events (argument validation with its one synchronisation
included).  Brute force runs where points x faces <= 5e10.  Each configuration also checks BVH == brute force bitwise
where both run.  The card name and power limit are read in the same run.  One JSON line per configuration.

usage: python scripts/bench_sdf.py [reps]"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from diffsound_b200 import native
from oracle.mesh_sdf import icosphere

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
assert torch.cuda.is_available(), "bench_sdf.py needs a CUDA device"
dev = torch.device("cuda:0")


def card():
    name = torch.cuda.get_device_name(dev)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        power, clock = (s.strip() for s in r.stdout.strip().split(","))
    except Exception as e:        # the query is informational; the times stand without it
        power, clock = f"unavailable ({type(e).__name__})", "unavailable"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, n):
    fn()                                   # warm-up: module load, arena growth, CUB temp sizing
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with native.prof(["sdf_build", "sdf_query"]) as pr:
        e0.record()
        for _ in range(n):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        stages = pr.read()
    ms = {k: v["ms"] / v["count"] for k, v in stages.items()}
    return out, e0.elapsed_time(e1) / n, ms.get("sdf_build"), ms.get("sdf_query")


info = card()
grid = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                            "grid64_tets.npz"))["vertices"].astype(np.float32) * np.float32(1.5)
rng = np.random.default_rng(20261020)
points = {"grid64x1.5": grid, "random2M": rng.uniform(-0.75, 0.75, (2_000_000, 3)).astype(np.float32)}
for level in (5, 6, 7, 8):
    v, f = icosphere(level, 0.6)
    tv, tf = torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev)
    for pname, p in points.items():
        tp = torch.from_numpy(p).to(dev)
        row = {"bench": "mesh_sdf", "mesh": f"icosphere{level}", "faces": int(len(f)), "points": pname,
               "n_points": int(len(p)), "reps": reps}
        bvh, row["bvh_call_ms"], row["bvh_build_ms"], row["bvh_query_ms"] = timed(
            lambda: native.mesh_sdf(tv, tf, tp), reps)
        row["inside"] = int((bvh > 0).sum())
        if len(p) * len(f) <= 5e10:
            brute, row["brute_call_ms"], _, row["brute_query_ms"] = timed(
                lambda: native.mesh_sdf(tv, tf, tp, brute_force=True), 1)
            row["bvh_equals_brute"] = bool(torch.equal(bvh, brute))
        row.update(info)
        print(json.dumps(row), flush=True)
