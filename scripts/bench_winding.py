"""Generalised winding number of a triangle mesh (csrc/sdf.cu: ds_mesh_winding_number) and the signed distance signed by it
(ds_mesh_sdf_winding), timed on the device after a warm-up.

Workloads of scripts/bench_sdf.py: radius-0.6 icospheres of 20 480, 81 920, 327 680 and 1 310 720 triangles, at the 64
background grid x 1.5 (36 562 points) and at 2 M seeded random points.  Per configuration:
  * ds_mesh_winding_number in BVH mode (whole call, and the library's sdf_winding stage: moments, point order and
    traversal) and in brute-force mode where points x faces <= 5e10, with max and mean |w_bvh - w_brute|;
  * ds_mesh_sdf_winding against ds_mesh_sdf, alternating call by call so that their times are comparable, and whether
    the two outputs are bitwise equal (they must be: the sphere is closed and outward).
Each time is the mean over `reps` calls of the whole call between two CUDA events (argument validation with its one
synchronisation included).  The card name and power limit are read in the same run.  One JSON line per configuration.

usage: python scripts/bench_winding.py [reps]"""
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
assert torch.cuda.is_available(), "bench_winding.py needs a CUDA device"
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


def timed_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return out, e0.elapsed_time(e1)


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
        wn = lambda: native.mesh_winding_number(tv, tf, tp)
        parity = lambda: native.mesh_sdf(tv, tf, tp)
        winding = lambda: native.mesh_sdf(tv, tf, tp, sign="winding")
        w, a, b = wn(), parity(), winding()                    # warm-up: module load, arena growth, CUB sizing
        torch.cuda.synchronize()
        t_wn, t_par, t_win = [], [], []
        with native.prof(["sdf_winding"]) as pr:
            for _ in range(reps):
                t_wn.append(timed_ms(wn)[1])
            stage = pr.read()["sdf_winding"]
        for _ in range(reps):
            t_par.append(timed_ms(parity)[1])
            t_win.append(timed_ms(winding)[1])
        row = {"bench": "mesh_winding", "mesh": f"icosphere{level}", "faces": int(len(f)), "points": pname,
               "n_points": int(len(p)), "reps": reps,
               "wn_bvh_call_ms": float(np.mean(t_wn)), "wn_bvh_call_ms_min": float(np.min(t_wn)),
               "wn_bvh_stage_ms": stage["ms"] / stage["count"],
               "sdf_parity_call_ms": float(np.mean(t_par)), "sdf_parity_call_ms_min": float(np.min(t_par)),
               "sdf_winding_call_ms": float(np.mean(t_win)), "sdf_winding_call_ms_min": float(np.min(t_win)),
               "sdf_winding_equals_parity": bool(torch.equal(a, b)), "inside": int((b > 0).sum())}
        if len(p) * len(f) <= 5e10:
            wb, row["wn_brute_call_ms"] = timed_ms(lambda: native.mesh_winding_number(tv, tf, tp, brute_force=True))
            err = (w.double() - wb.double()).abs()
            row["w_err_max"], row["w_err_mean"] = float(err.max()), float(err.mean())
        row.update(info)
        print(json.dumps(row), flush=True)
