"""Triangle-mesh SDF with its gradient (csrc/sdf.cu): ds_mesh_sdf, ds_mesh_sdf_nearest (the forward that also records
the nearest face) and ds_mesh_sdf_backward, timed on the device after a warm-up.

Workloads of scripts/bench_sdf.py: radius-0.6 icospheres of 20 480, 81 920, 327 680 and 1 310 720 triangles, at the 64
background grid x 1.5 (36 562 points) and at 2 M seeded random points.  ds_mesh_sdf and ds_mesh_sdf_nearest run in the
same process, alternating call by call, so that their times are comparable; the backward (both outputs, a seeded random
upstream gradient) runs after them.  Each time is the mean over `reps` calls of the whole call between two CUDA events
(argument validation with its one synchronisation included).  Each configuration also checks that the nearest-face
forward returns the same sdf bitwise.  The card name and power limit are read in the same run.  One JSON line per
configuration.

usage: python scripts/bench_sdf_grad.py [reps]"""
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
assert torch.cuda.is_available(), "bench_sdf_grad.py needs a CUDA device"
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
        g = torch.from_numpy(np.random.default_rng(level).standard_normal(len(p)).astype(np.float32)).to(dev)
        plain = lambda: native.mesh_sdf(tv, tf, tp)
        nearest = lambda: native.mesh_sdf_nearest(tv, tf, tp)
        base, (sdf, face) = plain(), nearest()                    # warm-up: module load, arena growth, CUB sizing
        back = lambda: native.mesh_sdf_backward(tv, tf, tp, face, sdf, g)
        back()
        torch.cuda.synchronize()
        t_plain, t_near, t_back = [], [], []
        for _ in range(reps):
            t_plain.append(timed_ms(plain)[1])
            t_near.append(timed_ms(nearest)[1])
        for _ in range(reps):
            t_back.append(timed_ms(back)[1])
        row = {"bench": "mesh_sdf_grad", "mesh": f"icosphere{level}", "faces": int(len(f)), "points": pname,
               "n_points": int(len(p)), "reps": reps,
               "sdf_call_ms": float(np.mean(t_plain)), "sdf_call_ms_min": float(np.min(t_plain)),
               "nearest_call_ms": float(np.mean(t_near)), "nearest_call_ms_min": float(np.min(t_near)),
               "backward_call_ms": float(np.mean(t_back)), "backward_call_ms_min": float(np.min(t_back)),
               "nearest_sdf_equals_sdf": bool(torch.equal(sdf, base))}
        row.update(info)
        print(json.dumps(row), flush=True)
