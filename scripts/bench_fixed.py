"""Clamped against free modal solves of the bench cube (DiffSoundObj.fix_nodes; csrc/fixed.cu).

Workload: the order-2 Kuhn cube of bench.py (32^3 cells x 6 tets, 32 modes, steel), once free and once with its z = 0 face
clamped (every node with z = 0, corner and mid-edge).  One object per case, solved cold (no warm start) like bench.py's
step: assembly, coarse assembly, eigen-solve.  The two cases alternate for REPS rounds after a warm-up of each, so drift of
the shared host hits both alike; per-solve times are CUDA events around each solve.  Reported per case: the mean, min and
max per-solve ms, the LOBPCG and nested (P1) iterations, and from an untimed profiled solve the device time of the
`fix_nodes` class (ds_fix_nodes_km on both levels, and the masking launches inside ds_lobpcg).  ds_fix_nodes_km on the
fine level is also timed alone over 50 launches.  The card name and power limit are read in the same run.  One JSON line
per case and one for the kernel.

usage: python scripts/bench_fixed.py [out.jsonl]"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from diffsound_b200 import native
from diffsound_b200.diffelastic.diff_model import DiffSoundObj
from diffsound_b200.diffelastic.material_model import MatSet
from oracle import modal_oracle as mo

assert torch.cuda.is_available(), "bench_fixed.py needs a CUDA device"
dev = torch.device("cuda:0")
REPS = 6


def card():
    name = torch.cuda.get_device_name(dev)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        power, clock = (s.strip() for s in r.stdout.strip().split(","))
    except Exception as e:        # the query is informational; the times stand without it
        power, clock = f"unavailable ({type(e).__name__})", "unavailable"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def solve(obj):
    obj._warm = []
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    obj.eigen_decomposition()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main(out_path):
    v, t = mo.kuhn_cube(32)
    objs = {}
    for case in ("free", "clamped_z0"):
        obj = DiffSoundObj(v.to(dev), t.to(dev), mode_num=32, order=2, mat=MatSet.Steel)
        if case != "free":
            obj.fix_nodes(obj.tetmesh.vertices[:, 2] == 0.0)
        objs[case] = obj
    for obj in objs.values():
        solve(obj)
        solve(obj)
    times = {c: [] for c in objs}
    stats = {}
    for _ in range(REPS):
        for c, obj in objs.items():
            times[c].append(solve(obj))
            stats[c] = obj.eig_stats
    info = card()
    lines = []
    for c, obj in objs.items():
        with native.prof(classes=["fix_nodes"]) as pf:
            solve(obj)
        p = pf.read().get("fix_nodes", {"ms": 0.0, "count": 0})
        s = stats[c]
        ts = times[c]
        lines.append(dict(case=c, n_dofs=obj.deform.pattern.n, fixed_nodes=int(obj._n_fixed if obj.fixed_nodes is not None
                                                                                  else 0),
                          modes=obj.mode_num, solve_ms_mean=sum(ts) / len(ts), solve_ms_min=min(ts), solve_ms_max=max(ts),
                          solve_ms=ts, lobpcg_iterations=s["iterations"], nested_iterations=s.get("nested_iterations"),
                          fix_nodes_class_ms=p["ms"], fix_nodes_class_launches=p["count"], **info))
    obj = objs["clamped_z0"]
    pat = obj.deform.pattern
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    native.fix_nodes_km(pat, obj._fixed_u8, obj._Kval, obj._Mblk)
    torch.cuda.synchronize()
    a.record()
    for _ in range(50):
        native.fix_nodes_km(pat, obj._fixed_u8, obj._Kval, obj._Mblk)
    b.record()
    torch.cuda.synchronize()
    us = a.elapsed_time(b) / 50 * 1e3
    bytes_min = pat.nnzb * 4 + (pat.n_nodes + 1) * 4 + pat.n_nodes   # bcol + brow + mask, read once
    lines.append(dict(case="ds_fix_nodes_km", n_nodes=pat.n_nodes, nnzb=pat.nnzb, us=us,
                      read_GBps=bytes_min / (us * 1e-6) / 1e9, **info))
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")
            print(json.dumps(ln))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "profiles/fixed_bench.jsonl")
