"""Free against supported modal solves of the bench cube (DiffSoundObj.set_supports; csrc/support.cu).

Workload: the order-2 Kuhn cube of bench.py (32^3 cells x 6 tets, 32 modes, steel), once free and resting on its z = 0
face on a 10 mm elastic pad at three pad moduli (rubber-like 2 MPa, 20 MPa, 200 MPa; supports.pad_stiffness, nu = 0.45).
One object per case, solved cold (no warm start) like bench.py's step.  The cases alternate for REPS rounds after a
warm-up of each, so drift of the shared host hits all alike; per-solve times are CUDA events around each solve.  Reported
per case: mean / min / max per-solve ms, LOBPCG and nested iterations, the preconditioner that finished the solve, the
lowest eigenvalue, the device time of the `support` class in one profiled solve and the time of get_vals() + backward.
The three support kernels are also timed alone over 50 launches each.  The card name and power limit are read in the same
run.  One JSON line per case and per kernel.

usage: python scripts/bench_supports.py [out.jsonl]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch

from bench_fixed import card, solve
from diffsound_b200 import native
from diffsound_b200.diffelastic.diff_model import DiffSoundObj
from diffsound_b200.diffelastic.material_model import MatSet
from diffsound_b200.diffelastic.supports import pad_stiffness
from oracle import modal_oracle as mo

dev = torch.device("cuda:0")
REPS = 5
PADS = {"pad_2MPa": 2e6, "pad_20MPa": 2e7, "pad_200MPa": 2e8}


def timed(fn, n=1):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main(out_path):
    v, t = mo.kuhn_cube(32)
    objs = {}
    for case in ["free"] + list(PADS):
        leaf = v.to(dev).requires_grad_(True)
        obj = DiffSoundObj(leaf, t.to(dev), mode_num=32, order=2, mat=MatSet.Steel)
        obj.leaf = leaf
        if case != "free":
            faces = obj.surface()[0]
            kn, kt = pad_stiffness(PADS[case], 0.45, 0.01)
            obj.set_supports((obj.tetmesh.vertices[faces][:, :, 2] == 0.0).all(dim=1), kn, kt)
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
        with native.prof(classes=["support"]) as pf:
            solve(obj)
        p = pf.read().get("support", {"ms": 0.0, "count": 0})
        g = torch.ones(obj.mode_num, device=dev)
        grad_ms = timed(lambda: torch.autograd.grad((obj.get_vals()[:, 0] * g).sum(), obj.leaf, retain_graph=True), 5)
        s = stats[c]
        ts = times[c]
        lines.append(dict(case=c, n_dofs=obj.deform.pattern.n, support_faces=0 if obj._sup is None else obj._sup["fine"].S,
                          modes=obj.mode_num, solve_ms_mean=sum(ts) / len(ts), solve_ms_min=min(ts), solve_ms_max=max(ts),
                          solve_ms=ts, lobpcg_iterations=s["iterations"], nested_iterations=s.get("nested_iterations"),
                          preconditioner=s.get("precond", "fp32 two-level"), lambda_min=float(obj.eigenvalues[0]),
                          support_class_ms=p["ms"], support_class_launches=p["count"], get_vals_backward_ms=grad_ms,
                          **info))
    obj = objs["pad_20MPa"]
    d, f, su = obj.deform, obj._sup["fine"], obj._sup_used
    gk = torch.ones(obj.mode_num, dtype=torch.float64, device=dev)
    kernels = {
        "ds_support_km": lambda: native.support_km(obj._verts32, d.tets_i32, d.pattern, f, su["kn"], su["kt"], obj._Kval),
        "ds_support_grad": lambda: native.support_grad(obj._verts32, d.tets_i32, f, su["kn"], su["kt"], obj.U_hat, gk),
        "ds_support_energies": lambda: native.support_energies(obj._verts32, d.tets_i32, f, su["kn"], su["kt"], obj.U_hat),
    }
    for name, fn in kernels.items():
        lines.append(dict(case=name, support_faces=f.S, incidence_rows=f.R, modes=obj.mode_num, us=timed(fn, 50) * 1e3,
                          **info))
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")
            print(json.dumps(ln))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "profiles/supports_bench.jsonl")
