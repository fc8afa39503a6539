"""Modal solves of the bench cube with and without a material field (DiffSoundObj.set_material_field), and the field
kernels timed alone.

Workload: the order-2 Kuhn cube of bench.py (32^3 cells x 6 tets = 196 608 P2 tets, 32 modes, steel).  Cases, one object
each, solved cold (no warm start) like bench.py's step -- assembly, coarse assembly, eigen-solve:
  homogeneous   no field;
  constant      a field equal to steel everywhere (same K and M bit for bit: the cost of the field path alone);
  two           steel for x < 1/2, wood above (material_field_from_regions);
  inclusion     steel with a 100x stiffer cube [0.3, 0.7]^3 inside.
The cases alternate for REPS rounds after a warm-up of each, so drift of the shared host hits all alike; per-solve times
are CUDA events around each solve.  Per case: mean / min / max ms, LOBPCG and nested (P1) iterations and whether the FP64
preconditioner was taken.  Then, over 50 launches each with CUDA events: the fine assembly scalar against field
(ds_assemble_km_tets / _field) and the P1 coarse assembly (ds_assemble_km / _field), and ds_material_field_grad at k = 32
and 64 against ds_eigval_grad_shape (k = 32, the solved modes).  Registers and spills of the new instantiations come from
the ptxas log of the build.  The card name and power limit are read in the same run.  One JSON line per record.

usage: python scripts/bench_material_field.py [out.jsonl]"""
import glob
import json
import os
import re
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from diffsound_b200 import native
from diffsound_b200.diffelastic.diff_model import DiffSoundObj, material_field_from_regions
from diffsound_b200.diffelastic.material_model import MatSet
from diffsound_b200.diffelastic.shape_func import CORNER_LOCAL
from oracle import modal_oracle as mo

assert torch.cuda.is_available(), "bench_material_field.py needs a CUDA device"
dev = torch.device("cuda:0")
REPS = 5
LAUNCHES = 50


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


def timed(fn):
    """ms per launch of fn over LAUNCHES launches, after one warm-up."""
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(LAUNCHES):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / LAUNCHES


def field(obj, case):
    T = obj.tetmesh.tets.shape[0]
    rho, E, nu = MatSet.Steel[:3]
    c = obj.tetmesh.vertices.detach().double()[obj.tetmesh.tets[:, list(CORNER_LOCAL[2])]].mean(1)
    full = lambda x: torch.full((T,), x, dtype=torch.float64, device=dev)
    if case == "constant":
        return full(E), full(nu), full(rho)
    if case == "two":
        return material_field_from_regions((c[:, 0] > 0.5).long(), [MatSet.Steel, MatSet.Wood])
    core = ((c > 0.3) & (c < 0.7)).all(1)
    return torch.where(core, 100.0 * E, E), full(nu), full(rho)


def ptxas_records():
    """registers / spills of the new kernel instantiations from the build's ptxas logs (diffsound_b200/csrc/build)."""
    out = []
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for path in sorted(glob.glob(os.path.join(root, "diffsound_b200", "csrc", "build", "*.ptxas.txt"))):
        text = open(path).read()
        for m in re.finditer(r"Function properties for (\S+)\n(.*?)ptxas info\s+: Used (\d+) registers", text, re.S):
            name, body, regs = m.group(1), m.group(2), int(m.group(3))
            if "k_material_field" in name or re.search(r"k_(assemble_rows|assemble_rows_tets2|eigval_grad_shape)I(Li\dE)?Li1EE", name):
                spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", body)
                out.append(dict(case="ptxas", kernel=name, registers=regs,
                                spill_stores=int(spill.group(1)) if spill else None,
                                spill_loads=int(spill.group(2)) if spill else None))
    return out


def main(out_path):
    v, t = mo.kuhn_cube(32)
    objs = {}
    for case in ("homogeneous", "constant", "two", "inclusion"):
        obj = DiffSoundObj(v.to(dev), t.to(dev), mode_num=32, order=2, mat=MatSet.Steel)
        if case != "homogeneous":
            obj.set_material_field(*field(obj, case))
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
        s, ts = stats[c], times[c]
        lines.append(dict(case=c, n_dofs=obj.deform.pattern.n, tets=obj.deform.num_tets, modes=obj.mode_num,
                          solve_ms_mean=sum(ts) / len(ts), solve_ms_min=min(ts), solve_ms_max=max(ts), solve_ms=ts,
                          lobpcg_iterations=s["iterations"], nested_iterations=s.get("nested_iterations"),
                          precond=s.get("precond", "fp32"), **info))
    # kernels alone, on the two-material object
    obj = objs["two"]
    d = obj.deform
    f = obj._field_used
    fld = (f["mu"], f["lam"], f["rho"])
    mu, lam = obj._lame_used
    rho = obj._density_used
    pat, v32 = d.pattern, obj._verts32
    K, Mb, geom = torch.empty_like(obj._Kval), torch.empty_like(obj._Mblk), torch.empty_like(obj._geom)
    co = d.coarse
    ms = dict(
        assemble_fine_scalar=timed(lambda: native.assemble_km(v32, d.tets_i32, 2, pat, mu, lam, d.ctab, d.mtab(rho), Kval=K,
                                                              Mblk=Mb, geom=geom)),
        assemble_fine_field=timed(lambda: native.assemble_km(v32, d.tets_i32, 2, pat, 0.0, 0.0, d.ctab, d.m32(), Kval=K,
                                                             Mblk=Mb, geom=geom, field=fld)),
        assemble_coarse_scalar=timed(lambda: co.assemble(v32, mu, lam, co.ctab, d.coarse_mtab(rho))),
        assemble_coarse_field=timed(lambda: co.assemble(v32, 0.0, 0.0, co.ctab, d.m32(1), field=fld)))
    inc_ptr, inc = d.incidence
    U, lamv = obj.U_hat, obj.eigenvalues
    g = 1.0 / lamv
    tet_grad = torch.empty(d.num_tets * 12, dtype=torch.float64, device=dev)
    ms["grad_shape_k32"] = timed(lambda: native.eigval_grad_shape(v32, d.tets_i32, 2, mu, lam, d.ctab, d.mtab(rho), U, lamv,
                                                                  g, inc_ptr, inc, tet_grad=tet_grad))
    ms["grad_shape_field_k32"] = timed(lambda: native.eigval_grad_shape_field(v32, d.tets_i32, 2, fld, d.ctab, d.mtab(1.0), U,
                                                                              lamv, g, inc_ptr, inc, tet_grad=tet_grad))
    ms["material_field_grad_k32"] = timed(lambda: native.material_field_grad(v32, d.tets_i32, 2, d.m32(), d.wsum, U, lamv, g))
    U64 = torch.randn(pat.n, 64, dtype=torch.float64, device=dev)
    lam64 = torch.rand(64, dtype=torch.float64, device=dev) + 1.0
    ms["material_field_grad_k64"] = timed(lambda: native.material_field_grad(v32, d.tets_i32, 2, d.m32(), d.wsum, U64, lam64,
                                                                             lam64))
    ms["element_energies_k32"] = timed(lambda: native.element_energies(v32, d.tets_i32, 2, d.m32(), d.wsum, U, fld))
    lines.append(dict(case="kernels", tets=d.num_tets, n_nodes=pat.n_nodes, nnzb=pat.nnzb, launches=LAUNCHES,
                      ms_per_launch=ms, **info))
    lines.extend(ptxas_records())
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")
            print(json.dumps(ln))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "profiles/material_field_bench.jsonl")
