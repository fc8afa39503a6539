"""Modal solves of the bench cube with and without an elasticity-tensor field (DiffSoundObj.set_elasticity_field), and the
tensor kernels timed alone.

Workload: the order-2 Kuhn cube of bench.py (32^3 cells x 6 tets = 196 608 P2 tets, 32 modes).  Cases, one object each,
solved cold (no warm start) like bench.py's step -- assembly, coarse assembly, eigen-solve:
  homogeneous   steel, no field;
  isotropic     a tensor field equal to steel everywhere (isotropic_stiffness): the cost of the tensor path alone;
  wood          wood-like orthotropic constants (illustrative, not measured wood data) with a random grain rotation per
                tet, density 500 (a worst case: grain directions uncorrelated from tet to tet);
  wood_x        the same constants with the grain along x everywhere (one piece of straight-grained wood).
The cases alternate for REPS rounds after a warm-up of each, so drift of the shared host hits all alike; per-solve times
are CUDA events around each solve.  Per case: mean / min / max ms, LOBPCG and nested (P1) iterations and which
preconditioner ran.  Then, over 50 launches each with CUDA events: the fine assembly scalar / Lame field / tensor field
(ds_assemble_km_tets, _field, _tensor), the P1 coarse assembly (ds_assemble_km, _field, _tensor), ds_elasticity_field_grad
at k = 32 and 64, ds_eigval_grad_shape_tensor against ds_eigval_grad_shape (k = 32, the solved modes) and
ds_element_energies_tensor.  Registers and spills of the tensor instantiations come from the ptxas log of the build.  The
card name and power limit are read in the same run.  One JSON line per record.

usage: python scripts/bench_elasticity_field.py [out.jsonl]"""
import glob
import json
import os
import re
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from diffsound_b200 import native
from diffsound_b200.diffelastic import anisotropic as an
from diffsound_b200.diffelastic.diff_model import DiffSoundObj, _lame
from diffsound_b200.diffelastic.material_model import MatSet
from oracle import modal_oracle as mo
from scripts.bench_material_field import card, solve, timed

assert torch.cuda.is_available(), "bench_elasticity_field.py needs a CUDA device"
dev = torch.device("cuda:0")
REPS = 5
WOOD = (1.2e10, 8e8, 5e8, 0.4, 0.45, 0.5, 7e8, 6e8, 5e7)      # E1 E2 E3 nu12 nu13 nu23 G12 G13 G23, illustrative


def random_rotations(n, seed):
    q = torch.randn(n, 4, dtype=torch.float64, device=dev, generator=torch.Generator(device=dev).manual_seed(seed))
    q = q / q.norm(dim=1, keepdim=True)
    w, x, y, z = q.unbind(1)
    return torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                        2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                        2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], dim=1).reshape(n, 3, 3)


def ptxas_records():
    """registers / spills of the tensor instantiations (MAT_TENSOR = 2) and k_elasticity_field from the build's ptxas
    logs (diffsound_b200/csrc/build)."""
    out = []
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for path in sorted(glob.glob(os.path.join(root, "diffsound_b200", "csrc", "build", "*.ptxas.txt"))):
        text = open(path).read()
        for m in re.finditer(r"Function properties for (\S+)\n(.*?)ptxas info\s+: Used (\d+) registers", text, re.S):
            name, body, regs = m.group(1), m.group(2), int(m.group(3))
            if ("k_elasticity_field" in name or re.search(r"k_assemble_rows_tets2ILi2E", name)
                    or re.search(r"k_(assemble_rows|eigval_grad_shape)ILi\dELi2E", name)):
                spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", body)
                out.append(dict(case="ptxas", kernel=name, registers=regs,
                                spill_stores=int(spill.group(1)) if spill else None,
                                spill_loads=int(spill.group(2)) if spill else None))
    return out


def main(out_path):
    v, t = mo.kuhn_cube(32)
    rho_s, E_s, nu_s = MatSet.Steel[:3]
    objs = {}
    for case in ("homogeneous", "isotropic", "wood", "wood_x"):
        obj = DiffSoundObj(v.to(dev), t.to(dev), mode_num=32, order=2, mat=MatSet.Steel)
        T = obj.deform.num_tets
        if case == "isotropic":
            obj.set_elasticity_field(an.isotropic_stiffness(E_s, nu_s).to(dev).expand(T, 6, 6))
        elif case in ("wood", "wood_x"):
            C = an.orthotropic_stiffness(*WOOD).to(dev).expand(T, 6, 6)
            if case == "wood":
                C = an.rotate_stiffness(C, random_rotations(T, 0))
            obj.set_elasticity_field(C, torch.full((T,), 500.0, dtype=torch.float64, device=dev))
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
    # kernels alone, on the wood object
    obj = objs["wood"]
    d = obj.deform
    tu = obj._tensor_used
    ten = (tu["C21"], tu["rho"])
    T = d.num_tets
    mu, lam = _lame(E_s, nu_s)
    f64 = dict(dtype=torch.float64, device=dev)
    fld = (torch.full((T,), mu, **f64), torch.full((T,), lam, **f64), tu["rho"])
    pat, v32 = d.pattern, obj._verts32
    K, Mb, geom = torch.empty_like(obj._Kval), torch.empty_like(obj._Mblk), torch.empty_like(obj._geom)
    co = d.coarse
    ms = dict(
        assemble_fine_scalar=timed(lambda: native.assemble_km(v32, d.tets_i32, 2, pat, mu, lam, d.ctab, d.mtab(500.0), Kval=K,
                                                              Mblk=Mb, geom=geom)),
        assemble_fine_field=timed(lambda: native.assemble_km(v32, d.tets_i32, 2, pat, 0.0, 0.0, d.ctab, d.m32(), Kval=K,
                                                             Mblk=Mb, geom=geom, field=fld)),
        assemble_fine_tensor=timed(lambda: native.assemble_km(v32, d.tets_i32, 2, pat, 0.0, 0.0, d.ctab, d.m32(), Kval=K,
                                                              Mblk=Mb, geom=geom, tensor=ten)),
        assemble_coarse_scalar=timed(lambda: co.assemble(v32, mu, lam, co.ctab, d.coarse_mtab(500.0))),
        assemble_coarse_field=timed(lambda: co.assemble(v32, 0.0, 0.0, co.ctab, d.m32(1), field=fld)),
        assemble_coarse_tensor=timed(lambda: co.assemble(v32, 0.0, 0.0, co.ctab, d.m32(1), tensor=ten)))
    inc_ptr, inc = d.incidence
    U, lamv = obj.U_hat, obj.eigenvalues
    g = 1.0 / lamv
    tet_grad = torch.empty(T * 12, **f64)
    ms["grad_shape_k32"] = timed(lambda: native.eigval_grad_shape(v32, d.tets_i32, 2, mu, lam, d.ctab, d.mtab(500.0), U, lamv,
                                                                  g, inc_ptr, inc, tet_grad=tet_grad))
    ms["grad_shape_tensor_k32"] = timed(lambda: native.eigval_grad_shape_tensor(v32, d.tets_i32, 2, ten, d.ctab, d.mtab(1.0),
                                                                                U, lamv, g, inc_ptr, inc, tet_grad=tet_grad))
    ms["elasticity_field_grad_k32"] = timed(lambda: native.elasticity_field_grad(v32, d.tets_i32, 2, d.m32(), d.wsum, U, lamv,
                                                                                 g))
    U64 = torch.randn(pat.n, 64, **f64)
    lam64 = torch.rand(64, **f64) + 1.0
    ms["elasticity_field_grad_k64"] = timed(lambda: native.elasticity_field_grad(v32, d.tets_i32, 2, d.m32(), d.wsum, U64,
                                                                                 lam64, lam64))
    ms["element_energies_tensor_k32"] = timed(lambda: native.element_energies_tensor(v32, d.tets_i32, 2, d.m32(), d.wsum, U,
                                                                                     ten))
    lines.append(dict(case="kernels", tets=T, n_nodes=pat.n_nodes, nnzb=pat.nnzb, launches=50, ms_per_launch=ms, **info))
    lines.extend(ptxas_records())
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")
            print(json.dumps(ln))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "profiles/elasticity_field_bench.jsonl")
