"""Modal gains on the device (csrc/gains.cu), stage by stage.

Workloads: the order-2 Kuhn cube of bench.py (32^3 cells, 196 608 tets) and a tetrahedralised radius-0.5 sphere
(tetrahedralize of the analytic SDF at edge length 0.025, promoted to order 2), each at k = 32 and 64 modes.  The
timed kernels read U in place and do not depend on its values, so U is a seeded random fp64 block of the solver's shape
(n_dofs x k, row-major).  Point sets: every boundary node (corner and mid-edge), and 10^6 random points on the boundary.
Stages, each the mean over 20 launches between two CUDA events after a warm-up: the boundary build
(ds_tet_boundary_*), the nearest-face lookup (ds_mesh_sdf_nearest over the corner-node boundary faces),
ds_modal_gains and ds_modal_gains_backward (each including its validation pass and synchronisation).  Reported with
the bytes of U gathered (P x npe x 3 x k x 8).  The card name and power limit are read in the same run.  One JSON line
per configuration.

usage: python scripts/bench_modal_gains.py [out.jsonl]"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from diffsound_b200 import native
from diffsound_b200.diffelastic.mesh import TetMesh
from diffsound_b200.diffelastic.tetrahedralize import tetrahedralize
from oracle import modal_oracle as mo

assert torch.cuda.is_available(), "bench_modal_gains.py needs a CUDA device"
dev = torch.device("cuda:0")
REPS = 20


def card():
    name = torch.cuda.get_device_name(dev)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        power, clock = (s.strip() for s in r.stdout.strip().split(","))
    except Exception as e:        # the query is informational; the times stand without it
        power, clock = f"unavailable ({type(e).__name__})", "unavailable"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(REPS):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / REPS, out


def workloads():
    v, t = mo.kuhn_cube(32)
    yield "kuhn_cube32", TetMesh(v.to(dev), t.to(dev)).to_high_order(2)
    m = tetrahedralize(lambda p: 0.5 - p.norm(dim=1), edge_length=0.025, bounds=((-0.6,) * 3, (0.6,) * 3))
    yield "sphere_h0.025", TetMesh(m.vertices, m.tets).to_high_order(2)


def point_sets(verts, faces, gen):
    a, b, c = (verts[faces[:, i].long()] for i in range(3))
    nodes = torch.unique(torch.cat([a, b, c, (a + b) / 2, (b + c) / 2, (c + a) / 2]), dim=0)
    area = torch.linalg.cross(b - a, c - a).norm(dim=1).double()
    f = torch.multinomial(area, 1_000_000, replacement=True, generator=gen)
    L = -torch.log(torch.rand(1_000_000, 3, device=dev, generator=gen, dtype=torch.float64))
    L = (L / L.sum(1, keepdim=True)).float()
    rand = L[:, :1] * a[f] + L[:, 1:2] * b[f] + L[:, 2:] * c[f]
    return {"boundary_nodes": nodes.contiguous(), "random_1e6": rand.contiguous()}


def main():
    out = open(sys.argv[1], "w") if len(sys.argv) > 1 else sys.stdout
    info = card()
    gen = torch.Generator(device=dev).manual_seed(0)
    for name, mesh in workloads():
        verts = mesh.vertices.detach().float().contiguous()
        tets = mesh.tets.to(torch.int32).contiguous()
        t_bnd, bnd = timed(lambda: native.tet_boundary(verts, tets, 2))
        faces64 = bnd[0].long()
        for pname, pts in point_sets(verts, bnd[0], gen).items():
            t_near, (_, face) = timed(lambda: native.mesh_sdf_nearest(verts, faces64, pts))
            for k in (32, 64):
                U = torch.randn(3 * verts.shape[0], k, dtype=torch.float64, device=dev, generator=gen)
                up = torch.randn(pts.shape[0], k, dtype=torch.float32, device=dev, generator=gen)
                t_fwd, _ = timed(lambda: native.modal_gains(verts, tets, 2, bnd, pts, face, None, U))
                t_bwd, _ = timed(lambda: native.modal_gains_backward(verts, tets, 2, bnd, pts, face, None, U, up))
                P = pts.shape[0]
                gathered = P * 10 * 3 * k * 8
                row = dict(workload=name, tets=int(tets.shape[0]), nodes=int(verts.shape[0]),
                           boundary_faces=int(bnd[0].shape[0]), points=pname, P=int(P), k=k,
                           boundary_ms=round(t_bnd, 4), nearest_ms=round(t_near, 4), gains_ms=round(t_fwd, 4),
                           gains_backward_ms=round(t_bwd, 4), U_bytes_gathered=gathered,
                           U_block_bytes=int(U.numel() * 8), gains_GBps=round(gathered / t_fwd / 1e6, 1), **info)
                out.write(json.dumps(row) + "\n")
                out.flush()


if __name__ == "__main__":
    main()
