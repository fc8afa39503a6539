"""Signed distance from points to a triangle mesh on the device (csrc/sdf.cu, native.mesh_sdf, DMTetGeometry.apply_sdf(path))
against the fp64 numpy oracle (oracle/mesh_sdf.py: brute-force distance, sign from the generalised winding number).

Bars: distance |d_gpu - d_ref| <= 2.5e-7 max(|d_ref|, 1e-6 diag); sign equal wherever |d_ref| >= 1e-6 diag on closed meshes
(on open meshes the three-ray vote and the winding number are different definitions); BVH and brute force bitwise equal;
flipped faces and unshared vertices bitwise equal to the indexed mesh."""
import os
import types

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import mesh_sdf as ms

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _grid(res):
    if res == 16:
        d = np.load(os.path.join(GOLDEN, "meshes.npz"))
        return d["grid16_verts"], d["grid16_tets"].astype(np.int64)
    if res == 32:
        d = np.load(os.path.join(GOLDEN, "mesh_grid32.npz"))
        return d["verts"], d["tets"].astype(np.int64)
    d = np.load(os.path.join(GOLDEN, "grid64_tets.npz"))
    return d["vertices"].astype(np.float32), d["indices"].astype(np.int64)


def _points(res):
    return _grid(res)[0].astype(np.float32) * np.float32(1.5)


def _concat(*meshes):
    vs, fs, n = [], [], 0
    for v, f in meshes:
        vs.append(v)
        fs.append(f + n)
        n += len(v)
    return np.concatenate(vs), np.concatenate(fs)


def _lshape():
    occ = np.zeros((2, 2, 2), dtype=bool)
    occ[0, 0, 0] = occ[1, 0, 0] = occ[0, 1, 0] = occ[0, 0, 1] = True
    return ms.voxel_mesh(occ, (-0.375, -0.375, -0.28125), (0.375, 0.375, 0.375))   # face planes through grid16 vertices


def _shell():
    ov, of = ms.icosphere(4, 0.6)
    iv, if_ = ms.icosphere(3, 0.3)
    return _concat((ov, of), (iv, if_[:, ::-1].copy()))


MESHES = {
    "triangle": lambda: (np.float32([[-0.3, -0.2, 0.05], [0.4, -0.1, 0.1], [0.0, 0.5, -0.05]]), np.int64([[0, 1, 2]])),
    "degenerate": lambda: (np.float32([[-0.4, 0, 0], [0, 0, 0], [0.4, 0, 0], [0.1, 0.2, 0.3], [0.2, -0.3, 0.1]]),
                           np.int64([[0, 1, 2], [3, 3, 4], [4, 4, 4], [0, 3, 4]])),
    "ico3": lambda: ms.icosphere(3, 0.6),
    "ico4": lambda: ms.icosphere(4, 0.6),
    "ico5": lambda: ms.icosphere(5, 0.6),
    "torus": lambda: ms.torus(),
    "lshape": _lshape,
    "two_spheres": lambda: _concat(ms.icosphere(3, 0.3, (-0.35, 0.0, 0.0)), ms.icosphere(3, 0.3, (0.35, 0.05, 0.0))),
    "shell": _shell,
}
OPEN = {"triangle", "degenerate"}


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _sdf(v, f, p, brute_force=False):
    from diffsound_b200 import native
    return native.mesh_sdf(_t(v), _t(f), _t(p), brute_force=brute_force)


# every mesh at the 16 and 32 grids, except ico5 x grid32 (20 480 faces x 6 641 points: over a minute of numpy oracle)
ORACLE_CASES = [(n, r) for n in MESHES for r in (16, 32) if (n, r) != ("ico5", 32)]


@pytest.mark.parametrize("name,res", ORACLE_CASES)
def test_mesh_sdf_matches_oracle(name, res):
    v, f = MESHES[name]()
    p = _points(res)
    ref, _ = ms.mesh_sdf(v, f, p)
    got = _sdf(v, f, p).cpu().numpy().astype(np.float64)
    diag = float(np.linalg.norm(p.max(0).astype(np.float64) - p.min(0)))
    err = np.abs(np.abs(got) - np.abs(ref))
    assert np.all(err <= 2.5e-7 * np.maximum(np.abs(ref), 1e-6 * diag)), float(err.max())
    if name not in OPEN:
        far = np.abs(ref) >= 1e-6 * diag
        bad = np.nonzero((got[far] > 0) != (ref[far] > 0))[0]
        assert bad.size == 0, (bad.size, p[far][bad[:5]], ref[far][bad[:5]])
        assert (got > 0).any() and (got < 0).any()


@pytest.mark.parametrize("name", ["ico4", "torus", "lshape", "shell", "degenerate"])
def test_orientation_and_duplicated_vertices_do_not_change_the_result(name):
    v, f = MESHES[name]()
    p = _points(32)
    base = _sdf(v, f, p)
    flipped = _sdf(v, f[:, ::-1].copy(), p)
    soup = _sdf(v[f].reshape(-1, 3), np.arange(3 * len(f), dtype=np.int64).reshape(-1, 3), p)
    assert torch.equal(base, flipped)
    assert torch.equal(base, soup)


@pytest.mark.parametrize("name", ["ico7", "ico8", "torus"])
def test_bvh_equals_brute_force_bitwise(name):
    """The minimum and the crossing counts do not depend on the visit order: any difference means the tree pruned the
    nearest triangle or a crossed one."""
    v, f = ms.icosphere(int(name[3:]), 0.6) if name.startswith("ico") else ms.torus(nu=384, nv=192)
    p = _points(64)
    bvh = _sdf(v, f, p)
    brute = _sdf(v, f, p, brute_force=True)
    assert torch.equal(bvh, brute), int((bvh != brute).sum())
    assert (bvh > 0).any() and (bvh < 0).any()


def test_apply_sdf_path_end_to_end(tmp_path):
    from diffsound_b200 import native
    from diffsound_b200.diffelastic.mesh import read_obj
    from diffsound_b200.dmtet.geometry.dmtet_thickness import DMTetGeometry
    v, f = ms.icosphere(4, 0.6)
    path = tmp_path / "sphere.obj"
    ms.write_obj(str(path), v, f)
    FLAGS = types.SimpleNamespace(mode_num=8, order=1, mat="Steel", out_dir="/tmp", without_tensorboard=True)
    geo = DMTetGeometry(64, 1.5, FLAGS, grid=_grid(64))
    geo.apply_sdf(str(path))
    rv, rf = read_obj(str(path))
    ref = DMTetGeometry(64, 1.5, FLAGS, grid=_grid(64))
    ref.apply_sdf(native.mesh_sdf(_t(rv), _t(rf), ref.verts))
    assert torch.equal(geo.sdf, ref.sdf)
    assert torch.equal(geo.marching_tets.max_thickness, ref.marching_tets.max_thickness)
    # against the sphere: within the Hausdorff distance between the sphere and the inscribed polyhedron
    tri = rv.astype(np.float64)[rf]
    n = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    h = np.abs(np.einsum("ij,ij->i", n, tri[:, 0])) / np.linalg.norm(n, axis=1)
    gv = geo.verts.cpu().numpy().astype(np.float64)
    analytic = 0.6 - np.linalg.norm(gv, axis=1)
    assert np.abs(geo.sdf.cpu().numpy() - analytic).max() <= (0.6 - h.min()) + 1e-6
    # one thickness step at order 1: getMesh -> eigen-solve -> loss, gradient to the thickness logits
    target = geo.get_eigenvalues(thickness_coef=1.0)
    loss = geo.tick(target, 0, FLAGS)
    loss.backward()
    grad = geo.marching_tets.thickness_coef.probablity.grad
    assert torch.isfinite(loss).item() and grad is not None and torch.isfinite(grad).all().item()


def test_cabi_errors_leave_the_device_usable():
    import ctypes as C
    from diffsound_b200 import _lib, native
    lib = _lib.load()
    ws = native.workspace(DEV)
    v, f = ms.icosphere(2, 0.6)
    p = _points(16)
    tv, tf, tp = _t(v), _t(f), _t(p)
    out = torch.empty(len(p), dtype=torch.float32, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(verts, faces, pts, mode=0):
        ptr = (lambda t: None if t is None else C.c_void_p(t.data_ptr()))
        return lib.ds_mesh_sdf(ws.handle, ptr(verts), len(v), ptr(faces), len(f), ptr(pts), len(p), mode, ptr(out), st)

    bad_f = tf.clone()
    bad_f[5, 1] = len(v)
    assert call(tv, bad_f, tp) == -2 and "face 5" in _lib.last_error()
    bad_f[5, 1] = -1
    assert call(tv, bad_f, tp) == -2 and "face 5" in _lib.last_error()
    nan_v = tv.clone()
    nan_v[3, 0] = float("nan")
    assert call(nan_v, tf, tp) == -2 and "vertex 3" in _lib.last_error()
    inf_p = tp.clone()
    inf_p[7, 2] = float("inf")
    assert call(tv, tf, inf_p) == -2 and "query point 7" in _lib.last_error()
    assert call(None, tf, tp) == -2 and "null" in _lib.last_error()
    assert call(tv, tf, tp, mode=3) == -2 and "unknown mode" in _lib.last_error()
    torch.cuda.synchronize()
    assert torch.equal(native.mesh_sdf(tv, tf, tp), native.mesh_sdf(tv, tf, tp, brute_force=True))
