"""Gradient of the triangle-mesh signed distance on the device (csrc/sdf.cu: ds_mesh_sdf_nearest, ds_mesh_sdf_backward;
native.mesh_sdf_nearest / mesh_sdf_backward; dmtet/geometry/mesh_sdf.py; DMTetGeometry.apply_sdf((verts, faces))) against
the fp64 numpy oracle (tests/mesh_sdf_grad_ref.py: mesh_sdf_grad, on the distance and sign of oracle/mesh_sdf.py).

Bars: forward sdf bitwise equal to ds_mesh_sdf; at points whose closest point is unambiguous, grad_points within 1e-6
(where |sdf| >= 1e-6 diag) and grad_verts within 1e-6 rel-L2 of the oracle; the translation and homogeneity identities
to fp32 rounding; face ids and both gradients bitwise equal between BVH and brute force, run to run, and for flipped
faces; a thickness-loop step's mesh gradient against central differences of the fp64 eigenvalues."""
import os
import types

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import mesh_sdf as ms
import mesh_sdf_grad_ref as gr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# ---- the meshes and grids of test_mesh_sdf_gpu.py ------------------------------------------------------------------
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
    "torus": lambda: ms.torus(),
    "lshape": _lshape,
    "two_spheres": lambda: _concat(ms.icosphere(3, 0.3, (-0.35, 0.0, 0.0)), ms.icosphere(3, 0.3, (0.35, 0.05, 0.0))),
    "shell": _shell,
}


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _nearest(v, f, p, brute_force=False):
    from diffsound_b200 import native
    return native.mesh_sdf_nearest(_t(v), _t(f), _t(p), brute_force=brute_force)


def _backward(v, f, p, face, sdf, g):
    from diffsound_b200 import native
    return native.mesh_sdf_backward(_t(v), _t(f), _t(p), face, sdf, _t(np.asarray(g, dtype=np.float32)))


def _unambiguous(v, f, p, diag):
    """points whose faces within 1e-6 diag of the minimum distance all have the same closest point (oracle, fp64)."""
    tris = v.astype(np.float32).astype(np.float64)[f]
    pp = p.astype(np.float64)
    ok = np.ones(len(p), dtype=bool)
    n = max(1, (1 << 17) // len(f))
    for s in range(0, len(p), n):
        d = np.sqrt(ms.point_triangle_d2(pp[s:s + n], tris))
        rows, cols = np.nonzero(d <= d.min(1, keepdims=True) + 1e-6 * diag)
        c, _ = gr.closest_on_triangles(pp[s + rows], *(tris[cols, k] for k in range(3)))
        c0, _ = gr.closest_on_triangles(pp[s:s + n], *(tris[d.argmin(1), k] for k in range(3)))
        far = np.zeros(len(d), dtype=bool)
        np.logical_or.at(far, rows, np.abs(c - c0[rows]).max(1) > 1e-9 * diag)
        ok[s:s + n] = ~far
    return ok


@pytest.mark.parametrize("res", [16, 32])
@pytest.mark.parametrize("name", list(MESHES))
def test_nearest_forward_is_mesh_sdf_bitwise(name, res):
    from diffsound_b200 import native
    v, f = MESHES[name]()
    p = _points(res)
    base = native.mesh_sdf(_t(v), _t(f), _t(p))
    sdf, face = _nearest(v, f, p)
    sdf_b, face_b = _nearest(v, f, p, brute_force=True)
    assert torch.equal(sdf, base) and torch.equal(sdf_b, base)
    assert torch.equal(face, face_b)
    assert int(face.min()) >= 0 and int(face.max()) < len(f)
    # the recorded face reaches the minimum distance, and is the lowest index that does
    ref = gr.mesh_sdf_grad(v, f, p)
    assert np.array_equal(face.cpu().numpy(), ref["face"]) or _ties_only(v, f, p, face.cpu().numpy(), ref["face"])


def _ties_only(v, f, p, got, ref):
    """the kernel's and the oracle's face differ only where their fp64 distances round to a tie differently."""
    tris = v.astype(np.float32).astype(np.float64)[f]
    bad = np.nonzero(got != ref)[0]
    dg = ms.point_triangle_d2(p[bad], tris)
    rows = np.arange(len(bad))
    return np.allclose(dg[rows, got[bad]], dg[rows, ref[bad]], rtol=1e-12, atol=1e-30)


@pytest.mark.parametrize("res", [16, 32])
@pytest.mark.parametrize("name", list(MESHES))
def test_backward_matches_oracle(name, res):
    v, f = MESHES[name]()
    p = _points(res)
    diag = float(np.linalg.norm(p.max(0).astype(np.float64) - p.min(0)))
    sdf, face = _nearest(v, f, p)
    s = sdf.cpu().numpy().astype(np.float64)
    ref_sdf, _ = ms.mesh_sdf(v, f, p)
    keep = _unambiguous(v, f, p, diag) & (np.abs(ref_sdf) >= 1e-6 * diag)
    assert keep.sum() >= len(p) // 4, keep.sum()
    g = np.random.default_rng(7).standard_normal(len(p)).astype(np.float32).astype(np.float64) * keep
    # the oracle's sign is the winding number, the kernel's the ray parity (they differ on open meshes): the oracle
    # gets g s_kernel s_oracle so that both compute g s_kernel u
    g_or = g * np.sign(s) * np.sign(ref_sdf)
    ref = gr.mesh_sdf_grad(v, f, p, g_or)
    gv, gp = _backward(v, f, p, face, sdf, g.astype(np.float32))
    gp, gv = gp.cpu().numpy().astype(np.float64), gv.cpu().numpy().astype(np.float64)
    assert np.abs(gp - ref["grad_points"]).max() <= 1e-6, np.abs(gp - ref["grad_points"]).max()
    rel = np.linalg.norm(gv - ref["grad_verts"]) / np.linalg.norm(ref["grad_verts"])
    assert rel <= 1e-6, rel
    assert not gv[np.setdiff1d(np.arange(len(v)), f[face.cpu().numpy()[keep]].reshape(-1))].any()


@pytest.mark.parametrize("name", list(MESHES))
def test_backward_identities(name):
    """sum_V grad_verts + sum_P grad_points = 0 (translation) and sum v . grad_verts + sum p . grad_points = sum g sdf
    (homogeneity of degree 1), at every point, for a random upstream gradient."""
    v, f = MESHES[name]()
    p = _points(32)
    sdf, face = _nearest(v, f, p)
    g = np.random.default_rng(11).standard_normal(len(p)).astype(np.float32)
    gv, gp = _backward(v, f, p, face, sdf, g)
    gv, gp = gv.cpu().double(), gp.cpu().double()
    tv, tp = torch.from_numpy(v).double(), torch.from_numpy(p).double()
    mag = float(np.abs(g).sum())
    eps = 2.0 ** -24
    assert float((gv.sum(0) + gp.sum(0)).abs().max()) <= 8 * eps * mag
    scale = float(np.abs(p).max())
    euler = float((tv * gv).sum() + (tp * gp).sum())
    assert abs(euler - float((g.astype(np.float64) * sdf.cpu().double().numpy()).sum())) <= 16 * eps * mag * scale


@pytest.mark.parametrize("name", ["ico7", "ico8", "torus"])
def test_bvh_equals_brute_force_bitwise(name):
    v, f = ms.icosphere(int(name[3:]), 0.6) if name.startswith("ico") else ms.torus(nu=384, nv=192)
    p = _points(64)
    g = np.random.default_rng(3).standard_normal(len(p)).astype(np.float32)
    sdf, face = _nearest(v, f, p)
    sdf_b, face_b = _nearest(v, f, p, brute_force=True)
    assert torch.equal(sdf, sdf_b) and torch.equal(face, face_b), int((face != face_b).sum())
    gv, gp = _backward(v, f, p, face, sdf, g)
    gv_b, gp_b = _backward(v, f, p, face_b, sdf_b, g)
    assert torch.equal(gv, gv_b) and torch.equal(gp, gp_b)
    gv2, gp2 = _backward(v, f, p, face, sdf, g)                # run to run
    assert torch.equal(gv, gv2) and torch.equal(gp, gp2)
    assert bool(gv.abs().sum() > 0) and bool(gp.abs().sum() > 0)


@pytest.mark.parametrize("name", ["ico4", "torus", "lshape", "shell", "degenerate"])
def test_flipped_faces_bitwise_and_soup_sums(name):
    v, f = MESHES[name]()
    p = _points(32)
    g = np.random.default_rng(5).standard_normal(len(p)).astype(np.float32)
    sdf, face = _nearest(v, f, p)
    gv, gp = _backward(v, f, p, face, sdf, g)
    fl = f[:, ::-1].copy()
    sdf_f, face_f = _nearest(v, fl, p)
    assert torch.equal(sdf, sdf_f) and torch.equal(face, face_f)
    gv_f, gp_f = _backward(v, fl, p, face_f, sdf_f, g)
    assert torch.equal(gv, gv_f) and torch.equal(gp, gp_f)
    # triangle soup: every corner its own vertex; summed over the copies of a vertex, the indexed mesh's gradient
    sv, sf = v[f].reshape(-1, 3), np.arange(3 * len(f), dtype=np.int64).reshape(-1, 3)
    sdf_s, face_s = _nearest(sv, sf, p)
    assert torch.equal(sdf, sdf_s)
    gv_s, gp_s = _backward(sv, sf, p, face_s, sdf_s, g)
    assert torch.equal(gp, gp_s)
    summed = torch.zeros_like(gv, dtype=torch.float64).index_add_(0, _t(f.reshape(-1)), gv_s.double())
    err = float((summed - gv.double()).norm() / gv.double().norm())
    assert err <= 1e-6, err


def _flags():
    return types.SimpleNamespace(mode_num=8, order=1, mat="Steel", out_dir="/tmp", without_tensorboard=True)


def test_apply_sdf_mesh_without_grad_equals_path(tmp_path):
    from diffsound_b200.dmtet.geometry.dmtet_thickness import DMTetGeometry
    from diffsound_b200.diffelastic.mesh import read_obj
    v, f = ms.icosphere(4, 0.6)
    path = tmp_path / "sphere.obj"
    ms.write_obj(str(path), v, f)
    rv, rf = read_obj(str(path))
    a = DMTetGeometry(32, 1.5, _flags(), grid=_grid(32))
    a.apply_sdf(str(path))
    b = DMTetGeometry(32, 1.5, _flags(), grid=_grid(32))
    b.apply_sdf((_t(rv), _t(rf)))
    assert torch.equal(a.sdf, b.sdf) and not b.sdf.requires_grad
    assert torch.equal(a.marching_tets.max_thickness, b.marching_tets.max_thickness)
    assert b._sdf_mesh is None


def test_apply_sdf_mesh_gradient_is_the_backward_of_the_sdf_gradient():
    from diffsound_b200 import native
    from diffsound_b200.dmtet.geometry.dmtet_thickness import DMTetGeometry
    v, f = ms.icosphere(3, 0.6)
    geo = DMTetGeometry(32, 1.5, _flags(), grid=_grid(32))
    tv = _t(v).requires_grad_(True)
    tf = _t(f)
    geo.apply_sdf((tv, tf))
    target = geo.get_eigenvalues(thickness_coef=0.8)
    for it in range(2):                 # each tick samples the mesh again and builds a fresh graph
        tv.grad = None
        loss = geo.tick(target, it, _flags())
        geo.sdf.retain_grad()
        loss.backward()
        g_sdf = geo.sdf.grad
        assert g_sdf is not None and bool(g_sdf.abs().sum() > 0)
        sdf, face = native.mesh_sdf_nearest(tv.detach(), tf, geo.verts.contiguous())
        assert torch.equal(sdf, geo.sdf.detach())
        gv, _ = native.mesh_sdf_backward(tv.detach(), tf, geo.verts.contiguous(), face, sdf, g_sdf.contiguous(),
                                         want_points=False)
        assert torch.equal(tv.grad, gv)


def test_end_to_end_mesh_gradient_matches_central_differences(monkeypatch):
    """d loss / d t of one thickness-loop step along (a) a uniform scaling of the mesh, (b) a seeded smooth field, against
    central differences of the same loss evaluated from the solver's fp64 eigenvalues."""
    from diffsound_b200.diffelastic.diff_model import DiffSoundObj
    from diffsound_b200.dmtet.geometry.dmtet_thickness import DMTetGeometry
    # residual tolerance 1e-6 (default 1e-5): eigenvalue errors ~1e-12 relative, far below the differences taken here
    # (1e-8 is beyond what the solver reaches on these meshes: Rayleigh-Ritz breakdown)
    monkeypatch.setattr(DiffSoundObj, "eig_tol", 1e-6)
    v, f = ms.icosphere(3, 0.6)
    v64 = v.astype(np.float64)
    coef = 0.8
    geo = DMTetGeometry(32, 1.5, _flags(), grid=_grid(32))
    geo.marching_tets.thickness_coef = lambda: torch.tensor(coef, device=DEV)
    with torch.no_grad():
        geo.apply_sdf((_t(v), _t(f)))
        target = geo.get_eigenvalues() * 1.05
    gpts = geo.verts.detach().cpu().numpy()
    rng = np.random.default_rng(17)
    a, ph = rng.standard_normal((3, 3)), rng.uniform(0, 2 * np.pi, (3, 3))
    fields = {"scale": v64, "smooth": 0.3 * np.stack([np.sin(v64 @ a[k] * 3 + ph[k, 0]) for k in range(3)], 1)}

    def step(vv, grad=False):
        tv = _t(vv.astype(np.float32)).requires_grad_(grad)
        geo.apply_sdf((tv, _t(f)))
        obj = geo.getMesh()
        obj.eigen_decomposition()
        lam = obj.eigenvalues.detach().cpu().numpy()
        tets = obj.tetmesh.tets.cpu().numpy()
        g_sdf = None
        if grad:
            vals = obj.get_vals()
            loss = ((vals - target) ** 2 / target ** 2).mean()
            geo.sdf.retain_grad()
            loss.backward()
            g_sdf = geo.sdf.grad.cpu().double().numpy()
        return lam, tets, tv.grad, geo.sdf.detach().cpu().numpy().astype(np.float64), g_sdf

    lam0, tets0, grad0, s0, g_sdf = step(v64, grad=True)
    g0 = grad0.cpu().double().numpy()
    # get_vals() is the eigenvalues (fp32, with the shape gradient): the same loss from the solver's fp64 eigenvalues
    tgt = target.detach().cpu().numpy().astype(np.float64)[:, 0]
    loss64 = lambda lam: float((((lam - tgt) ** 2) / tgt ** 2).mean())
    thick = coef * s0.max()
    for fname, dv in fields.items():
        # rate of each grid value along dv (oracle weights), margin to 0 and to the thickness
        r = gr.mesh_sdf_grad(v64, f, gpts)
        rate = -np.einsum("pk,pkd,pd->p", r["bary"], dv[f[r["face"]]], r["grad_points"])
        rmax = np.abs(rate).max()
        margin = np.minimum(np.abs(s0), np.where(s0 > 0, np.abs(s0 - thick), np.inf))
        h = 0.25 * float((margin / (np.abs(rate) + coef * rmax + 1e-30)).min())
        vp, vm = (v64 + h * dv).astype(np.float32), (v64 - h * dv).astype(np.float32)
        hi = step(vp.astype(np.float64))
        lo = step(vm.astype(np.float64))
        assert np.array_equal(hi[1], tets0) and np.array_equal(lo[1], tets0), fname
        fd = (loss64(hi[0]) - loss64(lo[0])) / (2 * h)
        # along the perturbation the kernel sees (the vertices are rounded to fp32)
        an = float((g0 * (vp.astype(np.float64) - vm.astype(np.float64)) / (2 * h)).sum())
        # the sampled values at +-h are rounded to fp32 (half an ulp, 2^-24 |sdf| relative, each), carried to the loss
        # by d loss / d sdf; twice that for the fp32 edge interpolation after it
        tol = 2 * float((np.abs(g_sdf) * 2.0 ** -24 * np.abs(s0)).sum()) / h + 1e-5 * abs(an)
        print(f"{fname}: h {h:.3e} autograd {an:.9e} central {fd:.9e} rel {abs(fd - an) / abs(an):.2e} tol {tol:.2e}")
        assert abs(fd - an) <= tol, (fname, an, fd, tol)


def test_cabi_errors_leave_the_device_usable():
    import ctypes as C
    from diffsound_b200 import _lib, native
    lib = _lib.load()
    ws = native.workspace(DEV)
    v, f = ms.icosphere(2, 0.6)
    p = _points(16)
    tv, tf, tp = _t(v), _t(f), _t(p)
    out = torch.empty(len(p), dtype=torch.float32, device=DEV)
    face = torch.empty(len(p), dtype=torch.int32, device=DEV)
    g = torch.ones(len(p), dtype=torch.float32, device=DEV)
    gv = torch.empty(len(v), 3, dtype=torch.float32, device=DEV)
    gp = torch.empty(len(p), 3, dtype=torch.float32, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ptr = (lambda t: None if t is None else C.c_void_p(t.data_ptr()))

    def near(verts, faces, pts, fo=face, mode=0):
        return lib.ds_mesh_sdf_nearest(ws.handle, ptr(verts), len(v), ptr(faces), len(f), ptr(pts), len(p), mode, ptr(out),
                                       ptr(fo), st)

    def back(verts, faces, pts, fi):
        return lib.ds_mesh_sdf_backward(ws.handle, ptr(verts), len(v), ptr(faces), len(f), ptr(pts), len(p), ptr(fi),
                                        ptr(out), ptr(g), ptr(gv), ptr(gp), st)

    bad_f = tf.clone()
    bad_f[5, 1] = len(v)
    assert near(tv, bad_f, tp) == -2 and "face 5" in _lib.last_error()
    assert near(None, tf, tp) == -2 and "null" in _lib.last_error()
    assert near(tv, tf, tp, fo=None) == -2 and "null" in _lib.last_error()
    assert near(tv, tf, tp, mode=3) == -2 and "unknown mode" in _lib.last_error()
    nan_v = tv.clone()
    nan_v[3, 0] = float("nan")
    assert near(nan_v, tf, tp) == -2 and "vertex 3" in _lib.last_error()
    assert near(tv, tf, tp) == 0
    assert back(tv, bad_f, tp, face) == -2 and "face 5" in _lib.last_error()
    assert back(tv, tf, tp, None) == -2 and "null" in _lib.last_error()
    inf_p = tp.clone()
    inf_p[7, 2] = float("inf")
    assert back(tv, tf, inf_p, face) == -2 and "query point 7" in _lib.last_error()
    for bad in (len(f), -1):
        bad_face = face.clone()
        bad_face[9] = bad
        assert back(tv, tf, tp, bad_face) == -2 and "point 9 has nearest face" in _lib.last_error()
    torch.cuda.synchronize()
    s1, f1 = native.mesh_sdf_nearest(tv, tf, tp)
    s2, f2 = native.mesh_sdf_nearest(tv, tf, tp, brute_force=True)
    assert torch.equal(s1, s2) and torch.equal(f1, f2)
    a = native.mesh_sdf_backward(tv, tf, tp, f1, s1, g)
    b = native.mesh_sdf_backward(tv, tf, tp, f2, s2, g)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
