"""Generalised winding number of a triangle mesh on the device and the signed distance signed by it (csrc/sdf.cu:
ds_mesh_winding_number, ds_mesh_sdf_winding; native.mesh_winding_number, mesh_sdf(..., sign="winding");
dmtet/geometry/mesh_sdf.py; DMTetGeometry.apply_sdf(..., sign="winding")) against the fp64 numpy oracle
(oracle/mesh_sdf.py: winding_number, the exact sum of the Van Oosterom-Strackee solid angles).

Meshes: those of test_mesh_sdf_gpu.py, plus an icosphere with a cap of faces removed (open), two overlapping icospheres
(self-intersecting), an inverted icosphere and an unshared-vertex soup.  Points within 1e-6 of the bounding-box diagonal
from the surface are left out wherever w is compared.  Bars: exact mode within 2e-6 of the oracle, BVH mode within 0.05;
both modes bitwise reproducible, bitwise -w for flipped faces and bitwise equal for the soup; |sdf| and the nearest face
bitwise those of ds_mesh_sdf_nearest, and the whole sdf bitwise that of ds_mesh_sdf on closed, consistently oriented
meshes."""
import functools
import types

import numpy as np
import pytest
import torch

from oracle import mesh_sdf as ms
import mesh_sdf_grad_ref as gr
import test_mesh_sdf_gpu as base
import test_mesh_sdf_grad_gpu as tg

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
_t = base._t


def _holed():
    v, f = ms.icosphere(3, 0.6)
    return v, f[v[f].mean(1)[:, 2] < 0.3]          # the cap above z = 0.3 removed: a hole of radius about 0.5


def _overlap():
    return base._concat(ms.icosphere(3, 0.4, (-0.15, 0.0, 0.0)), ms.icosphere(3, 0.4, (0.2, 0.05, 0.0)))


def _inverted():
    v, f = ms.icosphere(3, 0.6)
    return v, f[:, ::-1].copy()


def _soup():
    v, f = ms.torus()
    return v[f].reshape(-1, 3), np.arange(3 * len(f), dtype=np.int64).reshape(-1, 3)


MESHES = dict(base.MESHES, holed=_holed, overlap=_overlap, inverted=_inverted, soup=_soup)
NEW = ("holed", "overlap")
CLOSED = ("ico3", "ico4", "ico5", "torus", "lshape", "two_spheres", "shell", "inverted", "soup")


@functools.lru_cache(maxsize=None)
def _mesh(name):
    return MESHES[name]()


@functools.lru_cache(maxsize=None)
def _pts(kind):
    if kind == "random":
        return np.random.default_rng(20261020).uniform(-0.9, 0.9, (1000, 3)).astype(np.float32)
    return base._points(int(kind))


@functools.lru_cache(maxsize=None)
def _oracle(name, kind):
    """(distance fp64, exact winding number fp64, mask of points at least 1e-6 diag from the surface)."""
    v, f = _mesh(name)
    p = _pts(kind)
    sdf, w = ms.mesh_sdf(v, f, p)
    diag = float(np.linalg.norm(p.max(0).astype(np.float64) - p.min(0)))
    return np.abs(sdf), w, np.abs(sdf) >= 1e-6 * diag


def _wn(v, f, p, brute_force=False):
    from diffsound_b200 import native
    return native.mesh_winding_number(_t(v), _t(f), _t(p), brute_force=brute_force)


def _sdfw(v, f, p, brute_force=False):
    from diffsound_b200 import native
    return native.mesh_sdf_nearest(_t(v), _t(f), _t(p), brute_force=brute_force, sign="winding")


# the oracle is brute force in numpy: ico5 only at the 16 grid (see test_mesh_sdf_gpu.py)
CASES = [(n, k) for n in MESHES for k in ("16", "32", "random") if n != "ico5" or k == "16"]


@pytest.mark.parametrize("name,kind", CASES)
def test_winding_number_matches_oracle(name, kind):
    v, f = _mesh(name)
    p = _pts(kind)
    _, ref, far = _oracle(name, kind)
    exact = _wn(v, f, p, brute_force=True).cpu().numpy().astype(np.float64)
    bvh = _wn(v, f, p).cpu().numpy().astype(np.float64)
    e_exact = float(np.abs(exact - ref)[far].max())
    e_bvh = np.abs(bvh - ref)[far]
    print(f"{name} {kind}: exact max {e_exact:.3e}; bvh max {e_bvh.max():.3e} mean {e_bvh.mean():.3e}")
    assert e_exact <= 2e-6, e_exact
    assert e_bvh.max() <= 0.05, float(e_bvh.max())


@pytest.mark.parametrize("name", ["ico4", "torus", "shell", "degenerate", "holed", "overlap"])
def test_winding_number_is_reproducible_and_orientation_odd(name):
    v, f = _mesh(name)
    p = np.concatenate([_pts("32"), _pts("random")])
    for bf in (False, True):
        w = _wn(v, f, p, bf)
        assert torch.equal(w, _wn(v, f, p, bf))
        assert torch.equal(_wn(v, f[:, ::-1].copy(), p, bf), -w)
        soup = _wn(v[f].reshape(-1, 3), np.arange(3 * len(f), dtype=np.int64).reshape(-1, 3), p, bf)
        assert torch.equal(soup, w)


def _morton_order(cent):
    """face order of the BVH build for fp32 centroids (F, 3): k_morton_codes (fp32 box, 10 bits per axis) and a stable
    sort by code, restated in numpy."""
    lo, hi = cent.min(0), cent.max(0)
    ext = hi - lo
    t = np.clip(np.where(ext > 0, (cent - lo) / np.where(ext > 0, ext, np.float32(1)), np.float32(0)), 0, 1)
    q = (t.astype(np.float32) * np.float32(1023)).astype(np.uint32)
    code = np.zeros(len(cent), dtype=np.uint32)
    for d in range(3):
        v = q[:, d]
        v = (v | (v << 16)) & 0x030000FF
        v = (v | (v << 8)) & 0x0300F00F
        v = (v | (v << 4)) & 0x030C30C3
        v = (v | (v << 2)) & 0x09249249
        code |= v << (2 - d)
    return np.argsort(code, kind="stable")


def test_winding_number_is_orientation_odd_where_written_centroids_reorder_the_tree():
    """On this mesh the centroids summed in written corner order, (a + b + c) / 3 in fp32, round differently for flipped
    or rotated faces, enough to change the Morton order of the faces; the winding jobs build their tree from the sorted
    corners, so flipping gives bitwise -w and rotating the corners bitwise w in both modes."""
    v, f = ms.icosphere(7, 0.6)
    third = np.float32(1.0 / 3.0)
    written = lambda ff: (v[ff[:, 0]] + v[ff[:, 1]] + v[ff[:, 2]]) * third
    flipped, rotated = f[:, ::-1].copy(), f[:, [1, 2, 0]].copy()
    base_order = _morton_order(written(f))
    assert not np.array_equal(_morton_order(written(flipped)), base_order)
    assert not np.array_equal(_morton_order(written(rotated)), base_order)
    p = _pts("32")
    for bf in (False, True):
        w = _wn(v, f, p, bf)
        assert torch.equal(_wn(v, flipped, p, bf), -w)
        assert torch.equal(_wn(v, rotated, p, bf), w)
        assert (w > 0.5).any() and (w < 0.5).any()


@pytest.mark.parametrize("name", list(MESHES))
def test_sdf_winding_distances_and_faces_are_those_of_mesh_sdf(name):
    from diffsound_b200 import native
    v, f = _mesh(name)
    p = _pts("32")
    tv, tf, tp = _t(v), _t(f), _t(p)
    for bf in (False, True):
        plain = native.mesh_sdf(tv, tf, tp, brute_force=bf)
        _, face = native.mesh_sdf_nearest(tv, tf, tp, brute_force=bf)
        sdf, face_w = _sdfw(v, f, p, bf)
        assert torch.equal(sdf.abs(), plain.abs())
        assert torch.equal(face_w, face)
        assert torch.equal(native.mesh_sdf(tv, tf, tp, brute_force=bf, sign="winding"), sdf)     # face_out NULL
        assert not bool((sdf == 0).logical_and(torch.signbit(sdf)).any())                        # +0 on the surface
        if name in CLOSED:
            assert torch.equal(sdf, plain)


@pytest.mark.parametrize("kind", ["16", "32", "random"])
@pytest.mark.parametrize("name", NEW)
def test_winding_sign_on_open_and_self_intersecting_meshes(name, kind):
    from diffsound_b200 import native
    v, f = _mesh(name)
    p = _pts(kind)
    _, w, far = _oracle(name, kind)
    rule = np.abs(w) >= 0.5
    parity = native.mesh_sdf(_t(v), _t(f), _t(p)).cpu().numpy() > 0
    for bf, margin in ((True, 1e-6), (False, 0.05)):
        got = _sdfw(v, f, p, bf)[0].cpu().numpy() > 0
        sel = far & (np.abs(np.abs(w) - 0.5) > margin)
        assert sel.sum() >= len(p) // 2
        bad = np.nonzero(got[sel] != rule[sel])[0]
        assert bad.size == 0, (bad.size, p[sel][bad[:5]], w[sel][bad[:5]])
        # the reason for the option: the ray parity gets some of these points wrong
        assert (parity[sel] != rule[sel]).sum() > 0


def test_winding_sign_gradient_matches_the_reference():
    """backward of mesh_sdf(..., sign="winding") on the self-intersecting mesh against mesh_sdf_grad_ref.py with the
    reference's sign replaced by the winding rule (tolerances of test_mesh_sdf_grad_gpu.py)."""
    from diffsound_b200.dmtet.geometry.mesh_sdf import mesh_sdf
    v, f = _mesh("overlap")
    p = _pts("32")
    diag = float(np.linalg.norm(p.max(0).astype(np.float64) - p.min(0)))
    ref_sdf, w = ms.mesh_sdf(v, f, p)
    s_rule = np.where(np.abs(w) >= 0.5, 1.0, -1.0)
    keep = tg._unambiguous(v, f, p, diag) & (np.abs(ref_sdf) >= 1e-6 * diag)
    assert keep.sum() >= len(p) // 4 and (s_rule[keep] != np.sign(ref_sdf[keep])).any()
    g = np.random.default_rng(7).standard_normal(len(p)).astype(np.float32).astype(np.float64) * keep
    ref = gr.mesh_sdf_grad(v, f, p, g * s_rule * np.sign(ref_sdf))      # the reference then computes g s_rule u
    tv, tp = _t(v).requires_grad_(True), _t(p).requires_grad_(True)
    sdf = mesh_sdf(tv, _t(f), tp, sign="winding")
    assert np.array_equal(np.sign(sdf.detach().cpu().numpy()[keep]), s_rule[keep])
    (sdf * _t(g.astype(np.float32))).sum().backward()
    gp, gv = tp.grad.cpu().numpy().astype(np.float64), tv.grad.cpu().numpy().astype(np.float64)
    assert np.abs(gp - ref["grad_points"]).max() <= 1e-6, np.abs(gp - ref["grad_points"]).max()
    rel = np.linalg.norm(gv - ref["grad_verts"]) / np.linalg.norm(ref["grad_verts"])
    assert rel <= 1e-6, rel


def _flags():
    return types.SimpleNamespace(mode_num=8, order=1, mat="Steel", out_dir="/tmp", without_tensorboard=True)


def test_apply_sdf_winding_end_to_end(tmp_path):
    from diffsound_b200 import native
    from diffsound_b200.diffelastic.mesh import read_obj
    from diffsound_b200.dmtet.geometry.dmtet_thickness import DMTetGeometry
    v, f = _holed()
    path = tmp_path / "holed.obj"
    ms.write_obj(str(path), v, f)
    rv, rf = read_obj(str(path))
    geo = DMTetGeometry(32, 1.5, _flags(), grid=base._grid(32))
    geo.apply_sdf(str(path), sign="winding")
    assert torch.equal(geo.sdf, native.mesh_sdf(_t(rv), _t(rf), geo.verts.contiguous(), sign="winding"))
    target = geo.get_eigenvalues(thickness_coef=1.0)
    loss = geo.tick(target, 0, _flags())
    loss.backward()
    grad = geo.marching_tets.thickness_coef.probablity.grad
    assert torch.isfinite(loss).item() and grad is not None and torch.isfinite(grad).all().item()
    # the mesh form with a gradient to the vertices: the sign is kept for the resampling of every getMesh()
    geo = DMTetGeometry(32, 1.5, _flags(), grid=base._grid(32))
    tv = _t(v).requires_grad_(True)
    geo.apply_sdf((tv, _t(f)), sign="winding")
    target = geo.get_eigenvalues(thickness_coef=0.8) * 1.05
    loss = geo.tick(target, 0, _flags())
    assert torch.equal(geo.sdf.detach(), native.mesh_sdf(tv.detach(), _t(f), geo.verts.contiguous(), sign="winding"))
    loss.backward()
    assert tv.grad is not None and bool(torch.isfinite(tv.grad).all()) and bool(tv.grad.abs().sum() > 0)
    # sampled values carry no mesh to take a winding number of; an unknown sign is an error in every form
    with pytest.raises(ValueError):
        geo.apply_sdf(torch.zeros(geo.verts.shape[0], device=DEV), sign="winding")
    with pytest.raises(ValueError):
        geo.apply_sdf(lambda x: x[:, 0], sign="winding")
    for arg in (str(path), (_t(v), _t(f)), torch.zeros(geo.verts.shape[0], device=DEV)):
        with pytest.raises(ValueError):
            geo.apply_sdf(arg, sign="majority")


def test_cabi_errors_leave_the_device_usable():
    import ctypes as C
    from diffsound_b200 import _lib, native
    lib = _lib.load()
    ws = native.workspace(DEV)
    v, f = ms.icosphere(2, 0.6)
    p = _pts("16")
    tv, tf, tp = _t(v), _t(f), _t(p)
    out = torch.empty(len(p), dtype=torch.float32, device=DEV)
    face = torch.empty(len(p), dtype=torch.int32, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ptr = (lambda t: None if t is None else C.c_void_p(t.data_ptr()))

    def wn(verts, faces, pts, o=out, mode=0, V=len(v), F=len(f), P=len(p)):
        return lib.ds_mesh_winding_number(ws.handle, ptr(verts), V, ptr(faces), F, ptr(pts), P, mode, ptr(o), st)

    def sw(verts, faces, pts, o=out, mode=0, V=len(v), F=len(f), P=len(p)):
        return lib.ds_mesh_sdf_winding(ws.handle, ptr(verts), V, ptr(faces), F, ptr(pts), P, mode, ptr(o), ptr(face), st)

    bad_f = tf.clone()
    bad_f[5, 1] = len(v)
    neg_f = tf.clone()
    neg_f[5, 1] = -1
    nan_v = tv.clone()
    nan_v[3, 0] = float("nan")
    inf_p = tp.clone()
    inf_p[7, 2] = float("inf")
    for call in (wn, sw):
        for mode in (0, 1):
            assert call(tv, bad_f, tp, mode=mode) == -2 and "face 5" in _lib.last_error()
            assert call(tv, neg_f, tp, mode=mode) == -2 and "face 5" in _lib.last_error()
            assert call(nan_v, tf, tp, mode=mode) == -2 and "vertex 3" in _lib.last_error()
            assert call(tv, tf, inf_p, mode=mode) == -2 and "query point 7" in _lib.last_error()
        assert call(None, tf, tp) == -2 and "null" in _lib.last_error()
        assert call(tv, None, tp) == -2 and "null" in _lib.last_error()
        assert call(tv, tf, None) == -2 and "null" in _lib.last_error()
        assert call(tv, tf, tp, o=None) == -2 and "null" in _lib.last_error()
        assert call(tv, tf, tp, F=0) == -2 and "empty mesh" in _lib.last_error()
        assert call(tv, tf, tp, V=0) == -2 and "empty mesh" in _lib.last_error()
        assert call(tv, tf, tp, mode=3) == -2 and "unknown mode" in _lib.last_error()
        assert call(tv, tf, tp, P=0) == 0
    torch.cuda.synchronize()
    a, b = native.mesh_winding_number(tv, tf, tp), native.mesh_winding_number(tv, tf, tp, brute_force=True)
    assert float((a - b).abs().max()) <= 0.05
    s1, f1 = native.mesh_sdf_nearest(tv, tf, tp, sign="winding")
    s2, f2 = native.mesh_sdf_nearest(tv, tf, tp)
    assert torch.equal(s1, s2) and torch.equal(f1, f2)
    with pytest.raises(ValueError):
        native.mesh_sdf(tv, tf, tp, sign="odd")
