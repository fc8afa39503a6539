"""Modal gains on the device (csrc/gains.cu; native.tet_boundary / modal_gains / modal_gains_backward;
DiffSoundObj.surface / modal_gains / impulse_response) against the fp64 oracle (oracle/modal_gains.py) and closed forms.

Bars: boundary faces, owners and local faces equal to the oracle's, in the same order, also after shuffling the tets and
rotating their corners, and bitwise reproducible; gains within 2e-6 of max |g| of the oracle's at orders 1 and 2, with
the same value from every face that shares an edge or a vertex; an affine displacement field interpolated exactly; the
rigid-body closed form to 1e-5; the free-free beam's first bending mode (end / centre gain -1.6452, nodal line at
0.2242 L) to 2 %; the backward against central differences of the oracle; impulse_response bitwise reciprocal and
sign-invariant, within 1e-4 (relative L2) of the fp64 formula, with alpha / beta gradients matching finite
differences; the strike point recovered from its sound; the C-ABI error paths."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import modal_gains as mg
import test_modal_gains_cpu as tc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _native():
    from diffsound_b200 import native
    return native


def _boundary(v, t, order):
    nat = _native()
    out = nat.tet_boundary(torch.tensor(v, dtype=torch.float32, device=DEV),
                           torch.tensor(np.ascontiguousarray(t), dtype=torch.int32, device=DEV), order)
    return tuple(x.cpu().numpy().astype(np.int64) for x in out)


def _assert_boundary_equal(v, t, order):
    got = _boundary(v, t, order)
    ref = mg.boundary_faces(v, t, order)
    for g, r in zip(got, ref):
        assert np.array_equal(g, r)
    return got


def _sphere_mesh(h=0.12):
    from diffsound_b200.diffelastic.tetrahedralize import tetrahedralize
    m = tetrahedralize(lambda p: 0.5 - p.norm(dim=1), edge_length=h, bounds=((-0.6,) * 3, (0.6,) * 3))
    return m.vertices.detach().cpu().numpy(), m.tets.cpu().numpy().astype(np.int64)


def test_boundary_equals_oracle(meshes):
    for name, (v, t) in meshes.items():
        _assert_boundary_equal(v, t, 1)
    v, t = tc.promote(*tc.kuhn_box((3, 2, 4), (1.0, 0.5, 0.8)), 2)
    got = _assert_boundary_equal(v, t, 2)
    for _ in range(2):                                    # bitwise run to run
        assert all(np.array_equal(a, b) for a, b in zip(got, _boundary(v, t, 2)))
    v, t = _sphere_mesh()
    got = _assert_boundary_equal(v, t, 1)
    tc.check_surface(v, got[0], tc.tet_volume(v, t))
    # tet order and corner rotation do not change the faces; owners / local faces follow the tets
    rng = np.random.default_rng(0)
    perm = rng.permutation(len(t))
    rot = t[perm][:, [1, 2, 0, 3]]
    got2 = _assert_boundary_equal(v, rot, 1)
    assert np.array_equal(got2[0], got[0])
    assert np.array_equal(perm[got2[1]], got[1])


def _obj(v, t, order, mode_num=8):
    from diffsound_b200.diffelastic.diff_model import DiffSoundObj
    from diffsound_b200.diffelastic.material_model import MatSet
    obj = DiffSoundObj(torch.tensor(v, device=DEV), torch.tensor(t, device=DEV), mode_num=mode_num, order=order,
                       mat=MatSet.Steel)
    obj.eigen_decomposition()
    return obj


def _kernel_gains(obj, pts, face, dirs=None, U=None):
    nat = _native()
    U = obj.U_hat if U is None else U
    p = torch.tensor(pts, dtype=torch.float32, device=DEV)
    f = torch.tensor(face, dtype=torch.int32, device=DEV)
    d = None if dirs is None else torch.tensor(dirs, dtype=torch.float32, device=DEV)
    g, cp = nat.modal_gains(obj._verts32, obj.deform.tets_i32, obj.tetmesh.order, obj._boundary(), p, f, d, U)
    return g.cpu().numpy().astype(np.float64), cp.cpu().numpy().astype(np.float64)


def _mesh_np(obj):
    return obj._verts32.cpu().numpy(), obj.tetmesh.tets.cpu().numpy(), tuple(x.cpu().numpy() for x in obj.surface())


def _test_points(v, faces, rng, n=40):
    """points near the surface, on it, on shared edges and on shared vertices"""
    vd = v.astype(np.float64)
    f = faces[rng.choice(len(faces), n)]
    a, b, c = vd[f[:, 0]], vd[f[:, 1]], vd[f[:, 2]]
    nrm = np.cross(b - a, c - a)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    L = rng.dirichlet(np.ones(3), n)
    on = L[:, :1] * a + L[:, 1:2] * b + L[:, 2:] * c
    near = on + 0.01 * rng.normal(size=(n, 1)) * nrm
    return {"near": near, "on": on, "edge": 0.5 * (a + b), "vertex": a}


@pytest.mark.parametrize("order", [1, 2])
def test_gains_match_oracle(order):
    v, t = tc.kuhn_box((3, 3, 2), (1.0, 0.8, 0.5))
    obj = _obj(v, t, order)
    pv, pt, bnd = _mesh_np(obj)
    U = obj.U_hat.cpu().numpy()
    rng = np.random.default_rng(order)
    for kind, pts in _test_points(pv, bnd[0], rng).items():
        g = obj.modal_gains(torch.tensor(pts, dtype=torch.float32, device=DEV)).detach().cpu().numpy()
        _, face = _native().mesh_sdf_nearest(obj._verts32, obj.surface()[0], torch.tensor(pts, dtype=torch.float32,
                                                                                             device=DEV))
        face = face.cpu().numpy()
        ref, xs, _ = mg.gains(pv, pt, order, bnd, pts.astype(np.float32), face, U)
        scale = np.abs(ref).max()
        assert np.abs(g - ref).max() <= 2e-6 * scale, kind
        assert np.allclose(obj.last_strike_points.cpu().numpy(), xs, atol=1e-6)
        if kind in ("edge", "vertex"):
            # the same value from every face that holds the point (a fixed direction: the normals differ)
            d = rng.normal(size=(len(pts), 3))
            g0, _ = _kernel_gains(obj, pts, face, d)
            for i, p in enumerate(pts.astype(np.float32)):
                for f in np.nonzero((bnd[0] == _vid(pv, p)).any(axis=1) if kind == "vertex" else
                                    _edge_faces(pv, bnd[0], p))[0]:
                    gi, _ = _kernel_gains(obj, p[None], [f], d[i:i + 1])
                    assert np.abs(gi[0] - g0[i]).max() <= 2e-6 * scale


def _vid(v, p):
    return int(np.argmin(np.abs(v - p).sum(axis=1)))


def _edge_faces(v, faces, p):
    """faces that hold point p (the midpoint of one of their edges)"""
    vd = v.astype(np.float64)
    mids = [0.5 * (vd[faces[:, i]] + vd[faces[:, (i + 1) % 3]]) for i in range(3)]
    return np.any([np.abs(m - p).max(axis=1) < 1e-6 for m in mids], axis=0)


@pytest.mark.parametrize("order", [1, 2])
def test_affine_field_exact(order):
    v, t = tc.promote(*tc.kuhn_box((3, 2, 2), (1.0, 0.7, 0.6)), order)
    rng = np.random.default_rng(3)
    A, b = rng.normal(size=(4, 3, 3)), rng.normal(size=(4, 3))
    U = np.einsum("kij,nj->nik", A, v.astype(np.float64)) + b.T[None]          # (n, 3, 4)
    Ut = torch.tensor(U.reshape(-1, 4), dtype=torch.float64, device=DEV)
    bnd = tuple(torch.tensor(x, dtype=torch.int32, device=DEV) for x in mg.boundary_faces(v, t, order))
    pts = _test_points(v, bnd[0].cpu().numpy(), rng)["near"]
    face = _native().mesh_sdf_nearest(torch.tensor(v, device=DEV), bnd[0].long(), torch.tensor(pts, dtype=torch.float32,
                                                                                                   device=DEV))[1]
    d = rng.normal(size=pts.shape)
    g, cp = _native().modal_gains(torch.tensor(v, device=DEV), torch.tensor(t, dtype=torch.int32, device=DEV), order, bnd,
                                  torch.tensor(pts, dtype=torch.float32, device=DEV), face,
                                  torch.tensor(d, dtype=torch.float32, device=DEV), Ut)
    x = cp.cpu().numpy().astype(np.float64)
    ref = np.einsum("pi,kij,pj->pk", d.astype(np.float32), A, x) + d.astype(np.float32) @ b.T
    assert np.abs(g.cpu().numpy() - ref).max() <= 1e-5 * np.abs(ref).max()


def _rigid_closed_form(v, t, rho, x, d):
    X = v.astype(np.float64)[t[:, :4]]
    vol = np.abs(np.einsum("ij,ij->i", X[:, 1] - X[:, 0], np.cross(X[:, 2] - X[:, 0], X[:, 3] - X[:, 0]))) / 6
    V = vol.sum()
    com = (vol[:, None] * X.mean(axis=1)).sum(axis=0) / V
    Y = X - com
    S = sum(vol[i] / 20 * (Y[i].T @ Y[i] + np.outer(Y[i].sum(0), Y[i].sum(0))) for i in range(len(vol)))
    I = rho * (np.trace(S) * np.eye(3) - S)
    rd = np.cross(x - com, d)
    return 1.0 / (rho * V) + np.einsum("pi,ij,pj->p", rd, np.linalg.inv(I), rd)


@pytest.mark.parametrize("order", [1, 2])
def test_rigid_body_closed_form(order):
    v, t = tc.kuhn_box((3, 2, 2), (1.0, 0.6, 0.4))
    obj = _obj(v, t, order, mode_num=4)
    pv, pt, bnd = _mesh_np(obj)
    rng = np.random.default_rng(4)
    pts = _test_points(pv, bnd[0], rng)["on"]
    d = rng.normal(size=pts.shape)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    face = _native().mesh_sdf_nearest(obj._verts32, obj.surface()[0], torch.tensor(pts, dtype=torch.float32, device=DEV))[1]
    g, cp = _kernel_gains(obj, pts, face.cpu().numpy(), d, U=obj.U_hat_full[:, :6])
    ref = _rigid_closed_form(v, t, obj.material_model.mat.density, cp, d.astype(np.float32).astype(np.float64))
    assert np.abs((g ** 2).sum(axis=1) / ref - 1).max() <= 1e-5


def test_beam_first_bending_mode():
    L, W, H = 1.0, 0.05, 0.025
    v, t = tc.kuhn_box((40, 4, 2), (L, W, H))
    obj = _obj(v, t, 2, mode_num=4)
    xs = np.array([0.0, 0.2242 * L, 0.5 * L])
    pts = np.stack([xs, np.full(3, W / 2), np.full(3, H)], axis=1)
    g = obj.modal_gains(torch.tensor(pts, dtype=torch.float32, device=DEV),
                        torch.tensor([[0.0, 0.0, 1.0]] * 3, device=DEV)).detach().cpu().numpy()
    m = int(np.argmax(np.abs(g[0])))
    assert m == 0, g                                      # the lowest mode bends in the thin direction
    ratio = g[0, m] / g[2, m]
    assert abs(ratio / -1.6452 - 1) <= 0.02, ratio
    assert abs(g[1, m]) <= 0.02 * abs(g[0, m])


@pytest.mark.parametrize("order", [1, 2])
def test_backward_matches_central_differences(order):
    v, t = tc.kuhn_box((2, 2, 2), (1.0, 0.8, 0.6))
    obj = _obj(v, t, order, mode_num=6)
    pv, pt, bnd = _mesh_np(obj)
    U = obj.U_hat.cpu().numpy()
    rng = np.random.default_rng(5)
    pts = _test_points(pv, bnd[0], rng, n=12)["near"].astype(np.float32)
    ptst = torch.tensor(pts, device=DEV)
    face = _native().mesh_sdf_nearest(obj._verts32, obj.surface()[0], ptst)[1]
    fn = face.cpu().numpy()
    up = rng.normal(size=(len(pts), 6)).astype(np.float32)
    for dirs in (None, rng.normal(size=pts.shape).astype(np.float32)):
        dt = None if dirs is None else torch.tensor(dirs, device=DEV)
        gp, gd = _native().modal_gains_backward(obj._verts32, obj.deform.tets_i32, order, obj._boundary(), ptst, face, dt,
                                                obj.U_hat, torch.tensor(up, device=DEV))
        gp = gp.cpu().numpy()
        h = 1e-5
        fd = np.zeros((len(pts), 3))
        for c in range(3):
            e = np.zeros(3)
            e[c] = h
            gplus = mg.gains(pv, pt, order, bnd, pts + e, fn, U, dirs)[0]
            gminus = mg.gains(pv, pt, order, bnd, pts - e, fn, U, dirs)[0]
            fd[:, c] = ((gplus - gminus) * up).sum(axis=1) / (2 * h)
        assert np.abs(gp - fd).max() <= 1e-4 * np.abs(fd).max()
        _, _, regions = mg.gains(pv, pt, order, bnd, pts, fn, U)
        for i, r in enumerate(regions):
            if r == "face":
                a, b, c = pv[bnd[0][fn[i]]].astype(np.float64)
                n = np.cross(b - a, c - a)
                assert abs(gp[i] @ n) <= 1e-5 * np.linalg.norm(gp[i]) * np.linalg.norm(n) + 1e-30
        if dirs is not None:
            gd = gd.cpu().numpy()
            for c in range(3):
                e = np.zeros_like(dirs)
                e[:, c] = 1
                gc, _ = _kernel_gains(obj, pts, fn, e)
                assert np.abs(gd[:, c] - (gc * up).sum(axis=1)).max() <= 1e-5 * np.abs(gd).max()


def _fp64_response(obj, gs, gp, T, sr, alpha, beta, round32=False):
    """the formula in fp64; round32: from the fp32 damping and frequency the synth kernel is given"""
    lam = obj.eigenvalues.cpu().numpy()
    c = 0.5 * (alpha + beta * lam)
    w = np.sqrt(lam - c * c)
    if round32:
        c = c.astype(np.float32).astype(np.float64)
        w = 2 * np.pi * (w / (2 * np.pi)).astype(np.float32).astype(np.float64)
    tt = (np.arange(T) + 1) / sr                          # the synth's sample times
    amp = gs * gp / w
    return np.einsum("pk,kt->pt", amp, np.exp(-np.outer(c, tt)) * np.sin(np.outer(w, tt)))


def test_impulse_response():
    v, t = tc.kuhn_box((3, 2, 2), (0.3, 0.2, 0.15))
    obj = _obj(v, t, 2, mode_num=8)
    rng = np.random.default_rng(6)
    pv, _, bnd = _mesh_np(obj)
    s = torch.tensor(_test_points(pv, bnd[0], rng, 3)["on"], dtype=torch.float32, device=DEV)
    p = torch.tensor(_test_points(pv, bnd[0], rng, 3)["on"], dtype=torch.float32, device=DEV)
    T, sr = 4000, 44100.0
    y = obj.impulse_response(s, T, sr, pickup=p)
    assert torch.equal(y, obj.impulse_response(p, T, sr, pickup=s))
    gs = obj.modal_gains(s).detach().cpu().numpy().astype(np.float64)
    gp = obj.modal_gains(p).detach().cpu().numpy().astype(np.float64)
    mat = obj.material_model.mat
    ref = _fp64_response(obj, gs, gp, T, sr, mat.alpha, mat.beta, round32=True)
    assert np.linalg.norm(y.cpu().numpy() - ref) <= 1e-4 * np.linalg.norm(ref)
    # the sign of each eigenvector does not matter
    obj._X.neg_()
    try:
        assert torch.equal(y, obj.impulse_response(s, T, sr, pickup=p))
    finally:
        obj._X.neg_()
    # alpha / beta gradients
    a = torch.tensor(float(mat.alpha), dtype=torch.float64, device=DEV, requires_grad=True)
    b = torch.tensor(float(mat.beta), dtype=torch.float64, device=DEV, requires_grad=True)
    w = torch.tensor(rng.normal(size=(3, T)), dtype=torch.float32, device=DEV)
    (obj.impulse_response(s, T, sr, pickup=p, alpha=a, beta=b) * w).sum().backward()
    wn = w.cpu().numpy()
    for var, base, grad in ((0, mat.alpha, a.grad), (1, mat.beta, b.grad)):
        h = 1e-3 * base
        args = [mat.alpha, mat.beta]
        args[var] = base + h
        plus = (_fp64_response(obj, gs, gp, T, sr, *args) * wn).sum()
        args[var] = base - h
        minus = (_fp64_response(obj, gs, gp, T, sr, *args) * wn).sum()
        fd = (plus - minus) / (2 * h)
        assert abs(float(grad) - fd) <= 1e-3 * abs(fd), (var, float(grad), fd)


def _l_block():
    """an L-shaped Kuhn block with unequal arms (no in-plane symmetry): a 12 x 9 x 2 grid of cells of size h = 1/12 over
    1 x 0.75 x 1/6 with the corner x > 0.5, y > 0.375 removed"""
    h = 1.0 / 12
    v, t = tc.kuhn_box((12, 9, 2), (1.0, 0.75, 2 * h))
    c = v[t].mean(axis=1)
    t = t[~((c[:, 0] > 0.5) & (c[:, 1] > 0.375))]
    used, t = np.unique(t, return_inverse=True)
    return v[used], t.reshape(-1, 4), h


def test_strike_point_recovery():
    # The hidden point and the start are on the top face, away from its mirror image through the mid-thickness plane.
    # Adam's second-moment memory is shortened (beta2 = 0.99) so that the large gradients of the first steps do not
    # stall the descent along the flat valley near the minimum.
    v, t, h = _l_block()
    H = 2 * h
    obj = _obj(v, t, 2, mode_num=16)
    T, sr = 4096, 44100.0
    x_true = torch.tensor([[0.3, 0.2, H]], device=DEV)
    target = obj.impulse_response(x_true, T, sr).detach()
    x_true = obj.last_strike_points.clone()
    x = torch.tensor([[0.3 + 1.6 * h, 0.2 + 1.2 * h, H]], device=DEV, requires_grad=True)     # 2 h away
    opt = torch.optim.Adam([x], lr=0.05 * h, betas=(0.9, 0.99))
    sched = torch.optim.lr_scheduler.ExponentialLR(opt, 0.99)
    scale = float((target ** 2).sum())
    for _ in range(200):
        opt.zero_grad()
        loss = ((obj.impulse_response(x, T, sr) - target) ** 2).sum() / scale
        loss.backward()
        opt.step()
        sched.step()
    with torch.no_grad():
        obj.modal_gains(x)
    x_found = obj.last_strike_points
    assert float((x_found - x_true).norm()) < 0.1 * h, (x_found, x_true, float(loss))


def test_cabi_error_paths():
    from diffsound_b200 import _lib
    lib = _lib.load()
    nat = _native()
    ws = nat.workspace(DEV).handle
    st = nat._stream()
    v, t = tc.kuhn_box((2, 1, 1))
    tv = torch.tensor(v, device=DEV)
    tt = torch.tensor(t, dtype=torch.int32, device=DEV)
    n = C.c_int64(0)
    p = nat._p
    cnt = lambda verts, tets, T, order: lib.ds_tet_boundary_count(ws, p(verts), verts.shape[0], p(tets) if tets is not None
                                                                   else None, T, order, C.byref(n), st)
    assert cnt(tv, tt, len(t), 3) == -2 and "order 3" in _lib.last_error()
    assert cnt(tv, None, len(t), 1) == -2 and "null" in _lib.last_error()
    assert cnt(tv, tt, 0, 1) == -2 and "empty" in _lib.last_error()
    bad = tt.clone()
    bad[3, 2] = 99
    assert cnt(tv, bad, len(t), 1) == -2 and "tet 3" in _lib.last_error()
    nanv = tv.clone()
    nanv[4, 0] = float("nan")
    assert cnt(nanv, tt, len(t), 1) == -2 and "node 4" in _lib.last_error()
    three = torch.cat([tt, tt[:1], tt[:1]])
    assert cnt(tv, three, len(three), 1) == -2 and "non-conforming" in _lib.last_error()
    assert lib.ds_tet_boundary_fill(ws, None, None, None, st) == -2
    bnd = nat.tet_boundary(tv, tt, 1)
    U = torch.randn(3 * len(v), 4, dtype=torch.float64, device=DEV)
    pts = tv[:5].clone()
    face = torch.zeros(5, dtype=torch.int32, device=DEV)
    gout = torch.empty(5, 4, device=DEV)
    cp = torch.empty(5, 3, device=DEV)
    gp = torch.empty(5, 3, device=DEV)

    def gains(fn, order=1, pts=pts, face=face, dirs=None, k=4, ldu=4, U=U, tets=tt):
        head = [ws, p(tv), tv.shape[0], p(tets) if tets is not None else None, len(t), order, p(bnd[0]), p(bnd[1]),
                p(bnd[2]), bnd[0].shape[0], p(pts), p(face), p(dirs), pts.shape[0], p(U) if U is not None else None, ldu, k]
        if fn == "fwd":
            return lib.ds_modal_gains(*head, p(gout), p(cp), st)
        return lib.ds_modal_gains_backward(*head, p(gout), p(gp), None, st)

    for fn in ("fwd", "bwd"):
        assert gains(fn) == 0
        assert gains(fn, order=0) == -2 and "order 0" in _lib.last_error()
        assert gains(fn, tets=None) == -2 and "null" in _lib.last_error()
        assert gains(fn, U=None) == -2 and "null" in _lib.last_error()
        assert gains(fn, k=0) == -2 and "mode block" in _lib.last_error()
        assert gains(fn, ldu=3) == -2 and "mode block" in _lib.last_error()
        f2 = face.clone()
        f2[2] = bnd[0].shape[0]
        assert gains(fn, face=f2) == -2 and "point 2" in _lib.last_error()
        f2[2] = -1
        assert gains(fn, face=f2) == -2 and "point 2" in _lib.last_error()
        p2 = pts.clone()
        p2[3, 1] = float("inf")
        assert gains(fn, pts=p2) == -2 and "point 3" in _lib.last_error()
        d2 = torch.ones(5, 3, device=DEV)
        d2[1, 2] = float("nan")
        assert gains(fn, dirs=d2) == -2 and "direction 1" in _lib.last_error()
