"""The fp64 modal-gains oracle (oracle/modal_gains.py) on its own: boundary extraction, shape functions and the point
gradient.  No GPU.

Bars: the boundary of Kuhn boxes and the golden meshes is a closed 2-manifold (Euler characteristic 2 where the body is
a ball), its area is the box surface, and sum_f area_f (n_f . e_x) centroid_f,x equals the volume (outward orientation);
P2 interpolation reproduces quadratics and P1 affine fields to rounding; the point gradient matches central differences
in the face, edge and vertex regions of the closest-point map."""
import itertools

import numpy as np
import pytest
import torch

from oracle import modal_gains as mg
from oracle import modal_oracle as mo


def kuhn_box(n, size=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0)):
    """Kuhn triangulation of an n[0] x n[1] x n[2] cell grid over the box origin + [0, size]: six tets per cell."""
    nx, ny, nz = n
    ax = [np.linspace(o, o + s, k + 1) for o, s, k in zip(origin, size, n)]
    gx, gy, gz = np.meshgrid(*ax, indexing="ij")
    verts = np.stack([gx, gy, gz], axis=-1).reshape(-1, 3).astype(np.float32)
    vid = lambda i, j, k: (i * (ny + 1) + j) * (nz + 1) + k
    ii, jj, kk = np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij")
    base = np.stack([ii, jj, kk], axis=-1).reshape(-1, 3)
    tets = []
    for perm in itertools.permutations(range(3)):
        p = base.copy()
        ids = [vid(*p.T)]
        for a in perm:
            p = p.copy()
            p[:, a] += 1
            ids.append(vid(*p.T))
        tets.append(np.stack(ids, axis=1))
    return verts, np.concatenate(tets).astype(np.int64)


def promote(verts, tets, order):
    pv, pt = mo.promote(torch.from_numpy(verts), torch.from_numpy(tets), order)
    return pv.numpy(), pt.numpy()


def tet_volume(verts, tets, order=1):
    X = verts.astype(np.float64)[tets[:, list(mg.CORNER_LOCAL[order])]]
    return np.abs(np.einsum("ij,ij->i", X[:, 1] - X[:, 0], np.cross(X[:, 2] - X[:, 0], X[:, 3] - X[:, 0]))).sum() / 6


def check_surface(verts, faces, volume, area=None, euler=2):
    v = verts.astype(np.float64)
    edges = np.sort(np.concatenate([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]]), axis=1)
    ue, cnt = np.unique(edges, axis=0, return_counts=True)
    assert (cnt == 2).all(), "boundary is not a closed 2-manifold"
    # every directed edge once: consistently oriented
    directed = np.concatenate([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]])
    assert len(np.unique(directed, axis=0)) == len(directed)
    if euler is not None:
        assert len(np.unique(faces)) - len(ue) + len(faces) == euler
    a, b, c = v[faces[:, 0]], v[faces[:, 1]], v[faces[:, 2]]
    cr = np.cross(b - a, c - a)
    areas = 0.5 * np.linalg.norm(cr, axis=1)
    if area is not None:
        assert abs(areas.sum() - area) <= 1e-6 * area          # fp32 vertices
    cent = (a + b + c) / 3
    flux = (0.5 * cr[:, 0] * cent[:, 0]).sum()
    assert abs(flux - volume) <= 1e-9 * volume, (flux, volume)


@pytest.mark.parametrize("order", [1, 2])
@pytest.mark.parametrize("n,size", [((3, 3, 3), (1.0, 1.0, 1.0)), ((5, 2, 3), (1.0, 0.3, 0.45)), ((1, 1, 1), (2.0, 1.0, 0.5))])
def test_boundary_kuhn_box(n, size, order):
    v, t = kuhn_box(n, size)
    pv, pt = promote(v, t, order)
    faces, owner, local = mg.boundary_faces(pv, pt, order)
    nx, ny, nz = n
    assert len(faces) == 4 * (nx * ny + ny * nz + nx * nz)
    sx, sy, sz = size
    assert abs(tet_volume(pv, pt, order) - sx * sy * sz) <= 1e-6 * sx * sy * sz
    check_surface(pv, faces, tet_volume(pv, pt, order), 2 * (sx * sy + sy * sz + sx * sz))
    # owner / local name the face: its corners are the owning tet's corners other than `local`
    cn = pt[:, list(mg.CORNER_LOCAL[order])]
    for f in range(len(faces)):
        assert sorted(faces[f]) == sorted(np.delete(cn[owner[f]], local[f]))


def test_boundary_golden(meshes):
    for name, (v, t) in meshes.items():
        faces, owner, local = mg.boundary_faces(v, t, 1)
        edges = np.unique(np.sort(np.concatenate([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]]), axis=1), axis=0)
        chi = len(np.unique(faces)) - len(edges) + len(faces)
        assert chi % 2 == 0 and chi <= 2, (name, chi)
        check_surface(v, faces, tet_volume(v, t), euler=None)


def test_boundary_rejects_nonconforming():
    v, t = kuhn_box((1, 1, 1))
    with pytest.raises(ValueError):
        mg.boundary_faces(v, np.concatenate([t, t[:1]]), 1)


def _p2_nodes(X):
    """physical positions of the 10 P2 nodes of the tet with corners X (4, 3)."""
    return np.array([X[l] if l == m else 0.5 * (X[l] + X[m]) for l, m in mg.P2_NODES])


def test_shape_functions_reproduce_polynomials():
    rng = np.random.default_rng(0)
    X = rng.normal(size=(4, 3))
    A, b, Q = rng.normal(size=3), rng.normal(), rng.normal(size=(3, 3))
    quad = lambda x: x @ Q @ x + A @ x + b
    aff = lambda x: A @ x + b
    nodes2 = _p2_nodes(X)
    for _ in range(20):
        L = rng.dirichlet(np.ones(4))
        x = L @ X
        assert abs(mg.shape_fn(L, 2) @ np.array([quad(p) for p in nodes2]) - quad(x)) < 1e-12 * (1 + abs(quad(x)))
        assert abs(mg.shape_fn(L, 1) @ np.array([aff(p) for p in X]) - aff(x)) < 1e-12 * (1 + abs(aff(x)))
        # partition of unity and the gradient of the interpolant of a quadratic
        assert abs(mg.shape_fn(L, 2).sum() - 1) < 1e-14
        dN = mg.shape_grad(L, 2) @ mg.barycentric_grad(X)
        grad = np.array([quad(p) for p in nodes2]) @ dN
        assert np.allclose(grad, (Q + Q.T) @ x + A, atol=1e-10)


def _region_points(verts, faces, f):
    """one query point per region of face f: above its centroid, beyond edge (0, 1), beyond corner 0."""
    v = verts.astype(np.float64)
    a, b, c = v[faces[f, 0]], v[faces[f, 1]], v[faces[f, 2]]
    n = np.cross(b - a, c - a)
    n /= np.linalg.norm(n)
    g = (a + b + c) / 3
    m = 0.5 * (a + b)
    out_e = m - g
    return {"face": g + 0.03 * n + 0.01 * (b - a),
            "edge": m + 0.4 * out_e + 0.02 * n + 0.1 * (b - a),
            "vertex": a + 0.3 * (a - g) + 0.02 * n}


@pytest.mark.parametrize("order", [1, 2])
def test_point_gradient_central_differences(order):
    v, t = kuhn_box((2, 2, 2))
    pv, pt = promote(v, t, order)
    bnd = mg.boundary_faces(pv, pt, order)
    rng = np.random.default_rng(1)
    U = rng.normal(size=(3 * len(pv), 5))
    up = rng.normal(size=(1, 5))
    for f in (0, 7, len(bnd[0]) - 1):
        for region, p in _region_points(pv, bnd[0], f).items():
            for dirs in (None, rng.normal(size=(1, 3))):
                _, _, reg = mg.gains(pv, pt, order, bnd, [p], [f], U, dirs)
                assert reg[0] == region
                gp, gd = mg.gains_grad(pv, pt, order, bnd, [p], [f], U, up, dirs)
                h = 1e-6
                fd = np.zeros(3)
                for c in range(3):
                    e = np.zeros(3)
                    e[c] = h
                    gplus = mg.gains(pv, pt, order, bnd, [p + e], [f], U, dirs)[0]
                    gminus = mg.gains(pv, pt, order, bnd, [p - e], [f], U, dirs)[0]
                    fd[c] = ((gplus - gminus) @ up[0])[0] / (2 * h)
                assert np.allclose(gp[0], fd, atol=1e-6 * (1 + np.abs(fd).max())), (region, gp[0], fd)
                if region == "vertex":
                    assert np.all(gp[0] == 0)
                if dirs is not None:
                    for c in range(3):
                        e = np.zeros((1, 3))
                        e[0, c] = 1.0
                        assert np.isclose(gd[0, c], mg.gains(pv, pt, order, bnd, [p], [f], U, e)[0][0] @ up[0])
