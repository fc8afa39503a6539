"""Modal gains of a tet mesh at surface points, in plain fp64 numpy: the definition csrc/gains.cu is tested against.

With mass-normalised mode shapes (U^T M U = I), a unit impulse at surface point x in direction d excites mode m with
gain g_m(x, d) = d . u_m(x), u_m(x) the P1 / P2 interpolation of column m of U at x.

- boundary_faces: the triangles of exactly one tet, found by counting sorted corner triples, in ascending triple order,
  oriented so that (b - a) x (c - a) points away from the owning tet's opposite corner.
- closest_point: Ericson's vertex / edge / face region analysis (Real-Time Collision Detection 5.1.5).
- shape_fn / shape_grad: P1 / P2 shape functions in the local node order of shape_func.P2_NODES, and dN/dL.
- gains / gains_grad: the gains at the closest point of a given boundary face, and their gradient to the query point
  (through the closest-point map: I - n n^T on the face, t t^T on an edge, 0 at a vertex) and to the direction.
"""
import numpy as np

P2_NODES = ((0, 0), (0, 1), (1, 1), (1, 2), (2, 2), (2, 0), (0, 3), (1, 3), (2, 3), (3, 3))
CORNER_LOCAL = {1: (0, 1, 2, 3), 2: (0, 2, 4, 9)}


def boundary_faces(verts, tets, order=1):
    """(faces (F, 3), owner (F,), local (F,)) int64; a face shared by more than two tets raises ValueError."""
    verts = np.asarray(verts, dtype=np.float64)
    corners = np.asarray(tets, dtype=np.int64)[:, list(CORNER_LOCAL[order])]
    T = corners.shape[0]
    faces, owner, local = [], [], []
    for f in range(4):
        faces.append(np.delete(corners, f, axis=1))
        owner.append(np.arange(T))
        local.append(np.full(T, f))
    tri = np.sort(np.concatenate(faces), axis=1)
    owner, local = np.concatenate(owner), np.concatenate(local)
    # stable lexicographic order of the sorted triples, ties by face index 4 t + f (== the kernel's stable LSD passes)
    fidx = 4 * owner + local
    o = np.lexsort((fidx, tri[:, 2], tri[:, 1], tri[:, 0]))
    tri, owner, local = tri[o], owner[o], local[o]
    _, inv, cnt = np.unique(tri, axis=0, return_inverse=True, return_counts=True)
    if cnt.max() > 2:
        raise ValueError("non-conforming mesh: a face is shared by more than two tets")
    keep = cnt[inv.reshape(-1)] == 1
    tri, owner, local = tri[keep].copy(), owner[keep], local[keep]
    a, b, c = verts[tri[:, 0]], verts[tri[:, 1]], verts[tri[:, 2]]
    s = verts[corners[owner, local]]
    det = np.einsum("ij,ij->i", np.cross(b - a, c - a), s - a)
    flip = det > 0
    tri[flip, 1], tri[flip, 2] = tri[flip, 2], tri[flip, 1].copy()
    return tri, owner, local


def closest_point(p, a, b, c):
    """(closest point, barycentric weights on (a, b, c), region 'vertex' | 'edge' | 'face') of triangle abc to p."""
    p, a, b, c = (np.asarray(x, dtype=np.float64) for x in (p, a, b, c))
    ab, ac, ap = b - a, c - a, p - a
    d1, d2 = ab @ ap, ac @ ap
    if d1 <= 0 and d2 <= 0:
        return a, np.array([1.0, 0, 0]), "vertex"
    bp = p - b
    d3, d4 = ab @ bp, ac @ bp
    if d3 >= 0 and d4 <= d3:
        return b, np.array([0, 1.0, 0]), "vertex"
    vc = d1 * d4 - d3 * d2
    if vc <= 0 and d1 >= 0 and d3 <= 0:
        t = d1 / (d1 - d3)
        return a + t * ab, np.array([1 - t, t, 0]), "edge"
    cp = p - c
    d5, d6 = ab @ cp, ac @ cp
    if d6 >= 0 and d5 <= d6:
        return c, np.array([0, 0, 1.0]), "vertex"
    vb = d5 * d2 - d1 * d6
    if vb <= 0 and d2 >= 0 and d6 <= 0:
        t = d2 / (d2 - d6)
        return a + t * ac, np.array([1 - t, 0, t]), "edge"
    va = d3 * d6 - d5 * d4
    if va <= 0 and d4 - d3 >= 0 and d5 - d6 >= 0:
        t = (d4 - d3) / ((d4 - d3) + (d5 - d6))
        return b + t * (c - b), np.array([0, 1 - t, t]), "edge"
    den = va + vb + vc
    v, w = vb / den, vc / den
    return a + v * ab + w * ac, np.array([1 - v - w, v, w]), "face"


def shape_fn(L, order):
    """N_a(L) for one point: (4,) or (10,)."""
    L = np.asarray(L, dtype=np.float64)
    if order == 1:
        return L.copy()
    return np.array([L[l] * (2 * L[l] - 1) if l == m else 4 * L[l] * L[m] for l, m in P2_NODES])


def shape_grad(L, order):
    """dN_a / dL_l for one point: (npe, 4)."""
    L = np.asarray(L, dtype=np.float64)
    if order == 1:
        return np.eye(4)
    out = np.zeros((10, 4))
    for a, (l, m) in enumerate(P2_NODES):
        if l == m:
            out[a, l] = 4 * L[l] - 1
        else:
            out[a, l] += 4 * L[m]
            out[a, m] += 4 * L[l]
    return out


def barycentric_grad(X):
    """grad_x L_j (4, 3) of the tet with corners X (4, 3)."""
    J = (X[1:] - X[0]).T
    Ji = np.linalg.inv(J)
    return np.vstack([-Ji.sum(axis=0), Ji])


def _point(verts, tets, order, bnd, p, f):
    faces, owner, local = bnd
    tri = faces[f]
    A, B, C = verts[tri[0]], verts[tri[1]], verts[tri[2]]
    x, w, region = closest_point(p, A, B, C)
    t = owner[f]
    cn = tets[t, list(CORNER_LOCAL[order])]
    L = np.zeros(4)
    for j in range(4):
        if j != local[f]:
            L[j] = w[list(tri).index(cn[j])]
    n = np.cross(B - A, C - A)
    n = n / np.linalg.norm(n)
    if region == "face":
        P = np.eye(3) - np.outer(n, n)
    elif region == "edge":
        k = [i for i in range(3) if w[i] != 0]
        e = verts[tri[k[1]]] - verts[tri[k[0]]]
        e = e / np.linalg.norm(e)
        P = np.outer(e, e)
    else:
        P = np.zeros((3, 3))
    return x, L, n, P, tets[t], verts[cn], region


def gains(verts, tets, order, bnd, points, face, U, dirs=None):
    """(g (P, k), closest points (P, 3), regions) in fp64."""
    verts = np.asarray(verts, dtype=np.float64)
    tets = np.asarray(tets, dtype=np.int64)
    U = np.asarray(U, dtype=np.float64)
    P = len(points)
    g = np.zeros((P, U.shape[1]))
    xs = np.zeros((P, 3))
    regions = []
    for i in range(P):
        x, L, n, _, nodes, _, region = _point(verts, tets, order, bnd, np.asarray(points[i], np.float64), face[i])
        d = n if dirs is None else np.asarray(dirs[i], np.float64)
        N = shape_fn(L, order)
        u = U.reshape(-1, 3, U.shape[1])[nodes]                   # (npe, 3, k)
        g[i] = np.einsum("a,c,ack->k", N, d, u)
        xs[i] = x
        regions.append(region)
    return g, xs, regions


def gains_grad(verts, tets, order, bnd, points, face, U, up, dirs=None):
    """(grad_points (P, 3), grad_dirs (P, 3)) of sum(up * gains) in fp64."""
    verts = np.asarray(verts, dtype=np.float64)
    tets = np.asarray(tets, dtype=np.int64)
    U = np.asarray(U, dtype=np.float64)
    P = len(points)
    gp, gd = np.zeros((P, 3)), np.zeros((P, 3))
    for i in range(P):
        x, L, n, Pj, nodes, X, _ = _point(verts, tets, order, bnd, np.asarray(points[i], np.float64), face[i])
        d = n if dirs is None else np.asarray(dirs[i], np.float64)
        u = U.reshape(-1, 3, U.shape[1])[nodes]                   # (npe, 3, k)
        dN = shape_grad(L, order) @ barycentric_grad(X)           # (npe, 3) physical gradients
        s = np.einsum("c,ack,k->a", d, u, up[i])
        gp[i] = Pj @ (s @ dN)
        gd[i] = np.einsum("a,ack,k->c", shape_fn(L, order), u, up[i])
    return gp, gd
