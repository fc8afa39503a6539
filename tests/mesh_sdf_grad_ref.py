"""fp64 numpy reference for the gradient of the triangle-mesh signed distance (ds_mesh_sdf_backward, csrc/sdf.cu), built on
the distance and sign of oracle/mesh_sdf.py.

Nearest face = first index at the minimum fp64 squared distance (point_triangle_d2); its closest point c and barycentric
weights b from the oracle's own case split (plane projection when the point projects inside the face, else the nearest
edge, the first of ab, bc, ca on ties; degenerate faces: their edges); d sdf / d p = s u and d sdf / d v_k = -s b_k u
with u = (p - c) / |p - c| and s the oracle's sign.  `dtype` = np.float64 keeps the inputs exact (finite differences);
the default rounds them to fp32 first, as the kernel sees them.
"""
import numpy as np

from oracle import mesh_sdf as ms


def mesh_sdf(verts, faces, points, dtype=np.float32, pairs_per_chunk=1 << 17):
    """signed distance fp64 (P,) as oracle/mesh_sdf.py's mesh_sdf (positive inside: odd rounded winding number), with
    the inputs rounded to `dtype` instead of always to fp32."""
    tris = np.asarray(verts, dtype=dtype)[np.asarray(faces)]
    pts = np.asarray(points, dtype=dtype)
    n = max(1, pairs_per_chunk // max(1, len(tris)))
    d = np.empty(len(pts))
    w = np.empty(len(pts))
    for s in range(0, len(pts), n):
        d[s:s + n] = np.sqrt(ms.point_triangle_d2(pts[s:s + n], tris).min(axis=1))
        w[s:s + n] = ms.winding_number(pts[s:s + n], tris)
    inside = np.rint(np.abs(w)).astype(np.int64) % 2 == 1
    return np.where(inside, d, -d)


def _edge_closest(p, a, b):
    """closest points (n, 3) of the segments [a, b] to p and their parameters t (n,) (a point when a == b)."""
    ab = b - a
    l2 = np.einsum("ij,ij->i", ab, ab)
    with np.errstate(invalid="ignore", divide="ignore"):
        t = np.where(l2 > 0, np.einsum("ij,ij->i", p - a, ab) / np.where(l2 > 0, l2, 1.0), 0.0)
    t = np.clip(t, 0.0, 1.0)
    return a + t[:, None] * ab, t


def closest_on_triangles(p, A, B, C):
    """closest point (n, 3) and barycentric weights (n, 3) on (A, B, C) of each row's triangle to p, fp64, by the case
    split of point_triangle_d2: plane projection when p projects inside the (non-degenerate) face, else the nearest
    edge (the first of ab, bc, ca on ties)."""
    p, A, B, C = (np.asarray(x, dtype=np.float64) for x in (p, A, B, C))
    n = np.cross(B - A, C - A)
    nn = np.einsum("ij,ij->i", n, n)

    def side(e, q):
        return np.einsum("ij,ij->i", np.cross(e, q), n) >= 0

    inside = side(B - A, p - A) & side(C - B, p - B) & side(A - C, p - C) & (nn > 0)
    nns = np.where(nn > 0, nn, 1.0)
    h = np.einsum("ij,ij->i", n, p - A) / nns
    cp = p - h[:, None] * n
    bary = np.stack([np.einsum("ij,ij->i", np.cross(C - B, cp - B), n), np.einsum("ij,ij->i", np.cross(A - C, cp - C), n),
                     np.einsum("ij,ij->i", np.cross(B - A, cp - A), n)], 1) / nns[:, None]
    cands = [_edge_closest(p, A, B), _edge_closest(p, B, C), _edge_closest(p, C, A)]
    d2 = np.stack([((p - c) ** 2).sum(1) for c, _ in cands], 1)
    k = np.argmin(d2, axis=1)
    rows = np.arange(len(p))
    ce = np.stack([c for c, _ in cands], 1)[rows, k]
    t = np.stack([t for _, t in cands], 1)[rows, k]
    we = np.zeros((len(p), 3))
    for e, (i, j) in enumerate(((0, 1), (1, 2), (2, 0))):
        m = k == e
        we[m, i] = 1.0 - t[m]
        we[m, j] = t[m]
    return np.where(inside[:, None], cp, ce), np.where(inside[:, None], bary, we)


def mesh_sdf_grad(verts, faces, points, grad=None, dtype=np.float32, pairs_per_chunk=1 << 17):
    """Nearest face, closest point, barycentric weights and the gradients of the signed distance, fp64, brute force.
    Returns a dict: sdf (P,), face (P,) (lowest index on ties), closest (P, 3), bary (P, 3) on the corners faces[face],
    grad_points (P, 3) = g s u and grad_verts (V, 3) = sum of -g s b_k u over the points (grad: upstream gradient (P,),
    default ones); both 0 where sdf == 0.  Inputs rounded to `dtype` first."""
    v = np.asarray(verts, dtype=dtype).astype(np.float64)
    f = np.asarray(faces, dtype=np.int64)
    p = np.asarray(points, dtype=dtype).astype(np.float64)
    g = np.ones(len(p)) if grad is None else np.asarray(grad, dtype=np.float64)
    tris = v[f]
    n = max(1, pairs_per_chunk // max(1, len(tris)))
    face = np.empty(len(p), dtype=np.int64)
    for s in range(0, len(p), n):
        face[s:s + n] = np.argmin(ms.point_triangle_d2(p[s:s + n], tris), axis=1)
    sdf = mesh_sdf(v, f, p, np.float64, pairs_per_chunk)
    c, b = closest_on_triangles(p, *(tris[face, k] for k in range(3)))
    r = p - c
    d = np.linalg.norm(r, axis=1)
    with np.errstate(invalid="ignore", divide="ignore"):
        gs = np.where((sdf != 0) & (d > 0), np.sign(sdf) * g / np.where(d > 0, d, 1.0), 0.0)
    gp = gs[:, None] * r
    gv = np.zeros_like(v)
    for k in range(3):
        np.add.at(gv, f[face, k], -b[:, k, None] * gp)
    return {"sdf": sdf, "face": face, "closest": c, "bary": b, "grad_points": gp, "grad_verts": gv}
