"""fp64 numpy restatement of the triangle-mesh signed distance (ds_mesh_sdf, csrc/sdf.cu), for the tests.

Distance: brute force over all faces; per face the distance to its plane when the point projects inside it, else to its
nearest edge (a different case split from the kernel's vertex / edge / face region analysis); degenerate faces (zero
cross product) as the union of their edges.
Sign: from the generalised winding number (sum of the Van Oosterom-Strackee solid angles / 4 pi) instead of the kernel's
ray parity, so that the two check each other on closed meshes: inside when the rounded winding number is odd (for an
outward-oriented closed mesh, w = 1 inside and 0 outside; the parity makes the test independent of face orientation and
counts a cavity bounded by a nested surface as outside, as ray parity does).

Also the test meshes: icospheres, a torus, unions of axis-aligned boxes (voxels), and OBJ writing.
"""
import numpy as np


def degenerate(tris):
    """faces whose fp64 cross product (B - A) x (C - A) is exactly zero: (F,) bool."""
    t = tris.astype(np.float64)
    n = np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0])
    return ~np.any(n != 0.0, axis=1)


def _faces(tris):
    t = tris.astype(np.float64)
    return [t[:, i, k][None] for i in range(3) for k in range(3)]      # ax ay az bx ... cz, each (1, F)


def _seg_d2(px, py, pz, ex, ey, ez):
    """squared distance from (px, py, pz) (relative to the segment start) to the segment [0, e]."""
    l2 = ex * ex + ey * ey + ez * ez
    with np.errstate(invalid="ignore", divide="ignore"):
        t = np.where(l2 > 0, (px * ex + py * ey + pz * ez) / np.where(l2 > 0, l2, 1.0), 0.0)
    np.clip(t, 0.0, 1.0, out=t)
    dx, dy, dz = px - t * ex, py - t * ey, pz - t * ez
    return dx * dx + dy * dy + dz * dz


def point_triangle_d2(p, tris):
    """squared distances (n, F) from points p (n, 3) to triangles tris (F, 3, 3), fp64: the distance to the face plane
    when the point projects inside the triangle, else the distance to the nearest edge (degenerate faces: their edges)."""
    p = p.astype(np.float64)
    px, py, pz = p[:, 0, None], p[:, 1, None], p[:, 2, None]
    ax, ay, az, bx, by, bz, cx, cy, cz = _faces(tris)
    abx, aby, abz, bcx, bcy, bcz, cax, cay, caz = bx - ax, by - ay, bz - az, cx - bx, cy - by, cz - bz, ax - cx, ay - cy, az - cz
    nx, ny, nz = aby * (cz - az) - abz * (cy - ay), abz * (cx - ax) - abx * (cz - az), abx * (cy - ay) - aby * (cx - ax)
    nn = nx * nx + ny * ny + nz * nz
    apx, apy, apz = px - ax, py - ay, pz - az
    bpx, bpy, bpz = px - bx, py - by, pz - bz
    cpx, cpy, cpz = px - cx, py - cy, pz - cz

    def side(ex, ey, ez, qx, qy, qz):        # ((e x q) . n) >= 0: q on the inner side of edge e
        return ((ey * qz - ez * qy) * nx + (ez * qx - ex * qz) * ny + (ex * qy - ey * qx) * nz) >= 0

    inside = side(abx, aby, abz, apx, apy, apz) & side(bcx, bcy, bcz, bpx, bpy, bpz) & side(cax, cay, caz, cpx, cpy, cpz)
    inside &= nn > 0
    with np.errstate(invalid="ignore", divide="ignore"):
        h = nx * apx + ny * apy + nz * apz
        plane = h * h / np.where(nn > 0, nn, 1.0)
    edges = np.minimum(np.minimum(_seg_d2(apx, apy, apz, abx, aby, abz), _seg_d2(bpx, bpy, bpz, bcx, bcy, bcz)),
                       _seg_d2(cpx, cpy, cpz, cax, cay, caz))
    return np.where(inside, plane, edges)


def winding_number(p, tris):
    """generalised winding number of the triangle soup at points p (n, 3): (n,) fp64."""
    p = p.astype(np.float64)
    px, py, pz = p[:, 0, None], p[:, 1, None], p[:, 2, None]
    ax, ay, az, bx, by, bz, cx, cy, cz = _faces(tris[~degenerate(tris)])
    ax, ay, az, bx, by, bz, cx, cy, cz = ax - px, ay - py, az - pz, bx - px, by - py, bz - pz, cx - px, cy - py, cz - pz
    la, lb, lc = np.sqrt(ax * ax + ay * ay + az * az), np.sqrt(bx * bx + by * by + bz * bz), np.sqrt(cx * cx + cy * cy + cz * cz)
    num = ax * (by * cz - bz * cy) + ay * (bz * cx - bx * cz) + az * (bx * cy - by * cx)
    den = (la * lb * lc + (ax * bx + ay * by + az * bz) * lc + (ax * cx + ay * cy + az * cz) * lb
           + (bx * cx + by * cy + bz * cz) * la)
    return (2.0 * np.arctan2(num, den)).sum(axis=1) / (4.0 * np.pi)


def mesh_sdf(verts, faces, points, pairs_per_chunk=1 << 17):
    """(signed distance fp64 (P,), winding number fp64 (P,)): positive inside (odd rounded winding number)."""
    tris = np.asarray(verts, dtype=np.float32)[np.asarray(faces)]
    pts = np.asarray(points, dtype=np.float32)
    n = max(1, pairs_per_chunk // max(1, len(tris)))
    d = np.empty(len(pts))
    w = np.empty(len(pts))
    for s in range(0, len(pts), n):
        d[s:s + n] = np.sqrt(point_triangle_d2(pts[s:s + n], tris).min(axis=1))
        w[s:s + n] = winding_number(pts[s:s + n], tris)
    inside = np.rint(np.abs(w)).astype(np.int64) % 2 == 1
    return np.where(inside, d, -d), w


# ---- test meshes -------------------------------------------------------------------------------------------------
def icosphere(level, radius=1.0, center=(0.0, 0.0, 0.0)):
    """icosahedron subdivided `level` times (20 * 4**level faces, outward), vertices on the sphere: (fp32 (V,3), int64 (F,3))."""
    g = (1.0 + 5.0 ** 0.5) / 2.0
    v = np.array([[-1, g, 0], [1, g, 0], [-1, -g, 0], [1, -g, 0], [0, -1, g], [0, 1, g], [0, -1, -g], [0, 1, -g],
                  [g, 0, -1], [g, 0, 1], [-g, 0, -1], [-g, 0, 1]], dtype=np.float64)
    f = np.array([[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2],
                  [10, 7, 6], [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11],
                  [6, 2, 10], [8, 6, 7], [9, 8, 1]], dtype=np.int64)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    for _ in range(level):
        e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
        key = np.minimum(e[:, 0], e[:, 1]) * len(v) + np.maximum(e[:, 0], e[:, 1])
        uk, inv = np.unique(key, return_inverse=True)
        mid = (v[uk // len(v)] + v[uk % len(v)]) / 2.0
        mid /= np.linalg.norm(mid, axis=1, keepdims=True)
        m = len(v) + inv.reshape(3, -1)
        v = np.concatenate([v, mid])
        a, b, c = f[:, 0], f[:, 1], f[:, 2]
        f = np.concatenate([np.stack([a, m[0], m[2]], 1), np.stack([b, m[1], m[0]], 1), np.stack([c, m[2], m[1]], 1),
                            np.stack([m[0], m[1], m[2]], 1)])
    return (v * radius + np.asarray(center)).astype(np.float32), f


def torus(R=0.45, r=0.15, nu=48, nv=24):
    """closed torus around the z axis, outward: (fp32 (V,3), int64 (F,3))."""
    u = np.arange(nu) * 2 * np.pi / nu
    w = np.arange(nv) * 2 * np.pi / nv
    U, W = np.meshgrid(u, w, indexing="ij")
    v = np.stack([(R + r * np.cos(W)) * np.cos(U), (R + r * np.cos(W)) * np.sin(U), r * np.sin(W)], -1).reshape(-1, 3)
    i, j = np.meshgrid(np.arange(nu), np.arange(nv), indexing="ij")
    a, b = i * nv + j, ((i + 1) % nu) * nv + j
    c, d = ((i + 1) % nu) * nv + (j + 1) % nv, i * nv + (j + 1) % nv
    f = np.concatenate([np.stack([a, b, c], -1).reshape(-1, 3), np.stack([a, c, d], -1).reshape(-1, 3)])
    return v.astype(np.float32), f.astype(np.int64)


def voxel_mesh(occ, origin, spacing):
    """closed outward surface of the union of the filled cells of the boolean grid occ (nx, ny, nz), cell (i, j, k) =
    origin + [i, i + 1] x [j, j + 1] x [k, k + 1] * spacing; two triangles per boundary face, vertices shared."""
    occ = np.pad(np.asarray(occ, dtype=bool), 1)
    quads = []
    for ax in range(3):
        a1, a2 = (ax + 1) % 3, (ax + 2) % 3
        lo = np.transpose(occ, (ax, a1, a2))
        for s in range(lo.shape[0] - 1):
            diff = lo[s].astype(int) - lo[s + 1].astype(int)        # +1: filled below, outward normal +ax
            for (u, w) in zip(*np.nonzero(diff)):
                corner = [0, 0, 0]
                corner[ax] = s
                corner[a1], corner[a2] = u - 1, w - 1
                c = np.array(corner)
                e1, e2 = np.eye(3, dtype=int)[a1], np.eye(3, dtype=int)[a2]
                q = [c, c + e1, c + e1 + e2, c + e2]
                quads.append(q if diff[u, w] > 0 else q[::-1])
    pts = np.array([p for q in quads for p in q])
    uniq, inv = np.unique(pts, axis=0, return_inverse=True)
    inv = inv.reshape(-1, 4)
    f = np.concatenate([inv[:, [0, 1, 2]], inv[:, [0, 2, 3]]])
    v = np.asarray(origin, dtype=np.float64) + uniq * np.asarray(spacing, dtype=np.float64)
    return v.astype(np.float32), f.astype(np.int64)


def box_sdf(p, lo, hi):
    """analytic signed distance to the box [lo, hi] (positive inside), fp64."""
    p = np.asarray(p, dtype=np.float64)
    c, h = (np.asarray(lo) + np.asarray(hi)) / 2.0, (np.asarray(hi) - np.asarray(lo)) / 2.0
    q = np.abs(p - c) - h
    outside = np.linalg.norm(np.maximum(q, 0.0), axis=1)
    inside = np.minimum(q.max(axis=1), 0.0)
    return -(outside + inside)


def write_obj(path, verts, faces):
    with open(path, "w") as f:
        for x in verts:
            f.write("v %.9g %.9g %.9g\n" % (x[0], x[1], x[2]))
        for t in faces:
            f.write("f %d %d %d\n" % (t[0] + 1, t[1] + 1, t[2] + 1))
