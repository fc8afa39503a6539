"""Reference for objects on elastic supports (DiffSoundObj.set_supports), built without the kernels' tables.

A support face f (the face opposite tet corner `local` of tet `owner`) with normal / tangential stiffness per unit area
k_n, k_t adds  K_s,f[a, b] = int_f N_a N_b dA ((k_n - k_t) n n^T + k_t I)  over its P1 / P2 nodes.  Here the face integral
is a 6-point triangle rule exact to degree 4 (Dunavant / Strang-Fix), applied to the face's own P1 / P2 shape functions in
the face's barycentric coordinates; the geometry is affine from the three corners.  K_s is added to
`oracle.modal_oracle.assemble`'s K and the pencil is solved by shift-invert ARPACK (clamped dofs deleted as in
tests/fixed_oracle.py).  Energies and gradients are torch fp64 autograd of the same integrals: d lambda_i = u_i^T dK_s u_i.
"""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla
import torch

# degree-4 rule on the reference triangle: (barycentrics, weight as a fraction of the area)
_A1, _W1 = 0.44594849091596488632, 0.22338158967801146570
_A2, _W2 = 0.091576213509770743460, 0.10995174365532186764
QUAD4 = [((1 - 2 * _A1, _A1, _A1), _W1), ((_A1, 1 - 2 * _A1, _A1), _W1), ((_A1, _A1, 1 - 2 * _A1), _W1),
         ((1 - 2 * _A2, _A2, _A2), _W2), ((_A2, 1 - 2 * _A2, _A2), _W2), ((_A2, _A2, 1 - 2 * _A2), _W2)]

# tet-local P2 node of the edge between tet corners (l, m) (local order v0 m01 v1 m12 v2 m02 m03 m13 m23 v3)
_P2_EDGE = {(0, 1): 1, (1, 2): 3, (0, 2): 5, (0, 3): 6, (1, 3): 7, (2, 3): 8}
_CORNER = {1: (0, 1, 2, 3), 2: (0, 2, 4, 9)}


def face_shape(L, order):
    """Face shape functions at barycentrics L (3,): corners 0, 1, 2 then (P2) edges (0,1), (1,2), (0,2)."""
    if order == 1:
        return np.array(L, dtype=np.float64)
    l0, l1, l2 = L
    return np.array([l0 * (2 * l0 - 1), l1 * (2 * l1 - 1), l2 * (2 * l2 - 1), 4 * l0 * l1, 4 * l1 * l2, 4 * l0 * l2])


def face_mass_ref(order):
    """int N_a N_b dA over a face of unit area, by QUAD4."""
    nf = 3 if order == 1 else 6
    Mf = np.zeros((nf, nf))
    for L, w in QUAD4:
        N = face_shape(L, order)
        Mf += w * np.outer(N, N)
    return Mf


def face_nodes(tets, order, owner, local):
    """(S, nf) node ids of the support faces in face_shape's order."""
    tets = np.asarray(tets)
    out = []
    for t, f in zip(np.asarray(owner), np.asarray(local)):
        cj = [j for j in range(4) if j != f]
        row = [tets[t, _CORNER[order][j]] for j in cj]
        if order == 2:
            row += [tets[t, _P2_EDGE[tuple(sorted((cj[a], cj[b])))]] for a, b in ((0, 1), (1, 2), (0, 2))]
        out.append(row)
    return np.array(out, dtype=np.int64)


def face_energy(verts, nodes, kn, kt, U, order):
    """(S, k) u_i^T K_s,f u_i as a torch fp64 function of verts (V, 3), kn, kt (S,) and U (n, k)."""
    verts = torch.as_tensor(verts, dtype=torch.float64)
    nodes = torch.as_tensor(nodes)
    kn = torch.as_tensor(kn, dtype=torch.float64)
    kt = torch.as_tensor(kt, dtype=torch.float64)
    U = torch.as_tensor(U, dtype=torch.float64)
    Mf = torch.as_tensor(face_mass_ref(order))
    p = verts[nodes[:, :3]]
    a = 0.5 * torch.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0], dim=1)
    A = a.norm(dim=1)
    n = a / A[:, None]
    u = U.reshape(-1, 3, U.shape[1])[nodes]                     # (S, nf, 3, k)
    W = torch.einsum("ab,sack,sbdk->skcd", Mf, u, u)            # (S, k, 3, 3) int u u^T dA / A
    nn = torch.einsum("skcd,sc,sd->sk", W, n, n)
    tr = W.diagonal(dim1=2, dim2=3).sum(-1)
    return A[:, None] * ((kn - kt)[:, None] * nn + kt[:, None] * tr)


def support_matrix(verts, tets, order, owner, local, kn, kt):
    """K_s (n, n) scipy CSR, fp64."""
    verts = np.asarray(verts, dtype=np.float64)
    nodes = face_nodes(tets, order, owner, local)
    Mf = face_mass_ref(order)
    kn = np.broadcast_to(np.asarray(kn, dtype=np.float64), (nodes.shape[0],))
    kt = np.broadcast_to(np.asarray(kt, dtype=np.float64), (nodes.shape[0],))
    rows, cols, vals = [], [], []
    for s, fn in enumerate(nodes):
        p = verts[fn[:3]]
        a = 0.5 * np.cross(p[1] - p[0], p[2] - p[0])
        A = np.linalg.norm(a)
        n = a / A
        S = (kn[s] - kt[s]) * np.outer(n, n) + kt[s] * np.eye(3)
        blk = np.kron(A * Mf, S)                                   # (3 nf, 3 nf), dof (a, c) at 3 a + c
        dofs = (3 * fn[:, None] + np.arange(3)).reshape(-1)
        rows.append(np.repeat(dofs, dofs.size))
        cols.append(np.tile(dofs, dofs.size))
        vals.append(blk.reshape(-1))
    n_dof = 3 * verts.shape[0]
    return sp.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n_dof, n_dof)).tocsr()


def eig_supported(K, M, Ks, k, fixed_nodes=None, sigma=0.0):
    """Lowest k pairs of (K + Ks) u = lambda M u (clamped dofs deleted): (lam (k,), U (n, k) M-orthonormal)."""
    Kt = (K + Ks).tocsr()
    n = Kt.shape[0]
    free = np.arange(n)
    if fixed_nodes is not None:
        fixed = np.zeros(n // 3, dtype=bool)
        fixed[np.asarray(fixed_nodes)] = True
        free = np.flatnonzero(np.repeat(~fixed, 3))
    Kr = Kt[free][:, free]
    Mr = M.tocsr()[free][:, free]
    Kr.eliminate_zeros()
    Mr.eliminate_zeros()
    lam, Ur = spla.eigsh(Kr, M=Mr, k=k, sigma=sigma)
    order = np.argsort(lam)
    U = np.zeros((n, k))
    U[free] = Ur[:, order]
    return lam[order], U


def support_grads(verts, tets, order, owner, local, kn, kt, U, g):
    """Gradient of sum_i g_i u_i^T K_s u_i: ((S,) to kn, (S,) to kt, (V, 3) to the vertices)."""
    nodes = face_nodes(tets, order, owner, local)
    S = nodes.shape[0]
    v = torch.as_tensor(np.asarray(verts), dtype=torch.float64).clone().requires_grad_(True)
    a = torch.as_tensor(np.broadcast_to(np.asarray(kn, dtype=np.float64), (S,)).copy()).requires_grad_(True)
    b = torch.as_tensor(np.broadcast_to(np.asarray(kt, dtype=np.float64), (S,)).copy()).requires_grad_(True)
    e = face_energy(v, nodes, a, b, U, order)
    (e * torch.as_tensor(np.asarray(g), dtype=torch.float64)).sum().backward()
    return a.grad.numpy(), b.grad.numpy(), v.grad.numpy()


def rigid_fields(verts):
    """(n, 6) fp64: unit translations, then rotations about the centroid (x, y, z axes)."""
    p = np.asarray(verts, dtype=np.float64)
    p = p - p.mean(0)
    n = p.shape[0]
    R = np.zeros((3 * n, 6))
    for c in range(3):
        R[c::3, c] = 1.0
    R[1::3, 3], R[2::3, 3] = -p[:, 2], p[:, 1]
    R[0::3, 4], R[2::3, 4] = p[:, 2], -p[:, 0]
    R[0::3, 5], R[1::3, 5] = -p[:, 1], p[:, 0]
    return R
