"""Reference for objects with one elasticity tensor per tet (DiffSoundObj.set_elasticity_field), on the CPU.

Independent of the kernels' ctab contraction: the element stiffness is K_e = sum_q w_q |det A| B_q^T C_t B_q with the
6 x 3npe strain-displacement matrix B (Voigt order 11, 22, 33, 23, 13, 12, engineering shear strains) at the four points
of the degree-2 rule of `material_field_oracle` (exact for these integrands), with the same fp32 -> fp64 geometry.  M is
the one of `material_field_oracle.assemble_field`.  The strain Grams E_t,i = int_t eps_V(u_i) eps_V(u_i)^T dV come from the
same B, so d lambda_i / dC_t = E_t,i; the vertex gradient is taken by torch autograd with U and lambda constant."""
import numpy as np
import scipy.sparse as sp
import torch

import fixed_oracle as fo
import material_field_oracle as mf
from oracle import modal_oracle as mo

# (row of eps_V, displacement component c, derivative direction j): eps_V[row] += du_c / dx_j
_B_TERMS = ((0, 0, 0), (1, 1, 1), (2, 2, 2), (3, 1, 2), (3, 2, 1), (4, 0, 2), (4, 2, 0), (5, 0, 1), (5, 1, 0))


def _grad_n(verts, tets, order):
    """material_field_oracle._grad_n (grad_x N_a at the degree-2 rule's points, and w |det A|).  fp32 vertices give the
    kernels' geometry (fp32 differences, fp64 inverse); fp64 vertices keep the geometry in fp64 throughout."""
    if verts.dtype != torch.float64:
        return mf._grad_n(verts, tets, order)
    c = mo.CORNERS[order]
    v1, v2, v3, v4 = (verts[tets[:, i]] for i in c)
    A = torch.stack([v1 - v4, v2 - v4, v3 - v4], dim=2)
    dL = torch.tensor([[1, 0, 0], [0, 1, 0], [0, 0, 1], [-1, -1, -1]], dtype=torch.float64)
    g = (mo.shape_fn_grad(mf._KEAST, order) @ dL).unsqueeze(0) @ torch.linalg.inv(A).unsqueeze(1)
    w = float(mo.gauss_rule(3)[1].astype(np.float64).sum()) / 4.0 if order == 1 else 1.0 / 24.0
    return g, torch.abs(torch.linalg.det(A))[:, None] * w


def strain_matrix(g):
    """B (..., 6, 3 npe) from the shape-function gradients g (..., npe, 3): eps_V = B u_e, u_e = (u_a,c) a-major."""
    npe = g.shape[-2]
    B = torch.zeros(g.shape[:-2] + (6, npe, 3), dtype=g.dtype)
    for row, c, j in _B_TERMS:
        B[..., row, :, c] = B[..., row, :, c] + g[..., :, j]
    return B.reshape(g.shape[:-2] + (6, 3 * npe))


def element_stiffness(verts, tets, order, C):
    """(T, 3npe, 3npe) fp64 sum_q w_q B_q^T C_t B_q; C (T, 6, 6) fp64."""
    g, w = _grad_n(verts, tets, order)                       # (T, Q, npe, 3), (T, Q) with |det A|
    B = strain_matrix(g)                                     # (T, Q, 6, 3npe)
    return torch.einsum("tq,tqia,tij,tqjb->tab", w, B, torch.as_tensor(C, dtype=torch.float64), B)


def element_mass(verts, tets, order, density):
    """(T, 3npe, 3npe) fp64 with the entries double(float32(m_ab) * float32(rho_t)) * |6V|."""
    npe = mo.NPE[order]
    tab = (mo.element_mass_table(order)[None] * torch.as_tensor(density).to(torch.float32)[:, None, None]).double()
    Me = tab * mo.tet_det64(verts, tets, order)[:, None, None]
    eye = torch.eye(3, dtype=torch.float64)
    return (Me[:, :, None, :, None] * eye[None, None, :, None, :]).reshape(-1, 3 * npe, 3 * npe)


def assemble_tensor(verts, tets, order, C, density, batch=4096):
    """K, M (scipy CSR, the pattern of mo.assemble) with per-tet C (T, 6, 6) fp64 and density (T,)."""
    n = 3 * verts.shape[0]
    C = torch.as_tensor(C, dtype=torch.float64)
    density = torch.as_tensor(density)
    crow, col, _, _ = mo.pattern(tets, verts.shape[0])
    rows_of = np.repeat(np.arange(n, dtype=np.int64), np.diff(crow))
    keys = rows_of * n + col
    kv = np.zeros(col.size)
    mv = np.zeros(col.size)
    for s in range(0, tets.shape[0], batch):
        sl = slice(s, min(s + batch, tets.shape[0]))
        d = mo.element_dofs(tets[sl]).numpy().astype(np.int64)
        slot = np.searchsorted(keys, (d[:, :, None] * n + d[:, None, :]).reshape(-1))
        Ke = element_stiffness(verts, tets[sl], order, C[sl])
        Me = element_mass(verts, tets[sl], order, density[sl])
        kv += np.bincount(slot, weights=Ke.detach().numpy().reshape(-1), minlength=col.size)
        mv += np.bincount(slot, weights=Me.detach().numpy().reshape(-1), minlength=col.size)
    return sp.csr_matrix((kv, col, crow), shape=(n, n)), sp.csr_matrix((mv, col, crow), shape=(n, n))


def strain_grams(verts, tets, order, U, batch=2048):
    """E (T, k, 6, 6) fp64: int_t eps_V(u_i) eps_V(u_i)^T dV of every tet t and column i of U."""
    Ut = torch.as_tensor(U, dtype=torch.float64)
    out = []
    for s in range(0, tets.shape[0], batch):
        t = tets[s:s + batch]
        g, w = _grad_n(verts, t, order)
        B = strain_matrix(g)
        ue = Ut[mo.element_dofs(t)]                          # (T, 3npe, k)
        eps = torch.einsum("tqia,tak->tqki", B, ue)          # (T, Q, k, 6)
        out.append(torch.einsum("tq,tqki,tqkj->tkij", w, eps, eps))
    return torch.cat(out)


def tensor_grads(verts, tets, order, density, U, lam, g):
    """(d/dC (T, 6, 6), d/drho (T,)) of sum_i g_i lambda_i."""
    E = strain_grams(verts, tets, order, U)
    gt = torch.as_tensor(g, dtype=torch.float64)
    gC = torch.einsum("k,tkij->tij", gt, E)
    _, _, q_m = mf.element_forms(verts, tets, order, U)
    grho = -(q_m @ (np.asarray(g, np.float64) * np.asarray(lam, np.float64)))
    return gC.numpy(), grho


def vertex_grad(verts, tets, order, C, density, U, lam, g, batch=4096):
    """d/d(verts) of sum_i g_i (u_i^T K u_i - lam_i u_i^T M u_i) with C fixed in world axes (torch autograd)."""
    v = torch.as_tensor(verts).detach().clone().requires_grad_(True)
    C = torch.as_tensor(C, dtype=torch.float64)
    density = torch.as_tensor(density)
    Ut = torch.as_tensor(U, dtype=torch.float64)
    lamt = torch.as_tensor(lam, dtype=torch.float64)
    gt = torch.as_tensor(g, dtype=torch.float64)
    total = torch.zeros((), dtype=torch.float64)
    for s in range(0, tets.shape[0], batch):
        sl = slice(s, min(s + batch, tets.shape[0]))
        ue = Ut[mo.element_dofs(tets[sl])]
        Ke = element_stiffness(v, tets[sl], order, C[sl])
        Me = element_mass(v, tets[sl], order, density[sl])
        qk = torch.einsum("tak,tab,tbk->k", ue, Ke, ue)
        qm = torch.einsum("tak,tab,tbk->k", ue, Me, ue)
        total = total + (gt * (qk - lamt * qm)).sum()
    total.backward()
    return v.grad


def eigs(K, M, k, mask=None):
    """Lowest k elastic pairs (lam (k,), U (n, k)): shift-invert ARPACK, the rigid six dropped; `fixed_oracle` when a clamp
    mask (n_nodes,) is given."""
    if mask is not None:
        return fo.eig_fixed(K, M, np.asarray(mask), k)
    lam, U, _, _ = mo.eig_arpack(K, M, k, sigma=-1e3)
    return lam, U
