"""Reference for objects with one material per tet (DiffSoundObj.set_material_field), on the CPU.

K and M are assembled like `oracle.modal_oracle.assemble`, with the element stiffness of tet t at its own (mu_t, lam_t) and
the element mass table rounded against its own fp32 density (float32(m_ab) * float32(rho_t), promoted): a constant field
reproduces `mo.assemble` exactly.  Eigenpairs come from shift-invert ARPACK (`fixed_oracle` for clamped objects).

The per-tet forms q_mu[t, i] = u_i^T K_mu,t u_i, q_lam[t, i] = u_i^T K_lam,t u_i, q_m[t, i] = u_i^T Mhat_t u_i are evaluated
independently of the kernels: element gradients from an fp64 inverse of the fp32 transform matrix and an fp64 degree-2
quadrature (exact for these integrands), the mass from the promoted fp32 table and |6V| of fp64 corners.  With them the
eigenvalue derivatives are d lam_i / d mu_t = q_mu, d lam_i / d lam_t = q_lam, d lam_i / d rho_t = -lam_i q_m."""
import numpy as np
import scipy.sparse as sp
import torch

from oracle import modal_oracle as mo

# degree-2 rule on the unit tet (volume 1/6): four points, weight 1/24 each
_A, _B = (5.0 - 5.0 ** 0.5) / 20.0, (5.0 + 3.0 * 5.0 ** 0.5) / 20.0
_KEAST = torch.tensor([[_B, _A, _A, _A], [_A, _B, _A, _A], [_A, _A, _B, _A], [_A, _A, _A, _B]], dtype=torch.float64)


def lame_t(youngs, poisson):
    """(mu_t, lam_t) fp64 tensors: the expression of diff_model._lame."""
    E = torch.as_tensor(youngs, dtype=torch.float64)
    nu = torch.as_tensor(poisson, dtype=torch.float64)
    return E / (2 * (1 + nu)), E * nu / ((1 + nu) * (1 - 2 * nu))


def assemble_field(verts, tets, order, youngs, poisson, density, batch=4096):
    """K, M (scipy CSR, the pattern of mo.assemble) with per-tet (T,) youngs, poisson (fp64) and density (fp32)."""
    n = 3 * verts.shape[0]
    mu_t, lam_t = lame_t(youngs, poisson)
    rho32 = torch.as_tensor(density).to(torch.float32)
    crow, col, _, _ = mo.pattern(tets, verts.shape[0])
    rows_of = np.repeat(np.arange(n, dtype=np.int64), np.diff(crow))
    keys = rows_of * n + col
    kv = np.zeros(col.size)
    mv = np.zeros(col.size)
    tab32 = mo.element_mass_table(order)
    npe = mo.NPE[order]
    eye = torch.eye(3, dtype=torch.float64)
    for s in range(0, tets.shape[0], batch):
        sl = slice(s, min(s + batch, tets.shape[0]))
        d = mo.element_dofs(tets[sl]).numpy().astype(np.int64)
        slot = np.searchsorted(keys, (d[:, :, None] * n + d[:, None, :]).reshape(-1))
        b5 = (-1, 1, 1, 1, 1)
        Ke = mo.element_stiffness(verts, tets, order, mu_t[sl].reshape(b5), lam_t[sl].reshape(b5), sl)
        tab = (tab32[None] * rho32[sl][:, None, None]).double()          # fp32 product per tet, then promoted
        Me = tab * mo.tet_det64(verts, tets[sl], order)[:, None, None]
        Me = (Me[:, :, None, :, None] * eye[None, None, :, None, :]).reshape(-1, 3 * npe, 3 * npe)
        kv += np.bincount(slot, weights=Ke.detach().numpy().reshape(-1), minlength=col.size)
        mv += np.bincount(slot, weights=Me.detach().numpy().reshape(-1), minlength=col.size)
    return sp.csr_matrix((kv, col, crow), shape=(n, n)), sp.csr_matrix((mv, col, crow), shape=(n, n))


def _grad_n(verts, tets, order):
    """grad_x N_a at the four points of the degree-2 rule, (T, 4, npe, 3) fp64, and the weights (T, 4)."""
    A = mo.transform_matrix(verts, tets, order).double()
    Ainv = torch.linalg.inv(A)
    dL = torch.tensor([[1, 0, 0], [0, 1, 0], [0, 0, 1], [-1, -1, -1]], dtype=torch.float64)
    dN = mo.shape_fn_grad(_KEAST, order) @ dL                            # (4, npe, 3)
    g = dN.unsqueeze(0) @ Ainv.unsqueeze(1)
    if order == 1:      # the kernels integrate the constant P1 integrand with the fp32 rule's weight sum, as the assembly
        w = float(np.float64(mo.gauss_rule(3)[1].astype(np.float64).sum())) / 4.0
    else:
        w = 1.0 / 24.0
    return g, torch.abs(torch.linalg.det(A))[:, None] * w


def element_forms(verts, tets, order, U, density=None, batch=4096):
    """(q_mu, q_lam, q_m), each (T, k) fp64.  q_m uses the unit-density table (double(m_ab)) or, with density (T,) given,
    the entries double(float32(m_ab) * float32(rho_t)) of the field assembly (then u_i^T M_t u_i)."""
    Ut = torch.as_tensor(U, dtype=torch.float64)
    tab32 = mo.element_mass_table(order)
    out = ([], [], [])
    for s in range(0, tets.shape[0], batch):
        sl = slice(s, min(s + batch, tets.shape[0]))
        t = tets[sl]
        ue = Ut[mo.element_dofs(t)].reshape(t.shape[0], -1, 3, Ut.shape[1])          # (T, npe, 3, k)
        g, w = _grad_n(verts, t, order)
        F = torch.einsum("taci,tqaj->tqicj", ue, g)                      # (T, Q, k, 3, 3): F[c][j] = du_c / dx_j
        phi_mu = (F * (F + F.transpose(-1, -2))).sum((-1, -2))
        tr = F.diagonal(dim1=-2, dim2=-1).sum(-1)
        out[0].append(torch.einsum("tq,tqi->ti", w, phi_mu))
        out[1].append(torch.einsum("tq,tqi->ti", w, tr * tr))
        if density is None:
            tab = tab32.double()[None].expand(t.shape[0], -1, -1)
        else:
            tab = (tab32[None] * torch.as_tensor(density).to(torch.float32)[sl][:, None, None]).double()
        ms = torch.einsum("tab,taci,tbci->ti", tab, ue, ue)
        out[2].append(ms * mo.tet_det64(verts, t, order)[:, None])
    return tuple(torch.cat(o).numpy() for o in out)


def field_grads(verts, tets, order, youngs, poisson, U, lam, g):
    """d/d(E_t, nu_t, rho_t) of sum_i g_i lambda_i: three (T,) fp64 arrays."""
    q_mu, q_la, q_m = element_forms(verts, tets, order, U)
    g = np.asarray(g, np.float64)
    gmu, gla = q_mu @ g, q_la @ g
    grho = -(q_m @ (g * np.asarray(lam, np.float64)))
    E = torch.as_tensor(youngs, dtype=torch.float64).clone().requires_grad_(True)
    nu = torch.as_tensor(poisson, dtype=torch.float64).clone().requires_grad_(True)
    mu_t, lam_t = lame_t(E, nu)
    (mu_t * torch.from_numpy(gmu) + lam_t * torch.from_numpy(gla)).sum().backward()
    return E.grad.numpy(), nu.grad.numpy(), grho


def vertex_grad(verts, tets, order, youngs, poisson, density, U, lam, g, batch=4096):
    """d/d(verts) of sum_i g_i (u_i^T K u_i - lam_i u_i^T M u_i) with the field (torch autograd; U, lam constant)."""
    v = verts.detach().clone().requires_grad_(True)
    mu_t, lam_t = lame_t(youngs, poisson)
    rho32 = torch.as_tensor(density).to(torch.float32)
    Ut = torch.as_tensor(U, dtype=torch.float64)
    lamt = torch.as_tensor(lam, dtype=torch.float64)
    gt = torch.as_tensor(g, dtype=torch.float64)
    tab32 = mo.element_mass_table(order)
    eye = torch.eye(3, dtype=torch.float64)
    npe = mo.NPE[order]
    total = torch.zeros((), dtype=torch.float64)
    for s in range(0, tets.shape[0], batch):
        sl = slice(s, min(s + batch, tets.shape[0]))
        ue = Ut[mo.element_dofs(tets[sl])]
        b5 = (-1, 1, 1, 1, 1)
        Ke = mo.element_stiffness(v, tets, order, mu_t[sl].reshape(b5), lam_t[sl].reshape(b5), sl)
        tab = (tab32[None] * rho32[sl][:, None, None]).double()
        Me = tab * mo.tet_det64(v, tets[sl], order)[:, None, None]
        Me = (Me[:, :, None, :, None] * eye[None, None, :, None, :]).reshape(-1, 3 * npe, 3 * npe)
        qk = torch.einsum("tak,tab,tbk->k", ue, Ke, ue)
        qm = torch.einsum("tak,tab,tbk->k", ue, Me, ue)
        total = total + (gt * (qk - lamt * qm)).sum()
    total.backward()
    return v.grad
