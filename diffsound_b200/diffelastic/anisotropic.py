"""Elasticity tensors for DiffSoundObj.set_elasticity_field: differentiable, batched torch helpers.

Convention (the one of csrc/assemble.cu and include/diffsound_sm100.h): a stiffness is a (..., 6, 6) matrix C in Voigt order
(11, 22, 33, 23, 13, 12) with engineering shear strains, eps_V = (e11, e22, e33, 2 e23, 2 e13, 2 e12) and sigma_V = C eps_V.
The strain energy density is 1/2 eps_V^T C eps_V.  C is given in the global (mesh) frame.
"""
import torch

# Voigt index pairs (i, j) of 11, 22, 33, 23, 13, 12
VOIGT_PAIRS = ((0, 0), (1, 1), (2, 2), (1, 2), (0, 2), (0, 1))


def _broadcast(*xs):
    ref = next((x for x in xs if torch.is_tensor(x)), None)
    kw = dict(dtype=torch.float64) if ref is None else dict(dtype=ref.dtype, device=ref.device)
    ts = [x if torch.is_tensor(x) else torch.tensor(float(x), **kw) for x in xs]
    return torch.broadcast_tensors(*ts)


def isotropic_stiffness(E, nu):
    """(..., 6, 6) C = lam 1 1^T (upper 3x3 block) + mu diag(2, 2, 2, 1, 1, 1) of Young's modulus E and Poisson's ratio nu
    (scalars or tensors, broadcast together)."""
    E, nu = _broadcast(E, nu)
    lam = E * nu / ((1 + nu) * (1 - 2 * nu))
    mu = E / (2 * (1 + nu))
    block = torch.zeros(6, 6, dtype=E.dtype, device=E.device)
    block[:3, :3] = 1
    diag = torch.stack([2 * mu, 2 * mu, 2 * mu, mu, mu, mu], dim=-1)
    return lam[..., None, None] * block + torch.diag_embed(diag)


def orthotropic_compliance(E1, E2, E3, nu12, nu13, nu23, G12, G13, G23):
    """(..., 6, 6) compliance S (eps_V = S sigma_V) of an orthotropic material in its own axes 1, 2, 3: S11 = 1/E1,
    S12 = -nu12/E1, S13 = -nu13/E1, S23 = -nu23/E2, S44 = 1/G23, S55 = 1/G13, S66 = 1/G12 (nu_ij: contraction along j
    under stress along i, so nu_ij / E_i = nu_ji / E_j)."""
    E1, E2, E3, nu12, nu13, nu23, G12, G13, G23 = _broadcast(E1, E2, E3, nu12, nu13, nu23, G12, G13, G23)
    z = torch.zeros_like(E1)
    rows = [
        [1 / E1, -nu12 / E1, -nu13 / E1, z, z, z],
        [-nu12 / E1, 1 / E2, -nu23 / E2, z, z, z],
        [-nu13 / E1, -nu23 / E2, 1 / E3, z, z, z],
        [z, z, z, 1 / G23, z, z],
        [z, z, z, z, 1 / G13, z],
        [z, z, z, z, z, 1 / G12],
    ]
    return torch.stack([torch.stack(r, dim=-1) for r in rows], dim=-2)


def orthotropic_stiffness(E1, E2, E3, nu12, nu13, nu23, G12, G13, G23):
    """(..., 6, 6) stiffness C = S^-1 of the orthotropic compliance S (orthotropic_compliance) in the material axes
    1, 2, 3 = x, y, z; turn it with rotate_stiffness.  Raises ValueError when the constants do not give a positive
    definite S (a material that would not store energy under every strain)."""
    S = orthotropic_compliance(E1, E2, E3, nu12, nu13, nu23, G12, G13, G23)
    _, info = torch.linalg.cholesky_ex(S.detach())
    if bool((info != 0).any()):
        raise ValueError("orthotropic_stiffness: the constants give a compliance that is not positive definite "
                         "(need E, G > 0 and |nu_ij| small enough, e.g. nu_ij^2 < E_i / E_j)")
    return torch.linalg.inv(S)


def bond_matrix(R):
    """(..., 6, 6) Bond matrix M of rotations R (..., 3, 3): sigma_V' = M sigma_V for sigma' = R sigma R^T.  Its entries are
    M[(i,j), (k,l)] = R_ik R_jl + R_il R_jk for k != l, R_ik R_jl for k == l."""
    i = torch.tensor([p[0] for p in VOIGT_PAIRS], device=R.device)
    j = torch.tensor([p[1] for p in VOIGT_PAIRS], device=R.device)
    off = (i != j).to(R.dtype)
    a = R[..., i[:, None], i[None, :]] * R[..., j[:, None], j[None, :]]
    b = R[..., i[:, None], j[None, :]] * R[..., j[:, None], i[None, :]]
    return a + b * off[None, :]


def rotate_stiffness(C, R):
    """C' = M C M^T (M = bond_matrix(R)): the stiffness of the material C turned by the rotations R (..., 3, 3), i.e.
    C'_ijkl = R_ia R_jb R_kc R_ld C_abcd.  A mesh whose vertices are turned by R keeps its spectrum when its C is turned
    with it.  Batched over the leading dimensions of C and R (broadcast); R is moved to C's device and dtype."""
    M = bond_matrix(R.to(device=C.device, dtype=C.dtype))
    return M @ C @ M.transpose(-1, -2)


def rotation_about(axis, angle):
    """(..., 3, 3) rotation by `angle` (radians, scalar or tensor) about the unit vector `axis` (3,), differentiable in
    the angle (Rodrigues' formula)."""
    angle = angle if torch.is_tensor(angle) else torch.tensor(float(angle), dtype=torch.float64)
    a = torch.as_tensor(axis, dtype=angle.dtype, device=angle.device)
    a = a / torch.linalg.norm(a)
    K = torch.zeros(3, 3, dtype=angle.dtype, device=angle.device)
    K[0, 1], K[0, 2], K[1, 2] = -a[2], a[1], -a[0]
    K = K - K.T
    s, c = torch.sin(angle)[..., None, None], torch.cos(angle)[..., None, None]
    eye = torch.eye(3, dtype=angle.dtype, device=angle.device)
    return eye + s * K + (1 - c) * (K @ K)
