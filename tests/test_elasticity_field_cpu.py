"""The CPU reference for elasticity-tensor fields (tests/elasticity_field_oracle.py), the stiffness helpers of
diffsound_b200.diffelastic.anisotropic and the host validation of DiffSoundObj.set_elasticity_field."""
import numpy as np
import pytest
import torch

import elasticity_field_oracle as eo
import material_field_oracle as mf
from oracle import modal_oracle as mo
from test_modal_gains_cpu import kuhn_box

from diffsound_b200.diffelastic import anisotropic as an
from diffsound_b200.diffelastic import diff_model as dm

# wood-like orthotropic constants (illustrative: E1 along the grain, 2 radial, 3 tangential)
WOOD = dict(E1=1.2e10, E2=8e8, E3=5e8, nu12=0.4, nu13=0.45, nu23=0.5, G12=7e8, G13=6e8, G23=5e7)
RHO = 500.0


def wood():
    return an.orthotropic_stiffness(*WOOD.values())


def random_rotations(n, seed):
    q = torch.randn(n, 4, dtype=torch.float64, generator=torch.Generator().manual_seed(seed))
    q = q / q.norm(dim=1, keepdim=True)
    w, x, y, z = q.unbind(1)
    return torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                        2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                        2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], dim=1).reshape(n, 3, 3)


def _mesh(order, n=2):
    v, t = mo.kuhn_cube(n)
    return mo.promote(v, t, order) if order == 2 else (v, t)


# ------------------------------------------------------------------ the oracle
@pytest.mark.parametrize("order", [1, 2])
def test_isotropic_tensor_matches_lame_oracle(order):
    pv, pt = _mesh(order)
    T = pt.shape[0]
    g = torch.Generator().manual_seed(order)
    E = 2e11 * (0.5 + torch.rand(T, dtype=torch.float64, generator=g))
    nu = 0.2 + 0.2 * torch.rand(T, dtype=torch.float64, generator=g)
    rho = 7800.0 * (0.5 + torch.rand(T, dtype=torch.float64, generator=g))
    K0, M0 = mf.assemble_field(pv, pt, order, E, nu, rho)
    C = an.isotropic_stiffness(E, nu)
    K1, M1 = eo.assemble_tensor(pv, pt, order, C, rho)
    assert np.array_equal(M1.data, M0.data)
    # P1: the same quadrature as assemble_field.  P2: assemble_field integrates with the reference's fp32 Gauss rule
    # (~5e-8 from exact), so the tensor elements are also held against the Lame element formula on the exact rule.
    assert np.abs(K1.data - K0.data).max() <= (1e-12 if order == 1 else 1e-6) * np.abs(K0.data).max()
    g, w = mf._grad_n(pv, pt, order)
    mu, lam = mf.lame_t(E, nu)
    gw = g * w[:, :, None, None]
    dot = torch.einsum("tqac,tqbc->tab", gw, g)
    outer = torch.einsum("tqac,tqbd->tacbd", gw, g)
    eye = torch.eye(3, dtype=torch.float64)
    Kl = (mu[:, None, None, None, None] * (dot[:, :, None, :, None] * eye[None, None, :, None, :] + outer.permute(0, 1, 4, 3, 2))
          + lam[:, None, None, None, None] * outer).reshape(T, 3 * g.shape[2], -1)
    Kt = eo.element_stiffness(pv, pt, order, C)
    assert (Kt - Kl).abs().max().item() <= 1e-12 * Kl.abs().max().item()


def test_rotating_mesh_and_tensor_keeps_the_spectrum():
    # fp64 vertices: rotated coordinates rounded to fp32 would move the geometry by ~6e-8
    pv, pt = _mesh(2)
    pv = pv.double()
    T = pt.shape[0]
    C = an.rotate_stiffness(wood().expand(T, 6, 6), random_rotations(T, 1))
    rho = torch.full((T,), RHO)
    K, M = eo.assemble_tensor(pv, pt, 2, C, rho)
    lam, _ = eo.eigs(K, M, 12)
    R = random_rotations(1, 2)[0]
    pv_r = pv @ R.T
    K_r, M_r = eo.assemble_tensor(pv_r, pt, 2, an.rotate_stiffness(C, R), rho)
    lam_r, _ = eo.eigs(K_r, M_r, 12)
    assert np.abs(lam_r / lam - 1).max() <= 1e-9


def orthotropic_bar(turned):
    """(verts, tets, C, rho) of a free-free P2 bar 0.4 x 0.02 x 0.02 m (length / width 20) of the WOOD constants, the
    fibres (axis 1) along the bar (x) or turned 90 degrees about the bar's normal z (axis 2 along x)."""
    v, t = kuhn_box((20, 1, 1), (0.4, 0.02, 0.02))
    pv, pt = mo.promote(torch.from_numpy(v), torch.from_numpy(t), 2)
    C = wood()
    if turned:
        C = an.rotate_stiffness(C, an.rotation_about([0, 0, 1], np.pi / 2))
    T = pt.shape[0]
    return pv, pt, C.expand(T, 6, 6), torch.full((T,), RHO, dtype=torch.float64)


def longitudinal_mode(lam, U, M):
    """(index, frequency) of the lowest mode whose kinetic energy is more than 80 % axial (x)."""
    ax = (U[0::3] * (M @ U)[0::3]).sum(0) / (U * (M @ U)).sum(0)
    i = int(np.argmax(ax > 0.8))
    assert ax[i] > 0.8
    return i, np.sqrt(lam[i]) / (2 * np.pi)


@pytest.mark.parametrize("turned", [False, True])
def test_orthotropic_bar_longitudinal_mode(turned):
    # uniaxial stress along the bar: the bar modulus is exactly 1 / S_xx of the compliance in the bar's frame
    pv, pt, C, rho = orthotropic_bar(turned)
    K, M = eo.assemble_tensor(pv, pt, 2, C, rho)
    lam, U = eo.eigs(K, M, 16)
    _, f = longitudinal_mode(lam, U, M)
    E_bar = WOOD["E2"] if turned else WOOD["E1"]
    f_ref = np.sqrt(E_bar / RHO) / (2 * 0.4)
    assert abs(f / f_ref - 1) <= 0.01, (f, f_ref)


def test_strain_grams_give_the_eigenvalues():
    pv, pt = _mesh(2)
    T = pt.shape[0]
    C = an.rotate_stiffness(wood().expand(T, 6, 6), random_rotations(T, 3))
    K, M = eo.assemble_tensor(pv, pt, 2, C, torch.full((T,), RHO))
    lam, U = eo.eigs(K, M, 8)
    E = eo.strain_grams(pv, pt, 2, U)
    assert np.abs(torch.einsum("tij,tkij->k", C, E).numpy() / lam - 1).max() <= 1e-9


# ------------------------------------------------------------------ the helpers
def test_orthotropic_stiffness_inverts_its_compliance():
    C = wood()
    S = an.orthotropic_compliance(*WOOD.values())
    assert torch.allclose(C @ S, torch.eye(6, dtype=torch.float64), atol=1e-12)
    assert torch.allclose(C, C.T, rtol=1e-14, atol=0)
    E, nu = 2e11, 0.3
    G = E / (2 * (1 + nu))
    iso = an.orthotropic_stiffness(E, E, E, nu, nu, nu, G, G, G)
    assert torch.allclose(iso, an.isotropic_stiffness(E, nu), rtol=1e-13, atol=1e-13 * E)
    with pytest.raises(ValueError):
        an.orthotropic_stiffness(1e10, 1e9, 1e9, 0.9, 0.9, 0.9, 1e9, 1e9, 1e9)
    with pytest.raises(ValueError):
        an.orthotropic_stiffness(1e10, -1e9, 1e9, 0.3, 0.3, 0.3, 1e9, 1e9, 1e9)


def test_rotations():
    E, nu = 7e10, 0.33
    iso = an.isotropic_stiffness(E, nu)
    R = random_rotations(5, 4)
    assert torch.allclose(an.rotate_stiffness(iso, R), iso.expand(5, 6, 6), rtol=0, atol=1e-12 * E)
    C = wood()
    Cz = an.rotate_stiffness(C, an.rotation_about([0, 0, 1], np.pi / 2))
    swap = [1, 0, 2, 4, 3, 5]              # 11 <-> 22, 23 <-> 13
    assert torch.allclose(Cz, C[swap][:, swap], rtol=0, atol=1e-12 * float(C.abs().max()))
    # the Bond matrix of a product is the product of the Bond matrices
    assert torch.allclose(an.bond_matrix(R[0] @ R[1]), an.bond_matrix(R[0]) @ an.bond_matrix(R[1]), atol=1e-13)


def test_helpers_gradcheck():
    E = torch.tensor(2.0, dtype=torch.float64, requires_grad=True)
    nu = torch.tensor(0.3, dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(an.isotropic_stiffness, (E, nu))
    consts = torch.tensor([12.0, 0.8, 0.5, 0.4, 0.45, 0.5, 0.7, 0.6, 0.05], dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(lambda c: an.orthotropic_stiffness(*c), (consts,))
    C = wood().detach() * 1e-9
    theta = torch.tensor(0.3, dtype=torch.float64, requires_grad=True)
    Cr = C.clone().requires_grad_(True)
    assert torch.autograd.gradcheck(lambda c, th: an.rotate_stiffness(c, an.rotation_about([0.2, 0.5, 1.0], th)),
                                    (Cr, theta))


# ------------------------------------------------------------------ validation
def test_elasticity_field_validation_errors():
    T = 10
    C = wood().expand(T, 6, 6).clone()
    dm.check_elasticity_field(T, "cpu", C)
    dm.check_elasticity_field(T, "cpu", C.float(), torch.full((T,), RHO))
    bad = []
    bad.append(C[:-1])                                      # shape
    bad.append(C.to(torch.float16))                         # dtype
    nan = C.clone()
    nan[3, 0, 0] = float("nan")
    bad.append(nan)
    asym = C.clone()
    asym[2, 0, 1] *= 1.01
    bad.append(asym)
    indef = C.clone()
    indef[4, 3, 3] = -1e8
    bad.append(indef)
    for c in bad:
        with pytest.raises(ValueError):
            dm.check_elasticity_field(T, "cpu", c)
    with pytest.raises(ValueError):                         # device
        dm.check_elasticity_field(T, "cuda:0", C)
    with pytest.raises(ValueError):                         # density
        dm.check_elasticity_field(T, "cpu", C, torch.full((T,), -1.0))
