"""Objects with one elasticity tensor per tet on the B200 (DiffSoundObj.set_elasticity_field, ds_assemble_km_tensor,
ds_assemble_km_tets_tensor, ds_eigval_grad_shape_tensor, ds_elasticity_field_grad, ds_element_energies_tensor) against the
Lame-field kernels and the CPU reference of tests/elasticity_field_oracle.py."""
import numpy as np
import pytest
import torch

import elasticity_field_oracle as eo
from oracle import modal_oracle as mo
from test_elasticity_field_cpu import RHO, WOOD, longitudinal_mode, orthotropic_bar, random_rotations
from test_modal_gains_cpu import kuhn_box

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _mods():
    from diffsound_b200 import native
    from diffsound_b200.diffelastic import anisotropic as an
    from diffsound_b200.diffelastic import diff_model as dm
    from diffsound_b200.diffelastic.material_model import MatSet
    return native, an, dm, MatSet


def _geometry(meshes, name):
    if name == "box":
        return kuhn_box((6, 3, 2), (0.3, 0.12, 0.06))
    if name.startswith("cube"):
        v, t = mo.kuhn_cube(int(name[4:]))
        return v.numpy(), t.numpy()
    return meshes[name]


def _obj(meshes, name, order, mode_num=16, leaf=False, verts=None, tets=None, **kw):
    _, _, dm, MatSet = _mods()
    if verts is None:
        verts, tets = _geometry(meshes, name)
    vt = torch.as_tensor(np.asarray(verts), dtype=torch.float32, device=DEV)
    if leaf:
        vt.requires_grad_(True)
    obj = dm.DiffSoundObj(vt, torch.as_tensor(np.asarray(tets), device=DEV).long(), mode_num=mode_num, order=order,
                          mat=MatSet.Wood, **kw)
    return obj, vt


def _wood_field(obj, seed=0):
    """(C (T, 6, 6), density (T,)) fp64: the wood-like orthotropic C turned by a random rotation per tet, density 500."""
    _, an, _, _ = _mods()
    T = obj.tetmesh.tets.shape[0]
    C = an.rotate_stiffness(an.orthotropic_stiffness(*WOOD.values()).expand(T, 6, 6), random_rotations(T, seed))
    return C.to(DEV), torch.full((T,), RHO, dtype=torch.float64, device=DEV)


def _host(obj):
    return obj.tetmesh.vertices.detach().cpu(), obj.tetmesh.tets.cpu().long()


def _oracle(obj, C, rho, k, mask=None):
    pv, pt = _host(obj)
    K, M = eo.assemble_tensor(pv, pt, obj.tetmesh.order, C.detach().cpu(), rho.detach().cpu())
    lam, U = eo.eigs(K, M, k, None if mask is None else mask.cpu().numpy())
    return lam, U, K, M, pv, pt


def _check_modes(obj, lam, U, M):
    """eigenvalues <= 1e-6 rel, M-orthonormality <= 1e-10, and every cluster of close eigenvalues spans the reference's
    subspace (its principal cosines within 1e-6 of 1)."""
    got = obj.eigenvalues.cpu().numpy()
    assert np.abs(got / lam - 1).max() <= 1e-6, np.abs(got / lam - 1).max()
    Ug = obj.U_hat.cpu().numpy()
    G = Ug.T @ (M @ Ug)
    assert np.abs(G - np.eye(G.shape[0])).max() <= 1e-10
    i = 0
    while i < len(lam):
        j = i + 1
        while j < len(lam) and lam[j] / lam[j - 1] - 1 < 1e-3:
            j += 1
        if j < len(lam) or i == 0:            # a cluster cut by the last wanted mode is not a subspace of both
            s = np.linalg.svd(U[:, i:j].T @ (M @ Ug[:, i:j]), compute_uv=False)
            assert s.min() >= 1 - 1e-6, (i, j, s)
        i = j


# ------------------------------------------------------------------ 1. isotropic tensor field = Lame field
@pytest.mark.parametrize("name,order", [("cube3", 1), ("cube3", 2), ("box", 1), ("box", 2), ("bowl", 1), ("bowl", 2)])
def test_isotropic_tensor_assembly_matches_lame_field(meshes, name, order):
    native, an, dm, _ = _mods()
    obj, _ = _obj(meshes, name, order)
    d = obj.deform
    T = d.num_tets
    g = torch.Generator(device=DEV).manual_seed(order)
    E = 1e10 * (0.5 + torch.rand(T, dtype=torch.float64, device=DEV, generator=g))
    nu = 0.2 + 0.2 * torch.rand(T, dtype=torch.float64, device=DEV, generator=g)
    rho = (500.0 * (0.5 + torch.rand(T, dtype=torch.float64, device=DEV, generator=g))).float()
    mu, lam = dm._lame(E, nu)
    C21 = an.isotropic_stiffness(E, nu)[:, dm._IU[0], dm._IU[1]].contiguous()
    v32 = d.verts_f32()
    for kernel in (["rows", "tets"] if order == 2 else ["rows"]):
        K0, M0 = native.assemble_km(v32, d.tets_i32, order, d.pattern, 0.0, 0.0, d.ctab, d.m32(), kernel=kernel,
                                    field=(mu, lam, rho))
        K1, M1 = native.assemble_km(v32, d.tets_i32, order, d.pattern, 0.0, 0.0, d.ctab, d.m32(), kernel=kernel,
                                    tensor=(C21, rho))
        assert (K1 - K0).abs().max().item() <= 1e-13 * K0.abs().max().item(), kernel
        assert torch.equal(M0, M1), kernel
    if order == 2:
        co = d.coarse
        co.assemble(v32, 0.0, 0.0, co.ctab, d.m32(1), field=(mu, lam, rho))
        K0, M0 = co.Kval.clone(), co.Mblk.clone()
        co.assemble(v32, 0.0, 0.0, co.ctab, d.m32(1), tensor=(C21, rho))
        assert (co.Kval - K0).abs().max().item() <= 1e-13 * K0.abs().max().item()
        assert torch.equal(M0, co.Mblk)


# ------------------------------------------------------------------ 2. anisotropic assembly against the reference
@pytest.mark.parametrize("name,order", [("cube3", 1), ("cube3", 2), ("bowl", 1)])
def test_tensor_assembly_vs_oracle(meshes, name, order):
    obj, _ = _obj(meshes, name, order)
    C, rho = _wood_field(obj)
    obj.set_elasticity_field(C, rho)
    obj.update_mass_matrix(RHO)
    pv, pt = _host(obj)
    K, M = eo.assemble_tensor(pv, pt, order, C.cpu(), rho.cpu())
    Kg = obj.stiff_matrix.values().cpu().numpy()
    Mg = obj.mass_matrix.values().cpu().numpy()
    # P1: the same quadrature (the constant integrand times the fp32 rule's weight sum).  P2: the kernels' S_ab come from
    # the reference's fp32 Gauss rule (ctab), the reference integrates exactly: ~5e-8 apart, as for the Lame kernels.
    tol = 1e-12 if order == 1 else 2e-6
    assert np.abs(Kg - K.data).max() <= tol * np.abs(K.data).max()
    assert np.abs(Mg - M.data).max() <= 1e-12 * np.abs(M.data).max()
    if order == 2:      # both fine kernels (they sum the contributions of a slot in different orders)
        native, _, _, _ = _mods()
        d = obj.deform
        t = obj._tensor_used
        K0, M0 = native.assemble_km(obj._verts32, d.tets_i32, 2, d.pattern, 0.0, 0.0, d.ctab, d.m32(), kernel="rows",
                                    tensor=(t["C21"], t["rho"]))
        assert (K0 - obj._Kval).abs().max().item() <= 1e-13 * K0.abs().max().item()
        assert (M0 - obj._Mblk).abs().max().item() <= 1e-13 * M0.abs().max().item()


# ------------------------------------------------------------------ 3. kernels with a random U
@pytest.mark.parametrize("name,order", [("cube3", 1), ("cube3", 2), ("bowl", 1)])
@pytest.mark.parametrize("k", [16, 64])
def test_tensor_kernels_with_random_modes(meshes, name, order, k):
    native, _, dm, _ = _mods()
    obj, _ = _obj(meshes, name, order)
    C, rho = _wood_field(obj, seed=k)
    obj.set_elasticity_field(C, rho)
    obj.update_mass_matrix(RHO)
    d = obj.deform
    t = obj._tensor_used
    gen = torch.Generator(device=DEV).manual_seed(k)
    wide = torch.randn(d.pattern.n, k + 8, dtype=torch.float64, device=DEV, generator=gen)
    U = wide[:, 3:3 + k]
    lam = 1e6 * (1.0 + torch.rand(k, dtype=torch.float64, device=DEV, generator=gen))
    g = torch.randn(k, dtype=torch.float64, device=DEV, generator=gen)
    G21, Grho = native.elasticity_field_grad(obj._verts32, d.tets_i32, order, d.m32(), d.wsum, U, lam, g)
    strain, kinetic = native.element_energies_tensor(obj._verts32, d.tets_i32, order, d.m32(), d.wsum, U, (t["C21"], t["rho"]))
    pv, pt = _host(obj)
    E = eo.strain_grams(pv, pt, order, U.cpu().numpy())                                   # (T, k, 6, 6)
    want = torch.einsum("k,tkij->tij", g.cpu(), E)
    got = G21.cpu()[:, dm._VOIGT_UNPACK]
    assert (got - want).abs().max().item() <= 1e-12 * want.abs().max().item()
    # the density column is the one of the Lame-field kernel on the same U
    Gf = native.material_field_grad(obj._verts32, d.tets_i32, order, d.m32(), d.wsum, U, lam, g)
    assert (Grho - Gf[:, 2]).abs().max().item() <= 1e-14 * Gf[:, 2].abs().max().item()
    s_want = torch.einsum("tij,tkij->tk", t["C"].cpu(), E)
    assert (strain.cpu() - s_want).abs().max().item() <= 1e-12 * s_want.abs().max().item()
    # summed over the tets: the quadratic forms of the assembled operator (P2: fp32 Gauss rule of the assembly, ~5e-8)
    Uc = U.contiguous()
    KU, MU = native.spmm_k_and_m(d.pattern, obj._Kval, obj._Mblk, Uc)
    uku, umu = (Uc * KU).sum(0), (Uc * MU).sum(0)
    assert ((strain.sum(0) - uku).abs() / uku.abs()).max().item() <= (1e-12 if order == 1 else 2e-7)
    assert ((kinetic.sum(0) - umu).abs() / umu.abs()).max().item() <= 1e-12
    # no atomics: a second run is bitwise equal
    G21b, Grhob = native.elasticity_field_grad(obj._verts32, d.tets_i32, order, d.m32(), d.wsum, U, lam, g)
    s2, k2 = native.element_energies_tensor(obj._verts32, d.tets_i32, order, d.m32(), d.wsum, U, (t["C21"], t["rho"]))
    assert torch.equal(G21, G21b) and torch.equal(Grho, Grhob) and torch.equal(strain, s2) and torch.equal(kinetic, k2)


# ------------------------------------------------------------------ 4. eigenpairs against the reference
def _report(obj, label):
    s = obj.eig_stats
    print(f"{label}: iterations {s['iterations']} nested {s.get('nested_iterations')} precond {s.get('precond', 'fp32')}")


@pytest.mark.parametrize("name,order", [("box", 1), ("box", 2), ("cube3", 2), ("bowl", 2)])
def test_tensor_eigenpairs_vs_oracle(meshes, name, order):
    obj, _ = _obj(meshes, name, order)
    C, rho = _wood_field(obj, seed=5)
    obj.set_elasticity_field(C, rho)
    obj.eigen_decomposition()
    _report(obj, f"{name} o{order} wood")
    lam, U, _, M, _, _ = _oracle(obj, C, rho, obj.mode_num)
    _check_modes(obj, lam, U, M)


def test_tensor_fp64_clamp_and_locked_batches(meshes):
    fp64, _ = _obj(meshes, "box", 2)
    fp64._sliver = True                     # the sliver policy: straight to the FP64 Chebyshev preconditioner
    C, rho = _wood_field(fp64, seed=6)
    fp64.set_elasticity_field(C, rho)
    fp64.eigen_decomposition()
    assert fp64.eig_stats.get("precond") == "fp64"
    lam, U, _, M, _, _ = _oracle(fp64, C, rho, fp64.mode_num)
    _check_modes(fp64, lam, U, M)
    clamp, _ = _obj(meshes, "box", 2)
    v = clamp.tetmesh.vertices.detach()
    mask = v[:, 0] <= v[:, 0].min() + 1e-6
    C, rho = _wood_field(clamp, seed=7)
    clamp.fix_nodes(mask)
    clamp.set_elasticity_field(C, rho)
    clamp.eigen_decomposition()
    _report(clamp, "box o2 clamped wood")
    lam, U, _, M, _, _ = _oracle(clamp, C, rho, clamp.mode_num, mask)
    _check_modes(clamp, lam, U, M)
    assert float(clamp.U_hat[clamp._fixed_u8.repeat_interleave(3).bool()].abs().max()) == 0.0
    big, _ = _obj(meshes, "box", 2, mode_num=64)
    C, rho = _wood_field(big, seed=8)
    big.set_elasticity_field(C, rho)
    big.eigen_decomposition()
    assert big.eig_stats.get("batches", 1) >= 2
    _report(big, "box o2 wood, 64 modes")
    lam, U, _, M, _, _ = _oracle(big, C, rho, 64)
    _check_modes(big, lam, U, M)


# ------------------------------------------------------------------ 5. gradients through get_vals()
@pytest.mark.parametrize("name,order", [("box", 2), ("bowl", 1), ("cube3", 1)])
def test_tensor_gradients_vs_oracle(meshes, name, order):
    native, _, dm, _ = _mods()
    obj, _ = _obj(meshes, name, order, leaf=True)
    C, rho = (x.clone().requires_grad_(True) for x in _wood_field(obj, seed=9))
    obj.set_elasticity_field(C, rho)
    obj.eigen_decomposition()
    gw = (1.0 / obj.eigenvalues).float()
    pverts = obj.tetmesh.vertices
    pverts.retain_grad()
    (obj.get_vals()[:, 0] * gw).sum().backward()
    lam_h, U_h, _, _, pv, pt = _oracle(obj, C, rho, obj.mode_num)
    gh = gw.double().cpu().numpy()
    rC, rrho = eo.tensor_grads(pv, pt, order, rho.detach().cpu(), U_h, lam_h, gh)
    for got, want in ((C.grad, rC), (rho.grad, rrho)):
        err = np.linalg.norm(got.cpu().numpy() - want) / np.linalg.norm(want)
        assert err <= 1e-5, err
    rv = eo.vertex_grad(pv, pt, order, C.detach().cpu(), rho.detach().cpu(), U_h, lam_h, gh).numpy()
    err = np.linalg.norm(pverts.grad.cpu().numpy() - rv) / np.linalg.norm(rv)
    assert err <= 1e-5, err
    # lambda_i = sum_t <C_t, E_t,i>: strain energy is quadratic in eps
    d = obj.deform
    for i in range(0, obj.mode_num, 5):
        e = torch.zeros(obj.mode_num, dtype=torch.float64, device=DEV)
        e[i] = 1.0
        G21, _ = native.elasticity_field_grad(obj._verts32, d.tets_i32, order, d.m32(), d.wsum, obj.U_hat, obj.eigenvalues, e)
        s = (obj._tensor_used["C"] * G21[:, dm._VOIGT_UNPACK]).sum().item()
        li = obj.eigenvalues[i].item()
        assert abs(s / li - 1) <= (1e-10 if order == 1 else 2e-7), (i, s / li - 1)
    # two backward passes are bitwise equal
    g1 = torch.autograd.grad((obj.get_vals()[:, 0] * gw).sum(), (C, rho))
    g2 = torch.autograd.grad((obj.get_vals()[:, 0] * gw).sum(), (C, rho))
    assert all(torch.equal(a, b) for a, b in zip(g1, g2))


def _solve(meshes, C, rho, name="cube3", order=1, verts=None, tets=None, mode_num=16):
    obj, _ = _obj(meshes, name, order, mode_num=mode_num, verts=verts, tets=tets)
    obj.eig_tol = 1e-9
    obj.set_elasticity_field(C, rho)
    obj.eigen_decomposition()
    return obj


def test_tensor_gradients_vs_central_differences(meshes):
    """d lambda / d(entries of a shared C0), d/d(the nine orthotropic constants) and d/d(grain angle), each through the
    helpers and get_vals(), against central differences of re-solved eigenvalues."""
    _, an, _, _ = _mods()
    obj0, _ = _obj(meshes, "cube3", 1)
    T = obj0.tetmesh.tets.shape[0]
    R = random_rotations(T, 11).to(DEV)
    rho = torch.full((T,), RHO, dtype=torch.float64, device=DEV)
    consts = torch.tensor(list(WOOD.values()), dtype=torch.float64, device=DEV)
    theta0 = 0.4
    axis = [0.3, 0.2, 1.0]

    def build(c, th):
        C0 = an.orthotropic_stiffness(*c)
        return an.rotate_stiffness(an.rotate_stiffness(C0, an.rotation_about(axis, th)).expand(T, 6, 6), R)

    c = consts.clone().requires_grad_(True)
    th = torch.tensor(theta0, dtype=torch.float64, device=DEV, requires_grad=True)
    obj = _solve(meshes, build(c, th), rho)
    w = torch.linspace(1.0, 2.0, obj.mode_num, device=DEV)
    (obj.get_vals()[:, 0] * w).sum().backward()

    def f(cc, tt):
        o = _solve(meshes, build(cc, tt).detach(), rho)
        return float((o.eigenvalues * w.double()).sum())

    for j in (0, 1, 3, 6, 8):                   # E1, E2, nu12, G12, G23
        h = 1e-4 * float(consts[j])
        cp, cm = consts.clone(), consts.clone()
        cp[j] += h
        cm[j] -= h
        fd = (f(cp, theta0) - f(cm, theta0)) / (2 * h)
        assert abs(float(c.grad[j]) / fd - 1) <= 1e-5, (j, float(c.grad[j]), fd)
    h = 1e-4
    fd = (f(consts, theta0 + h) - f(consts, theta0 - h)) / (2 * h)
    assert abs(float(th.grad) / fd - 1) <= 1e-5, (float(th.grad), fd)
    # entries of one C0 shared by every tet (symmetric perturbations)
    def fC(X):
        return float((_solve(meshes, X.expand(T, 6, 6), rho).eigenvalues * w.double()).sum())

    C0 = an.orthotropic_stiffness(*consts).detach().requires_grad_(True)
    obj = _solve(meshes, C0.expand(T, 6, 6), rho)
    (obj.get_vals()[:, 0] * w).sum().backward()
    for (a, b) in ((0, 0), (1, 2), (3, 3), (0, 5)):
        h = 1e-4 * float(C0[a, a])
        D = torch.zeros(6, 6, dtype=torch.float64, device=DEV)
        D[a, b] = D[b, a] = h
        fd = (fC(C0.detach() + D) - fC(C0.detach() - D)) / (2 * h)
        an_ = float(C0.grad[a, b] + (C0.grad[b, a] if a != b else 0.0))
        # against the largest entry: C16 is zero in C0 and its derivative ~1e-5 of the others, where O(h^2) terms show
        assert abs(an_ - fd) <= 1e-5 * float(C0.grad.abs().max()), ((a, b), an_, fd)


# ------------------------------------------------------------------ 6. isotropic tensors = the Lame material field
@pytest.mark.parametrize("order", [1, 2])
def test_isotropic_tensor_field_matches_material_field(meshes, order):
    _, an, _, _ = _mods()
    ref, _ = _obj(meshes, "box", order)
    T = ref.tetmesh.tets.shape[0]
    g = torch.Generator(device=DEV).manual_seed(3)
    E0 = 1e10 * (0.5 + torch.rand(T, dtype=torch.float64, device=DEV, generator=g))
    nu0 = 0.2 + 0.2 * torch.rand(T, dtype=torch.float64, device=DEV, generator=g)
    rho0 = 500.0 * (0.5 + torch.rand(T, dtype=torch.float64, device=DEV, generator=g))
    E1, nu1, r1 = (x.clone().requires_grad_(True) for x in (E0, nu0, rho0))
    ref.eig_tol = 1e-9
    ref.set_material_field(E1, nu1, r1)
    ref.eigen_decomposition()
    w = (1.0 / ref.eigenvalues).float()
    (ref.get_vals()[:, 0] * w).sum().backward()
    E2, nu2, r2 = (x.clone().requires_grad_(True) for x in (E0, nu0, rho0))
    obj, _ = _obj(meshes, "box", order)
    obj.eig_tol = 1e-9
    obj.set_elasticity_field(an.isotropic_stiffness(E2, nu2), r2)
    obj.eigen_decomposition()
    assert ((obj.eigenvalues / ref.eigenvalues - 1).abs().max().item()) <= 1e-10
    (obj.get_vals()[:, 0] * w).sum().backward()
    for a, b in ((E1, E2), (nu1, nu2), (r1, r2)):
        err = (torch.linalg.norm(b.grad - a.grad) / torch.linalg.norm(a.grad)).item()
        assert err <= 1e-8, err


# ------------------------------------------------------------------ 7. rotation invariance on the device
def test_rotating_mesh_and_tensor_on_the_device(meshes):
    _, an, _, _ = _mods()
    v, t = _geometry(meshes, "box")
    obj, _ = _obj(meshes, "box", 2)
    C, rho = _wood_field(obj, seed=12)
    a = _solve(meshes, C, rho, "box", 2)
    # the cyclic turn x -> y -> z -> x moves fp32 vertices exactly; a general rotation rounds them (~6e-8 of the geometry)
    for R, tol in ((torch.tensor([[0., 0., 1.], [1., 0., 0.], [0., 1., 0.]], dtype=torch.float64), 1e-9),
                   (random_rotations(1, 13)[0], 3e-7)):
        vr = (torch.from_numpy(np.asarray(v, np.float64)) @ R.T).float().numpy()
        b = _solve(meshes, an.rotate_stiffness(C, R.to(DEV)), rho, "box", 2, verts=vr, tets=t)
        err = (b.eigenvalues / a.eigenvalues - 1).abs().max().item()
        assert err <= tol, (err, tol)


# ------------------------------------------------------------------ 8. element energies, refusals, clearing
def test_element_energies_refusals_and_clearing(meshes):
    native, an, dm, _ = _mods()
    obj, _ = _obj(meshes, "box", 1)
    C, rho = _wood_field(obj, seed=14)
    obj.set_elasticity_field(C, rho)
    obj.eigen_decomposition()
    strain, kinetic = obj.element_energies()
    T = obj.tetmesh.tets.shape[0]
    assert strain.shape == kinetic.shape == (T, obj.mode_num)
    assert ((strain.sum(0) - obj.eigenvalues).abs() / obj.eigenvalues).max().item() <= 1e-8
    assert (kinetic.sum(0) - 1).abs().max().item() <= 1e-8
    with pytest.raises(NotImplementedError):
        obj.stiff_func(torch.zeros(obj.deform.pattern.n, 1, device=DEV))
    from diffsound_b200.parallel.rowpart_lobpcg import eigen_decomposition_rowpart
    with pytest.raises(NotImplementedError):
        eigen_decomposition_rowpart(obj)
    E = torch.full((T,), 1e10, dtype=torch.float64, device=DEV)
    with pytest.raises(ValueError):
        obj.set_material_field(youngs=E)
    # validation at every assembly: a tensor made indefinite in place is caught
    C2 = C.clone()
    obj.set_elasticity_field(C2)
    C2[0, 3, 3] = -1.0
    with pytest.raises(ValueError):
        obj.eigen_decomposition()
    # cleared: the homogeneous object bitwise
    obj.set_elasticity_field(None)
    obj.eigen_decomposition()
    leaf_obj, v1 = _obj(meshes, "box", 1, leaf=True)
    leaf_obj.set_elasticity_field(C, rho)
    leaf_obj.eigen_decomposition()
    leaf_obj.set_elasticity_field(None)
    leaf_obj.eigen_decomposition()
    ref, v0 = _obj(meshes, "box", 1, leaf=True)
    ref.eigen_decomposition()
    assert torch.equal(obj._Kval, ref._Kval) and torch.equal(obj._Mblk, ref._Mblk)
    assert torch.equal(obj.eigenvalues, ref.eigenvalues)
    w = (1.0 / ref.eigenvalues).float()
    (ref.get_vals()[:, 0] * w).sum().backward()
    (leaf_obj.get_vals()[:, 0] * w).sum().backward()
    assert torch.equal(v0.grad, v1.grad)
    # errors
    fresh, _ = _obj(meshes, "cube3", 1)
    Tf = fresh.tetmesh.tets.shape[0]
    Cf, _ = _wood_field(fresh)
    for bad in (Cf[:-1], Cf.cpu(), Cf.half(), torch.where(torch.arange(Tf, device=DEV)[:, None, None] == 3, float("nan"), Cf)):
        with pytest.raises(ValueError):
            fresh.set_elasticity_field(bad)
    fresh.set_material_field(youngs=torch.full((Tf,), 1e10, dtype=torch.float64, device=DEV))
    with pytest.raises(ValueError):
        fresh.set_elasticity_field(Cf)
    tl, _ = _obj(meshes, "cube3", 1, mat_model=dm.TrainableLinear)
    with pytest.raises(ValueError):
        tl.set_elasticity_field(Cf)


# ------------------------------------------------------------------ 9. the orthotropic bar
def test_orthotropic_bar_on_the_device(meshes):
    f = {}
    for turned in (False, True):
        _, _, C, rho = orthotropic_bar(turned)                  # one C and density for the whole bar
        v, t = kuhn_box((20, 1, 1), (0.4, 0.02, 0.02))
        obj, _ = _obj(meshes, None, 2, verts=v, tets=t)
        C, rho = C.to(DEV), rho.to(DEV)
        obj.set_elasticity_field(C, rho)
        obj.eigen_decomposition()
        lam, U, _, M, _, _ = _oracle(obj, C, rho, obj.mode_num)
        _check_modes(obj, lam, U, M)
        _, f[turned] = longitudinal_mode(obj.eigenvalues.cpu().numpy(), obj.U_hat.cpu().numpy(), M)
    ratio = f[False] / f[True]
    assert abs(ratio / np.sqrt(WOOD["E1"] / WOOD["E2"]) - 1) <= 5e-3, ratio
