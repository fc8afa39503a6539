"""Objects made of more than one material on the B200 (DiffSoundObj.set_material_field, ds_assemble_km_field,
ds_assemble_km_tets_field, ds_eigval_grad_shape_field, ds_material_field_grad, ds_element_energies) against the homogeneous
kernels and the CPU reference of tests/material_field_oracle.py."""
import numpy as np
import pytest
import torch

import fixed_oracle as fo
import material_field_oracle as mf
from oracle import modal_oracle as mo
from test_modal_gains_cpu import kuhn_box

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _mods():
    from diffsound_b200 import native
    from diffsound_b200.diffelastic import diff_model as dm
    from diffsound_b200.diffelastic.material_model import MatSet
    return native, dm, MatSet


def _geometry(meshes, name):
    if name == "box":
        return kuhn_box((6, 3, 2), (0.3, 0.12, 0.06))
    if name.startswith("cube"):
        v, t = mo.kuhn_cube(int(name[4:]))
        return v.numpy(), t.numpy()
    return meshes[name]


def _obj(meshes, name, order, mode_num=16, leaf=False, mat_model=None):
    _, dm, MatSet = _mods()
    v, t = _geometry(meshes, name)
    vt = torch.as_tensor(np.asarray(v), dtype=torch.float32, device=DEV)
    if leaf:
        vt.requires_grad_(True)
    kw = {} if mat_model is None else dict(mat_model=mat_model)
    return dm.DiffSoundObj(vt, torch.as_tensor(np.asarray(t), device=DEV).long(), mode_num=mode_num, order=order,
                           mat=MatSet.Steel, **kw), vt


def _centroids(obj):
    from diffsound_b200.diffelastic.shape_func import CORNER_LOCAL
    v = obj.tetmesh.vertices.detach().double()
    return v[obj.tetmesh.tets[:, list(CORNER_LOCAL[obj.tetmesh.order])]].mean(1)


def _field(obj, kind, seed=0):
    """(youngs, poisson, density) fp64 CUDA tensors of one of the test fields."""
    _, dm, MatSet = _mods()
    T = obj.tetmesh.tets.shape[0]
    c = _centroids(obj)
    rho, E, nu = MatSet.Steel[:3]
    if kind == "constant":
        return (torch.full((T,), E, dtype=torch.float64, device=DEV), torch.full((T,), nu, dtype=torch.float64, device=DEV),
                torch.full((T,), rho, dtype=torch.float64, device=DEV))
    if kind == "two":                       # steel | wood across the middle of the longest axis
        ax = int(torch.argmax(c.max(0).values - c.min(0).values))
        mid = 0.5 * (c[:, ax].max() + c[:, ax].min())
        return dm.material_field_from_regions((c[:, ax] > mid).long(), [MatSet.Steel, MatSet.Wood])
    if kind == "random":                    # log-normal: E x [0.3, 3], nu in [0.2, 0.4], rho x [0.5, 2]
        g = torch.Generator(device=DEV).manual_seed(seed)
        u = torch.rand(3, T, dtype=torch.float64, device=DEV, generator=g)
        return (E * torch.exp(np.log(0.3) + u[0] * np.log(10.0)), 0.2 + 0.2 * u[1],
                rho * torch.exp(np.log(0.5) + u[2] * np.log(4.0)))
    if kind == "inclusion":                 # a 100x stiffer core
        lo, hi = c.min(0).values, c.max(0).values
        core = (((c - 0.5 * (lo + hi)) / (hi - lo)).abs() < 0.2).all(1)
        youngs = torch.where(core, 100.0 * E, E)
        return youngs, torch.full((T,), nu, dtype=torch.float64, device=DEV), torch.full((T,), rho, dtype=torch.float64,
                                                                                         device=DEV)
    raise ValueError(kind)


def _host(obj):
    return obj.tetmesh.vertices.detach().cpu(), obj.tetmesh.tets.cpu().long()


def _cpu(f):
    return tuple(x.detach().cpu() for x in f)


# ------------------------------------------------------------------ 1. a constant field is the homogeneous object
@pytest.mark.parametrize("name,order", [("cube3", 1), ("cube3", 2), ("box", 2), ("bowl", 1), ("bowl", 2)])
def test_constant_field_assembly_is_bitwise_homogeneous(meshes, name, order):
    native, dm, MatSet = _mods()
    obj, _ = _obj(meshes, name, order)
    d = obj.deform
    rho, E, nu = MatSet.Steel[:3]
    mu, lam = dm._lame(E, nu)
    T = d.num_tets
    f64 = dict(dtype=torch.float64, device=DEV)
    field = (torch.full((T,), mu, **f64), torch.full((T,), lam, **f64), torch.full((T,), rho, dtype=torch.float32, device=DEV))
    v32 = d.verts_f32()
    kernels = ["rows", "tets"] if order == 2 else ["rows"]
    for kernel in kernels:
        K0, M0 = native.assemble_km(v32, d.tets_i32, order, d.pattern, mu, lam, d.ctab, d.mtab(rho), kernel=kernel)
        K1, M1 = native.assemble_km(v32, d.tets_i32, order, d.pattern, 0.0, 0.0, d.ctab, d.m32(), kernel=kernel, field=field)
        assert torch.equal(K0, K1) and torch.equal(M0, M1), kernel
    if order == 2:
        co = d.coarse
        co.assemble(v32, mu, lam, co.ctab, d.coarse_mtab(rho))
        K0, M0 = co.Kval.clone(), co.Mblk.clone()
        co.assemble(v32, 0.0, 0.0, co.ctab, d.m32(1), field=field)
        assert torch.equal(K0, co.Kval) and torch.equal(M0, co.Mblk)


@pytest.mark.parametrize("name,order", [("cube3", 2), ("bowl", 1)])
def test_constant_field_solve_and_gradients(meshes, name, order):
    native, dm, _ = _mods()
    ref, v0 = _obj(meshes, name, order, leaf=True)
    ref.eigen_decomposition()
    gw = (1.0 / ref.eigenvalues).float()
    (ref.get_vals()[:, 0] * gw).sum().backward()
    obj, v1 = _obj(meshes, name, order, leaf=True)
    youngs, poisson, density = (x.clone().requires_grad_(True) for x in _field(obj, "constant"))
    obj.set_material_field(youngs, poisson, density)
    obj.eigen_decomposition()
    assert torch.equal(obj._Kval, ref._Kval) and torch.equal(obj._Mblk, ref._Mblk)
    err = ((obj.eigenvalues - ref.eigenvalues).abs() / ref.eigenvalues).max().item()
    assert err <= 1e-12, err
    (obj.get_vals()[:, 0] * gw).sum().backward()
    gerr = (torch.linalg.norm(v1.grad - v0.grad) / torch.linalg.norm(v0.grad)).item()
    assert gerr <= 1e-7, gerr                   # one fp32 rounding of the mass table product (m_ab * rho)
    # the per-tet (mu, lam) forms sum to the global material forms
    d = obj.deform
    g = torch.rand(obj.mode_num, dtype=torch.float64, device=DEV)
    G = native.material_field_grad(obj._verts32, d.tets_i32, order, d.m32(), d.wsum, obj.U_hat, obj.eigenvalues, g)
    q_mu, q_la, _ = native.eigval_quadforms_material(obj._verts32, d.tets_i32, order, d.mtab(obj._density_used), d.wsum,
                                                     obj.U_hat)
    for got, want in ((G[:, 0].sum(), (g * q_mu).sum()), (G[:, 1].sum(), (g * q_la).sum())):
        assert abs(got.item() - want.item()) <= 1e-12 * abs(want.item())


# ------------------------------------------------------------------ 2. assembly against the reference
@pytest.mark.parametrize("name,order", [("cube3", 1), ("cube3", 2), ("bowl", 1)])
@pytest.mark.parametrize("kind", ["two", "random"])
def test_field_assembly_vs_oracle(meshes, name, order, kind):
    obj, _ = _obj(meshes, name, order)
    f = _field(obj, kind)
    obj.set_material_field(*f)
    obj.update_mass_matrix(7850.0)
    pv, pt = _host(obj)
    E, nu, rho = _cpu(f)
    K, M = mf.assemble_field(pv, pt, order, E, nu, rho)
    Kg = obj.stiff_matrix.values().cpu().numpy()
    Mg = obj.mass_matrix.values().cpu().numpy()
    assert np.abs(Kg - K.data).max() <= 2e-6 * np.abs(K.data).max()
    assert np.abs(Mg - M.data).max() <= 1e-12 * np.abs(M.data).max()


# ------------------------------------------------------------------ 3. kernels with a random U
@pytest.mark.parametrize("name,order", [("cube3", 1), ("cube3", 2), ("bowl", 1)])
@pytest.mark.parametrize("k", [16, 32, 64])
def test_field_kernels_with_random_modes(meshes, name, order, k):
    native, _, _ = _mods()
    obj, _ = _obj(meshes, name, order)
    E, nu, rho = _field(obj, "random", seed=k)
    obj.set_material_field(E, nu, rho)
    obj.update_mass_matrix(7850.0)
    d = obj.deform
    f = obj._field_used
    n = d.pattern.n
    gen = torch.Generator(device=DEV).manual_seed(k)
    wide = torch.randn(n, k + 8, dtype=torch.float64, device=DEV, generator=gen)
    U = wide[:, 3:3 + k]                                      # read in place through its leading dimension
    lam = 1e6 * (1.0 + torch.rand(k, dtype=torch.float64, device=DEV, generator=gen))
    g = torch.randn(k, dtype=torch.float64, device=DEV, generator=gen)
    G = native.material_field_grad(obj._verts32, d.tets_i32, order, d.m32(), d.wsum, U, lam, g)
    strain, kinetic = native.element_energies(obj._verts32, d.tets_i32, order, d.m32(), d.wsum, U, (f["mu"], f["lam"], f["rho"]))
    pv, pt = _host(obj)
    Uh = U.cpu().numpy()
    q_mu, q_la, q_m = mf.element_forms(pv, pt, order, Uh)
    gh, lh = g.cpu().numpy(), lam.cpu().numpy()
    want = np.stack([q_mu @ gh, q_la @ gh, -(q_m @ (gh * lh))], axis=1)
    Gh = G.cpu().numpy()
    for c in range(3):
        assert np.abs(Gh[:, c] - want[:, c]).max() <= 1e-12 * np.abs(want[:, c]).max(), c
    mu_t, lam_t = f["mu"].cpu().numpy(), f["lam"].cpu().numpy()
    s_want = mu_t[:, None] * q_mu + lam_t[:, None] * q_la
    k_want = mf.element_forms(pv, pt, order, Uh, density=rho.cpu())[2]
    assert np.abs(strain.cpu().numpy() - s_want).max() <= 1e-12 * np.abs(s_want).max()
    assert np.abs(kinetic.cpu().numpy() - k_want).max() <= 1e-12 * np.abs(k_want).max()
    # summed over the tets: the quadratic forms of the assembled operator (P1: same quadrature; P2: the assembly's fp32
    # Gauss rule against the exact one, ~5e-8) and of M (the same table entries)
    Uc = U.contiguous()
    KU, MU = native.spmm_k_and_m(d.pattern, obj._Kval, obj._Mblk, Uc)
    uku, umu = (Uc * KU).sum(0), (Uc * MU).sum(0)
    tol_k = 1e-12 if order == 1 else 2e-7
    assert ((strain.sum(0) - uku).abs() / uku.abs()).max().item() <= tol_k
    assert ((kinetic.sum(0) - umu).abs() / umu.abs()).max().item() <= 1e-12
    # no atomics: a second run is bitwise equal
    G2 = native.material_field_grad(obj._verts32, d.tets_i32, order, d.m32(), d.wsum, U, lam, g)
    s2, k2 = native.element_energies(obj._verts32, d.tets_i32, order, d.m32(), d.wsum, U, (f["mu"], f["lam"], f["rho"]))
    assert torch.equal(G, G2) and torch.equal(strain, s2) and torch.equal(kinetic, k2)


# ------------------------------------------------------------------ 4. eigenvalues against ARPACK
def _oracle_eigs(obj, f, k, mask=None):
    pv, pt = _host(obj)
    E, nu, rho = _cpu(f)
    K, M = mf.assemble_field(pv, pt, obj.tetmesh.order, E, nu, rho)
    if mask is not None:
        lam, U = fo.eig_fixed(K, M, mask.cpu().numpy(), k)
    else:
        lam, U, _, _ = mo.eig_arpack(K, M, k, sigma=-1e3)
    return lam, U, pv, pt


def _report(obj, label):
    s = obj.eig_stats
    print(f"{label}: iterations {s['iterations']} nested {s.get('nested_iterations')} precond {s.get('precond', 'fp32')}")


@pytest.mark.parametrize("name,order", [("box", 2), ("bowl", 1)])
@pytest.mark.parametrize("kind", ["two", "random", "inclusion"])
def test_field_eigenvalues_vs_arpack(meshes, name, order, kind):
    ref, _ = _obj(meshes, name, order)
    ref.eigen_decomposition()
    _report(ref, f"{name} o{order} homogeneous")
    obj, _ = _obj(meshes, name, order)
    f = _field(obj, kind)
    obj.set_material_field(*f)
    obj.eigen_decomposition()
    _report(obj, f"{name} o{order} {kind}")
    lam, _, _, _ = _oracle_eigs(obj, f, obj.mode_num)
    err = (np.abs(obj.eigenvalues.cpu().numpy() - lam) / lam).max()
    assert err <= 1e-6, err


def test_field_with_clamp_batches_and_fp64(meshes):
    """fix_nodes + a field; more modes than one block holds (batched solve); the FP64 preconditioner path."""
    obj, _ = _obj(meshes, "box", 2, mode_num=44)
    f = _field(obj, "two")
    obj.set_material_field(*f)
    obj.eigen_decomposition()
    _report(obj, "box o2 two, 44 modes")
    lam, _, _, _ = _oracle_eigs(obj, f, 44)
    assert (np.abs(obj.eigenvalues.cpu().numpy() - lam) / lam).max() <= 1e-6
    clamp, _ = _obj(meshes, "box", 1)
    v = clamp.tetmesh.vertices.detach()
    mask = v[:, 0] <= v[:, 0].min() + 1e-6
    fc = _field(clamp, "random")
    clamp.fix_nodes(mask)
    clamp.set_material_field(*fc)
    clamp.eigen_decomposition()
    _report(clamp, "box o1 clamped random")
    lam, _, _, _ = _oracle_eigs(clamp, fc, clamp.mode_num, mask)
    assert (np.abs(clamp.eigenvalues.cpu().numpy() - lam) / lam).max() <= 1e-6
    fp64, _ = _obj(meshes, "box", 2)
    fp64._sliver = True                     # the sliver policy: straight to the FP64 Chebyshev preconditioner
    fr = _field(fp64, "random")
    fp64.set_material_field(*fr)
    fp64.eigen_decomposition()
    assert fp64.eig_stats.get("precond") == "fp64"
    lam, _, _, _ = _oracle_eigs(fp64, fr, fp64.mode_num)
    assert (np.abs(fp64.eigenvalues.cpu().numpy() - lam) / lam).max() <= 1e-6


# ------------------------------------------------------------------ 5. gradients through get_vals()
@pytest.mark.parametrize("name,order", [("box", 2), ("bowl", 1), ("cube3", 1)])
def test_field_gradients_vs_oracle(meshes, name, order):
    obj, _ = _obj(meshes, name, order, leaf=True)
    E, nu, rho = (x.clone().requires_grad_(True) for x in _field(obj, "random", seed=7))
    obj.set_material_field(E, nu, rho)
    obj.eigen_decomposition()
    lam = obj.eigenvalues
    gw = (1.0 / lam).float()
    pverts = obj.tetmesh.vertices                       # the promoted nodes the reference differentiates
    pverts.retain_grad()
    (obj.get_vals()[:, 0] * gw).sum().backward()
    lam_h, U_h, pv, pt = _oracle_eigs(obj, (E, nu, rho), obj.mode_num)
    gh = gw.double().cpu().numpy()
    rE, rnu, rrho = mf.field_grads(pv, pt, order, E.detach().cpu(), nu.detach().cpu(), U_h, lam_h, gh)
    for got, want in ((E.grad, rE), (nu.grad, rnu), (rho.grad, rrho)):
        err = np.linalg.norm(got.cpu().numpy() - want) / np.linalg.norm(want)
        assert err <= 1e-5, err
    with mo.inverse_precision(torch.float64):          # the kernel's arithmetic (test_grad_synth_gpu: fp32-inverse floor)
        rv = mf.vertex_grad(pv, pt, order, E.detach().cpu(), nu.detach().cpu(), rho.detach().cpu(), U_h, lam_h, gh).numpy()
    err = np.linalg.norm(pverts.grad.cpu().numpy() - rv) / np.linalg.norm(rv)
    assert err <= 1e-5, err
    # Euler identities on the solved modes: lambda is homogeneous of degree 1 in E and -1 in rho.  The per-tet forms
    # integrate exactly; K of a quadratic mesh uses the fp32 Gauss rule (~5e-8 apart).  M holds float32(m_ab) *
    # float32(rho_t) per table entry, the rho gradient the exact product: one fp32 rounding (2^-24 = 6e-8) apart at most.
    # Only the field inputs are differentiated here: the promotion of a quadratic mesh's vertices is a graph the first
    # backward above has already consumed.
    for i in range(0, obj.mode_num, 5):
        gE, gR = torch.autograd.grad(obj.get_vals()[i, 0], (E, rho))
        li = lam[i].item()
        sE = (E.detach() * gE).sum().item()
        sR = (rho.detach() * gR).sum().item()
        assert abs(sE / li - 1) <= (1e-8 if order == 1 else 2e-7), (i, sE / li - 1)     # measured P1: <= 5e-14
        assert abs(sR / li + 1) <= 6e-8, (i, sR / li + 1)     # measured: <= 8.6e-9 (cube3), 5.6e-10 (bowl)
        print(f"{name} o{order} mode {i}: Euler E {sE / li - 1:.2e}, rho {sR / li + 1:.2e}")


def test_element_energies_of_solved_modes(meshes):
    obj, _ = _obj(meshes, "box", 1)
    obj.set_material_field(*_field(obj, "two"))
    obj.eigen_decomposition()
    strain, kinetic = obj.element_energies()
    T = obj.tetmesh.tets.shape[0]
    assert strain.shape == kinetic.shape == (T, obj.mode_num) and strain.dtype == torch.float64
    lam = obj.eigenvalues
    assert ((strain.sum(0) - lam).abs() / lam).max().item() <= 1e-8
    assert (kinetic.sum(0) - 1).abs().max().item() <= 1e-8
    # the strike response runs on the composite's M-normalised modes
    y = obj.impulse_response(torch.tensor([[0.15, 0.06, 0.06]], device=DEV), 512, 44100.0)
    assert y.shape == (1, 512) and bool(torch.isfinite(y).all()) and float(y.abs().max()) > 0
    obj.set_material_field(None)
    assert obj.material_field is None and obj._field_used is None


# ------------------------------------------------------------------ 6. warm start across a field change
def test_warm_start_after_field_change(meshes):
    obj, _ = _obj(meshes, "box", 2)
    E, nu, rho = _field(obj, "random", seed=3)
    obj.set_material_field(E, nu, rho)
    obj.eigen_decomposition()
    with torch.no_grad():
        E.mul_(1.01)                                    # an optimiser step in place
        rho.mul_(0.99)
    assert len(obj._warm) == 1
    obj.eigen_decomposition()
    assert obj.eig_stats.get("nested_iterations", 0) == 0       # warm: no nested start
    cold, _ = _obj(meshes, "box", 2)
    cold.set_material_field(E.clone(), nu.clone(), rho.clone())
    cold.eigen_decomposition()
    err = ((obj.eigenvalues - cold.eigenvalues).abs() / cold.eigenvalues).max().item()
    assert err <= 1e-6, err


# ------------------------------------------------------------------ 7. errors
def test_field_errors(meshes):
    _, dm, _ = _mods()
    obj, _ = _obj(meshes, "cube3", 1)
    T = obj.tetmesh.tets.shape[0]
    E, nu, rho = _field(obj, "constant")
    for kw in (dict(youngs=E[:-1]), dict(youngs=E.cpu()), dict(density=-rho), dict(poisson=nu + 0.3),
               dict(youngs=torch.where(torch.arange(T, device=DEV) == 3, float("nan"), E))):
        with pytest.raises(ValueError):
            obj.set_material_field(**kw)
    assert obj.material_field is None
    # a field changed in place to an invalid value is caught at the next assembly
    E2 = E.clone()
    obj.set_material_field(youngs=E2)
    E2[0] = -1.0
    with pytest.raises(ValueError):
        obj.eigen_decomposition()
    obj.set_material_field(youngs=E)
    with pytest.raises(NotImplementedError):
        obj.stiff_func(torch.zeros(obj.deform.pattern.n, 1, device=DEV))
    from diffsound_b200.parallel.rowpart_lobpcg import eigen_decomposition_rowpart
    with pytest.raises(NotImplementedError):
        eigen_decomposition_rowpart(obj)
    tl, _ = _obj(meshes, "cube3", 1, mat_model=dm.TrainableLinear)
    with pytest.raises(ValueError):
        tl.set_material_field(youngs=E)
