"""Objects on elastic supports on the B200 (DiffSoundObj.set_supports, ds_support_km / _grad / _energies) against the
kernel-free reference of tests/support_oracle.py."""
import numpy as np
import pytest
import torch

import support_oracle as so
from oracle import modal_oracle as mo
from test_fixed_gpu import _check_modes, _sphere
from test_modal_gains_cpu import kuhn_box

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _mods():
    from diffsound_b200 import native
    from diffsound_b200.diffelastic.diff_model import DiffSoundObj
    from diffsound_b200.diffelastic.material_model import MatSet
    return native, DiffSoundObj, MatSet


def _obj(v, t, order, mode_num, leaf=False):
    _, DiffSoundObj, MatSet = _mods()
    vt = torch.as_tensor(np.asarray(v), dtype=torch.float32, device=DEV)
    if leaf:
        vt.requires_grad_(True)
    return DiffSoundObj(vt, torch.as_tensor(np.asarray(t), device=DEV).long(), mode_num=mode_num, order=order,
                        mat=MatSet.Steel), vt


def _bottom(obj, frac=0.0):
    """Mask over surface() of the faces whose corners all lie within frac * height of the lowest z."""
    faces = obj.surface()[0]
    z = obj.tetmesh.vertices.detach()[:, 2]
    tol = 1e-6 + frac * float(z.max() - z.min())
    return (z[faces] <= z.min() + tol).all(dim=1)


def _bar():
    return kuhn_box((16, 3, 2), (0.5, 0.06, 0.04))


def _oracle(obj, fmask, kn, kt, k, fixed=None):
    _, _, MatSet = _mods()
    rho, E, nu = MatSet.Steel[:3]
    pv = obj.tetmesh.vertices.detach().cpu()
    pt = obj.tetmesh.tets.cpu().long()
    _, owner, local = (x.cpu().numpy() for x in obj.surface())
    sel = fmask.cpu().numpy()
    K, M = mo.assemble(pv, pt, obj.tetmesh.order, E, nu, rho)
    Ks = so.support_matrix(pv.double().numpy(), pt.numpy(), obj.tetmesh.order, owner[sel], local[sel], kn, kt)
    lam, U = so.eig_supported(K, M, Ks, k, fixed)
    return K, M, Ks, lam, U, owner[sel], local[sel]


def _kval_of(pattern, A):
    """A (scipy) read at the pattern's (row, col) positions, in Kval order."""
    r, c = (x.cpu().numpy() for x in pattern.coo_indices())
    A = A.tocoo()
    n = A.shape[1]
    key = A.row.astype(np.int64) * n + A.col
    order = np.argsort(key, kind="stable")
    ukey, start = np.unique(key[order], return_index=True)
    val = np.add.reduceat(A.data[order], start)
    want = r * n + c
    pos = np.searchsorted(ukey, want).clip(0, ukey.size - 1)
    return np.where(ukey[pos] == want, val[pos], 0.0)


def _bitwise_symmetric(pattern, Kval):
    r, c = pattern.coo_indices()
    n = pattern.n
    key = r * n + c
    tkey = c * n + r
    order = torch.argsort(key)
    pos = torch.searchsorted(key[order], tkey)
    return torch.equal(Kval, Kval[order[pos]])


@pytest.mark.parametrize("order", [1, 2])
def test_support_km_against_oracle(order):
    native, _, _ = _mods()
    v, t = _bar()
    obj, _ = _obj(v, t, order, 12)
    obj.update_stiff_matrix()
    fm = _bottom(obj)
    kn = torch.linspace(2e9, 4e9, int(fm.sum()), dtype=torch.float64, device=DEV)
    obj.set_supports(fm, kn, 5e8)
    # the spring bed alone: the kernel run on a zero Kval (K - K0 would carry the volume part's rounding)
    Kz = native.support_km(obj._verts32, obj.deform.tets_i32, obj.deform.pattern, obj._sup["fine"], obj._sup_used["kn"],
                           obj._sup_used["kt"], torch.zeros_like(obj._Kval))
    Ks = Kz.cpu().numpy()
    pv = obj.tetmesh.vertices.detach().cpu().double().numpy()
    _, own, loc = (x.cpu().numpy() for x in obj.surface())
    sel = fm.cpu().numpy()
    Kref = so.support_matrix(pv, obj.tetmesh.tets.cpu().numpy(), order, own[sel], loc[sel], kn.cpu().numpy(), 5e8)
    ref = _kval_of(obj.deform.pattern, Kref)
    assert np.abs(Ks - ref).max() <= 1e-13 * np.abs(ref).max()
    # blocks (i, j) and (j, i) receive the same values in the same order: a symmetric K stays bitwise so
    assert _bitwise_symmetric(obj.deform.pattern, Kz)
    K1 = obj._Kval.clone()
    obj.update_stiff_matrix()
    assert torch.equal(obj._Kval, K1)                      # bitwise reproducible
    if order == 2:                                          # the P1 coarse level: corner nodes, coarse numbering
        c = obj.deform.coarse
        mu, la = obj._lame_used
        mt = obj.deform.coarse_mtab(obj._density_used)
        c.fixed = None
        c.assemble(obj._verts32, mu, la, c.ctab, mt, supports=(obj._support_faces_coarse(), obj._sup_used["kn"],
                                                               obj._sup_used["kt"]))
        Kcz = native.support_km(c.verts, c.tets, c.pattern, obj._support_faces_coarse(), obj._sup_used["kn"],
                                obj._sup_used["kt"], torch.zeros_like(c.Kval))
        cv = c.verts.double().cpu().numpy()
        Kcref = so.support_matrix(cv, c.tets.cpu().numpy(), 1, own[sel], loc[sel], kn.cpu().numpy(), 5e8)
        refc = _kval_of(c.pattern, Kcref)
        assert np.abs(Kcz.cpu().numpy() - refc).max() <= 1e-13 * np.abs(refc).max()
        assert _bitwise_symmetric(c.pattern, Kcz)


@pytest.mark.parametrize("name,order,k,fp64", [("bar", 1, 16, False), ("bar", 2, 16, False), ("bowl", 2, 12, False),
                                               ("sphere", 1, 12, False), ("bar", 2, 16, True), ("bar", 2, 64, False)])
def test_eigenpairs_against_oracle(meshes, name, order, k, fp64):
    v, t = _bar() if name == "bar" else (_sphere() if name == "sphere" else meshes[name])
    obj, _ = _obj(v, t, order, k)
    obj.fp64_fallback = True
    if fp64:
        obj.sliver_ratio = 2.0          # every mesh counts as sliver-laden: straight to the FP64 preconditioner
    fm = _bottom(obj, 0.05 if name != "bar" else 0.0)
    obj.set_supports(fm, 3e9, 1e9)
    obj.eigen_decomposition()
    if fp64:
        assert obj.eig_stats["precond"] == "fp64"
    _, M, _, lam, U, _, _ = _oracle(obj, fm, 3e9, 1e9, k)
    _check_modes(obj, torch.zeros(obj.deform.num_nodes, dtype=torch.bool), lam, U, M)


@pytest.mark.parametrize("variant", ["clamps", "lame", "tensor"])
def test_supports_combine(variant):
    from diffsound_b200.diffelastic.anisotropic import isotropic_stiffness
    v, t = _bar()
    obj, _ = _obj(v, t, 2, 12)
    fm = _bottom(obj)
    fixed = None
    _, _, MatSet = _mods()
    rho, E, nu = MatSet.Steel[:3]
    T = obj.deform.num_tets
    if variant == "clamps":
        x = obj.tetmesh.vertices.detach()[:, 0]
        fixed = x >= x.max() - 1e-6
        obj.fix_nodes(fixed)
        obj.set_supports(fm, 3e9, 0.0)            # the clamps hold the sliding motions
    else:
        if variant == "lame":
            obj.set_material_field(torch.full((T,), E, dtype=torch.float64, device=DEV), None, None)
        else:
            obj.set_elasticity_field(isotropic_stiffness(torch.tensor(E, dtype=torch.float64),
                                                         torch.tensor(nu, dtype=torch.float64)).to(DEV).expand(T, 6, 6))
        obj.set_supports(fm, 3e9, 1e9)
    obj.eigen_decomposition()
    _, M, _, lam, U, _, _ = _oracle(obj, fm, 3e9, 0.0 if variant == "clamps" else 1e9, 12,
                                    None if fixed is None else fixed.cpu().numpy())
    _check_modes(obj, torch.zeros(obj.deform.num_nodes, dtype=torch.bool, device=DEV) if fixed is None else fixed,
                 lam, U, M)


def test_ordering_free_supported_clamped():
    v, t = _bar()
    lams = []
    for kn in (None, 1e8, 1e10, 1e12, 1e14, "clamp"):
        obj, _ = _obj(v, t, 2, 12)
        fm = _bottom(obj)
        if kn == "clamp":
            z = obj.tetmesh.vertices.detach()[:, 2]
            obj.fix_nodes(z <= z.min() + 1e-6)              # every node of the support faces, mid-edge nodes included
        elif kn is not None:
            obj.set_supports(fm, kn, kn / 3)
        obj.eigen_decomposition()
        lams.append(obj.eigenvalues.cpu().numpy())
    free = np.concatenate([np.zeros(6), lams[0]])[:12]     # the free object's six rigid modes at 0
    for a, b in zip([free] + lams[1:-1], lams[1:]):
        assert np.all(a <= b * (1 + 1e-9)), (a, b)
    # as the bed stiffens the spectrum closes in on the clamped one
    gaps = [np.abs(lam - lams[-1]).max() / lams[-1].max() for lam in lams[1:-1]]
    assert all(a > b for a, b in zip(gaps, gaps[1:])) and gaps[-1] <= 0.1, gaps


def test_rigid_limit_and_heave_gain():
    """A steel block on a soft bed (bed modes ~1e-6 of the first elastic one): the six lowest modes are the rigid-body pencil
    (R^T K_s R, R^T M R); the heave mode's gain at the top centre is 1 / sqrt(m)."""
    v, t = kuhn_box((4, 4, 4), (0.1, 0.1, 0.1))
    obj, _ = _obj(v, t, 2, 8)
    fm = _bottom(obj)
    kn, kt = 1e7, 4e6
    obj.set_supports(fm, kn, kt)
    obj.eigen_decomposition()
    _, _, Ks, _, _, _, _ = _oracle(obj, fm, kn, kt, 1)
    _, M = mo.assemble(obj.tetmesh.vertices.detach().cpu(), obj.tetmesh.tets.cpu().long(), 2, 1.0, 0.3,
                       float(obj.material_model.mat.density))
    import scipy.linalg as sla
    R = so.rigid_fields(obj.tetmesh.vertices.detach().cpu().double().numpy())
    lam_r = sla.eigh(R.T @ (Ks @ R), R.T @ (M @ R), eigvals_only=True)
    lam = obj.eigenvalues.cpu().numpy()[:6]
    assert np.abs(lam - lam_r).max() / lam_r.max() <= 1e-4, (lam, lam_r)
    mass = float(obj.material_model.mat.density) * 1e-3
    g = obj.modal_gains(torch.tensor([[0.05, 0.05, 0.1]], device=DEV)).abs()[0].cpu().numpy()
    heave = int(np.argmax(g[:6]))
    assert abs(g[heave] * np.sqrt(mass) - 1) <= 1e-3, g


@pytest.mark.parametrize("order", [1, 2])
def test_gradients_against_oracle_and_fd(order):
    v, t = _bar()
    obj, leaf = _obj(v, t, order, 12, leaf=True)
    fm = _bottom(obj)
    S = int(fm.sum())
    kn = torch.linspace(2e9, 3e9, S, dtype=torch.float64, device=DEV).requires_grad_(True)
    kt = torch.linspace(5e8, 8e8, S, dtype=torch.float64, device=DEV).requires_grad_(True)
    obj.set_supports(fm, kn, kt)
    obj.eigen_decomposition()
    g = torch.linspace(1.0, 2.0, 12, device=DEV)
    (obj.get_vals()[:, 0] * g / obj.eigenvalues.float()).sum().backward()
    gw = (g.double() / obj.eigenvalues).cpu().numpy()
    _, _, _, lam, U, own, loc = _oracle(obj, fm, kn.detach().cpu().numpy(), kt.detach().cpu().numpy(), 12)
    U_gpu = obj.U_hat.cpu().numpy()
    pv = obj.tetmesh.vertices.detach().cpu().double().numpy()
    pt = obj.tetmesh.tets.cpu().numpy()
    gn, gt, gv = so.support_grads(pv, pt, order, own, loc, kn.detach().cpu().numpy(), kt.detach().cpu().numpy(), U_gpu, gw)
    rel = lambda a, b: np.linalg.norm(a - b) / np.linalg.norm(b)
    assert rel(kn.grad.cpu().numpy(), gn) <= 1e-5 and rel(kt.grad.cpu().numpy(), gt) <= 1e-5
    _, _, MatSet = _mods()
    rho, E, nu = MatSet.Steel[:3]
    gvol = mo.eigval_grad_shape(obj.tetmesh.vertices.detach().cpu(), obj.tetmesh.tets.cpu().long(), order, E, nu, rho,
                                U_gpu, obj.eigenvalues.cpu().numpy(), gw).numpy()
    if order == 1:
        assert rel(leaf.grad.cpu().numpy(), gvol + gv) <= 1e-5
    # central differences of sum_i w_i lambda_i in one face's k_n
    s = S // 2
    h = 1e-3 * float(kn[s])
    vals = []
    for sgn in (1, -1):
        o2, _ = _obj(v, t, order, 12)
        k2 = kn.detach().clone()
        k2[s] += sgn * h
        o2.set_supports(fm, k2, kt.detach())
        o2.eigen_decomposition()
        vals.append(float((o2.eigenvalues * torch.as_tensor(gw, device=DEV)).sum()))
    fd = (vals[0] - vals[1]) / (2 * h)
    assert abs(fd - float(kn.grad[s])) <= 1e-5 * np.abs(gn).max(), (fd, float(kn.grad[s]))


@pytest.mark.parametrize("order,floor", [(1, 1e-8), (2, 3e-8)])
def test_euler_identity_and_energy_partition(order, floor):
    v, t = _bar()
    obj, _ = _obj(v, t, order, 12)
    _, _, MatSet = _mods()
    E = MatSet.Steel[1]
    T = obj.deform.num_tets
    youngs = torch.full((T,), E, dtype=torch.float64, device=DEV, requires_grad=True)
    obj.set_material_field(youngs, None, None)
    fm = _bottom(obj)
    S = int(fm.sum())
    kn = torch.full((S,), 3e9, dtype=torch.float64, device=DEV, requires_grad=True)
    kt = torch.full((S,), 1e9, dtype=torch.float64, device=DEV, requires_grad=True)
    obj.set_supports(fm, kn, kt)
    obj.eigen_decomposition()
    lam = obj.eigenvalues
    strain, _ = obj.element_energies()
    sup = obj.support_energies()
    assert sup.shape == (S, 12)
    assert float(((strain.sum(0) + sup.sum(0) - lam).abs() / lam).max()) <= floor
    for i in (0, 5, 11):
        for x in (youngs, kn, kt):
            x.grad = None
        obj.get_vals()[i, 0].backward()
        euler = (youngs * youngs.grad).sum() + (kn * kn.grad).sum() + (kt * kt.grad).sum()
        assert abs(float(euler) / float(lam[i]) - 1) <= floor, (i, float(euler), float(lam[i]))
    # get_undamped_freqs: still sqrt(lambda) / 2 pi (gt task: no add term; the support energy enters the material path)
    f = obj.get_undamped_freqs()[:, 0].double()
    assert torch.allclose(f, torch.sqrt(lam) / (2 * np.pi), rtol=1e-6)


def test_undamped_freqs_trainable():
    from diffsound_b200.diffelastic.diff_model import TrainableLinear
    _, DiffSoundObj, MatSet = _mods()
    v, t = _bar()
    obj = DiffSoundObj(torch.as_tensor(v, device=DEV), torch.as_tensor(t, device=DEV), mode_num=12, order=1,
                       mat=MatSet.Steel, mat_model=TrainableLinear, task="material")
    obj.init_material_coeffs(steps=200, verbose=False)
    obj.set_supports(_bottom(obj), 3e9, 1e9)
    obj.eigen_decomposition()
    f = obj.get_undamped_freqs()[:, 0].double()
    assert torch.allclose(f, torch.sqrt(obj.eigenvalues) / (2 * np.pi), rtol=1e-5)


def test_refusals_and_clear_is_bitwise():
    native, _, _ = _mods()
    v, t = _bar()
    ref, _ = _obj(v, t, 2, 12)
    ref.eigen_decomposition()
    obj, _ = _obj(v, t, 2, 12)
    fm = _bottom(obj)
    with pytest.raises(ValueError, match="rigid motion"):
        obj.set_supports(fm, 3e9, 0.0)                     # a flat bed without shear: the object slides
    assert obj.supports is None
    with pytest.raises(ValueError, match=">= 0"):
        obj.set_supports(fm, -1.0, 1.0)
    with pytest.raises(ValueError, match="mask"):
        obj.set_supports(fm[:-1], 1.0, 1.0)
    with pytest.raises(ValueError, match="shape"):
        obj.set_supports(fm, torch.ones(3, device=DEV), 1.0)
    obj.set_supports(fm, 3e9, 1e9)
    obj.eigen_decomposition()
    with pytest.raises(NotImplementedError):
        obj.stiff_func(torch.zeros(obj.deform.pattern.n, device=DEV))
    from diffsound_b200.parallel.rowpart_lobpcg import eigen_decomposition_rowpart
    with pytest.raises(NotImplementedError, match="supports"):
        eigen_decomposition_rowpart(obj, [DEV])
    # in-place change to an invalid value is caught at the next assembly
    kn = torch.full((int(fm.sum()),), 3e9, dtype=torch.float64, device=DEV)
    obj.set_supports(fm, kn, 1e9)
    kn[0] = float("nan")
    with pytest.raises(ValueError, match="non-finite"):
        obj.eigen_decomposition()
    obj.set_supports(None)
    obj.eigen_decomposition()
    assert torch.equal(obj.eigenvalues, ref.eigenvalues) and torch.equal(obj.U_hat, ref.U_hat)
    assert torch.equal(obj._Kval, ref._Kval)
    # C-ABI argument errors
    lib = native._lib.load()
    f = native.SupportFaces(obj.deform.tets_i32, 2, obj.surface()[1][fm], obj.surface()[2][fm])
    k = torch.ones(f.S, dtype=torch.float64, device=DEV)
    p = native._p
    rc = lib.ds_support_km(p(obj._verts32), p(obj.deform.tets_i32), obj.deform.num_tets, 3, obj.deform.num_nodes,
                           p(f.owner), p(f.local), f.S, p(k), p(k), p(f.inc_node), p(f.inc_ptr), p(f.inc), f.R,
                           p(obj.deform.pattern.brow), p(obj.deform.pattern.bcol), None, obj.deform.pattern.nnzb,
                           p(obj._Kval), None)
    assert rc == -2 and "order" in native._lib.last_error()
    rc = lib.ds_support_energies(p(obj._verts32), p(obj.deform.tets_i32), obj.deform.num_tets, 2, obj.deform.num_nodes,
                                 p(f.owner), p(f.local), 0, p(k), p(k), p(obj.U_hat_full.contiguous()), 12, 12, p(k), None)
    assert rc == -2 and "support face count" in native._lib.last_error()
    rc = lib.ds_support_grad(p(obj._verts32), p(obj.deform.tets_i32), obj.deform.num_tets, 2, obj.deform.num_nodes,
                             p(f.owner), p(f.local), f.S, p(k), p(k), None, 12, 12, p(k), None, None, None, 0, None, None,
                             None, None)
    assert rc == -2 and "null" in native._lib.last_error()
