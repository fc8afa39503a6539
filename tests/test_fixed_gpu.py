"""Clamped objects on the B200 (DiffSoundObj.fix_nodes, ds_fix_nodes_km, ds_lobpcg_opts.fixed) against the reduced-pencil
reference of tests/fixed_oracle.py."""
import numpy as np
import pytest
import torch

import fixed_oracle as fo
from oracle import modal_oracle as mo
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


def _oracle(obj, mask, k):
    _, _, MatSet = _mods()
    rho, E, nu = MatSet.Steel[:3]
    pv = obj.tetmesh.vertices.detach().cpu()
    pt = obj.tetmesh.tets.cpu().long()
    K, M = mo.assemble(pv, pt, obj.tetmesh.order, E, nu, rho)
    lam, U = fo.eig_fixed(K, M, mask.cpu().numpy(), k)
    return K, M, lam, U, pv, pt


def _face_x0(obj):
    v = obj.tetmesh.vertices.detach()
    return v[:, 0] <= v[:, 0].min() + 1e-6


def _bar(order=1, cells=(24, 3, 2)):
    v, t = kuhn_box(cells, (1.0, 0.1, 0.05))
    return v, t


def _sphere():
    from diffsound_b200.diffelastic.tetrahedralize import tetrahedralize
    a = 0.1
    mesh = tetrahedralize(lambda p: a - p.norm(dim=1), edge_length=0.02, bounds=((-a,) * 3, (a,) * 3))
    return mesh.vertices.detach().cpu().numpy(), mesh.tets.cpu().numpy()


def _mesh(meshes, name):
    if name == "sphere":
        return _sphere()
    return meshes[name]


def _mask(obj, name):
    v = obj.tetmesh.vertices.detach()
    if name == "bowl":                                  # the base disc, through the shell's thickness
        r = torch.hypot(v[:, 0], v[:, 1])
        return r < 0.25 * r.max()
    if name == "sphere":                                # a cap
        return v[:, 2] > 0.08
    return _face_x0(obj)


def _check_modes(obj, mask, lam_ref, U_ref, M):
    lam = obj.eigenvalues.cpu().numpy()
    # eig_tol 1e-5 on the relative residual gives eigenvalue errors ~1e-10; 1e-6 leaves room for the fp32 preconditioner's
    # stopping point and the oracle's own ARPACK tolerance
    err = np.abs(lam - lam_ref) / lam_ref
    assert err.max() <= 1e-6, (err.max(), lam[:4], lam_ref[:4])
    U = obj.U_hat.cpu().numpy()
    fixed_rows = np.repeat(mask.cpu().numpy(), 3)
    assert np.all(U[fixed_rows] == 0.0)                 # exactly, not approximately
    G = U.T @ (M @ U)
    assert np.abs(G - np.eye(U.shape[1])).max() <= 1e-10
    # subspaces of (near-)equal eigenvalues agree with the oracle's.  The angle of a computed invariant subspace is bounded
    # by its residual over the gap to the rest of the spectrum (Davis-Kahan): eig_tol * lambda / gap, here with 10x slack
    k = lam_ref.size
    start = 0
    while start < k:
        end = start + 1
        while end < k and lam_ref[end] - lam_ref[end - 1] < 1e-4 * lam_ref[end]:
            end += 1
        if end < k:                                     # a cluster cut at the end of the block is not compared
            gap = lam_ref[end] - lam_ref[end - 1]
            if start > 0:
                gap = min(gap, lam_ref[start] - lam_ref[start - 1])
            s = np.linalg.svd(U_ref[:, start:end].T @ (M @ U[:, start:end]), compute_uv=False)
            sin = np.sqrt(max(0.0, 1.0 - s.min() ** 2))
            assert sin <= 10 * obj.eig_tol * lam_ref[end - 1] / gap, (start, end, s, gap)
        start = end


def test_operator_blocks_zero_and_rest_bitwise(meshes):
    native, _, _ = _mods()
    v, t = meshes["grid16"]
    obj, _ = _obj(v, t, 2, 16)
    mask = _face_x0(obj)
    obj.update_stiff_matrix()
    K0, M0 = obj._Kval.clone(), obj._Mblk.clone()
    obj.fix_nodes(mask)                                   # re-assembles, clamped
    pat = obj.deform.pattern
    crow, col = pat.csr()
    rows = torch.repeat_interleave(torch.arange(pat.n, device=DEV), crow[1:] - crow[:-1])
    ni, nj = rows // 3, col // 3
    touch = touch_fine = (ni != nj) & (mask[ni] | mask[nj])
    assert bool(touch.any())
    assert bool((obj._Kval[touch] == 0.0).all())
    assert torch.equal(obj._Kval[~touch], K0[~touch])
    brows = torch.repeat_interleave(torch.arange(pat.n_nodes, device=DEV), pat.brow[1:] - pat.brow[:-1]).long()
    bcol = pat.bcol.long()
    btouch = (brows != bcol) & (mask[brows] | mask[bcol])
    assert bool((obj._Mblk[btouch] == 0.0).all()) and torch.equal(obj._Mblk[~btouch], M0[~btouch])
    # coarse (P1) level: the fine mask at the corner nodes
    c = obj.deform.coarse
    mu, la = obj._lame_used
    mt = obj.deform.coarse_mtab(obj._density_used)
    c.fixed = None
    c.assemble(obj._verts32, mu, la, c.ctab, mt)
    Kc0, Mc0 = c.Kval.clone(), c.Mblk.clone()
    cmask = mask[c.corner_nodes]
    c.fixed = cmask.to(torch.uint8).contiguous()
    c.assemble(obj._verts32, mu, la, c.ctab, mt)
    cp = c.pattern
    brows = torch.repeat_interleave(torch.arange(cp.n_nodes, device=DEV), cp.brow[1:] - cp.brow[:-1]).long()
    bcol = cp.bcol.long()
    btouch = (brows != bcol) & (cmask[brows] | cmask[bcol])
    assert bool(btouch.any())
    assert bool((c.Mblk[btouch] == 0.0).all()) and torch.equal(c.Mblk[~btouch], Mc0[~btouch])
    ccrow, ccol = cp.csr()
    rows = torch.repeat_interleave(torch.arange(cp.n, device=DEV), ccrow[1:] - ccrow[:-1])
    ni, nj = rows // 3, ccol // 3
    touch = (ni != nj) & (cmask[ni] | cmask[nj])
    assert bool((c.Kval[touch] == 0.0).all()) and torch.equal(c.Kval[~touch], Kc0[~touch])
    # the unit stiffnesses of stiff_func carry the same clamp
    Kmu, Kla = obj._unit_stiffness()
    assert bool((Kmu[touch_fine] == 0.0).all()) and bool((Kla[touch_fine] == 0.0).all())
    assert bool((Kmu[~touch_fine] != 0.0).any()) and bool((Kla[~touch_fine] != 0.0).any())


@pytest.mark.parametrize("name,order,k", [("cube2", 2, 12), ("cube3", 1, 12), ("cube3", 2, 16),
                                          ("grid16", 1, 16), ("grid16", 2, 16), ("bowl", 2, 16), ("sphere", 2, 16)])
def test_eigenpairs_match_oracle(meshes, name, order, k):
    v, t = _mesh(meshes, name)
    obj, _ = _obj(v, t, order, k)
    mask = _mask(obj, name)
    obj.fix_nodes(mask)
    obj.eigen_decomposition()
    K, M, lam_ref, U_ref, _, _ = _oracle(obj, mask, k)
    _check_modes(obj, mask, lam_ref, U_ref, M)


@pytest.mark.parametrize("variant", ["two_level_nested", "two_level", "chebyshev", "fp64", "locked64"])
def test_solver_paths_match_oracle(meshes, variant):
    v, t = meshes["grid16"]
    k = 64 if variant == "locked64" else 16
    obj, _ = _obj(v, t, 2, k)
    if variant == "two_level":
        obj.nested_start = False
    elif variant == "chebyshev":
        obj.two_level = False
    elif variant == "fp64":
        obj._has_slivers = lambda: True               # straight to the FP64 Chebyshev preconditioner
    mask = _face_x0(obj)
    obj.fix_nodes(mask)
    obj.eigen_decomposition()
    if variant == "fp64":
        assert obj.eig_stats.get("precond") == "fp64"
    if variant == "locked64":
        assert obj.eig_stats["batches"] == 2
    if variant == "two_level_nested":
        assert obj.eig_stats["nested_iterations"] > 0
    K, M, lam_ref, U_ref, _, _ = _oracle(obj, mask, k)
    _check_modes(obj, mask, lam_ref, U_ref, M)


def _bar_obj(k=8, leaf=True):
    v, t = _bar()
    obj, vt = _obj(v, t, 1, k, leaf=leaf)
    return obj, vt, v, t


def test_shape_gradient_against_oracle_and_differences():
    _, _, MatSet = _mods()
    rho, E, nu = MatSet.Steel[:3]
    k = 8
    obj, leaf, v, t = _bar_obj(k)
    mask = _face_x0(obj)
    obj.fix_nodes(mask)
    obj.eigen_decomposition()
    _, M, lam_ref, U_ref, pv, pt = _oracle(obj, mask, k)
    g = 1.0 / lam_ref
    vals = obj.get_vals()
    (vals[:, 0] * torch.as_tensor(g, device=DEV, dtype=torch.float32)).sum().backward()
    gref = mo.eigval_grad_shape(pv, pt, 1, E, nu, rho, U_ref, lam_ref, g).numpy()
    grad = leaf.grad.cpu().numpy()
    err = np.linalg.norm(grad - gref) / np.linalg.norm(gref)
    # the modes of the bar are simple (b != h), so the gradient is sign-invariant and the oracle's is the same quantity;
    # the kernel rounds once to fp32
    assert err <= 1e-5, err
    # central differences of sum g_i lambda_i with the clamp held on the same nodes, on a free tip node, an interior
    # node and a fixed node (moving a clamped node still changes its elements)
    m0 = mask.clone()
    tip = int(np.argmax(v[:, 0] + v[:, 1] + v[:, 2]))
    fixed_node = int(torch.nonzero(m0)[3])
    mid = int(np.argmin(np.abs(v[:, 0] - 0.5) + np.abs(v[:, 1] - 0.05) + np.abs(v[:, 2])))
    for node, axis in [(tip, 2), (mid, 0), (fixed_node, 0)]:
        f = []
        hs = []
        for s in (+1, -1):
            vp = v.copy()
            vp[node, axis] = np.float32(v[node, axis] + s * 5e-4)
            hs.append(float(vp[node, axis]) - float(v[node, axis]))
            o, _ = _obj(vp, t, 1, k)
            o.fix_nodes(m0)
            o.eigen_decomposition()
            f.append(float((o.eigenvalues.cpu().numpy() * g).sum()))
        fd = (f[0] - f[1]) / (hs[0] - hs[1])
        # O(h^2) truncation: a 5e-4 step moves a node by ~1-2 % of its element size, so the quotient is good to ~1e-3
        assert abs(fd - grad[node, axis]) <= 3e-3 * np.abs(grad).max(), (node, axis, fd, grad[node, axis])
    assert abs(grad[fixed_node]).max() > 0


def test_material_forms_and_stiff_func_against_oracle():
    k = 8
    obj, _, v, t = _bar_obj(k, leaf=False)
    mask = _face_x0(obj)
    obj.fix_nodes(mask)
    obj.eigen_decomposition()
    K, M, lam_ref, U_ref, pv, pt = _oracle(obj, mask, k)
    q_mu, q_la, q_m = (x.cpu().numpy() for x in obj._material_forms())
    r_mu, r_la = mo.material_quadforms(pv, pt, 1, U_ref)
    # quadratic forms of simple modes do not depend on the eigenvector signs.  Each one alone is first order in the
    # eigenvector error (~ eig_tol lambda / gap, 1e-4 bounds it on the bar); their Lame-weighted sum is the Rayleigh
    # quotient, second order, hence 1e-6
    np.testing.assert_allclose(q_mu, r_mu, rtol=1e-4)
    np.testing.assert_allclose(q_la, r_la, rtol=1e-4)
    np.testing.assert_allclose(q_m, 1.0, rtol=1e-9)
    mu, la = obj._lame_used
    np.testing.assert_allclose(mu * q_mu + la * q_la, lam_ref, rtol=1e-6)
    f = obj.get_undamped_freqs()
    np.testing.assert_allclose(f[:, 0].cpu().numpy(), np.sqrt(lam_ref) / (2 * np.pi), rtol=1e-6)
    # stiff_func is mu K_mu + lam K_lam of the clamped K
    x = torch.randn(obj.deform.pattern.n, 3, dtype=torch.float64, device=DEV, generator=torch.Generator(DEV).manual_seed(0))
    y = obj.stiff_func(x).cpu().numpy()
    Kc = fo.constrain(K, mask.cpu().numpy())
    ref = Kc @ x.cpu().numpy()
    # stiff_func multiplies K_mu and K_lam by the fp32 Lame scalars, the oracle assembles K with fp64 ones
    assert np.linalg.norm(y - ref) <= 1e-6 * np.linalg.norm(ref)


def test_strike_on_the_clamped_face_is_silent():
    k = 8
    obj, _, v, t = _bar_obj(k, leaf=False)
    mask = _face_x0(obj)
    obj.fix_nodes(mask)
    obj.eigen_decomposition()
    pts = torch.tensor([[-0.01, 0.05, 0.025], [-0.01, 0.02, 0.01]], device=DEV)
    g = obj.modal_gains(pts)
    assert bool((g == 0.0).all())
    tip = torch.tensor([[1.01, 0.05, 0.025]], device=DEV)
    assert bool((obj.modal_gains(tip).abs() > 0).any())
    y = obj.impulse_response(torch.tensor([[0.9, 0.05, 0.06]], device=DEV), 4000, 44100.0,
                             pickup=torch.tensor([[1.01, 0.05, 0.025]], device=DEV))
    assert y.shape == (1, 4000) and bool(torch.isfinite(y).all()) and float(y.abs().max()) > 0


def test_clear_clamp_is_bitwise_free(meshes):
    v, t = meshes["cube3"]
    a, _ = _obj(v, t, 2, 12)
    b, _ = _obj(v, t, 2, 12)
    a.fix_nodes(_face_x0(a))
    a.eigen_decomposition()
    lam_c = a.eigenvalues.clone()
    a.fix_nodes(None)
    a.eigen_decomposition()
    b.eigen_decomposition()
    assert torch.equal(a.eigenvalues, b.eigenvalues)
    assert torch.equal(a.U_hat, b.U_hat)
    assert not torch.equal(lam_c, b.eigenvalues)


def test_fix_nodes_device_and_rowpart_rejection(meshes):
    v, t = meshes["cube3"]
    obj, _ = _obj(v, t, 2, 12)
    mask = _face_x0(obj)
    with pytest.raises(ValueError, match="on cpu"):
        obj.fix_nodes(mask.cpu())
    obj.fix_nodes(mask)
    from diffsound_b200.parallel.rowpart_lobpcg import eigen_decomposition_rowpart
    with pytest.raises(NotImplementedError, match="clamped"):
        eigen_decomposition_rowpart(obj)
