"""GPU parity tests of the FP32 preconditioner kernels (csrc/precond32.cu, csrc/pmg.cu) behind the C-ABI.

The oracle for the SpMM modes is the FP64 product of the same assembled matrix (scipy CSR from
oracle.modal_oracle on the CPU); tolerance 2e-6 of the result norm (fp32 storage of K and X, fp32
accumulation over <= ~80 blocks per row).  The coarse-level integer tables are compared bit-exactly
with a numpy restatement of the quadratic -> linear hierarchy (reference local node order,
/root/reference/src/diffelastic/mesh.py:139-154).
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import modal_oracle as mo

pytestmark = pytest.mark.gpu

STEEL = (7850.0, 2.0e11, 0.29)
DEV = "cuda:0"


def _assembled(v, t, order):
    from diffsound_b200 import native
    from diffsound_b200.diffelastic import mass_matrix as mmx
    pv, pt = mo.promote(torch.as_tensor(v), torch.as_tensor(t), order)
    verts = pv.to(DEV).contiguous()
    tets = pt.to(torch.int32).to(DEV).contiguous()
    pat = native.Pattern(tets, verts.shape[0])
    mu, lam = mo.lame(STEEL[1], STEEL[2])
    Kval, Mblk = native.assemble_km(verts, tets, order, pat, mu, lam, mmx.stiffness_contraction_table(order).to(DEV),
                                    mmx.mass_density_table(order, STEEL[0]).to(DEV))
    crow, col = pat.csr()
    K = sp.csr_matrix((Kval.cpu().numpy(), col.cpu().numpy(), crow.cpu().numpy()), shape=(pat.n, pat.n))
    return pv, pt, verts, tets, pat, Kval, Mblk, K


def _wheel(nring):
    """nring tets around one edge: the edge's nodes get ~5*nring neighbours at order 2, far more
    than any other row (a very unbalanced row for the ticketed row sweep of k_spmm32v)."""
    ang = np.linspace(0, 2 * np.pi, nring, endpoint=False)
    ring = np.stack([np.cos(ang), np.sin(ang), 0.5 + 0.1 * np.cos(3 * ang)], 1)
    v = np.concatenate([[[0, 0, 0], [0, 0, 1.0]], ring]).astype(np.float32)
    t = np.array([[0, 1, 2 + i, 2 + (i + 1) % nring] for i in range(nring)], dtype=np.int64)
    return v, t


@pytest.mark.parametrize("mesh,order", [("cube3", 2), ("grid16", 1), ("bowl", 2), ("wheel", 2)])
@pytest.mark.parametrize("ncols", [16, 32, 48, 64])
def test_spmm32_modes(meshes, mesh, order, ncols):
    from diffsound_b200 import native
    v, t = _wheel(120) if mesh == "wheel" else meshes[mesh]
    _, _, _, _, pat, Kval, Mblk, K = _assembled(v, t, order)
    if mesh == "wheel":
        deg = np.diff(pat.brow.cpu().numpy())
        assert deg.max() > 400, "the wheel must have a very long row"
    rec, invD = native.k32_pack(pat, Kval)
    g = torch.Generator(device=DEV).manual_seed(1)
    X = torch.randn(pat.n, ncols, device=DEV, generator=g)
    R = torch.randn(pat.n, ncols, device=DEV, generator=g) * float(np.abs(K.data).max())
    Zp = torch.randn(pat.n, ncols, device=DEV, generator=g)
    AX = K @ X.cpu().numpy().astype(np.float64)
    scale = np.linalg.norm(AX)

    y = native.spmm32(pat, rec, X, mode=0)
    assert np.linalg.norm(y.cpu().numpy() - AX) <= 2e-6 * scale
    y = native.spmm32(pat, rec, X, mode=1, R=R)
    ref = R.cpu().numpy().astype(np.float64) - AX
    assert np.linalg.norm(y.cpu().numpy() - ref) <= 2e-6 * (scale + np.linalg.norm(ref))

    # block-Jacobi inverse
    nb = pat.n_nodes
    D = np.zeros((nb, 3, 3))
    Kc = K.tocsr()
    for c in range(3):
        for d in range(3):
            D[:, c, d] = np.asarray(Kc[np.arange(nb) * 3 + c, np.arange(nb) * 3 + d]).ravel()
    Di = np.linalg.inv(D)
    got = invD.cpu().numpy().reshape(nb, 3, 3)
    assert np.abs(got - Di).max() <= 1e-5 * np.abs(Di).max()

    # one Chebyshev step, out aliasing Zprev
    ab, cc = 0.37, 0.81
    out = Zp.clone()
    native.spmm32(pat, rec, X, mode=2, R=R, invD=invD, Zprev=out, ab=ab, cc=cc, out=out)
    res = (R.cpu().numpy().astype(np.float64) - AX).reshape(nb, 3, ncols)
    dr = np.einsum("ncd,ndk->nck", Di, res).reshape(pat.n, ncols)
    x64 = X.cpu().numpy().astype(np.float64)
    ref = x64 + ab * (x64 - Zp.cpu().numpy()) + cc * dr
    assert np.linalg.norm(out.cpu().numpy() - ref) <= 4e-6 * np.linalg.norm(ref)


def _coarse_numpy(pt, n_nodes):
    t = pt.numpy()
    corners = np.unique(t[:, [0, 2, 4, 9]])
    cid = -np.ones(n_nodes, dtype=np.int64)
    cid[corners] = np.arange(corners.size)
    par = np.zeros((n_nodes, 2), dtype=np.int64)
    par[corners, 0] = par[corners, 1] = cid[corners]
    for mloc, (a, b) in {1: (0, 2), 3: (2, 4), 5: (4, 0), 6: (0, 9), 7: (2, 9), 8: (4, 9)}.items():
        ca, cb = cid[t[:, a]], cid[t[:, b]]
        par[t[:, mloc], 0] = np.minimum(ca, cb)
        par[t[:, mloc], 1] = np.maximum(ca, cb)
    ctets = cid[t[:, [0, 2, 4, 9]]]
    return corners, cid, par, ctets


@pytest.mark.parametrize("mesh", ["cube3", "grid16", "bowl"])
def test_coarse_level_tables(meshes, mesh):
    from diffsound_b200 import native
    v, t = meshes[mesh]
    pv, pt, verts, tets, pat, _, _, _ = _assembled(v, t, 2)
    cl = native.CoarseLevel(verts, tets)
    corners, cid, par, ctets = _coarse_numpy(pt, pv.shape[0])
    assert cl.n_nodes == corners.size
    assert np.array_equal(cl.cid.cpu().numpy(), cid)
    assert np.array_equal(cl.tets.cpu().numpy(), ctets)
    assert np.array_equal(cl.parents.cpu().numpy().reshape(-1, 2), par)
    assert np.array_equal(cl.verts.cpu().numpy(), pv.numpy()[corners])
    assert np.array_equal(cl.corner_nodes.cpu().numpy(), corners)
    # gather lists of P^T: stable sort of the flattened parent table
    flat = par.reshape(-1)
    order = np.argsort(flat, kind="stable")
    assert np.array_equal(cl.rlist.cpu().numpy(), order // 2)
    assert np.array_equal(cl.rptr.cpu().numpy(), np.searchsorted(flat[order], np.arange(corners.size + 1)))
    # the coarse pattern is the order-1 pattern of the corner mesh
    crow, col, brow, bcol = mo.pattern(torch.as_tensor(ctets), corners.size)
    assert np.array_equal(cl.pattern.brow.cpu().numpy(), brow)
    assert np.array_equal(cl.pattern.bcol.cpu().numpy(), bcol)


@pytest.mark.parametrize("ncols", [16, 48])
def test_transfer_operators(meshes, ncols):
    from diffsound_b200 import native
    v, t = meshes["grid16"]
    pv, pt, verts, tets, pat, _, _, _ = _assembled(v, t, 2)
    cl = native.CoarseLevel(verts, tets)
    _, _, par, _ = _coarse_numpy(pt, pv.shape[0])
    nf, nc = pv.shape[0], cl.n_nodes
    Pn = sp.csr_matrix((np.full(2 * nf, 0.5), (np.repeat(np.arange(nf), 2), par.reshape(-1))), shape=(nf, nc))
    P = sp.kron(Pn, sp.identity(3), format="csr")
    g = torch.Generator(device=DEV).manual_seed(2)
    res = torch.randn(3 * nf, ncols, device=DEV, generator=g)
    zc = torch.randn(3 * nc, ncols, device=DEV, generator=g)
    z = torch.randn(3 * nf, ncols, device=DEV, generator=g)
    rc = native.pmg_restrict32(cl, res)
    ref = P.T @ res.cpu().numpy().astype(np.float64)
    assert np.abs(rc.cpu().numpy() - ref).max() <= 1e-5 * np.abs(ref).max()
    z0 = z.cpu().numpy().astype(np.float64)
    native.pmg_prolong_add32(cl, zc, z)
    ref = z0 + P @ zc.cpu().numpy().astype(np.float64)
    assert np.abs(z.cpu().numpy() - ref).max() <= 1e-6 * np.abs(ref).max()


def test_galerkin_coarse_operator_is_p1_stiffness(meshes):
    """P^T K_P2 P equals the P1 stiffness matrix assembled on the corner mesh (the reason the coarse
    level can be assembled directly): <= 1e-5 relative (fp32 quadrature tables of the two orders)."""
    from diffsound_b200 import native
    from diffsound_b200.diffelastic import mass_matrix as mmx
    v, t = meshes["cube3"]
    pv, pt, verts, tets, pat, Kval, Mblk, K = _assembled(v, t, 2)
    cl = native.CoarseLevel(verts, tets)
    mu, lam = mo.lame(STEEL[1], STEEL[2])
    cl.assemble(verts, mu, lam, mmx.stiffness_contraction_table(1).to(DEV), mmx.mass_density_table(1, STEEL[0]).to(DEV))
    crow, col = cl.pattern.csr()
    Kc = sp.csr_matrix((cl.Kval.cpu().numpy(), col.cpu().numpy(), crow.cpu().numpy()), shape=(cl.pattern.n,) * 2)
    _, _, par, _ = _coarse_numpy(pt, pv.shape[0])
    nf, nc = pv.shape[0], cl.n_nodes
    Pn = sp.csr_matrix((np.full(2 * nf, 0.5), (np.repeat(np.arange(nf), 2), par.reshape(-1))), shape=(nf, nc))
    P = sp.kron(Pn, sp.identity(3), format="csr")
    G = (P.T @ K @ P).toarray()
    assert np.abs(G - Kc.toarray()).max() <= 1e-5 * np.abs(G).max()


@pytest.mark.parametrize("mesh,two_level,nested", [("grid16", True, True), ("grid16", True, False), ("grid16", False, False),
                                                   ("bowl", True, True)])
def test_eigensolver_two_level_matches_arpack(meshes, mesh, two_level, nested):
    """LOBPCG with the FP32 two-level (or one-level Chebyshev) preconditioner reproduces the ARPACK
    spectrum of the oracle's matrices to 1e-6 relative (north-star tolerance) on quadratic meshes."""
    from diffsound_b200.diffelastic.diff_model import DiffSoundObj
    from diffsound_b200.diffelastic.material_model import MatSet
    v, t = meshes[mesh]
    k = 16
    obj = DiffSoundObj(torch.as_tensor(v).to(DEV), torch.as_tensor(t).to(DEV), mode_num=k, order=2, mat=MatSet.Steel)
    obj.two_level = two_level
    obj.nested_start = nested
    obj.eigen_decomposition()
    assert obj.eig_stats["two_level"] == two_level
    assert (obj.eig_stats["nested_iterations"] > 0) == nested
    pv, pt = mo.promote(torch.as_tensor(v), torch.as_tensor(t), 2)
    rho, E, nu = MatSet.Steel[:3]
    K, M = mo.assemble(pv, pt, 2, E, nu, rho)
    lam, _, _, _ = mo.eig_arpack(K, M, k)
    err = np.abs(obj.eigenvalues.cpu().numpy() - lam) / lam
    assert err.max() <= 1e-6, (err.max(), obj.eig_stats)


@pytest.mark.parametrize("name,order,ncols,degree", [("grid16", 2, 48, 12), ("grid16", 1, 32, 7), ("bowl", 1, 16, 40),
                                                     ("bowl", 2, 48, 3)])
def test_persistent_chebyshev_matches_stepwise(meshes, name, order, ncols, degree):
    """The cooperative one-launch Chebyshev solve (records in shared memory, grid barrier per step) against the same
    recurrence run as one SpMM launch per step: identical arithmetic, so the iterates agree to fp32 rounding, and both
    reduce the residual of K z = r."""
    from diffsound_b200 import _lib, native
    lib = _lib.load()
    v, t = meshes[name]
    _, _, _, _, pat, Kval, Mblk, K = _assembled(v, t, order)
    rec, invD = native.k32_pack(pat, Kval)
    g = torch.Generator(device=DEV).manual_seed(11)
    R = torch.randn(pat.n, ncols, device=DEV, generator=g) * float(np.abs(K.data).max())
    lmax, ratio = 2.8, 0.4 * degree * degree + 2.0
    n0 = lib.ds_launch_count()
    za = native.cheb32_solve(pat, rec, invD, R, degree, lmax, ratio, persistent=True)
    n1 = lib.ds_launch_count()
    zb = native.cheb32_solve(pat, rec, invD, R, degree, lmax, ratio, persistent=False)
    # launches: the row-chunk table, then the one cooperative kernel, or the Jacobi step and degree - 1 SpMM steps
    assert n1 - n0 == 2, "the persistent kernel did not run"
    assert lib.ds_launch_count() - n1 == 1 + degree
    assert torch.isfinite(za).all()
    scale = float(zb.abs().max())
    assert float((za - zb).abs().max()) <= 2e-5 * scale
    # and it is a contraction towards the solution: ||R - A z|| < ||R||
    res = native.spmm32(pat, rec, za, mode=1, R=R)
    assert float(res.norm()) < float(R.norm())
