"""The eigensolver's inner kernels one by one, through the C-ABI, against fp64 / high-precision host references.

Whole-solve tests compare eigenvalues with ARPACK at 1e-6; a kernel that is subtly wrong (K W accumulated in fp32, a
wrong Chebyshev coefficient, a Jacobi that stops early) can pass them, because LOBPCG converges to the eigenpairs of
whatever operator it is given.  Here each kernel meets a reference of its own operation:
  A  ds_spmm_dual_z32 (K Z, M Z from the fp32 search block)   scipy fp64, elementwise fp64 summation-error model
  B  ds_lobpcg_residual (R = KX - MX diag(lam), column sums)  numpy / math.fsum
  C  ds_eigh_generalized_f64 / _idx_f64 (Rayleigh-Ritz solve)  mpmath at 40 digits, scipy, exact construction
  D  ds_cheb32_solve (persistent and stepwise Chebyshev)       closed-form polynomial, textbook fp64 iteration
  E  the row-slab utilities of csrc/slab.cu                    numpy
Every bar states the value measured on an NVIDIA B200.  Helpers print what they measure (pytest -s shows it).
"""
import ctypes as C
import functools
import math
import os

import numpy as np
import pytest
import scipy.linalg
import scipy.sparse as sp
import scipy.sparse.linalg
import torch

import lobpcg_refs as refs
from conftest import GOLDEN
from oracle import modal_oracle as mo

pytestmark = pytest.mark.gpu

STEEL = (7850.0, 2.0e11, 0.29)
DEV = "cuda:0"
EPS = np.finfo(np.float64).eps
SENT = -7.25


def _lib():
    from diffsound_b200 import _lib as L
    return L.load()


def _check(rc, what):
    from diffsound_b200 import _lib as L
    L.check(rc, what)


def _p(t, offset=0):
    """device pointer of tensor t, `offset` elements in"""
    return C.c_void_p(t.data_ptr() + offset * t.element_size())


def _st():
    from diffsound_b200 import native
    return native._stream()


def _wheel(nring):
    """nring tets around one edge: the edge's nodes get ~5*nring neighbours at order 2, far more
    than any other row (a very unbalanced row for the ticketed row sweep of k_spmm32v)."""
    ang = np.linspace(0, 2 * np.pi, nring, endpoint=False)
    ring = np.stack([np.cos(ang), np.sin(ang), 0.5 + 0.1 * np.cos(3 * ang)], 1)
    v = np.concatenate([[[0, 0, 0], [0, 0, 1.0]], ring]).astype(np.float32)
    t = np.array([[0, 1, 2 + i, 2 + (i + 1) % nring] for i in range(nring)], dtype=np.int64)
    return v, t


@functools.lru_cache(maxsize=None)
def _mesh(name):
    if name == "wheel":
        return _wheel(120)
    if name == "tet":
        return np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=np.float32), np.array([[0, 1, 2, 3]])
    d = np.load(os.path.join(GOLDEN, "meshes.npz"))
    return d[f"{name}_verts"], d[f"{name}_tets"].astype(np.int64)


@functools.lru_cache(maxsize=None)
def _system(name, order):
    """(pattern, Kval, Mblk, K, M): the device operator and its scipy fp64 twin (same values)."""
    from diffsound_b200 import native
    from diffsound_b200.diffelastic import mass_matrix as mmx
    v, t = _mesh(name)
    pv, pt = mo.promote(torch.as_tensor(v), torch.as_tensor(t), order)
    verts = pv.to(DEV).contiguous()
    tets = pt.to(torch.int32).to(DEV).contiguous()
    pat = native.Pattern(tets, verts.shape[0])
    mu, lam = mo.lame(STEEL[1], STEEL[2])
    Kval, Mblk = native.assemble_km(verts, tets, order, pat, mu, lam, mmx.stiffness_contraction_table(order).to(DEV),
                                    mmx.mass_density_table(order, STEEL[0]).to(DEV))
    crow, col = pat.csr()
    crow, col = crow.cpu().numpy(), col.cpu().numpy()
    K = sp.csr_matrix((Kval.cpu().numpy(), col, crow), shape=(pat.n, pat.n))
    M = sp.csr_matrix((native.mass_expand(pat, Mblk).cpu().numpy(), col, crow), shape=(pat.n, pat.n))
    return pat, Kval, Mblk, K, M


# ---------------------------------------------------------------------------------------------------------------------
# A. ds_spmm_dual_z32
# ---------------------------------------------------------------------------------------------------------------------
def _spmm_dual_z32(pat, Kval, Mblk, bcolP, Z, m=48, ldy=None, off=None, ncols=None):
    """YK, YM written into columns [off, off + ncols) of (n x ld) buffers filled with SENT, as the drivers do
    (ld = 3m, offset m); returns (rc, YK, YM)."""
    from diffsound_b200 import native
    lib = _lib()
    ncols = Z.shape[1] if ncols is None else ncols
    ld = 3 * m if ldy is None else ldy
    off = m if off is None else off
    YK = torch.full((pat.n * ld + 8,), SENT, dtype=torch.float64, device=DEV)
    YM = torch.full((pat.n * ld + 8,), SENT, dtype=torch.float64, device=DEV)
    chunks = native.spmm32_chunks(pat)
    rc = lib.ds_spmm_dual_z32(_p(pat.brow), _p(bcolP), pat.n_nodes, pat.nnzb, _p(chunks), _p(Kval), _p(Mblk),
                              _p(Z), ncols, _p(YK, off), ld, _p(YM, off), ld, _st())
    torch.cuda.synchronize()
    view = lambda Y: Y[:pat.n * ld].view(pat.n, ld).cpu().numpy()
    return rc, view(YK), view(YM)


def _z_block(pat, ncols, seed, permuted, row_scale=False):
    """random fp32 block Z (exact in fp64) and its device copy in the gather numbering with the matching bcolP"""
    rng = np.random.default_rng(seed)
    nn = pat.n_nodes
    Z = rng.standard_normal((3 * nn, ncols)).astype(np.float32)
    if row_scale:
        Z = (Z * (10.0 ** rng.uniform(-3, 3, (3 * nn, 1)))).astype(np.float32)
    bcol = pat.bcol.cpu().numpy()
    if permuted:    # Morton-like private numbering: node j of Z lives at row inv[j] of the gathered block
        perm = rng.permutation(nn)
        inv = np.argsort(perm)
        Zg = Z.reshape(nn, 3, ncols)[perm].reshape(3 * nn, ncols)
        bcolP = inv[bcol].astype(np.int32)
    else:
        Zg, bcolP = Z, bcol.astype(np.int32)
    return Z, torch.tensor(Zg, device=DEV), torch.tensor(bcolP, device=DEV)


def _spmm_case(mesh, order, ncols, permuted, row_scale=False, seed=0):
    pat, Kval, Mblk, K, M = _system(mesh, order)
    Z, Zd, bcolP = _z_block(pat, ncols, seed, permuted, row_scale)
    rc, YK, YM = _spmm_dual_z32(pat, Kval, Mblk, bcolP, Zd)
    assert rc == 0, _lib().ds_last_error()
    m = 48
    Z64 = Z.astype(np.float64)
    worst = 0.0
    for Y, A in ((YK, K), (YM, M)):
        ref = A @ Z64
        bound = abs(A) @ np.abs(Z64)          # |A| |Z|: the scale of the fp64 summation error of each entry
        got = Y[:, m:m + ncols]
        nz = bound > 0
        assert np.all(got[~nz] == 0.0)
        worst = max(worst, float((np.abs(got - ref)[nz] / bound[nz]).max()) / EPS)
        assert (Y[:, :m] == SENT).all() and (Y[:, m + ncols:] == SENT).all(), "columns outside the block were written"
    return worst


@pytest.mark.parametrize("numbering", ["identity", "permuted"])
@pytest.mark.parametrize("ncols", [16, 32, 48])
@pytest.mark.parametrize("mesh,order", [("cube3", 1), ("cube3", 2), ("grid16", 2), ("bowl", 2), ("wheel", 2), ("tet", 1),
                                        ("tet", 2)])
def test_spmm_dual_z32_matches_fp64(mesh, order, ncols, numbering):
    """K Z and M Z of an fp32 block, accumulated in fp64: every entry within 64 eps |K| |Z| of the fp64 product
    (measured: <= 8.7 eps).  fp32 accumulation (~1e7 eps) or a lost / doubled odd block of a row (O(1)) fail it.  The
    wheel has a row of more than 400 blocks; a single tet has rows shorter than the 4 / 8 lane groups."""
    if mesh == "wheel":
        pat = _system(mesh, order)[0]
        assert int(np.diff(pat.brow.cpu().numpy()).max()) > 400
    worst = _spmm_case(mesh, order, ncols, numbering == "permuted")
    print(f"[spmm_dual_z32] {mesh} o{order} ncols {ncols} {numbering}: max err / (eps |K||Z|) = {worst:.2f}")
    assert worst <= 64.0


def test_spmm_dual_z32_rows_scaled_over_six_decades():
    """Rows of Z scaled across 1e-3 .. 1e3: the bar is elementwise, so small rows are not hidden by large ones
    (measured: <= 10.9 eps |K||Z|)."""
    for ncols in (16, 48):
        worst = _spmm_case("bowl", 2, ncols, True, row_scale=True, seed=5)
        print(f"[spmm_dual_z32] bowl o2 ncols {ncols} scaled rows: {worst:.2f}")
        assert worst <= 64.0


def test_spmm_dual_z32_rejects_bad_arguments():
    """ncols 64 (no instantiation), an odd leading dimension and an output that is not 16-byte aligned are refused
    before anything is written."""
    pat, Kval, Mblk, _, _ = _system("cube3", 2)
    _, Z64, bcolP = _z_block(pat, 64, 1, False)
    rc, YK, YM = _spmm_dual_z32(pat, Kval, Mblk, bcolP, Z64, ncols=64, m=64)
    assert rc != 0 and "ncols" in _lib().ds_last_error().decode()
    _, Z, bcolP = _z_block(pat, 16, 1, False)
    for kw in (dict(ldy=145), dict(off=49)):
        rc, YK, YM = _spmm_dual_z32(pat, Kval, Mblk, bcolP, Z, **kw)
        assert rc != 0 and "aligned" in _lib().ds_last_error().decode()
        assert (YK == SENT).all() and (YM == SENT).all()


# ---------------------------------------------------------------------------------------------------------------------
# B. ds_lobpcg_residual
# ---------------------------------------------------------------------------------------------------------------------
def _residual(KX, MX, lam, m, ldr):
    lib = _lib()
    n, ld = KX.shape
    R = torch.full((n, ldr), SENT, dtype=torch.float64, device=DEV)
    sums = torch.full((2 * m,), SENT, dtype=torch.float64, device=DEV)
    partial = torch.empty(296 * 2 * m, dtype=torch.float64, device=DEV)
    _check(lib.ds_lobpcg_residual(_p(KX), _p(MX), ld, m, n, _p(lam), _p(R), ldr, _p(sums), _p(partial), _st()),
           "ds_lobpcg_residual")
    return R.cpu().numpy(), sums.cpu().numpy()


@pytest.mark.parametrize("n", [1, 7, 1000, 100_003])
@pytest.mark.parametrize("m", [1, 16, 33, 48, 64])
def test_lobpcg_residual_matches_numpy(m, n):
    """R = KX - MX diag(lam) within 2 eps (|KX| + |lam MX|) per entry (one rounding after a fused multiply-add: measured
    <= 0.25 eps); the column sums of R^2 and MX^2 within 1e-13 relative of math.fsum (measured: <= 1.3e-15); columns
    [m, ldr) of R untouched; a second call gives the same bits (fixed reduction order)."""
    rng = np.random.default_rng(m * 1000 + n % 997)
    ld, ldr = m + 5, m + 3
    lam = np.geomspace(1e-3, 1e9, m) if m > 1 else np.array([3.7e5])
    MX = rng.standard_normal((n, ld))
    KX = MX * np.concatenate([lam, np.ones(ld - m)]) * (1 + 1e-6 * rng.standard_normal((n, ld)))   # a converging block
    KXd, MXd, lamd = (torch.tensor(a, device=DEV) for a in (KX, MX, lam))
    R, sums = _residual(KXd, MXd, lamd, m, ldr)
    ref = KX[:, :m] - MX[:, :m] * lam
    bound = np.abs(KX[:, :m]) + np.abs(lam * MX[:, :m])
    rel = float((np.abs(R[:, :m] - ref) / bound).max()) / EPS
    assert rel <= 2.0
    assert (R[:, m:] == SENT).all()
    exact_r = np.array([math.fsum((R[:, j] * R[:, j]).tolist()) for j in range(m)])
    exact_m = np.array([math.fsum((MX[:, j] * MX[:, j]).tolist()) for j in range(m)])
    srel = float(max((np.abs(sums[:m] - exact_r) / exact_r).max(), (np.abs(sums[m:] - exact_m) / exact_m).max()))
    print(f"[residual] m {m} n {n}: R err {rel:.2f} eps, sums rel err {srel:.2e}")
    assert srel <= 1e-13
    R2, sums2 = _residual(KXd, MXd, lamd, m, ldr)
    assert np.array_equal(sums, sums2) and np.array_equal(R, R2)


# ---------------------------------------------------------------------------------------------------------------------
# C. the small generalised eigen-solve
# ---------------------------------------------------------------------------------------------------------------------
EIG_NS = [2, 3, 16, 47, 48, 49, 96, 131, 143, 144]
SIGMAS = [-1e-6, 0.0, 1e5]
_sweeps = {"max": 0}


def _eigh(GK, GM, sigma, N=None, idx=None, ldc=None):
    """one call on device copies of host matrices (their row length is ldg); returns theta, C (ldc x ldc, host), info.
    C starts out as SENT everywhere."""
    lib = _lib()
    N = GK.shape[0] if N is None else N
    ldc = N if ldc is None else ldc
    GKd, GMd = torch.tensor(GK, device=DEV), torch.tensor(GM, device=DEV)
    ldg = GK.shape[1]
    theta = torch.full((N,), SENT, dtype=torch.float64, device=DEV)
    Cm = torch.full((ldc, ldc), SENT, dtype=torch.float64, device=DEV)
    scratch = torch.empty(lib.ds_eigh_scratch_elems(N), dtype=torch.float64, device=DEV)
    info = torch.full((2,), -1, dtype=torch.int32, device=DEV)
    if idx is None:
        _check(lib.ds_eigh_generalized_f64(_p(GKd), _p(GMd), N, ldg, float(sigma), _p(theta), _p(Cm), ldc, _p(scratch),
                                           _p(info), _st()), "ds_eigh_generalized_f64")
    else:
        arr = (C.c_int * N)(*idx)
        _check(lib.ds_eigh_generalized_idx_f64(_p(GKd), _p(GMd), N, ldg, arr, float(sigma), _p(theta), _p(Cm), ldc,
                                               _p(scratch), _p(info), _st()), "ds_eigh_generalized_idx_f64")
    info = info.cpu().numpy()
    if info[0] == 0:
        _sweeps["max"] = max(_sweeps["max"], int(info[1]))
    return theta.cpu().numpy(), Cm.cpu().numpy(), info


def _effective_shift(GK, GM, sigma):
    """the shift the solver factorises GK + s GM with: sigma >= 0 as given, sigma < 0 relative to the mean diagonal of
    D GK D, D = diag(GM)^-1/2 (the drivers pass -1e-6)"""
    if sigma >= 0:
        return sigma
    return -sigma * float(np.mean(np.abs(np.diag(GK)) / np.diag(GM)))


def _check_pencil(GK, GM, theta, Cm, info, res_bar=1e-12, orth_bar=1e-10):
    """info, sweeps, ascending theta, the residual of every column and GM-orthonormality; returns (res, orth)"""
    N = GK.shape[0]
    assert info[0] == 0, info
    assert 1 <= info[1] <= 24, f"Jacobi stopped at its sweep cap without converging: info {info}"
    assert np.all(np.diff(theta) >= 0)
    Cn = Cm[:N, :N]
    R = GK @ Cn - (GM @ Cn) * theta
    scale = (np.linalg.norm(GK, 2) + np.abs(theta) * np.linalg.norm(GM, 2)) * np.linalg.norm(Cn, axis=0)
    res = float((np.linalg.norm(R, axis=0) / scale).max())
    orth = float(np.abs(Cn.T @ GM @ Cn - np.eye(N)).max())
    assert res <= res_bar, res
    assert orth <= orth_bar, orth
    return res, orth


@functools.lru_cache(maxsize=None)
def _graded(N):
    GK, GM, rigid = refs.graded_pencil(N, 100 + N)
    ref = refs.mp_pencil_eigvals(GK, GM) if N <= 48 else None
    return GK, GM, rigid, ref


@pytest.mark.parametrize("sigma", SIGMAS)
@pytest.mark.parametrize("N", EIG_NS)
def test_eigh_graded_pencil_relative_accuracy(N, sigma):
    """Driver-like graded pencils (rigid-size values 1e-5 .. 1e-2 in the first slots, elastic 1e7 .. 1e9, W / P up to
    1e12).  theta + s is relatively accurate for every eigenvalue, s the effective shift, so the rigid-size values are
    relatively accurate at sigma = 0 and absolutely accurate to eps s otherwise: |theta - ref| <= 1e-13 (|ref| + s)
    (measured: 4.8e-15; rigid values at sigma = 0: 5.2e-16 relative) against mpmath at 40 digits for N <= 48; above,
    the rigid values against their exact construction and the rest against LAPACK within 1e-13 max|theta|.  Every
    column's residual <= 1e-12 (measured: 7.4e-14), C^T GM C = I within 1e-10 (measured: 1.0e-13)."""
    GK, GM, rigid, ref = _graded(N)
    theta, Cm, info = _eigh(GK, GM, sigma)
    res, orth = _check_pencil(GK, GM, theta, Cm, info)
    s = _effective_shift(GK, GM, sigma)
    nr = rigid.size
    if ref is not None:
        rel = np.abs(theta - ref) / (np.abs(ref) + s)
    else:
        w = scipy.linalg.eigh(GK, GM, eigvals_only=True)
        rel = np.concatenate([np.abs(theta[:nr] - rigid) / (rigid + s), np.abs(theta[nr:] - w[nr:]) / (np.abs(w).max() + s)])
    rrel = float((np.abs(theta[:nr] - rigid) / (rigid + s)).max())
    print(f"[eigh graded] N {N} sigma {sigma:g} s {s:.3g}: max rel(theta+s) {rel.max():.2e}, rigid {rrel:.2e}, "
          f"res {res:.2e}, orth {orth:.2e}, sweeps {info[1]}")
    assert rel.max() <= 1e-13
    assert rrel <= 1e-13


def test_eigh_graded_pencil_n96_against_mpmath():
    """One N = 96 graded pencil at the drivers' shift against mpmath (the 96-column solve of a 32-column block)."""
    GK, GM, rigid = refs.graded_pencil(96, 196)
    ref = refs.mp_pencil_eigvals(GK, GM)
    theta, Cm, info = _eigh(GK, GM, -1e-6)
    _check_pencil(GK, GM, theta, Cm, info)
    s = _effective_shift(GK, GM, -1e-6)
    rel = float((np.abs(theta - ref) / (np.abs(ref) + s)).max())
    print(f"[eigh graded] N 96 mpmath: max rel(theta+s) {rel:.2e}, sweeps {info[1]}")
    assert rel <= 1e-13


def _cluster_pencil(N, seed):
    """GK c = theta GM c with exact eigenvalue multiplicities 2 and 3 and a pair at relative gap 1e-10 (before the
    entries are rounded), well separated from the rest; returns GK, GM, eigenvalues, the index groups of the clusters"""
    rng = np.random.default_rng(seed)
    Q = rng.standard_normal((4 * N, N))
    GM = Q.T @ Q / (4 * N) + 0.1 * np.eye(N)
    ev = np.geomspace(1e7, 1e12, N)
    groups = []
    for start, mult, gap in ((N // 4, 2, 0.0), (N // 2, 3, 0.0), (3 * N // 4, 2, 1e-10)):
        ev[start:start + mult] = ev[start] * (1 + gap * np.arange(mult))
        groups.append(list(range(start, start + mult)))
    V = np.linalg.qr(rng.standard_normal((N, N)))[0]
    Lm = np.linalg.cholesky(GM)
    GK = Lm @ (V * ev) @ V.T @ Lm.T
    return (GK + GK.T) / 2, GM, ev, groups


@pytest.mark.parametrize("sigma", SIGMAS)
@pytest.mark.parametrize("N", [16, 47, 48, 49, 96, 131, 143, 144])
def test_eigh_clusters(N, sigma):
    """Exact double and triple eigenvalues and a pair at relative gap 1e-10: theta within 1e-13 (max|theta| + |sigma|) of
    LAPACK (measured: 5.6e-15); the cluster subspaces agree with LAPACK's by the distance of their GM-orthogonal
    projectors, <= 1e-10 (measured: 6.4e-12), although single vectors inside a cluster are arbitrary."""
    GK, GM, ev, groups = _cluster_pencil(N, 7 * N)
    theta, Cm, info = _eigh(GK, GM, sigma)
    res, orth = _check_pencil(GK, GM, theta, Cm, info)
    w, Z = scipy.linalg.eigh(GK, GM)
    err = float(np.abs(theta - w).max() / (np.abs(w).max() + abs(sigma)))
    dist = 0.0
    for g in groups:
        Pc = Cm[:N, g] @ Cm[:N, g].T @ GM
        Pz = Z[:, g] @ Z[:, g].T @ GM
        dist = max(dist, float(np.linalg.norm(Pc - Pz, 2)))
    print(f"[eigh clusters] N {N} sigma {sigma:g}: theta err {err:.2e}, projector dist {dist:.2e}, res {res:.2e}, "
          f"orth {orth:.2e}, sweeps {info[1]}")
    assert err <= 1e-13
    assert dist <= 1e-10


@pytest.mark.parametrize("sigma", SIGMAS)
@pytest.mark.parametrize("kappa", [1e6, 1e10, 1e13])
@pytest.mark.parametrize("N", [16, 48, 49, 144])
def test_eigh_ill_conditioned_gm(N, kappa, sigma):
    """GM of condition number kappa sharing its near-null directions with GK (as nearly dependent columns of [X W P] make
    them): the eigenvalues are still 1e7 .. 1e9, and perturbations of the stored entries move them by ~eps kappa.
    theta within 1e-17 kappa (max|theta| + |sigma|) of mpmath (N <= 48) / LAPACK (measured: <= 2.4e-18 kappa),
    C^T GM C = I within 2e-17 kappa (measured: <= 6.3e-18 kappa), every column's residual <= 1e-14 (measured:
    7.1e-17)."""
    GK, GM, ref = _ill_pencil(N, kappa)
    theta, Cm, info = _eigh(GK, GM, sigma)
    assert info[0] == 0 and 1 <= info[1] <= 24, info
    err = float(np.abs(theta - ref).max() / (np.abs(ref).max() + abs(sigma)))
    Cn = Cm[:N, :N]
    R = GK @ Cn - (GM @ Cn) * theta
    scale = (np.linalg.norm(GK, 2) + np.abs(theta) * np.linalg.norm(GM, 2)) * np.linalg.norm(Cn, axis=0)
    res = float((np.linalg.norm(R, axis=0) / scale).max())
    orth = float(np.abs(Cn.T @ GM @ Cn - np.eye(N)).max())
    print(f"[eigh ill GM] N {N} kappa {kappa:.0e} sigma {sigma:g}: theta err {err:.2e}, res {res:.2e}, orth {orth:.2e}, "
          f"sweeps {info[1]}")
    assert np.all(np.diff(theta) >= 0)
    assert err <= 1e-17 * kappa
    assert res <= 1e-14
    assert orth <= 2e-17 * kappa


@functools.lru_cache(maxsize=None)
def _ill_pencil(N, kappa):
    """GM with eigenvalues 1 .. 1/kappa, GK = L V diag(1e7 .. 1e9) V^T L^T (L = chol(GM)); eigenvalues of the stored
    pencil from mpmath (N <= 48) or LAPACK"""
    rng = np.random.default_rng(int(np.log10(kappa)) * 1000 + N)
    Q = np.linalg.qr(rng.standard_normal((N, N)))[0]
    GM = (Q * np.geomspace(1.0, 1.0 / kappa, N)) @ Q.T
    GM = (GM + GM.T) / 2
    V = np.linalg.qr(rng.standard_normal((N, N)))[0]
    Lm = np.linalg.cholesky(GM)
    GK = Lm @ (V * np.geomspace(1e7, 1e9, N)) @ V.T @ Lm.T
    GK = (GK + GK.T) / 2
    ref = refs.mp_pencil_eigvals(GK, GM) if N <= 48 else scipy.linalg.eigh(GK, GM, eigvals_only=True)
    return GK, GM, ref


@pytest.mark.parametrize("N", [2, 16, 49, 144])
def test_eigh_failure_codes(N):
    """An indefinite GM gives info[0] in [1, N]; GK + s GM indefinite gives info[0] >= 1000 -- at the drivers' relative
    shift -1e-6 a rigid-size eigenvalue of -1e-5 is not lifted when the mean diagonal of GK is O(1), nor at sigma = 0."""
    rng = np.random.default_rng(N)
    Q = np.linalg.qr(rng.standard_normal((N, N)))[0]
    GK = (Q * np.geomspace(1.0, 10.0, N)) @ Q.T
    d = np.geomspace(1.0, 2.0, N)
    d[N // 2] = -0.5
    GMi = (Q * d) @ Q.T
    for sigma in SIGMAS:
        _, _, info = _eigh((GK + GK.T) / 2, (GMi + GMi.T) / 2, sigma)
        assert 1 <= info[0] <= N, info
    V = np.linalg.qr(rng.standard_normal((N, N)))[0]
    ev = np.concatenate([[-1e-5], np.geomspace(1e-4, 1.0, N - 1)])
    GKi = (V * ev) @ V.T
    for sigma in (-1e-6, 0.0):
        _, _, info = _eigh((GKi + GKi.T) / 2, np.eye(N), sigma)
        assert info[0] >= 1000 and info[0] - 1000 <= N, info
    # a large enough shift lifts it; theta + sigma is then relatively accurate (the bar of the graded pencils)
    theta, _, info = _eigh((GKi + GKi.T) / 2, np.eye(N), 1e5)
    assert info[0] == 0 and abs(theta[0] + 1e-5) <= 1e-12 * (1e-5 + 1e5)


@pytest.mark.parametrize("N", [3, 48, 49, 131])
def test_eigh_input_contract(N):
    """Only the upper triangle is read (the lower one full of NaN changes no bit); ldg = 144 and ldc = 144 with N < 144
    (nothing outside the N x N blocks is read or written); two calls give the same bits."""
    GK, GM, _, _ = _graded(N)
    theta0, C0, info0 = _eigh(GK, GM, -1e-6)
    _check_pencil(GK, GM, theta0, C0, info0)
    low = np.tril_indices(N, -1)
    GKn, GMn = GK.copy(), GM.copy()
    GKn[low] = np.nan
    GMn[low] = np.nan
    theta1, C1, _ = _eigh(GKn, GMn, -1e-6)
    assert np.array_equal(theta0, theta1) and np.array_equal(C0, C1)
    GKw = np.full((144, 144), np.nan)
    GMw = np.full((144, 144), np.nan)
    iu = np.triu_indices(N)
    GKw[iu], GMw[iu] = GK[iu], GM[iu]
    theta2, C2, _ = _eigh(GKw, GMw, -1e-6, N=N, ldc=144)
    assert np.array_equal(theta0, theta2) and np.array_equal(C0, C2[:N, :N])
    assert (C2[N:, :] == SENT).all() and (C2[:, N:] == SENT).all()
    theta3, C3, _ = _eigh(GK, GM, -1e-6)
    assert np.array_equal(theta0, theta3) and np.array_equal(C0, C3)


@pytest.mark.parametrize("m,na,act", [(16, 11, [0, 3, 4, 9, 15]), (48, 48, list(range(48))), (32, 5, [])])
def test_eigh_idx_slots_match_compact(m, na, act):
    """The slot-map variant on the drivers' non-contiguous slots (X = [0, m), active W = [m, m + na), P at 2m + active
    columns) in 144 x 144 storage gives the bits of the compact problem; rows of C outside the slots keep their
    contents."""
    slots = list(range(m)) + [m + s for s in range(na)] + [2 * m + j for j in act]
    N = len(slots)
    GK, GM, _ = refs.graded_pencil(N, 100 + N)
    theta0, C0, info0 = _eigh(GK, GM, -1e-6)
    _check_pencil(GK, GM, theta0, C0, info0)
    GKw = np.full((144, 144), np.nan)
    GMw = np.full((144, 144), np.nan)
    sl = np.array(slots)
    iu = np.triu_indices(N)
    GKw[sl[iu[0]], sl[iu[1]]] = GK[iu]
    GMw[sl[iu[0]], sl[iu[1]]] = GM[iu]
    theta1, C1, info1 = _eigh(GKw, GMw, -1e-6, N=N, idx=slots, ldc=144)
    assert info1[0] == 0
    assert np.array_equal(theta0, theta1)
    assert np.array_equal(C1[sl, :N], C0)
    others = np.setdiff1d(np.arange(144), sl)
    assert (C1[others, :] == SENT).all() and (C1[:, N:] == SENT).all()


def test_eigh_sweeps_below_cap_report():
    """Runs after the pencils above (file order): the largest Jacobi sweep count any of them needed (measured: 14),
    below the cap of 24."""
    print(f"[eigh] largest sweep count over all pencils: {_sweeps['max']}")
    assert _sweeps["max"] <= 24


# ---------------------------------------------------------------------------------------------------------------------
# D. the Chebyshev preconditioner
# ---------------------------------------------------------------------------------------------------------------------
CHEB_DEGREES = [1, 2, 3, 12, 40, 64, 65]
CHEB_NCOLS = [16, 32, 48, 64]
CHP_MAX_DEGREE = 64


def _cheb(pat, rec, invD, R, degree, lmax, ratio, persistent):
    """(z, launches): the result and the number of library kernel launches of the call"""
    from diffsound_b200 import native
    lib = _lib()
    before = lib.ds_launch_count()
    z = native.cheb32_solve(pat, rec, invD, R, degree, lmax, ratio, persistent=persistent)
    return z, lib.ds_launch_count() - before


def _persistent_eligible(pat, degree, ncols):
    """the conditions of Level32::cheb under which all steps run in one cooperative launch"""
    lib = _lib()
    nchunks = lib.ds_spmm32_chunk_count(pat.n_nodes)
    avg = (lib.ds_k32_record_bytes(pat.nnzb) - 64) // nchunks
    return 3 <= degree <= CHP_MAX_DEGREE and nchunks >= 8 and avg <= 190 * 1024 and ncols in (16, 32, 48)


def _expected_launches(pat, degree, ncols, persistent):
    # the row-chunk table, then either the cooperative kernel or the Jacobi step and degree - 1 SpMM steps
    return 2 if persistent and _persistent_eligible(pat, degree, ncols) else 1 + degree


@functools.lru_cache(maxsize=None)
def _cube3_dense():
    """A y = mu D y for cube3 order 2 (dense), D the exact fp64 3x3 block diagonal"""
    from diffsound_b200 import native
    pat, Kval, _, K, _ = _system("cube3", 2)
    rec, invD = native.k32_pack(pat, Kval)
    D = refs.block_diagonal(K, pat.n_nodes)
    Dm = refs.block_diag_matrix(D).toarray()
    mu, Y = scipy.linalg.eigh(K.toarray(), Dm)
    return pat, rec, invD, Dm, mu, Y


@pytest.mark.parametrize("persistent", [True, False])
@pytest.mark.parametrize("where", ["above", "below"])
@pytest.mark.parametrize("ncols", CHEB_NCOLS)
def test_chebyshev_closed_form(ncols, where, persistent):
    """R = D Y for generalised eigenvectors A y = mu D y of cube3 order 2 (343 nodes: 11 row chunks, eligible for the
    persistent kernel): z = p_k(mu) y / ... with p_k the closed-form Chebyshev polynomial, for every degree, with lmax
    above the largest mu and just below it.  <= 1e-4 of each column's norm (fp32 records and arithmetic, the fp32
    rounding of R = D Y feeds every mode; measured: above 1.1e-5, below 1.6e-5), and the kernel launches show which path ran."""
    pat, rec, invD, Dm, mu, Y = _cube3_dense()
    assert _lib().ds_spmm32_chunk_count(pat.n_nodes) == 11
    sel = np.linspace(12, mu.size - 1, ncols).round().astype(int)      # skips the six rigid modes (mu ~ 0)
    lmax = 1.05 * mu.max() if where == "above" else 0.998 * mu.max()
    R = torch.tensor((Dm @ Y[:, sel]).astype(np.float32), device=DEV)
    worst = 0.0
    for degree in CHEB_DEGREES:
        ratio = 0.4 * degree * degree + 2.0
        z, launches = _cheb(pat, rec, invD, R, degree, lmax, ratio, persistent)
        assert launches == _expected_launches(pat, degree, ncols, persistent), (degree, launches)
        ref = Y[:, sel] * refs.cheb_closed_form(mu[sel], degree, lmax, ratio)[None, :]
        err = float((np.linalg.norm(z.cpu().numpy() - ref, axis=0) / np.linalg.norm(ref, axis=0)).max())
        worst = max(worst, err)
    print(f"[cheb closed form] ncols {ncols} lmax {where} persistent {persistent}: max column rel err {worst:.2e}")
    assert worst <= 1e-4


@functools.lru_cache(maxsize=None)
def _cheb_reference(name, order):
    """fp64 Chebyshev iterates 1 .. 65 (Saad, Alg. 12.1) for 64 random columns; lmax = 1.1 lambda_max(D^-1 K)"""
    from diffsound_b200 import native
    pat, Kval, _, K, _ = _system(name, order)
    rec, invD = native.k32_pack(pat, Kval)
    nn = pat.n_nodes
    D = refs.block_diagonal(K, nn)
    w, V = np.linalg.eigh(D)
    Dih = refs.block_diag_matrix(np.einsum("nij,nj,nkj->nik", V, 1.0 / np.sqrt(w), V))
    lmax = 1.1 * float(scipy.sparse.linalg.eigsh(Dih @ K @ Dih, k=1, which="LA", tol=1e-6,
                                                 v0=np.ones(3 * nn), return_eigenvectors=False)[0])
    Dinv = np.linalg.inv(D)
    apply_Dinv = lambda r: np.einsum("ncd,ndk->nck", Dinv, r.reshape(nn, 3, -1)).reshape(3 * nn, -1)
    rng = np.random.default_rng(3)
    R = rng.standard_normal((3 * nn, 64)).astype(np.float32)
    xs = refs.cheb_iterates(lambda v: K @ v, apply_Dinv, R.astype(np.float64), max(CHEB_DEGREES), lmax, 30.0)
    return pat, rec, invD, R, lmax, xs


@pytest.mark.parametrize("ncols", CHEB_NCOLS)
@pytest.mark.parametrize("name,order", [("grid16", 1), ("bowl", 1), ("bowl", 2)])
def test_chebyshev_matches_fp64_iteration(name, order, ncols):
    """Both paths against the textbook fp64 iteration on larger meshes, degrees 1 .. 65 (65 is above the persistent
    kernel's limit, ncols 64 is stepwise only): <= 1e-5 of each column's norm (measured: 7.8e-7), and every eligible
    case ran the persistent kernel (two launches: the row chunks and the cooperative kernel)."""
    pat, rec, invD, R, lmax, xs = _cheb_reference(name, order)
    Rd = torch.tensor(R[:, :ncols].copy(), device=DEV)
    worst, n_persistent = 0.0, 0
    for degree in CHEB_DEGREES:
        ref = xs[degree - 1][:, :ncols]
        for persistent in (True, False):
            z, launches = _cheb(pat, rec, invD, Rd, degree, lmax, 30.0, persistent)
            expect = _expected_launches(pat, degree, ncols, persistent)
            assert launches == expect, (degree, persistent, launches, expect)
            n_persistent += expect == 2 and degree > 1
            err = float((np.linalg.norm(z.cpu().numpy() - ref, axis=0) / np.linalg.norm(ref, axis=0)).max())
            worst = max(worst, err)
    print(f"[cheb fp64] {name} o{order} ncols {ncols}: max column rel err {worst:.2e}, persistent runs {n_persistent}")
    assert worst <= 1e-5
    assert n_persistent == (0 if ncols == 64 else 4)        # degrees 3, 12, 40 and 64 of the persistent calls


# ---------------------------------------------------------------------------------------------------------------------
# E. row-slab utilities
# ---------------------------------------------------------------------------------------------------------------------
def test_gather_cols_f32():
    """dst[:, s] = fp32(src[:, cols[s]]) in the order given, zero for count <= s < width: exact."""
    lib = _lib()
    rng = np.random.default_rng(0)
    n, lds = 3001, 48
    src = rng.standard_normal((n, lds)) * 10.0 ** rng.uniform(-5, 5, (n, lds))
    srcd = torch.tensor(src, device=DEV)
    for cols, width in (([7, 0, 47, 3, 3, 12, 40], 16), (list(range(47, -1, -1)), 48), ([5], 4), ([], 16)):
        dst = torch.full((n, width), SENT, dtype=torch.float32, device=DEV)
        arr = (C.c_int * max(1, len(cols)))(*cols)
        _check(lib.ds_gather_cols_f32(_p(srcd), lds, arr, len(cols), width, n, _p(dst), _st()), "ds_gather_cols_f32")
        ref = np.zeros((n, width), dtype=np.float32)
        ref[:, :len(cols)] = src[:, cols].astype(np.float32)
        assert np.array_equal(dst.cpu().numpy(), ref)


def test_widen_f32():
    """dst[:, off:off + width] = fp64(src) exactly (into a column block of a wider buffer), nothing else written."""
    lib = _lib()
    rng = np.random.default_rng(1)
    n = 2999
    for width, ldd, off in ((16, 48, 16), (48, 144, 48), (32, 96, 64)):
        src = (rng.standard_normal((n, width)) * 1e3).astype(np.float32)
        dst = torch.full((n, ldd), SENT, dtype=torch.float64, device=DEV)
        srcd = torch.tensor(src, device=DEV)
        _check(lib.ds_widen_f32(_p(srcd), width, n, _p(dst, off), ldd, _st()), "ds_widen_f32")
        got = dst.cpu().numpy()
        assert np.array_equal(got[:, off:off + width], src.astype(np.float64))
        assert (got[:, :off] == SENT).all() and (got[:, off + width:] == SENT).all()


@pytest.mark.parametrize("ncols", [4, 16, 48])
def test_jacobi32(ncols):
    """Out = cc invD R within 1e-6 of cc |invD| |R| per entry (fp32 products and sums; measured: 2.1e-7)."""
    from diffsound_b200 import native
    lib = _lib()
    pat, Kval, _, _, _ = _system("bowl", 1)
    _, invD = native.k32_pack(pat, Kval)
    nn = pat.n_nodes
    rng = np.random.default_rng(ncols)
    R = (rng.standard_normal((3 * nn, ncols)) * 1e6).astype(np.float32)
    out = torch.full((3 * nn, ncols), SENT, dtype=torch.float32, device=DEV)
    cc = 0.6180339887
    Rd = torch.tensor(R, device=DEV)
    _check(lib.ds_jacobi32(_p(invD), _p(Rd), nn, ncols, cc, _p(out), _st()), "ds_jacobi32")
    Di = invD.cpu().numpy().astype(np.float64).reshape(nn, 3, 3)
    R64 = R.astype(np.float64).reshape(nn, 3, ncols)
    ref = cc * np.einsum("ncd,ndk->nck", Di, R64).reshape(3 * nn, ncols)
    bound = cc * np.einsum("ncd,ndk->nck", np.abs(Di), np.abs(R64)).reshape(3 * nn, ncols)
    err = float((np.abs(out.cpu().numpy() - ref) / bound).max())
    print(f"[jacobi32] ncols {ncols}: {err:.2e}")
    assert err <= 1e-6


@pytest.mark.parametrize("m,wa", [(16, 16), (32, 21), (48, 48), (48, 1)])
def test_gram_insert(m, wa):
    """Rows and columns [m, 2m) of GK / GM from the strips (W-W block mirrored from its upper triangle, rows / columns
    of inactive W zero); every other entry untouched: exact."""
    lib = _lib()
    rng = np.random.default_rng(m + wa)
    N, ldg, lds = 3 * m, 144, 144
    G0 = [rng.standard_normal((ldg, ldg)) for _ in range(2)]
    Gs = [rng.standard_normal((lds, lds)) for _ in range(2)]
    Gd = [torch.tensor(g, device=DEV) for g in G0]
    Gsd = [torch.tensor(g, device=DEV) for g in Gs]      # kept alive: a freed temporary's memory is handed out again
    _check(lib.ds_gram_insert_f64(_p(Gd[0]), _p(Gd[1]), ldg, _p(Gsd[0]), _p(Gsd[1]), lds, m, wa, _st()), "ds_gram_insert_f64")
    for g0, gs, gd in zip(G0, Gs, Gd):
        ref = g0.copy()
        strip = np.zeros((m, N))
        strip[:wa] = gs[:wa, :N]
        ww = np.triu(gs[:wa, m:m + wa])
        ww = ww + np.triu(ww, 1).T
        strip[:wa, m:2 * m] = 0.0
        strip[:wa, m:m + wa] = ww
        ref[m:2 * m, :N] = strip
        ref[:N, m:2 * m] = strip.T
        assert np.array_equal(gd.cpu().numpy(), ref)


@pytest.mark.parametrize("N", [2, 48, 131, 144])
def test_sym_upper(N):
    """The lower triangle of the leading N x N block becomes the exact mirror of the upper one; nothing else changes."""
    lib = _lib()
    rng = np.random.default_rng(N)
    G0 = [rng.standard_normal((144, 144)) for _ in range(2)]
    Gd = [torch.tensor(g, device=DEV) for g in G0]
    _check(lib.ds_sym_upper_f64(_p(Gd[0]), _p(Gd[1]), 144, N, _st()), "ds_sym_upper_f64")
    for g0, gd in zip(G0, Gd):
        ref = g0.copy()
        blk = np.triu(g0[:N, :N])
        ref[:N, :N] = blk + np.triu(blk, 1).T
        assert np.array_equal(gd.cpu().numpy(), ref)


def test_pmg_prolong64():
    """x_i = 0.5 (xc[p0] + xc[p1]) in fp64, bit for bit, for the rows of a column block of width w (ld > w)."""
    from diffsound_b200 import native
    lib = _lib()
    v, t = _mesh("grid16")
    pv, pt = mo.promote(torch.as_tensor(v), torch.as_tensor(t), 2)
    cl = native.CoarseLevel(pv.to(DEV).contiguous(), pt.to(torch.int32).to(DEV).contiguous())
    nf, nc = pv.shape[0], cl.n_nodes
    par = cl.parents.cpu().numpy().reshape(nf, 2)
    rng = np.random.default_rng(2)
    for w, ldc, ldx in ((16, 16, 16), (48, 48, 48), (32, 48, 144)):
        xc = rng.standard_normal((3 * nc, ldc))
        x = torch.full((3 * nf, ldx), SENT, dtype=torch.float64, device=DEV)
        xcd = torch.tensor(xc, device=DEV)
        _check(lib.ds_pmg_prolong64(_p(cl.parents), nf, _p(xcd), ldc, w, _p(x), ldx, _st()),
               "ds_pmg_prolong64")
        xr = xc.reshape(nc, 3, ldc)[:, :, :w]
        ref = (0.5 * (xr[par[:, 0]] + xr[par[:, 1]])).reshape(3 * nf, w)
        got = x.cpu().numpy()
        assert np.array_equal(got[:, :w], ref)
        assert (got[:, w:] == SENT).all()


@pytest.mark.parametrize("ncols", [16, 48])
def test_pmg_restrict32_range(ncols):
    """Two ranges that split the fine nodes: each partial, and their sum, within 1e-6 of |P^T| |res| per entry of the fp64
    P^T res and of pmg_restrict32 (fp32 sums; measured: 2.1e-7); the whole range reproduces pmg_restrict32 bit for
    bit."""
    from diffsound_b200 import native
    lib = _lib()
    v, t = _mesh("grid16")
    pv, pt = mo.promote(torch.as_tensor(v), torch.as_tensor(t), 2)
    cl = native.CoarseLevel(pv.to(DEV).contiguous(), pt.to(torch.int32).to(DEV).contiguous())
    nf, nc = pv.shape[0], cl.n_nodes
    par = cl.parents.cpu().numpy().reshape(nf, 2)
    Pn = sp.csr_matrix((np.full(2 * nf, 0.5), (np.repeat(np.arange(nf), 2), par.reshape(-1))), shape=(nf, nc))
    P = sp.kron(Pn, sp.identity(3), format="csr")
    rng = np.random.default_rng(ncols)
    res = rng.standard_normal((3 * nf, ncols)).astype(np.float32)
    resd = torch.tensor(res, device=DEV)
    full = native.pmg_restrict32(cl, resd).cpu().numpy()

    def part(lo, hi):
        rc = torch.full((3 * nc, ncols), SENT, dtype=torch.float32, device=DEV)
        loc = resd[3 * lo:3 * hi].contiguous()
        _check(lib.ds_pmg_restrict32_range(_p(cl.rptr), _p(cl.rlist), nc, _p(loc), ncols, lo, hi, _p(rc), _st()),
               "ds_pmg_restrict32_range")
        return rc.cpu().numpy()

    assert np.array_equal(part(0, nf), full)
    split = nf // 3 + 7
    a, b = part(0, split), part(split, nf)
    res64 = res.astype(np.float64)
    bound = abs(P.T) @ np.abs(res64)
    perr = 0.0
    for lo, hi, got in ((0, split, a), (split, nf, b)):
        r = res64.copy()
        r[:3 * lo] = 0.0
        r[3 * hi:] = 0.0
        perr = max(perr, float((np.abs(got - P.T @ r) / bound).max()))
    err = float((np.abs(a.astype(np.float64) + b - P.T @ res64) / bound).max())
    ferr = float((np.abs(a.astype(np.float64) + b - full) / bound).max())
    print(f"[restrict32_range] ncols {ncols}: of |P^T||res|: partials {perr:.2e}, their sum vs P^T res {err:.2e}, "
          f"vs pmg_restrict32 {ferr:.2e}")
    assert perr <= 1e-6 and err <= 1e-6 and ferr <= 1e-6
