"""The host references of tests/test_lobpcg_kernels_gpu.py (tests/lobpcg_refs.py) checked against each other and
against their construction, without a GPU."""
import numpy as np
import pytest
import scipy.linalg

import lobpcg_refs as refs


@pytest.mark.parametrize("degree", [1, 2, 3, 12, 40, 64, 65])
@pytest.mark.parametrize("lmax", [2.8, 2.0])
def test_chebyshev_closed_form_matches_recurrence(degree, lmax):
    """Saad's Chebyshev iteration on a diagonal operator (D = I) reproduces the closed-form polynomial at every
    eigenvalue, inside the interval, below lmin and above lmax: <= 1e-12 relative (measured here: 2e-14)."""
    mu = np.concatenate([np.linspace(0.01, 2.9, 60), [2.0 / (0.4 * degree * degree + 2.0)]])
    ratio = 0.4 * degree * degree + 2.0
    xs = refs.cheb_iterates(lambda x: mu * x, lambda x: x, np.ones_like(mu), degree, lmax, ratio)
    assert len(xs) == degree
    for k in (1, degree // 2, degree):
        if k >= 1:
            cf = refs.cheb_closed_form(mu, k, lmax, ratio)
            assert np.max(np.abs(xs[k - 1] - cf) / np.abs(cf)) <= 1e-12


def test_chebyshev_iteration_uses_block_jacobi():
    """With a non-trivial block diagonal D the iterate is p(D^-1 A) D^-1 b, checked on the generalised eigenvectors
    A y = mu D y of a small SPD block matrix (R = D Y): <= 1e-11 relative."""
    rng = np.random.default_rng(0)
    n = 8
    B = rng.standard_normal((3 * n, 3 * n))
    A = B @ B.T + 3 * n * np.eye(3 * n)
    D = np.stack([A[3 * i:3 * i + 3, 3 * i:3 * i + 3] for i in range(n)])
    Dm = refs.block_diag_matrix(D).toarray()
    mu, Y = scipy.linalg.eigh(A, Dm)
    Dinv = np.linalg.inv(D)
    apply_Dinv = lambda r: np.einsum("ncd,ndk->nck", Dinv, r.reshape(n, 3, -1)).reshape(3 * n, -1)
    lmax = 1.05 * mu.max()
    x = refs.cheb_iterates(lambda v: A @ v, apply_Dinv, Dm @ Y, 12, lmax, 30.0)[-1]
    ref = Y * refs.cheb_closed_form(mu, 12, lmax, 30.0)[None, :]
    assert np.abs(x - ref).max() <= 1e-11 * np.abs(ref).max()


def test_mpmath_pencil_matches_scipy_when_well_conditioned():
    """mpmath at 40 digits against LAPACK on a well-conditioned pencil: <= 1e-13 relative (measured here: ~1e-15)."""
    rng = np.random.default_rng(1)
    N = 12
    Q = rng.standard_normal((3 * N, N))
    GM = Q.T @ Q / (3 * N) + 0.5 * np.eye(N)
    B = rng.standard_normal((N, N))
    GK = B @ B.T + N * np.eye(N)
    w = scipy.linalg.eigh(GK, GM, eigvals_only=True)
    wm = refs.mp_pencil_eigvals(GK, GM)
    assert np.max(np.abs(wm - w) / np.abs(w)) <= 1e-13


@pytest.mark.parametrize("N", [2, 3, 16, 48])
def test_graded_pencil_rigid_eigenvalues_match_construction(N):
    """The rigid-size eigenvalues of the stored graded pencil equal the constructed ones to relative rounding of the
    entries (<= 1e-13, measured here: 1.7e-16), while LAPACK cannot resolve them for N >= 16 (they sit 17 orders of
    magnitude below the largest eigenvalue): the graded pencils need the mpmath reference."""
    GK, GM, rigid = refs.graded_pencil(N, N)
    w = refs.mp_pencil_eigvals(GK, GM)
    nr = rigid.size
    assert np.max(np.abs(w[:nr] - rigid) / rigid) <= 1e-13
    assert w[nr] >= 1e6 and w[-1] <= 1e13
    if N >= 16:
        assert w[-1] >= 1e11
        ws = scipy.linalg.eigh(GK, GM, eigvals_only=True)
        assert np.max(np.abs(ws[:nr] - rigid) / rigid) > 1e-6
