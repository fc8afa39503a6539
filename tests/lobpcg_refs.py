"""Host references for the eigensolver's inner kernels (tests/test_lobpcg_kernels_gpu.py), pinned on the CPU by
tests/test_lobpcg_refs_cpu.py.

- `cheb_closed_form`: the block-Jacobi Chebyshev polynomial of degree k on [lmax / ratio, lmax] at an eigenvalue mu of
  D^-1 A, z = (1 - T_k((theta - mu) / delta) / T_k(theta / delta)) / mu, with T_k from cos / cosh (no recurrence).
- `cheb_iterates`: Chebyshev acceleration in fp64 as written in Saad, Iterative Methods for Sparse Linear Systems, 2nd ed.,
  Algorithm 12.1, from x_0 = 0 with the preconditioned residual D^-1 r.
- `graded_pencil`: a driver-like Rayleigh-Ritz pencil whose rigid-size eigenvalues are known exactly by construction.
- `mp_pencil_eigvals`: eigenvalues of a pencil as stored in fp64, at 40 significant digits (mpmath).
"""
import mpmath
import numpy as np
import scipy.sparse as sp


def cheb_T(k, x):
    """T_k(x) for real x, elementwise, from the trigonometric / hyperbolic closed forms."""
    x = np.asarray(x, dtype=np.float64)
    inside = np.abs(x) <= 1.0
    out = np.empty_like(x)
    out[inside] = np.cos(k * np.arccos(x[inside]))
    xo = x[~inside]
    out[~inside] = np.sign(xo) ** k * np.cosh(k * np.arccosh(np.abs(xo)))
    return out


def cheb_closed_form(mu, degree, lmax, ratio):
    """p(mu) with z = p(D^-1 A) D^-1 r: (1 - T_k((theta - mu)/delta) / T_k(theta/delta)) / mu, k = degree, mu != 0."""
    lmin = lmax / ratio
    theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
    mu = np.asarray(mu, dtype=np.float64)
    return (1.0 - cheb_T(degree, (theta - mu) / delta) / cheb_T(degree, np.array(theta / delta))) / mu


def cheb_iterates(apply_A, apply_Dinv, b, degree, lmax, ratio):
    """x_1 .. x_degree of Saad's Algorithm 12.1 for A x = b, preconditioned by D, from x_0 = 0 (a list)."""
    lmin = lmax / ratio
    theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
    sigma1 = theta / delta
    rho = 1.0 / sigma1
    x = np.zeros_like(b)
    r = b.copy()
    d = apply_Dinv(r) / theta
    out = []
    for _ in range(degree):
        x = x + d
        out.append(x.copy())
        r = r - apply_A(d)
        rho_new = 1.0 / (2.0 * sigma1 - rho)
        d = rho_new * rho * d + (2.0 * rho_new / delta) * apply_Dinv(r)
        rho = rho_new
    return out


def block_diagonal(K, n_nodes):
    """(n_nodes, 3, 3) diagonal blocks of a scalar-CSR matrix with 3 dofs per node."""
    Kc = sp.csr_matrix(K)
    D = np.zeros((n_nodes, 3, 3))
    idx = np.arange(n_nodes) * 3
    for c in range(3):
        for d in range(3):
            D[:, c, d] = np.asarray(Kc[idx + c, idx + d]).ravel()
    return D


def block_diag_matrix(D):
    """scipy block-diagonal matrix of (n, 3, 3) blocks."""
    n = D.shape[0]
    rows = np.repeat(np.arange(3 * n).reshape(n, 3), 3, axis=1).ravel()
    cols = np.tile(np.arange(3 * n).reshape(n, 3), (1, 3)).ravel()
    return sp.csr_matrix((D.ravel(), (rows, cols)), shape=(3 * n, 3 * n))


def _spd_unit_diag(n, rng, cond=10.0):
    """well-conditioned SPD matrix with unit diagonal (condition number about `cond`)."""
    Q = np.linalg.qr(rng.standard_normal((n, n)))[0]
    A = (Q * np.geomspace(1.0, cond, n)) @ Q.T
    d = 1.0 / np.sqrt(np.diag(A))
    return A * d[:, None] * d[None, :]


def graded_pencil(N, seed):
    """(GK, GM, rigid) shaped like the Rayleigh-Ritz pencil of the eigensolver: the first slots carry rigid-size
    eigenvalues (1e-5 .. 1e-2), then elastic values (1e7 .. 1e9), then W / P Rayleigh quotients up to 1e12.

    GK0 = diag(rigid) (+) S A S with S the square roots of the other scales and A a well-conditioned unit-diagonal SPD
    matrix; GM0 = I (+) (I + small symmetric perturbation).  Both are congruent with one unit upper-triangular T, which
    keeps GK graded (row i of GK only mixes in rows k <= i), so the small eigenvalues stay determined to relative accuracy
    by the stored entries.  The pencil's rigid eigenvalues are exactly `rigid` before the entries are rounded to fp64."""
    rng = np.random.default_rng(seed)
    nr = 6 if N >= 16 else max(1, N // 3)
    rigid = np.geomspace(1e-5, 1e-2, nr)
    rest = N - nr
    ne = (rest + 1) // 2
    scales = np.concatenate([np.geomspace(1e7, 1e9, ne), rng.permutation(np.geomspace(1e9, 1e12, rest - ne))])
    s = np.sqrt(scales)
    GK0 = np.zeros((N, N))
    GM0 = np.eye(N)
    GK0[:nr, :nr] = np.diag(rigid)
    GK0[nr:, nr:] = _spd_unit_diag(rest, rng) * s[:, None] * s[None, :]
    E = rng.standard_normal((rest, rest)) * (0.05 / np.sqrt(rest))
    GM0[nr:, nr:] += (E + E.T) / 2
    T = np.eye(N) + np.triu(rng.standard_normal((N, N)), 1) * (0.3 / np.sqrt(N))
    GK = T.T @ GK0 @ T
    GM = T.T @ GM0 @ T
    return (GK + GK.T) / 2, (GM + GM.T) / 2, rigid


def mp_pencil_eigvals(GK, GM, dps=40):
    """ascending eigenvalues of GK c = theta GM c (GM SPD) for the fp64 entries as stored, computed at `dps` digits:
    L = chol(GM), eigenvalues of L^-1 GK L^-T."""
    N = GK.shape[0]
    with mpmath.workdps(dps):
        A = mpmath.matrix(GK.tolist())
        L = mpmath.cholesky(mpmath.matrix(GM.tolist()))
        Li = mpmath.inverse(L)
        H = Li * A * Li.T
        for i in range(N):
            for j in range(i):
                H[i, j] = H[j, i] = (H[i, j] + H[j, i]) / 2
        E = mpmath.eigsy(H, eigvals_only=True)
        return np.array(sorted(float(e) for e in E))
