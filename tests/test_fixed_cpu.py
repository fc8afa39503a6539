"""Clamped objects on the host: the reference of the reduced pencil (tests/fixed_oracle.py) against beam theory and the
interlacing bounds, and the validation of a clamp mask (DiffSoundObj.fix_nodes)."""
import numpy as np
import pytest
import scipy.linalg
import torch

import fixed_oracle as fo
from oracle import modal_oracle as mo
from test_modal_gains_cpu import kuhn_box, promote

RHO, E, NU = 7850.0, 2.0e11, 0.29


def test_oracle_cantilever_matches_euler_bernoulli():
    L, b, h = 1.0, 0.1, 0.05                       # slender (L / h = 20), bending in the thin direction z
    v, t = kuhn_box((40, 4, 2), (L, b, h))
    pv, pt = promote(v, t, 2)
    K, M = mo.assemble(torch.from_numpy(pv), torch.from_numpy(pt), 2, E, NU, RHO)
    lam, U = fo.eig_fixed(K, M, pv[:, 0] <= 1e-6, 2)
    f = np.sqrt(lam[0]) / (2 * np.pi)
    f_eb = 1.8751 ** 2 * np.sqrt(E * (b * h ** 3 / 12) / (RHO * b * h * L ** 4)) / (2 * np.pi)
    # Measured: +0.33 %.  The 3-D clamp also holds the lateral (Poisson) contraction at the root, and shear deformation
    # (Timoshenko) lowers the frequency by O((h / L)^2); both are effects beam theory leaves out, and P2 with two layers
    # through the thickness adds well under 0.1 % here.  1 % bounds them with room; a wrong clamp (free-free 4.730^2 or a
    # hinged 1.875 -> pi / 2 root) would be off by far more.
    assert abs(f / f_eb - 1) < 1e-2, (f, f_eb)
    # the first mode bends in z: the displacement of the tip is along z
    tip = np.flatnonzero(pv[:, 0] >= L - 1e-6)
    uz, uy = np.abs(U[3 * tip + 2, 0]).max(), np.abs(U[3 * tip + 1, 0]).max()
    assert uz > 100 * uy


def test_interlacing_with_the_free_spectrum():
    v, t = mo.kuhn_cube(3)
    K, M = mo.assemble(v, t, 1, E, NU, RHO)
    fixed = np.flatnonzero(v[:, 0].numpy() == 0.0)
    n, nc = K.shape[0], fixed.size
    lam_free = scipy.linalg.eigh(K.toarray(), M.toarray(), eigvals_only=True)        # rigid six included
    free = fo.free_dofs(fixed, n // 3)
    lam_fix = scipy.linalg.eigh(K.toarray()[np.ix_(free, free)], M.toarray()[np.ix_(free, free)], eigvals_only=True)
    lam_arp, _ = fo.eig_fixed(K, M, fixed, 12)
    np.testing.assert_allclose(lam_arp, lam_fix[:12], rtol=1e-9)
    # Cauchy interlacing of a pencil restricted to a subspace of codimension 3 n_c; the slack is fp64 rounding of the
    # dense solver (the rigid eigenvalues of the free pencil are 0 to ~1e-9 of the largest)
    eps = 1e-9 * lam_free[-1]
    i = np.arange(lam_fix.size)
    assert np.all(lam_free[i] <= lam_fix + eps)
    j = i + 3 * nc < n
    assert np.all(lam_fix[j] <= lam_free[i[j] + 3 * nc] + eps)
    assert lam_fix[0] > 1e-3 * lam_free[6]           # no rigid motion left


def test_constrain_keeps_diagonal_blocks_and_pattern():
    v, t = mo.kuhn_cube(2)
    K, _ = mo.assemble(v, t, 1, E, NU, RHO)
    fixed = np.array([0, 1, 3])
    Kc = fo.constrain(K, fixed)
    assert np.array_equal(Kc.indptr, K.indptr) and np.array_equal(Kc.indices, K.indices)
    D, Dc = K.toarray(), Kc.toarray()
    nodes = np.arange(K.shape[0]) // 3
    touch = (nodes[:, None] != nodes[None, :]) & (np.isin(nodes, fixed)[:, None] | np.isin(nodes, fixed)[None, :])
    assert np.all(Dc[touch] == 0.0) and np.array_equal(Dc[~touch], D[~touch])


def test_mask_validation():
    from diffsound_b200.diffelastic.diff_model import check_fixed_mask
    v, _ = mo.kuhn_cube(3)
    face = v[:, 0] == 0.0
    check_fixed_mask(v, face)                        # a face: fine
    line = face & (v[:, 1] == 0.0)                   # the 4 nodes of one edge are collinear
    tri = line.clone()
    tri[int(torch.nonzero(face & (v[:, 1] == 1.0))[0])] = True
    check_fixed_mask(v, tri)
    with pytest.raises(ValueError, match="non-collinear"):
        check_fixed_mask(v, line)
    with pytest.raises(ValueError, match="non-collinear"):
        check_fixed_mask(v, torch.zeros(v.shape[0], dtype=torch.bool))
    with pytest.raises(ValueError, match="non-collinear"):
        check_fixed_mask(v, torch.arange(v.shape[0]) < 2)
    with pytest.raises(ValueError, match="shape"):
        check_fixed_mask(v, face[:-1])
    with pytest.raises(ValueError, match="shape"):
        check_fixed_mask(v, face[None, :])
    with pytest.raises(ValueError, match="boolean"):
        check_fixed_mask(v, face.to(torch.uint8))
