"""Reference for clamped objects (DiffSoundObj.fix_nodes): the eigenpairs of the pencil reduced to the free dofs.

The fixed dofs are deleted from the scipy matrices of `oracle.modal_oracle.assemble`; the reduced pencil is SPD, so
shift-invert ARPACK at sigma = 0 returns its lowest pairs.  The eigenvectors are scattered back with zeros on the fixed
rows, so `modal_oracle.eigval_grad_shape` / `material_quadforms` give the reference gradients of the clamped problem
(d lambda = u^T (dK - lambda dM) u with u zero on the fixed rows)."""
import numpy as np
import scipy.sparse.linalg as spla


def free_dofs(fixed_nodes, n_nodes):
    """Indices of the dofs of the nodes that are not fixed (fixed_nodes: bool (n_nodes,) or node ids)."""
    fixed = np.zeros(n_nodes, dtype=bool)
    fixed[np.asarray(fixed_nodes)] = True
    return np.flatnonzero(np.repeat(~fixed, 3))


def constrain(K, fixed_nodes):
    """K with every entry that couples a fixed node to another node set to an explicit zero (the pattern is kept): what
    ds_fix_nodes_km makes of the assembled matrix."""
    K = K.tocsr(copy=True)
    n_nodes = K.shape[0] // 3
    fixed = np.zeros(n_nodes, dtype=bool)
    fixed[np.asarray(fixed_nodes)] = True
    rows = np.repeat(np.arange(K.shape[0]), np.diff(K.indptr))
    ni, nj = rows // 3, K.indices // 3
    K.data[(ni != nj) & (fixed[ni] | fixed[nj])] = 0.0
    return K


def eig_fixed(K, M, fixed_nodes, k):
    """Lowest k pairs of the clamped pencil: (lam (k,), U (n, k) M-orthonormal with zero fixed rows)."""
    n = K.shape[0]
    free = free_dofs(fixed_nodes, n // 3)
    Kr = K.tocsr()[free][:, free]
    Mr = M.tocsr()[free][:, free]
    Kr.eliminate_zeros()
    Mr.eliminate_zeros()
    lam, Ur = spla.eigsh(Kr, M=Mr, k=k, sigma=0.0)
    order = np.argsort(lam)
    U = np.zeros((n, k))
    U[free] = Ur[:, order]
    return lam[order], U
