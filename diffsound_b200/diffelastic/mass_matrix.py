"""Reference-element tables: consistent mass and the stiffness contraction table.

API mirror of src/diffelastic/mass_matrix.py:9-31
(`calculate_element_mass_matrix`, `get_elememt_mass_matrix` -- the misspelling
is the reference's public name).  `stiffness_contraction_table` is new: it is
the constant the fused assembly kernel needs (see csrc/assemble.cu).
All tables are computed on the CPU, once per (order), and cached.
"""
import functools

import torch

from .gauss import generate_gauss_points_weights
from .shape_func import get_shape_function, get_shape_function_grad, NODES_PER_TET


@functools.lru_cache(maxsize=None)
def _rule(gauss_order):
    p, w = generate_gauss_points_weights(gauss_order)
    return torch.from_numpy(p), torch.from_numpy(w)


@functools.lru_cache(maxsize=None)
def _mass_table_cpu(fem_order, gauss_order):
    pts, wts = _rule(gauss_order)
    N = get_shape_function(pts, fem_order)
    v = NODES_PER_TET[fem_order]
    M = torch.zeros(v, v, dtype=torch.float32)
    for a in range(v):
        for b in range(v):
            M[a, b] = torch.sum(N[:, a] * N[:, b] * wts)
    return M


def calculate_element_mass_matrix(fem_order, gauss_order):
    """(nodes, nodes) fp32 table of int N_a N_b over the unit tet."""
    return _mass_table_cpu(fem_order, gauss_order).clone()


def get_elememt_mass_matrix(fem_order, device=None):
    """Flat (3 nodes)^2 fp32 element mass matrix, (table (x) I3), like the reference."""
    M = calculate_element_mass_matrix(fem_order, fem_order + 2)
    v = M.shape[0]
    full = (M[:, None, :, None] * torch.eye(3)[None, :, None, :]).reshape(3 * v, 3 * v)
    full = full.reshape(-1)
    return full.to(device) if device is not None else full


@functools.lru_cache(maxsize=None)
def stiffness_contraction_table(fem_order):
    """ctab[a, b, l, m] = sum_g w_g dN_a/dL_l(g) dN_b/dL_m(g), fp64 (nodes, nodes, 4, 4).

    Built from the fp32 rule and fp32 dN/dL the reference feeds into
    (dN/dL . dL/dxi) . A^-1 (deform.py:52-67), promoted to fp64 before the sum.
    """
    pts, wts = _rule(fem_order + 2)
    D = get_shape_function_grad(pts, fem_order).double()        # (G, nodes, 4)
    return torch.einsum("g,gal,gbm->ablm", wts.double(), D, D).contiguous()


def mass_density_table(fem_order, density):
    """mtab[a, b] = double(float32(m_ab) * float32(density)), fp64 (nodes, nodes):
    the factor the reference multiplies |6V| with (diff_model.py:299-303)."""
    return (_mass_table_cpu(fem_order, fem_order + 2) * density).double().contiguous()


def unit_mass_table32(fem_order):
    """m_ab fp32 (nodes, nodes): the unit-density table that the material-field kernels round against float32(rho_t) per tet,
    exactly as mass_density_table rounds against one density."""
    return _mass_table_cpu(fem_order, fem_order + 2).clone()
