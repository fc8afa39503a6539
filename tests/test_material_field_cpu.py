"""Material fields on the host: the reference (tests/material_field_oracle.py) against the homogeneous oracle and against
finite differences of ARPACK eigenvalues, the rounding rules a constant field relies on, and the validation and region
helpers of DiffSoundObj.set_material_field."""
import numpy as np
import pytest
import scipy.sparse.linalg as spla
import torch

import material_field_oracle as mf
from oracle import modal_oracle as mo

RHO, E, NU = 7850.0, 2.0e11, 0.29


def _mesh(order, N=2):
    v, t = mo.kuhn_cube(N)
    return mo.promote(v, t, order)


@pytest.mark.parametrize("order", [1, 2])
def test_constant_field_equals_homogeneous_oracle(order):
    pv, pt = _mesh(order)
    T = pt.shape[0]
    K, M = mo.assemble(pv, pt, order, E, NU, RHO)
    Kf, Mf = mf.assemble_field(pv, pt, order, torch.full((T,), E, dtype=torch.float64),
                               torch.full((T,), NU, dtype=torch.float64), torch.full((T,), RHO))
    assert np.array_equal(K.data, Kf.data) and np.array_equal(M.data, Mf.data)


def test_rounding_rules_of_a_constant_field():
    from diffsound_b200.diffelastic import diff_model as dm
    from diffsound_b200.diffelastic import mass_matrix as mmx
    for order in (1, 2):
        for rho in (7850.0, 750.0, 2700.0, 1190.0, 8000.0):
            ref = mmx.mass_density_table(order, rho)
            field = (mmx.unit_mass_table32(order) * torch.tensor(rho, dtype=torch.float32)).double()
            assert torch.equal(ref, field)
    for mat in ((E, NU), (1.1e10, 0.25), (1.4e9, 0.35), (7.2e10, 0.19)):
        mu, lam = dm._lame(*mat)
        mu_t, lam_t = dm._lame(torch.tensor([mat[0]], dtype=torch.float64), torch.tensor([mat[1]], dtype=torch.float64))
        assert float(mu_t) == mu and float(lam_t) == lam


def _eigs(K, M, k):
    Kz, Mz = K.copy(), M.copy()
    Kz.eliminate_zeros()
    Mz.eliminate_zeros()
    lam, U = spla.eigsh(Kz, M=Mz, k=k + 6, sigma=-1e3, tol=1e-14)     # K + 1e3 M: SPD with the rigid modes
    o = np.argsort(lam)
    return lam[o][6:], U[:, o][:, 6:]


@pytest.mark.parametrize("order", [1, 2])
def test_field_gradients_against_finite_differences(order):
    pv, pt = _mesh(order)
    T = pt.shape[0]
    rng = np.random.default_rng(3)
    youngs = torch.from_numpy(E * np.exp(rng.uniform(np.log(0.3), np.log(3), T)))
    poisson = torch.from_numpy(rng.uniform(0.2, 0.4, T))
    density = torch.from_numpy(RHO * np.exp(rng.uniform(np.log(0.5), np.log(2), T))).float()
    k = 4
    K, M = mf.assemble_field(pv, pt, order, youngs, poisson, density)
    lam, U = _eigs(K, M, k)
    g = 1.0 / lam
    gE, gnu, grho = mf.field_grads(pv, pt, order, youngs, poisson, U, lam, g)

    def loss(E_, nu_, rho_):
        return float(g @ _eigs(*mf.assemble_field(pv, pt, order, E_, nu_, rho_), k)[0])

    for t in (0, T // 3, T - 1):
        h = 1e-3
        Ep, Em = youngs.clone(), youngs.clone()
        Ep[t] *= 1 + h
        Em[t] *= 1 - h
        fd = (loss(Ep, poisson, density) - loss(Em, poisson, density)) / float(Ep[t] - Em[t])
        assert abs(fd - gE[t]) <= 1e-4 * abs(gE[t]), ("E", t, fd, gE[t])
        Np, Nm = poisson.clone(), poisson.clone()
        Np[t] += 1e-4
        Nm[t] -= 1e-4
        fd = (loss(youngs, Np, density) - loss(youngs, Nm, density)) / float(Np[t] - Nm[t])
        assert abs(fd - gnu[t]) <= 1e-4 * abs(gnu[t]), ("nu", t, fd, gnu[t])
        Rp, Rm = density.clone(), density.clone()
        Rp[t] *= 1 + h
        Rm[t] *= 1 - h
        fd = (loss(youngs, poisson, Rp) - loss(youngs, poisson, Rm)) / float(Rp[t].double() - Rm[t].double())
        assert abs(fd - grho[t]) <= 1e-4 * abs(grho[t]), ("rho", t, fd, grho[t])


def test_euler_identities_of_the_oracle():
    """lambda is homogeneous of degree 1 in E and of degree -1 in rho: sum_t E_t dlam/dE_t = lam, sum_t rho_t dlam/drho_t
    = -lam (the second up to the fp32 rounding of the mass table products)."""
    pv, pt = _mesh(2)
    T = pt.shape[0]
    rng = np.random.default_rng(4)
    youngs = torch.from_numpy(E * np.exp(rng.uniform(np.log(0.3), np.log(3), T)))
    poisson = torch.from_numpy(rng.uniform(0.2, 0.4, T))
    density = torch.from_numpy(RHO * np.exp(rng.uniform(np.log(0.5), np.log(2), T))).float()
    K, M = mf.assemble_field(pv, pt, 2, youngs, poisson, density)
    lam, U = _eigs(K, M, 3)
    for i in range(3):
        g = np.zeros(3)
        g[i] = 1.0
        gE, _, grho = mf.field_grads(pv, pt, 2, youngs, poisson, U, lam, g)
        assert abs(gE @ youngs.numpy() / lam[i] - 1) < 1e-6     # exact vs fp32-Gauss quadrature of K: ~1e-7
        assert abs(grho @ density.double().numpy() / lam[i] + 1) < 1e-6


def test_check_material_field_errors():
    from diffsound_b200.diffelastic.diff_model import check_material_field
    T = 5
    ok = torch.full((T,), 1.0, dtype=torch.float64)
    check_material_field(T, "cpu", ok, torch.full((T,), 0.3), ok.float())
    check_material_field(T, "cpu", None, None, None)
    bad = [
        dict(youngs=torch.ones(T + 1, dtype=torch.float64)),                       # shape
        dict(youngs=torch.ones(T, 1, dtype=torch.float64)),
        dict(youngs=torch.ones(T, dtype=torch.int64)),                             # dtype
        dict(youngs=np.ones(T)),                                                   # not a tensor
        dict(youngs=torch.tensor([1.0, 1.0, float("nan"), 1.0, 1.0])),             # NaN
        dict(density=torch.tensor([1.0, 1.0, float("inf"), 1.0, 1.0])),
        dict(youngs=torch.tensor([1.0, 1.0, 0.0, 1.0, 1.0])),                      # sign
        dict(density=torch.tensor([1.0, -1.0, 1.0, 1.0, 1.0])),
        dict(poisson=torch.tensor([0.3, 0.5, 0.3, 0.3, 0.3])),                     # range
        dict(poisson=torch.tensor([0.3, -1.0, 0.3, 0.3, 0.3])),
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            check_material_field(T, "cpu", **kw)
    with pytest.raises(ValueError):                                                # device
        check_material_field(T, "cuda:0", youngs=ok)


def test_material_field_from_regions():
    from diffsound_b200.diffelastic.diff_model import material_field_from_regions
    from diffsound_b200.diffelastic.material_model import MatSet
    labels = torch.tensor([0, 1, 1, 0, 2])
    youngs, poisson, density = material_field_from_regions(labels, [MatSet.Steel, MatSet.Wood, MatSet.Glass])
    assert youngs.dtype == poisson.dtype == density.dtype == torch.float64
    assert youngs.tolist() == [2.0e11, 1.1e10, 1.1e10, 2.0e11, 6.2e10]
    assert poisson.tolist() == [0.29, 0.25, 0.25, 0.29, 0.20]
    assert density.tolist() == [7850.0, 750.0, 750.0, 7850.0, 2600.0]
    for bad in (torch.tensor([0, 3]), torch.tensor([-1]), torch.tensor([0.0, 1.0]), torch.zeros(2, 2, dtype=torch.int64)):
        with pytest.raises(ValueError):
            material_field_from_regions(bad, [MatSet.Steel, MatSet.Wood, MatSet.Glass])
