"""The elastic-support reference (tests/support_oracle.py) against closed forms, central differences and the Winkler beam,
plus the host-side validation and helpers of DiffSoundObj.set_supports.  No GPU needed."""
import numpy as np
import pytest
import torch

import support_oracle as so
from oracle import modal_oracle as mo
from test_modal_gains_cpu import kuhn_box

RHO, E, NU = 7800.0, 2.0e11, 0.3


def boundary(tets, order):
    """(owner, local) of the faces that belong to one tet, in ascending sorted-corner-triple order."""
    c = np.asarray(tets)[:, list(so._CORNER[order])]
    seen = {}
    for t in range(c.shape[0]):
        for f in range(4):
            key = tuple(sorted(c[t, j] for j in range(4) if j != f))
            seen.setdefault(key, []).append((t, f))
    keys = sorted(k for k, v in seen.items() if len(v) == 1)
    return np.array([seen[k][0][0] for k in keys]), np.array([seen[k][0][1] for k in keys])


def faces_where(verts, tets, order, pred):
    owner, local = boundary(tets, order)
    nodes = so.face_nodes(tets, order, owner, local)
    keep = np.array([all(pred(verts[i]) for i in row[:3]) for row in nodes])
    return owner[keep], local[keep]


def test_face_mass_closed_forms():
    assert np.allclose(so.face_mass_ref(1) * 12, [[2, 1, 1], [1, 2, 1], [1, 1, 2]], atol=1e-13)
    m2 = so.face_mass_ref(2) * 180
    ref = np.array([[6, -1, -1, 0, -4, 0], [-1, 6, -1, 0, 0, -4], [-1, -1, 6, -4, 0, 0],
                    [0, 0, -4, 32, 16, 16], [-4, 0, 0, 16, 32, 16], [0, -4, 0, 16, 16, 32]], dtype=np.float64)
    assert np.abs(m2 - ref).max() <= 1e-12


@pytest.mark.parametrize("order", [1, 2])
def test_rigid_energies_of_a_flat_support(order):
    """Translations give k_n A and k_t A; rotations about in-plane axes give k_n times the second moments of area."""
    v, t = kuhn_box((3, 2, 2), (0.3, 0.2, 0.1))
    pv, pt = mo.promote(torch.from_numpy(v), torch.from_numpy(t), order)
    pv, pt = pv.double().numpy(), pt.numpy()
    owner, local = faces_where(pv, pt, order, lambda p: abs(p[2]) < 1e-9)
    kn, kt = 3.0e8, 1.0e8
    Ks = so.support_matrix(pv, pt, order, owner, local, kn, kt)
    R = so.rigid_fields(pv)
    G = R.T @ (Ks @ R)
    X, Y = pv[:, 0].max() - pv[:, 0].min(), pv[:, 1].max() - pv[:, 1].min()     # the fp32 box extents
    A = X * Y
    assert np.isclose(G[0, 0], kt * A, rtol=1e-12) and np.isclose(G[1, 1], kt * A, rtol=1e-12)
    assert np.isclose(G[2, 2], kn * A, rtol=1e-12)
    c = pv.mean(0)
    Ix = X * (Y ** 3 / 12 + Y * (Y / 2 - c[1]) ** 2)            # int (y - cy)^2 over the face [0, X] x [0, Y]
    Iy = Y * (X ** 3 / 12 + X * (X / 2 - c[0]) ** 2)
    # rotation about x: u = (0, -z', y'), z' = -c_z on the face; normal part k_n y'^2, tangential k_t z'^2.  The interior
    # grid lines sit at fp32 roundings of their ideal positions, which the closed form does not see: 1e-6
    assert np.isclose(G[3, 3], kn * Ix + kt * A * c[2] ** 2, rtol=1e-6)
    assert np.isclose(G[4, 4], kn * Iy + kt * A * c[2] ** 2, rtol=1e-6)


@pytest.mark.parametrize("order", [1, 2])
def test_oracle_gradients_central_differences(order):
    v, t = kuhn_box((4, 2, 2), (0.4, 0.1, 0.1))
    pv, pt = mo.promote(torch.from_numpy(v), torch.from_numpy(t), order)
    pvn, ptn = pv.double().numpy(), pt.numpy()
    owner, local = faces_where(pvn, ptn, order, lambda p: abs(p[2]) < 1e-9)
    S = owner.size
    rng = np.random.default_rng(0)
    kn = 1e9 * (1 + rng.random(S))
    kt = 3e8 * (1 + rng.random(S))
    K, M = mo.assemble(pv, pt, order, E, NU, RHO)
    k = 4

    def lam_of(kn_, kt_):
        return so.eig_supported(K, M, so.support_matrix(pvn, ptn, order, owner, local, kn_, kt_), k)[0]

    lam, U = so.eig_supported(K, M, so.support_matrix(pvn, ptn, order, owner, local, kn, kt), k)
    g = np.array([1.0, 0.5, -0.3, 0.2])
    gn, gt, gv = so.support_grads(pvn, ptn, order, owner, local, kn, kt, U, g)
    for s in (0, S // 2):
        for which, grad in ((0, gn), (1, gt)):
            h = 1e-4 * (kn[s] if which == 0 else kt[s])
            dp, dm = kn.copy(), kn.copy()
            ep, em = kt.copy(), kt.copy()
            if which == 0:
                dp[s] += h
                dm[s] -= h
            else:
                ep[s] += h
                em[s] -= h
            fd = (g @ lam_of(dp, ep) - g @ lam_of(dm, em)) / (2 * h)
            assert abs(fd - grad[s]) <= 1e-5 * np.abs(g * lam).sum() / kn[s] + 1e-6 * abs(grad[s]), (s, which, fd, grad[s])
    # vertex gradient: the energy of fixed modes under a moved corner node
    node = so.face_nodes(ptn, order, owner, local)[S // 2, 0]
    for c in range(3):
        h = 1e-6
        vp, vm = pvn.copy(), pvn.copy()
        vp[node, c] += h
        vm[node, c] -= h
        ep = so.face_energy(vp, so.face_nodes(ptn, order, owner, local), kn, kt, U, order).sum(0).numpy()
        em = so.face_energy(vm, so.face_nodes(ptn, order, owner, local), kn, kt, U, order).sum(0).numpy()
        fd = g @ (ep - em) / (2 * h)
        assert abs(fd - gv[node, c]) <= 1e-6 * np.abs(gv).max(), (c, fd, gv[node, c])


def _vertical_bending(U, pv, nmodes):
    """Indices of the modes whose displacement is mostly vertical and even across the bar's width (x-z bending)."""
    out = []
    ymid = 0.5 * (pv[:, 1].min() + pv[:, 1].max())
    lo, hi = pv[:, 1] < ymid - 1e-9, pv[:, 1] > ymid + 1e-9
    for i in range(nmodes):
        u = U[:, i].reshape(-1, 3)
        if (u[:, 2] ** 2).sum() < 0.8 * (u ** 2).sum():
            continue
        # even in y: the mirror image across the mid-plane carries the same vertical displacement
        if np.sign(u[lo, 2].sum()) == np.sign(u[hi, 2].sum()) and abs(u[lo, 2].sum()) > 0.5 * abs(u[hi, 2].sum()):
            out.append(i)
    return out


def test_winkler_bar_shift():
    """A P2 bar lying on its long bottom face (k_t = 0): its bending modes in the vertical plane shift by k_n / (rho h)
    (Euler-Bernoulli beam on a Winkler foundation; the 3-D bar differs by the beam model's error)."""
    L, b, h = 1.0, 0.04, 0.05
    v, t = kuhn_box((24, 2, 3), (L, b, h))
    pv, pt = mo.promote(torch.from_numpy(v), torch.from_numpy(t), 2)
    pvn, ptn = pv.double().numpy(), pt.numpy()
    owner, local = faces_where(pvn, ptn, 2, lambda p: abs(p[2]) < 1e-9)
    K, M = mo.assemble(pv, pt, 2, E, NU, RHO)
    shift = 1.0e6
    kn = shift * RHO * h
    lam_f, U_f = so.eig_supported(K, M, so.support_matrix(pvn, ptn, 2, owner, local, 0.0, 0.0), 20, sigma=-1.0)
    lam_s, U_s = so.eig_supported(K, M, so.support_matrix(pvn, ptn, 2, owner, local, kn, 0.0), 20, sigma=-1.0)
    bf = [i for i in _vertical_bending(U_f, pvn, 20) if lam_f[i] > 1.0]       # elastic modes of the free bar
    bs = _vertical_bending(U_s, pvn, 20)
    # heave and rock of the bar on its bed: k_n / (rho h) for a rigid bar; the elastic bar is 0.25 % softer in heave
    assert np.allclose(lam_s[bs[:2]], shift, rtol=5e-3), lam_s[bs[:2]]
    # first bending mode: the shift is 1.1 % short of k_n / (rho h) here (h / L = 0.05; the higher modes, shorter against
    # the height, move further from the beam model: 4.5 % and 8.5 %)
    free, supp = lam_f[bf[0]], lam_s[bs[2]]
    rel = abs((supp - free) - shift) / shift
    assert rel <= 1.5e-2, (free, supp, rel)


def test_pad_stiffness_gradcheck_and_values():
    from diffsound_b200.diffelastic.supports import pad_stiffness
    kn, kt = pad_stiffness(2.0e6, 0.3, 0.01)
    assert np.isclose(kn, 2.0e6 * 0.7 / (1.3 * 0.4 * 0.01)) and np.isclose(kt, 2.0e6 / (2.6 * 0.01))
    x = (torch.tensor([2.0e6, 5.0e6], dtype=torch.float64, requires_grad=True),
         torch.tensor([0.3, 0.45], dtype=torch.float64, requires_grad=True),
         torch.tensor([0.01, 0.02], dtype=torch.float64, requires_grad=True))
    assert torch.autograd.gradcheck(lambda E_, nu_, t_: pad_stiffness(E_, nu_, t_), x)


def test_stiffness_validation():
    from diffsound_b200.diffelastic.diff_model import check_support_stiffness
    kn, kt = check_support_stiffness(3, "cpu", 1.0, torch.tensor([1.0, 2.0, 3.0], dtype=torch.float32))
    assert kn.dtype == torch.float64 and torch.equal(kt, torch.tensor([1.0, 2.0, 3.0], dtype=torch.float64))
    for bad, msg in [((-1.0, 1.0), ">= 0"), ((float("nan"), 1.0), "non-finite"), ((torch.ones(2), 1.0), "shape"),
                     ((torch.ones(3, dtype=torch.int64), 1.0), "float"), (("x", 1.0), "float"),
                     ((1.0, torch.tensor([1.0, -1.0, 1.0])), ">= 0")]:
        with pytest.raises(ValueError, match=msg):
            check_support_stiffness(3, "cpu", *bad)


def test_rigid_check_matrix():
    """R^T K_s R of the host-side rigid-motion check: a flat face with k_t = 0 leaves three rigid motions free, one with
    k_t > 0 holds all six, and the matrix is the oracle's K_s over the same rigid fields."""
    from diffsound_b200.diffelastic.diff_model import support_rigid_matrix
    v, t = kuhn_box((3, 2, 2), (0.3, 0.2, 0.1))
    pv = v.astype(np.float64)
    owner, local = faces_where(pv, t, 1, lambda p: abs(p[2]) < 1e-9)
    nodes = so.face_nodes(t, 1, owner, local)
    p = torch.as_tensor(pv)[torch.as_tensor(nodes)]
    S = nodes.shape[0]
    for kt, free in ((0.0, 3), (1e8, 0)):
        G = support_rigid_matrix(p[:, 0], p[:, 1], p[:, 2], torch.full((S,), 3e8, dtype=torch.float64),
                                 torch.full((S,), kt, dtype=torch.float64))
        ev = torch.linalg.eigvalsh(G)
        assert int((ev <= 1e-10 * ev[-1]).sum()) == free
    # the same quadratic form as the oracle's K_s over rigid fields about the support centroid, rotations scaled by 1/L
    Ks = so.support_matrix(pv, t, 1, owner, local, 3e8, 1e8)
    corners = p.reshape(-1, 3).numpy()                   # every face's three corners, as the check weights them
    c = corners.mean(0)
    L = float(np.linalg.norm(corners - c, axis=1).max())
    R = so.rigid_fields(pv)
    q = pv - c
    R[1::3, 3], R[2::3, 3] = -q[:, 2], q[:, 1]
    R[0::3, 4], R[2::3, 4] = q[:, 2], -q[:, 0]
    R[0::3, 5], R[1::3, 5] = -q[:, 1], q[:, 0]
    R[:, 3:] /= L
    G = support_rigid_matrix(p[:, 0], p[:, 1], p[:, 2], torch.full((S,), 3e8, dtype=torch.float64),
                             torch.full((S,), 1e8, dtype=torch.float64)).numpy()
    Gref = R.T @ (Ks @ R)
    # the check's rotation columns are (-y, x, 0), (0, -z, y), (z, 0, -x): about z, x, y
    perm = [0, 1, 2, 5, 3, 4]
    Gp = Gref[np.ix_(perm, perm)]
    assert np.allclose(G, Gp, rtol=1e-10, atol=1e-12 * np.abs(Gp).max())
