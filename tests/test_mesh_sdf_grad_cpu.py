"""The fp64 numpy reference for the gradient of the triangle-mesh signed distance (tests/mesh_sdf_grad_ref.py, built on the
distance and sign of oracle/mesh_sdf.py), which the tests of ds_mesh_sdf_backward compare against: against central
differences of its own fp64 distance at points with a unique closest point, and the exact identities per point
(translation, Euler homogeneity of degree 1, unit point gradient)."""
import numpy as np
import pytest

from oracle import mesh_sdf as ms
import mesh_sdf_grad_ref as gr


def _bumpy_ico(level=1, seed=0):
    v, f = ms.icosphere(level, 0.6)
    rng = np.random.default_rng(seed)
    return (v.astype(np.float64) * (1.0 + 0.1 * rng.standard_normal((len(v), 1)))), f


MESHES = {
    # every closest-point region of one face: points all around it
    "triangle": lambda: (np.array([[-0.3, -0.2, 0.05], [0.4, -0.1, 0.1], [0.0, 0.5, -0.05]]), np.int64([[0, 1, 2]])),
    # a degenerate face (collinear corners): the union of its edges
    "degenerate": lambda: (np.array([[-0.4, 0.0, 0.0], [0.1, 0.05, 0.02], [0.4, 0.1, 0.04]]), np.int64([[0, 1, 2]])),
    "bumpy_ico1": _bumpy_ico,
}


def _points(n=400, seed=1):
    return np.random.default_rng(seed).uniform(-0.8, 0.8, (n, 3))


def _unique_closest(v, f, p, margin):
    """points whose nearest face is ahead of every face with a different closest point by `margin` in distance."""
    tris = v[f]
    d = np.sqrt(ms.point_triangle_d2(p, tris))
    best = d.min(1)
    out = []
    for i in range(len(p)):
        near = np.nonzero(d[i] <= best[i] + margin)[0]
        c, _ = gr.closest_on_triangles(np.repeat(p[i:i + 1], len(near), 0), *(tris[near, k] for k in range(3)))
        out.append(np.abs(c - c[0]).max() == 0.0 or len(near) == 1)
    return np.array(out) & (best > margin)


@pytest.mark.parametrize("name", list(MESHES))
def test_oracle_gradient_matches_central_differences(name):
    v, f = MESHES[name]()
    p = _points()
    keep = _unique_closest(v, f, p, 1e-3)
    p = p[keep]
    assert len(p) >= 50
    g = np.random.default_rng(2).standard_normal(len(p))
    ref = gr.mesh_sdf_grad(v, f, p, g, dtype=np.float64)
    rng = np.random.default_rng(3)
    h = 1e-6
    for _ in range(3):
        dv, dp = rng.standard_normal(v.shape), rng.standard_normal(p.shape)
        lp = g @ gr.mesh_sdf(v + h * dv, f, p + h * dp, dtype=np.float64)
        lm = g @ gr.mesh_sdf(v - h * dv, f, p - h * dp, dtype=np.float64)
        fd = (lp - lm) / (2 * h)
        an = (ref["grad_verts"] * dv).sum() + (ref["grad_points"] * dp).sum()
        assert abs(fd - an) <= 1e-6 * max(1.0, abs(an)), (fd, an)


@pytest.mark.parametrize("name", list(MESHES))
def test_oracle_gradient_identities(name):
    v, f = MESHES[name]()
    p = _points(seed=4)
    r = gr.mesh_sdf_grad(v, f, p, dtype=np.float64)
    assert np.all(r["bary"] >= -1e-12) and np.allclose(r["bary"].sum(1), 1.0, rtol=0, atol=1e-12)
    # per point: the corner gradients of its face and the point gradient
    corners = v[f[r["face"]]]                                         # (P, 3, 3)
    gvk = -r["bary"][:, :, None] * r["grad_points"][:, None, :]       # (P, 3 corners, 3)
    assert np.abs(gvk.sum(1) + r["grad_points"]).max() <= 1e-12                                     # translation
    euler = np.einsum("pkd,pkd->p", corners, gvk) + np.einsum("pd,pd->p", p, r["grad_points"])
    assert np.abs(euler - r["sdf"]).max() <= 1e-12                                                 # homogeneity
    nz = r["sdf"] != 0
    assert np.abs(np.linalg.norm(r["grad_points"][nz], axis=1) - 1.0).max() <= 1e-12             # |d sdf / d p| = 1
    # the accumulated vertex gradient is the sum of the corner gradients
    gv = np.zeros_like(v)
    np.add.at(gv, f[r["face"]].reshape(-1), gvk.reshape(-1, 3))
    assert np.allclose(gv, r["grad_verts"], rtol=0, atol=1e-12)


def test_oracle_nearest_face_takes_the_lowest_index_on_ties():
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=np.float64)
    f = np.int64([[1, 2, 3], [0, 1, 2], [0, 1, 3]])          # faces 1 and 2 share the edge 0-1
    r = gr.mesh_sdf_grad(v, f, np.array([[0.5, -0.5, -0.5]]), dtype=np.float64)
    assert r["face"][0] == 1
    assert np.allclose(r["closest"][0], [0.5, 0, 0]) and np.allclose(r["bary"][0], [0.5, 0.5, 0.0])


def test_oracle_sdf_default_is_fp32_rounded():
    v, f = _bumpy_ico()
    p = _points(50)
    d32, _ = ms.mesh_sdf(v, f, p)
    d32b = gr.mesh_sdf(v.astype(np.float32), f, p.astype(np.float32), dtype=np.float64)
    assert np.array_equal(d32, d32b)
