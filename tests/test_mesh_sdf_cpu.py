"""CPU tests of the triangle-mesh SDF support: the OBJ reader, the fp64 oracle against closed forms, and the argument
checks of ds_mesh_sdf that come back before any device work."""
import ctypes

import numpy as np
import pytest

from conftest import golden
from oracle import mesh_sdf as ms


def _write(tmp_path, text):
    p = tmp_path / "m.obj"
    p.write_text(text)
    return str(p)


def test_read_obj_fans_polygons_and_resolves_index_forms(tmp_path):
    from diffsound_b200.diffelastic.mesh import read_obj
    path = _write(tmp_path, """# header comment
o thing
mtllib none.mtl
v 0 0 0
v 1 0 0
v 1 1 0
v 0 1 0   # trailing comment
vt 0 0
vn 0 0 1
usemtl x
s off
f 1 2 3 4
v 2 0 0
v 3 0 0
v 3 1 0
v 2 2 0
v 1.5 1 0
f -5/1 -4/1/1 -3//1 -2/1/1 -1
g part
f 1/1/1 3//1 4/1
l 1 2
""")
    v, f = read_obj(path)
    assert v.dtype == np.float32 and v.shape == (9, 3)
    assert f.dtype == np.int64
    assert np.array_equal(f, [[0, 1, 2], [0, 2, 3], [4, 5, 6], [4, 6, 7], [4, 7, 8], [0, 2, 3]])
    assert np.array_equal(v[8], np.float32([1.5, 1, 0]))


def test_read_obj_errors(tmp_path):
    from diffsound_b200.diffelastic.mesh import read_obj
    with pytest.raises(FileNotFoundError):
        read_obj(str(tmp_path / "missing.obj"))
    with pytest.raises(ValueError):
        read_obj(_write(tmp_path, "v 0 0 0\nv 1 0 0\nv 0 1 0\n"))
    with pytest.raises(ValueError):
        read_obj(_write(tmp_path, "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 4\n"))
    with pytest.raises(ValueError):
        read_obj(_write(tmp_path, "v 0 0 0\nv 1 0 0\nv 0 1 0\nf -4 2 3\n"))
    with pytest.raises(ValueError):
        read_obj(_write(tmp_path, "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 0 1 2\n"))


def test_oracle_distance_in_each_voronoi_region_of_a_triangle():
    tri = np.float32([[[0, 0, 0], [1, 0, 0], [0, 1, 0]]])
    cases = [
        ((0.2, 0.2, 0.5), 0.5),                      # face
        ((-1, -1, 0.5), 1.5),                        # vertex A
        ((2, -1, 0), 2 ** 0.5),                      # vertex B
        ((-0.5, 2, 1), 1.5),                         # vertex C
        ((0.5, -2, 1), 5 ** 0.5),                    # edge AB
        ((-3, 0.5, 0), 3.0),                         # edge CA
        ((1, 1, 0.5), 0.75 ** 0.5),                  # edge BC
    ]
    p = np.float32([c[0] for c in cases])
    d = np.sqrt(ms.point_triangle_d2(p, tri)[:, 0])
    assert np.allclose(d, [c[1] for c in cases], rtol=1e-15, atol=0)
    # degenerate faces are their edges: collinear, and two coincident corners
    deg = np.float32([[[0, 0, 0], [1, 0, 0], [2, 0, 0]], [[0, 0, 0], [0, 0, 0], [0, 0, 2]]])
    assert ms.degenerate(deg).all()
    q = np.float32([[3, 0, 0], [1, 1, 0], [0, 3, 1]])
    d = np.sqrt(ms.point_triangle_d2(q, deg))
    assert np.allclose(d[:, 0], [1.0, 1.0, 10 ** 0.5], rtol=1e-15)
    assert np.allclose(d[:, 1], [3.0, 2 ** 0.5, 3.0], rtol=1e-15)


def test_oracle_box_against_analytic_sdf_on_grid16():
    """Box with its face planes through grid vertices (multiples of 1.5 / 16): many queries lie exactly on the planes."""
    v = golden("meshes")["grid16_verts"] * np.float32(1.5)
    lo, hi = np.array([-0.375, -0.1875, -0.5625]), np.array([0.28125, 0.46875, 0.09375])
    bv, bf = ms.voxel_mesh(np.ones((1, 1, 1)), lo, hi - lo)
    assert bf.shape == (12, 3)
    on_plane = np.any(np.isin(v, np.concatenate([lo, hi]).astype(np.float32)), axis=1)
    assert on_plane.sum() > 100
    s, _ = ms.mesh_sdf(bv, bf, v)
    ref = ms.box_sdf(v, lo, hi)
    assert np.abs(s - ref).max() <= 1e-15
    nz = ref != 0
    assert np.array_equal(np.sign(s[nz]), np.sign(ref[nz]))


def test_mesh_sdf_argument_checks_before_device_work():
    """V == 0, F == 0, a null pointer and an unknown mode come back as DS_ERR_ARG with a message; P == 0 returns 0
    without touching the device (no pointer is dereferenced on these paths, so a dummy workspace is enough)."""
    from diffsound_b200 import _lib
    lib = _lib.load()
    buf = ctypes.create_string_buffer(64)
    d = ctypes.cast(buf, ctypes.c_void_p)
    N = None
    cases = [
        (lambda: lib.ds_mesh_sdf(d, d, 0, d, 1, d, 1, 0, d, N), "empty mesh"),
        (lambda: lib.ds_mesh_sdf(d, d, 3, d, 0, d, 1, 0, d, N), "empty mesh"),
        (lambda: lib.ds_mesh_sdf(d, N, 3, d, 1, d, 1, 0, d, N), "null"),
        (lambda: lib.ds_mesh_sdf(N, d, 3, d, 1, d, 1, 0, d, N), "null"),
        (lambda: lib.ds_mesh_sdf(d, d, 3, d, 1, N, 1, 0, d, N), "null"),
        (lambda: lib.ds_mesh_sdf(d, d, 3, d, 1, d, 1, 0, N, N), "null"),
        (lambda: lib.ds_mesh_sdf(d, d, 3, d, 1, d, 1, 2, d, N), "unknown mode"),
        (lambda: lib.ds_mesh_sdf(d, d, 3, d, 1, d, 1, -1, d, N), "unknown mode"),
    ]
    for call, msg in cases:
        assert call() == -2
        assert msg in _lib.last_error()
    assert lib.ds_mesh_sdf(d, d, 3, d, 1, N, 0, 0, N, N) == 0
