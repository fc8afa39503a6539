"""CPU tests of the host-side logic: the C-ABI library loads and exports every declared symbol, the
constant tables, mesh promotion and I/O, and the product package never touches the oracle."""
import ctypes
import hashlib
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, golden


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "diffsound_sm100.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ds_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from diffsound_b200 import _lib
    syms = _header_symbols()
    assert len(syms) >= 25
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/diffsound_sm100.h but not exported"
    assert sorted(_lib.SIGNATURES) == syms, "ctypes table and header disagree"
    loaded = _lib.load()
    assert loaded.ds_version() >= 100
    assert isinstance(_lib.last_error(), str)


def test_cabi_rejects_bad_arguments_with_a_message():
    """Argument validation happens before any device work: null pointers, empty meshes and unsupported shapes
    come back as DS_ERR_ARG (-2) with a message in ds_last_error(), never as a crash (reference debug build:
    std::runtime_error -> RuntimeError, include/macro.h:109-124)."""
    from diffsound_b200 import _lib
    lib = _lib.load()
    N = None
    cases = [
        lambda: lib.ds_assemble_km(N, N, 0, 2, 0, 1.0, 1.0, N, N, N, N, N, N, 0, N, N, N, N),
        lambda: lib.ds_assemble_mass_coo(N, N, 4, 7, N, 1.0, N, N, N, N),                  # order 7
        lambda: lib.ds_spmm32(0, N, N, 10, 48, N, N, N, N, N, 0.0, 0.0, N, N),
        lambda: lib.ds_spmm32(5, N, N, 10, 48, N, N, N, N, N, 0.0, 0.0, N, N),             # unknown mode
        lambda: lib.ds_lobpcg(N, N, N, 10, N, N, N, N, 48, N, N, N, N, N),
        lambda: lib.ds_modal_synth_fwd(N, N, N, 0, 0, 0, 44100.0, N, N, N),
        lambda: lib.ds_unique_rows3_count(N, N, 0, N, N),
        lambda: lib.ds_rr_update_f64(N, N, N, 144, 144, 40, N, N, 48, 144, 10, N, N, N, 144, N),   # m = 40
        lambda: lib.ds_cheb32_solve(N, N, N, 10, 10, N, 48, 0, 1.0, 2.0, 1, N, N, N, N),
        lambda: lib.ds_gram_f64(N, 8, 12, N, 8, 8, 10, N, 8, N, N),                        # p not a multiple of 8
    ]
    for i, call in enumerate(cases):
        rc = call()
        assert rc == -2, (i, rc)
        msg = _lib.last_error()
        assert isinstance(msg, str) and len(msg) > 8, (i, msg)


def test_no_compute_without_gpu_and_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from diffsound_b200 import native
    with pytest.raises(RuntimeError):
        native._p(torch.zeros(3))
    from diffsound_b200.diffelastic.diff_model import DiffSoundObj
    with pytest.raises(RuntimeError):
        DiffSoundObj(torch.zeros(4, 3), torch.zeros(1, 4, dtype=torch.long))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "diffsound_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert "/root/reference" not in txt.replace("/root/reference/src", "REFDOC") or f.endswith((".cu", ".cuh")), f


def test_tables():
    from diffsound_b200.diffelastic import gauss, mass_matrix as mmx, shape_func as sf
    from oracle import modal_oracle as mo
    for order in (1, 2):
        pts, w = gauss.generate_gauss_points_weights(order + 2)
        opts, ow = mo.gauss_rule(order + 2)
        assert pts.dtype == np.float32 and np.array_equal(pts, opts) and np.array_equal(w, ow)
        L = torch.from_numpy(pts)
        assert torch.equal(sf.get_shape_function(L, order), mo.shape_fn(L, order))
        assert torch.equal(sf.get_shape_function_grad(L, order), mo.shape_fn_grad(L, order))
        assert torch.equal(mmx.calculate_element_mass_matrix(order, order + 2), mo.element_mass_table(order))
        npe = sf.NODES_PER_TET[order]
        full = mmx.get_elememt_mass_matrix(order)
        assert full.shape == (9 * npe * npe,) and full.dtype == torch.float32
        ct = mmx.stiffness_contraction_table(order)
        assert ct.shape == (npe, npe, 4, 4) and ct.dtype == torch.float64
        # sum over nodes of dN_a/dL_l is the derivative of the partition of unity: sum_a N_a = 1
        # (exactly 1 for order 1; for order 2 it is 4 sum(L) - 1 + ... = constant) -> rows sum consistently
        assert torch.allclose(ct, ct.permute(1, 0, 3, 2))
    assert abs(float(mmx.stiffness_contraction_table(1)[0, 0, 0, 0]) - 1 / 6) <= 1e-7


def test_tetmesh_promotion_needs_cuda(meshes):
    """The node numbering runs in csrc/mesh.cu: host tensors are refused, never renumbered on the CPU."""
    from diffsound_b200.diffelastic.mesh import TetMesh
    v, t = meshes["cube2"]
    m1 = TetMesh(torch.tensor(v), torch.tensor(t)).to_high_order(1)
    assert m1.order == 1
    with pytest.raises(RuntimeError, match="no CPU path"):
        TetMesh(torch.tensor(v), torch.tensor(t)).to_high_order(2)
    with pytest.raises(NotImplementedError):
        TetMesh(torch.tensor(v), torch.tensor(t)).to_high_order(3)


def test_msh_roundtrip(tmp_path, meshes):
    from diffsound_b200.diffelastic import mesh as M
    v, t = meshes["cube2"]
    p = str(tmp_path / "c.msh")
    M.write_msh(p, v, t, "tetra")
    pts, cells = M.read_msh(p)
    assert np.array_equal(pts.astype(np.float32), v) and np.array_equal(cells["tetra"], t)
    with pytest.raises(FileNotFoundError):
        M.TetMesh.from_triangle_mesh(str(tmp_path / "missing.obj"))


def test_bench_cube_matches_oracle_cube():
    import bench
    from oracle import modal_oracle as mo
    v, t = bench.kuhn_cube(3)
    ov, ot = mo.kuhn_cube(3)
    assert np.array_equal(v, ov.numpy()) and np.array_equal(t, ot.numpy())


def test_material_models_cpu_side():
    from diffsound_b200.diffelastic.diff_model import TrainableLinear, FixedLinear
    from diffsound_b200.diffelastic.material_model import Material, MatSet
    fl = FixedLinear(Material(MatSet.Steel))
    mu, lam = fl.lame()
    assert abs(mu - 2.0e11 / (2 * 1.29)) < 1 and abs(lam - 2.0e11 * 0.29 / (1.29 * 0.42)) < 1
    torch.manual_seed(0)
    tl = TrainableLinear(Material(MatSet.Ceramic))
    assert tl.youngs_list.shape == (16,) and tl.poisson_list.shape == (16,)
    assert float(tl.poisson_list[0]) == pytest.approx(0.01) and float(tl.poisson_list[-1]) == pytest.approx(0.499)
    assert len(list(tl.parameters())) == 2
    y = tl.youngs()
    assert y.dtype == torch.float32 and y.device.type == "cpu" and y.requires_grad
    bl = TrainableLinear(Material(MatSet.Ceramic), baseline=True)
    assert bl.poisson_list.shape == (1,) and float(bl.poisson()) == pytest.approx(0.19)
    F = torch.randn(5, 3, 3)
    P = fl.get_stress(F.double())
    ref = mu * (F.double() + F.double().transpose(1, 2)) + lam * torch.einsum("bii->b", F.double())[:, None, None] * torch.eye(3).double()
    assert torch.allclose(P, ref)


def test_bench_clock_sampler_summary():
    """bench.py's clocks field: median SM clock, maximum clock and the throttle reasons seen in any sample -- same record
    layout from the NVML path and from the nvidia-smi fallback (clocks.sm, clocks.max.sm, power, hw_slowdown,
    hw_thermal_slowdown, sw_thermal_slowdown, sw_power_cap)."""
    import bench
    s = bench.ClockSampler(0)          # no driver in the build container: falls back to the command-line path, no samples
    s.samples = [["1965", "1965", "0.0", "Not Active", "Not Active", "Not Active", "Not Active"],
                 ["1950", "1965", "0.0", "Not Active", "Not Active", "Not Active", "Active"],
                 ["1965", "1965", "0.0", "Not Active", "Not Active", "Not Active", "Not Active"]]
    out = s.summary()
    assert out["sm_mhz"] == 1965.0 and out["sm_max_mhz"] == 1965.0 and out["samples"] == 3
    assert out["reasons"] == ["sw_power_cap"]
    s.samples.append(["1200", "1965", "0.0", "Active", "Not Active", "Active", "Not Active"])
    assert s.summary()["reasons"] == ["hw_slowdown", "sw_thermal_slowdown"] + ["sw_power_cap"]
    s.samples = []
    assert s.summary()["sm_mhz"] is None and s.summary()["reasons"] == []


def test_bench_dump_outputs_bounded_and_seeded(tmp_path):
    """bench.py --dump-outputs: arrays are written whole while they fit; above the limit the large ones are cut to the same
    seeded row sample in every run, with the row ids beside them, and the files stay within the limit."""
    import bench
    rng = np.random.default_rng(1)
    arrays = {"eigenvalues": rng.standard_normal(32), "vertex_grad": rng.standard_normal((5000, 3)).astype(np.float32)}
    bench.dump_outputs(str(tmp_path / "whole"), arrays)
    assert sorted(os.listdir(tmp_path / "whole")) == ["eigenvalues.npy", "vertex_grad.npy"]
    for name, a in arrays.items():
        b = np.load(tmp_path / "whole" / (name + ".npy"))
        assert b.dtype == a.dtype and np.array_equal(a, b)
    limit = 40000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, limit=limit)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["eigenvalues.npy", "vertex_grad.npy", "vertex_grad_rows.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)
    rows = np.load(tmp_path / "a" / "vertex_grad_rows.npy").astype(np.int64)
    assert 1000 < rows.size < 5000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "vertex_grad.npy"), arrays["vertex_grad"][rows])
    assert np.array_equal(np.load(tmp_path / "a" / "eigenvalues.npy"), arrays["eigenvalues"])
    with pytest.raises(TypeError):
        bench.dump_outputs(str(tmp_path / "c"), {"tets": np.zeros((4, 4), dtype=np.int64)})
