"""Per-mesh FEM bookkeeping used by `DiffSoundObj`.

API mirror of src/diffelastic/deform.py:8-180 (`Deform`).  The reference
precomputes, per (tet, Gauss point), the shape-function gradients (T*G, N, 3)
fp32 = 1.5 GB and a dof index (T*G*N*3) int64 = 3 GB at 200k quadratic tets
(SURVEY.md section 8a rows a5-a7) and drives everything through them.  The
CUDA path needs none of that: geometry is affine per tet, so the kernels work
from the 4x3 matrix dL/dxi A^-1 recomputed on the fly and constant per-order
tables.  `Deform` here owns the device-side topology the kernels share:

  * int32 connectivity and the block-CSR sparsity pattern with per-slot
    contributor lists (`native.Pattern`, csrc/pattern.cu),
  * the corner incidence lists of the gradient gather (csrc/grad.cu),
  * the per-order constant tables.

The reference's heavy attributes (`shape_func_deriv`, `integration_weights`,
`stress_index`) remain available as lazily built torch tensors for API parity;
nothing in this package reads them.
"""
import torch

from .. import native
from . import mass_matrix as _mm
from .gauss import generate_gauss_points_weights
from .mesh import TetMesh
from .shape_func import get_shape_function_grad


class Deform:
    def __init__(self, tetmesh: TetMesh):
        self.tetmesh = tetmesh
        self.device = tetmesh.device
        if self.device.type != "cuda":
            raise RuntimeError("diffsound_b200: mesh tensors must live on a CUDA device (there is no CPU path)")
        pts, wts = generate_gauss_points_weights(tetmesh.order + 2)
        self.gauss_points = torch.tensor(pts, dtype=torch.float32, device=self.device)
        self.gauss_weights = torch.tensor(wts, dtype=torch.float32, device=self.device)
        self.num_guass_points = self.gauss_points.shape[0]
        self.num_nodes_per_tet = tetmesh.tets.shape[1]
        self.num_tets = tetmesh.tets.shape[0]
        self.num_nodes = tetmesh.vertices.shape[0]

    # ---- device-side topology shared by the kernels (built once per mesh) ----
    @property
    def tets_i32(self):
        if not hasattr(self, "_tets_i32"):
            self._tets_i32 = self.tetmesh.tets.to(torch.int32).contiguous()
        return self._tets_i32

    @property
    def pattern(self):
        if not hasattr(self, "_pattern"):
            self._pattern = native.Pattern(self.tets_i32, self.num_nodes)
        return self._pattern

    @property
    def incidence(self):
        if not hasattr(self, "_incidence"):
            self._incidence = native.corner_incidence(self.tets_i32, self.tetmesh.order, self.num_nodes)
        return self._incidence

    @property
    def coarse(self):
        """P1 level of a quadratic mesh (two-level eigensolver preconditioner); None for linear tets."""
        if self.tetmesh.order != 2:
            return None
        if not hasattr(self, "_coarse"):
            self._coarse = native.CoarseLevel(self.verts_f32(), self.tets_i32)
            self._coarse.ctab = _mm.stiffness_contraction_table(1).to(self.device)
            self._coarse.mtabs = {}
        return self._coarse

    def coarse_mtab(self, density):
        key = float(density)
        cache = self.coarse.mtabs
        if key not in cache:
            cache[key] = _mm.mass_density_table(1, key).to(self.device)
        return cache[key]

    @property
    def ctab(self):
        if not hasattr(self, "_ctab"):
            self._ctab = _mm.stiffness_contraction_table(self.tetmesh.order).to(self.device)
        return self._ctab

    @property
    def wsum(self):
        return float(_mm.stiffness_contraction_table(1)[0, 0, 0, 0]) if self.tetmesh.order == 1 else 1.0 / 6.0

    def mtab(self, density):
        key = float(density)
        cache = self.__dict__.setdefault("_mtab", {})
        if key not in cache:
            cache[key] = _mm.mass_density_table(self.tetmesh.order, key).to(self.device)
        return cache[key]

    def m32(self, order=None):
        """fp32 unit-density mass table of this mesh's order (or of `order`) on the device, for the material-field kernels."""
        order = self.tetmesh.order if order is None else order
        cache = self.__dict__.setdefault("_m32", {})
        if order not in cache:
            cache[order] = _mm.unit_mass_table32(order).to(self.device)
        return cache[order]

    def verts_f32(self):
        return self.tetmesh.vertices.detach().to(torch.float32).contiguous()

    # ---- reference attributes, kept for API parity (lazy; unused by this package) ----
    @property
    def B_matrix(self):
        return self.shape_func_deriv

    @property
    def shape_func_deriv(self):
        """(T*G, N, 3) fp32 = (dN/dL . dL/dxi) . A^-1 (deform.py:35-68)."""
        if not hasattr(self, "_shape_func_deriv"):
            A_inv = torch.inverse(self.tetmesh.transform_matrix)
            dL = torch.tensor([[1, 0, 0], [0, 1, 0], [0, 0, 1], [-1, -1, -1]], dtype=torch.float32, device=self.device)
            dN = get_shape_function_grad(self.gauss_points, self.tetmesh.order) @ dL       # (G, N, 3)
            B = dN.unsqueeze(0) @ A_inv.unsqueeze(1)                                        # (T, G, N, 3)
            self._shape_func_deriv = B.reshape(self.num_tets * self.num_guass_points, self.num_nodes_per_tet, 3)
        return self._shape_func_deriv

    @property
    def integration_weights(self):
        """(T*G, 1, 1) fp32 = w_g |det A| (deform.py:136-147)."""
        if not hasattr(self, "_integration_weights"):
            vol = torch.abs(torch.det(self.tetmesh.transform_matrix)).unsqueeze(1)
            self._integration_weights = (self.gauss_weights.unsqueeze(0) * vol).reshape(-1, 1, 1)
        return self._integration_weights

    @property
    def stress_index(self):
        """(T*G*N*3,) int64 dof ids 3*node + c (deform.py:113-125)."""
        if not hasattr(self, "_stress_index"):
            base = self.tetmesh.tets.unsqueeze(1).expand(-1, self.num_guass_points, -1)
            idx = base.unsqueeze(-1) * 3 + torch.arange(3, device=self.device)
            self._stress_index = idx.reshape(-1)
        return self._stress_index
