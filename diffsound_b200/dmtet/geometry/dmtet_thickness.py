"""Hollow-shell marching tetrahedra with a learnable thickness, as a TET mesh generator for the modal model.

API mirror of src/dmtet/geometry/dmtet_thickness.py:13-327 (`DMTet`, `DMTetGeometry`): same class / method / attribute
names (`marching_tets`, `thickness_coef`, `max_thickness`, `verts`, `indices`, `sdf`, `getMesh`,
`get_largest_connected_component`, `tick`, `get_eigenvalues`, `get_thickness`, `parameters`), same outputs in the same
order and numbering -- the tet order and vertex numbering this stage produces define the sparsity pattern of K and M.

What differs underneath: the integer work of the reference (`torch.unique` sorts of the edge list, boolean-mask
gathers through the 16-case tables, `torch.unique` of the flattened tets, and the GPU -> CPU round trip through
`scipy.sparse.csgraph.connected_components` with its Python loop over components) is three native calls
(`ds_mtet_*`, `ds_compact_ids_*`, `ds_tet_components_*`, csrc/mtet.cu).  The interpolation of the edge vertices stays
the reference's handful of element-wise fp32 torch operations (dmtet_thickness.py:133-148), in the same order, so the
positions are bit-identical and autograd reaches the thickness parameter.

`apply_sdf(path)` samples the signed distance of a triangle mesh (an OBJ file) at the grid vertices on the device
(`native.mesh_sdf`, csrc/sdf.cu: BVH nearest-triangle queries and ray-crossing parity) where the reference uses open3d's
`RaycastingScene` (dmtet_thickness.py:301-314; SURVEY.md section 8f-4); `apply_sdf` also takes the sampled values (a
tensor) or a callable evaluated at the grid vertices.  `apply_sdf((verts, faces))` takes the triangle mesh as tensors and
samples it through the differentiable `mesh_sdf` (mesh_sdf.py): with `verts.requires_grad` the mesh is sampled again on
every `getMesh()`, so the loss of a `tick()` reaches the triangle-mesh vertices.  `apply_sdf(..., sign="winding")` takes
the sign from the generalised winding number instead of the ray parity (open or self-intersecting meshes).  Not reproduced: the renderer's `mesh.Mesh` container
(return_triangle=True) is replaced by a plain namespace with `v_pos` / `t_pos_idx`.
"""
import os
import types

import numpy as np
import torch

from ... import native
from ...ddsp.oscillator import WeightedParam
from ...diffelastic.diff_model import DiffSoundObj
from ...diffelastic.material_model import MatSet
from ...diffelastic.mesh import read_obj
from .mesh_sdf import mesh_sdf


def _dev():
    if not torch.cuda.is_available():
        raise RuntimeError("diffsound_b200 needs a CUDA device (there is no CPU path)")
    return torch.device("cuda", torch.cuda.current_device())


class DMTet:
    def __init__(self):
        dev = _dev()
        # the reference's tables, kept as attributes (dmtet_thickness.py:15-76); the kernels hold their own copies
        self.triangle_table = torch.tensor(
            [[-1, -1, -1, -1, -1, -1], [1, 0, 2, -1, -1, -1], [4, 0, 3, -1, -1, -1], [1, 4, 2, 1, 3, 4], [3, 1, 5, -1, -1, -1],
             [2, 3, 0, 2, 5, 3], [1, 4, 0, 1, 5, 4], [4, 2, 5, -1, -1, -1], [4, 5, 2, -1, -1, -1], [4, 1, 0, 4, 5, 1],
             [3, 2, 0, 3, 5, 2], [1, 3, 5, -1, -1, -1], [4, 1, 2, 4, 3, 1], [3, 0, 4, -1, -1, -1], [2, 0, 1, -1, -1, -1],
             [-1, -1, -1, -1, -1, -1]], dtype=torch.long, device=dev)
        self.num_triangles_table = torch.tensor([0, 1, 1, 2, 1, 2, 2, 1, 1, 2, 2, 1, 2, 1, 1, 0], dtype=torch.long, device=dev)
        self.base_tet_edges = torch.tensor([0, 1, 0, 2, 0, 3, 1, 2, 1, 3, 2, 3], dtype=torch.long, device=dev)
        self.num_tets_table = torch.tensor([0, 1, 1, 3, 1, 3, 3, 3, 1, 3, 3, 3, 3, 3, 3, 1], dtype=torch.long, device=dev)
        self.tet_table = torch.tensor(
            [[-1] * 12, [0, 4, 5, 6] + [-1] * 8, [1, 4, 8, 7] + [-1] * 8, [7, 1, 8, 6, 5, 1, 7, 6, 5, 0, 1, 6],
             [2, 5, 7, 9] + [-1] * 8, [4, 0, 6, 7, 9, 0, 7, 6, 7, 0, 9, 2], [4, 1, 9, 8, 5, 1, 9, 4, 5, 1, 2, 9],
             [6, 0, 1, 2, 8, 6, 1, 2, 9, 6, 8, 2], [3, 6, 9, 8] + [-1] * 8, [5, 0, 4, 8, 5, 0, 8, 3, 5, 8, 9, 3],
             [1, 4, 7, 3, 4, 7, 6, 3, 9, 6, 7, 3], [0, 1, 5, 3, 5, 1, 9, 3, 5, 1, 7, 9], [5, 2, 3, 7, 3, 6, 5, 8, 3, 5, 7, 8],
             [0, 4, 7, 8, 0, 3, 8, 7, 0, 3, 7, 2], [4, 1, 2, 3, 4, 3, 2, 5, 4, 3, 5, 6], [0, 1, 2, 3] + [-1] * 8],
            dtype=torch.long, device=dev)
        # thickness coef in (0, 1) -> (0, max(self.sdf))
        self.thickness_list = torch.linspace(0, 1, steps=32)
        self.thickness_coef = WeightedParam(self.thickness_list)

    def sort_edges(self, edges_ex2):
        with torch.no_grad():
            order = (edges_ex2[:, 0] > edges_ex2[:, 1]).long().unsqueeze(dim=1)
            a = torch.gather(input=edges_ex2, index=order, dim=1)
            b = torch.gather(input=edges_ex2, index=1 - order, dim=1)
        return torch.stack([a, b], -1)

    def __call__(self, pos_nx3, sdf_n, tet_fx4, thickness_coef=None):
        if thickness_coef is None:
            thickness = self.thickness_coef() * self.max_thickness
        else:
            thickness = thickness_coef * self.max_thickness
        thickness = torch.as_tensor(thickness, dtype=torch.float32).to(pos_nx3.device)
        with torch.no_grad():
            sdf32 = sdf_n.detach().to(torch.float32).contiguous()
            # crossing edges (ascending unique (min, max) pairs), the tets of the shell over ids in [0, V + E), surface faces
            interp_v, all_tets, faces = native.marching_tets(sdf32, float(thickness), tet_fx4.to(torch.int64).contiguous())
        # ---- edge vertices: dmtet_thickness.py:133-148, operation for operation
        edges_to_interp = pos_nx3[interp_v.reshape(-1)].reshape(-1, 2, 3)
        edges_to_interp_sdf = sdf_n[interp_v.reshape(-1)].reshape(-1, 2, 1)
        both = (edges_to_interp_sdf[:, 0, 0] > 0) & (edges_to_interp_sdf[:, 1, 0] > 0)
        edges_to_interp_sdf = torch.where(both[:, None, None], edges_to_interp_sdf - thickness, edges_to_interp_sdf)
        edges_to_interp_sdf = torch.cat([edges_to_interp_sdf[:, :1], -edges_to_interp_sdf[:, 1:]], dim=1)
        denominator = edges_to_interp_sdf.sum(1, keepdim=True)
        edges_to_interp_sdf = torch.flip(edges_to_interp_sdf, [1]) / denominator
        verts = (edges_to_interp * edges_to_interp_sdf).sum(1)
        # ---- compaction of the used vertices (torch.unique(all_tets.reshape(-1), return_inverse=True), :195-199)
        all_verts = torch.cat([pos_nx3, verts], dim=0)
        with torch.no_grad():
            all_unique_tets, all_tets_tetmesh = native.compact_ids(all_tets, all_verts.shape[0])
        all_verts_tetmesh = all_verts[all_unique_tets]
        return verts, faces, all_verts_tetmesh, all_tets_tetmesh


class DMTetGeometry(torch.nn.Module):
    def __init__(self, grid_res, scale, FLAGS, grid=None):
        """grid (optional, not in the reference's signature): (vertices, indices) arrays of the background tet grid; default:
        data/tets/{grid_res}_tets.npz relative to the working directory, like the reference (dmtet_thickness.py:215)."""
        super().__init__()
        self.scale = scale
        self.FLAGS = FLAGS
        self.grid_res = grid_res
        self.marching_tets = DMTet()
        self.writer = None
        if not hasattr(FLAGS, "without_tensorboard"):
            try:
                from torch.utils.tensorboard import SummaryWriter
                self.writer = SummaryWriter(FLAGS.out_dir + "/tensorboard")
            except Exception:           # tensorboard is optional in this image
                self.writer = None
        if grid is None:
            tets = np.load("data/tets/{}_tets.npz".format(self.grid_res))
            grid = (tets["vertices"], tets["indices"])
        dev = _dev()
        self.base_verts = torch.tensor(np.asarray(grid[0]), dtype=torch.float32, device=dev)
        self.verts = self.base_verts * self.scale
        self.indices = torch.tensor(np.asarray(grid[1]), dtype=torch.long, device=dev)
        self.generate_edges()
        self.sdf = torch.zeros_like(self.verts[:, 0])
        self._sdf_mesh = None       # (verts, faces, sign) of apply_sdf((verts, faces), sign) when verts requires grad

    def generate_edges(self):
        """`all_edges` (unique sorted vertex pairs of the background grid, dmtet_thickness.py:225-230) is only read by the
        regularisers of the image experiments; it is built on first access."""
        self._all_edges = None

    @property
    def all_edges(self):
        if self._all_edges is None:
            with torch.no_grad():
                edges = torch.tensor([0, 1, 0, 2, 0, 3, 1, 2, 1, 3, 2, 3], dtype=torch.long, device=self.indices.device)
                all_edges = self.indices[:, edges].reshape(-1, 2)
                self._all_edges = torch.unique(torch.sort(all_edges, dim=1)[0], dim=0)
        return self._all_edges

    @torch.no_grad()
    def getAABB(self):
        return torch.min(self.verts, dim=0).values, torch.max(self.verts, dim=0).values

    def getMesh(self, return_triangle=False, thickness_coef=None):
        if self._sdf_mesh is not None:
            self._sample_mesh(*self._sdf_mesh)
        verts, faces, verts_tetmesh, tets_tetmesh = self.marching_tets(self.verts, self.sdf, self.indices, thickness_coef)
        if return_triangle:
            return types.SimpleNamespace(v_pos=verts, t_pos_idx=faces)
        verts_tetmesh, tets_tetmesh = self.get_largest_connected_component(verts_tetmesh, tets_tetmesh)
        mat = getattr(MatSet, self.FLAGS.mat) if hasattr(self.FLAGS, "mat") else MatSet.Ceramic
        return DiffSoundObj(verts_tetmesh, tets_tetmesh, mode_num=self.FLAGS.mode_num, order=self.FLAGS.order, mat=mat)

    def get_largest_connected_component(self, verts, tets):
        """Largest connected component of the tet mesh (dmtet_thickness.py:254-285), on the device: lock-free union-find
        over the tets instead of the SciPy round trip.  Same vertex subset, numbering and tet order."""
        n_components, kept, tets_out, _ = native.largest_tet_component(tets.contiguous(), verts.shape[0])
        self.last_n_components = n_components
        if n_components == 1:
            return verts, tets
        return verts[kept], tets_out

    def tick(self, target, it, FLAGS):
        sound_obj = self.getMesh()
        sound_obj.eigen_decomposition()
        vals = sound_obj.get_vals()
        audio_loss = ((vals - target) ** 2 / target ** 2).mean()
        print("thickness", self.marching_tets.thickness_coef().item(), "audio_loss", audio_loss.item())
        if self.writer is not None:
            self.writer.add_scalar("loss", audio_loss.item(), it)
            self.writer.add_scalar("thickness", self.marching_tets.thickness_coef().item(), it)
        return audio_loss

    def apply_sdf(self, sdf, sign="parity"):
        """`sdf`: path of a triangle mesh (OBJ), tensor of signed distances at `self.verts`, or a callable verts -> tensor.
        Signed distances are positive inside, the sign convention `apply_sdf` of the reference produces
        (dmtet_thickness.py:312).  A path is read with `read_obj` and sampled at `self.verts` by `native.mesh_sdf`: exact
        distance to the closest triangle, sign by ray-crossing parity (face orientation does not matter).  The mesh is
        used as given, in its own coordinates, with no rescaling or recentring.
        `sdf` = (verts (V, 3), faces (F, 3)) tensors: the triangle mesh, sampled by the differentiable `mesh_sdf`.  If
        verts.requires_grad, the geometry keeps the mesh and every `getMesh()` samples it again (and resets
        `max_thickness`), so each `tick()` builds a fresh graph down to verts; otherwise it is sampled once, like a path.
        `sign` (path and mesh forms): "parity", the ray-crossing parity, right for closed meshes that do not cross
        themselves whatever their face orientation; or "winding", inside where the generalised winding number |w| >= 1/2,
        for meshes with holes or cracks and for surfaces folded through themselves (their overlap stays solid), which
        needs consistently oriented faces.  A tensor or callable `sdf` takes only "parity"."""
        is_mesh = isinstance(sdf, (tuple, list)) and len(sdf) == 2
        is_path = isinstance(sdf, (str, os.PathLike))
        if native._sdf_sign(sign) and not (is_mesh or is_path):
            raise ValueError("apply_sdf: sign='winding' needs a triangle mesh (a path or (verts, faces)), not sampled values")
        self._sdf_mesh = None
        if is_mesh:
            verts, faces = sdf
            dev = self.verts.device
            verts = torch.as_tensor(verts, device=dev)
            faces = torch.as_tensor(faces, device=dev).to(torch.int64)
            if verts.requires_grad:
                self._sdf_mesh = (verts, faces, sign)
            self._sample_mesh(verts, faces, sign)
            return
        if is_path:
            v, f = read_obj(sdf)
            dev = self.verts.device
            sdf = native.mesh_sdf(torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev), self.verts.contiguous(),
                                  sign=sign)
        values = sdf(self.verts) if callable(sdf) else sdf
        self.sdf = torch.as_tensor(values, dtype=torch.float32).to(self.verts.device).reshape(-1)
        self.marching_tets.max_thickness = self.sdf.max()

    def _sample_mesh(self, verts, faces, sign):
        self.sdf = mesh_sdf(verts, faces, self.verts.contiguous(), sign=sign)
        self.marching_tets.max_thickness = self.sdf.max()

    def parameters(self):
        return self.marching_tets.thickness_coef.parameters()

    def get_eigenvalues(self, thickness_coef=None):
        with torch.no_grad():
            sound_obj = self.getMesh(thickness_coef=thickness_coef)
            sound_obj.eigen_decomposition()
            vals = sound_obj.get_vals()
        return vals

    def get_thickness(self):
        return self.marching_tets.thickness_coef()
