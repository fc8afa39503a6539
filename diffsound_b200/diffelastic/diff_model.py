"""Differentiable modal model: assemble K, M -> lowest modes -> differentiable eigenvalues.

API mirror of src/diffelastic/diff_model.py:17-399 (`FixedLinear`,
`TrainableLinear`, `build_model`, `DiffSoundObj`): same constructor arguments,
attribute names (`tetmesh, deform, material_model, mode_num, task, stiff_matrix,
mass_matrix, eigenvalues, U_hat, U_hat_full`), method names, output shapes and
dtypes, so the reference's experiment loops run against this class unchanged.

Underneath, every step is one or a few calls into libdiffsound_sm100.so:

  reference (torch eager / SciPy)                      here
  update_mass_matrix + update_stiff_matrix  (:184-312)  ds_assemble_km into a fixed block-CSR pattern
  eigen_decomposition_arpack (CPU eigsh)    (:335-369)  ds_lobpcg (device-resident, preconditioned)
  get_vals (sparse mm + autograd graph)     (:390-399)  ds_spmm_k_and_m / ds_gram_f64 forward,
                                                        ds_eigval_grad_shape backward
  get_undamped_freqs (fp32 matrix-free K U) (:371-388)  ds_eigval_quadforms_material once per
                                                        decomposition; lambda_i(E, nu) = mu q_mu + lam q_lam
There is no CPU fallback: tensors must be CUDA tensors and the library must load.
"""
import numpy as np
import torch
import torch.nn as nn

from .. import native
from ..ddsp.oscillator import WeightedParam, modal_synth
from .deform import Deform
from .mass_matrix import get_elememt_mass_matrix  # noqa: F401  (re-exported like the reference)
from .material_model import Material, MatSet
from .mesh import TetMesh


def _lame(youngs, poisson):
    lame_lambda = youngs * poisson / ((1 + poisson) * (1 - 2 * poisson))
    lame_mu = youngs / (2 * (1 + poisson))
    return lame_mu, lame_lambda


# packed upper triangle of a 6x6 Voigt matrix, row by row (the 21 values per tet the tensor kernels read), and back
_IU = torch.triu_indices(6, 6)
_VOIGT_UNPACK = torch.tensor([[min(i, j) * (11 - min(i, j)) // 2 + max(i, j) for j in range(6)] for i in range(6)])


def _stress(F, lame_mu, lame_lambda):
    """P = mu (F + F^T) + lambda tr(F) I   (diff_model.py:39-41)."""
    tr = F.diagonal(dim1=-2, dim2=-1).sum(-1)
    return lame_mu * (F + F.transpose(1, 2)) + lame_lambda * tr[:, None, None] * torch.eye(3, device=F.device, dtype=F.dtype)


class FixedLinear(nn.Module):
    """Linear elasticity with fixed E, nu ("gt" and shape tasks)."""

    def __init__(self, mat: Material):
        super().__init__()
        self.youngs = mat.youngs
        self.poisson = mat.poisson
        self.mat = mat

    def lame(self):
        return _lame(self.youngs, self.poisson)

    def forward(self, F: torch.Tensor):
        b, n, _, _ = F.shape
        return self.get_stress(F.reshape(b * n, 3, 3)).reshape(b, n, 3, 3)

    def get_stress(self, F):
        mu, lam = self.lame()
        return _stress(F, mu, lam)

    def jacobian_F(self):
        """d(stress)/dF at F = 0 as a (1,3,3,1,3,3) fp64 tensor (diff_model.py:44-48); closed form."""
        mu, lam = self.lame()
        return _jacobian(float(mu), float(lam))


class TrainableLinear(nn.Module):
    """Learnable E, nu as softplus-normalised mixes of 16 bins (diff_model.py:51-96).  Like the
    reference the parameters live on the CPU (WeightedParam.values_list is not a buffer)."""

    def __init__(self, mat: Material, bin_num=16, baseline=False):
        super().__init__()
        self.youngs_list = torch.exp(torch.linspace(np.log(mat.youngs / 10), np.log(mat.youngs * 10), bin_num))
        if baseline:
            self.poisson_list = torch.linspace(mat.poisson, mat.poisson, 1)
        else:
            self.poisson_list = torch.linspace(0.01, 0.499, bin_num)
        self.youngs = WeightedParam(self.youngs_list)
        self.poisson = WeightedParam(self.poisson_list)
        self.mat = mat

    def lame(self):
        return _lame(self.youngs(), self.poisson())

    def forward(self, F: torch.Tensor):
        b, n, _, _ = F.shape
        return self.get_stress(F.reshape(b * n, 3, 3)).reshape(b, n, 3, 3)

    def get_stress(self, F):
        mu, lam = self.lame()
        return _stress(F, mu.to(F.device), lam.to(F.device))

    def jacobian_F(self):
        mu, lam = self.lame()
        return _jacobian(float(mu), float(lam))


def _jacobian(mu, lam):
    dev = torch.device("cuda", torch.cuda.current_device())
    eye = torch.eye(3, dtype=torch.float64, device=dev)
    J = (mu * (torch.einsum("ik,jl->ijkl", eye, eye) + torch.einsum("il,jk->ijkl", eye, eye))
         + lam * torch.einsum("ij,kl->ijkl", eye, eye))
    return J.reshape(1, 3, 3, 1, 3, 3)


def build_model(mesh_dir, mode_num, order, mat, task, vertices=None, tets=None, scale_range=None, init_scale=None):
    if task == "material" or task == "mat_baseline":
        mat_model = TrainableLinear
    elif task == "gt":
        mat_model = FixedLinear
    else:
        raise ValueError("task not defined")
    model = DiffSoundObj(mesh_dir=mesh_dir, mode_num=mode_num, order=order, mat=mat, mat_model=mat_model, task=task)
    if task == "material" or task == "mat_baseline":
        model.init_material_coeffs()
    return model


def check_fixed_mask(vertices, mask):
    """Host validation of a clamp mask (DiffSoundObj.fix_nodes): a boolean (n_nodes,) tensor over `vertices` whose nodes
    contain three non-collinear points, so that the clamps remove all rigid motion.  Raises ValueError otherwise."""
    n_nodes = vertices.shape[0]
    if not torch.is_tensor(mask) or mask.dtype != torch.bool:
        raise ValueError("fix_nodes: mask must be a boolean tensor")
    if mask.shape != (n_nodes,):
        raise ValueError(f"fix_nodes: mask has shape {tuple(mask.shape)}, expected ({n_nodes},) over tetmesh.vertices")
    p = vertices.detach()[mask].double().cpu()
    sv = torch.linalg.svdvals(p - p.mean(0)) if p.shape[0] >= 3 else torch.zeros(2, dtype=torch.float64)
    # relative to the extent of the fixed set: fp32 coordinates of points on one line are collinear to ~1e-7
    if p.shape[0] < 3 or not bool(sv[1] > 1e-6 * sv[0]):
        raise ValueError(f"fix_nodes: the {p.shape[0]} fixed nodes do not contain three non-collinear points, so rigid "
                         "motion would remain; clamp a larger set or none (fix_nodes(None))")


def check_material_field(num_tets, device, youngs=None, poisson=None, density=None):
    """Host validation of a material field (DiffSoundObj.set_material_field): each given part is a finite fp32 / fp64
    (num_tets,) tensor on `device` with E > 0, -1 < nu < 0.5 and rho > 0.  Raises ValueError otherwise."""
    for name, t in (("youngs", youngs), ("poisson", poisson), ("density", density)):
        if t is None:
            continue
        if not torch.is_tensor(t) or t.dtype not in (torch.float32, torch.float64):
            raise ValueError(f"set_material_field: {name} must be a float32 or float64 tensor")
        if t.shape != (num_tets,):
            raise ValueError(f"set_material_field: {name} has shape {tuple(t.shape)}, expected ({num_tets},): one value per "
                             "row of tetmesh.tets")
        if t.device != torch.device(device):
            raise ValueError(f"set_material_field: {name} is on {t.device}, the mesh on {device}")
        x = t.detach()
        if not bool(torch.isfinite(x).all()):
            raise ValueError(f"set_material_field: {name} has non-finite values")
        if name == "poisson":
            ok = bool(((x > -1) & (x < 0.5)).all())
            cond = "-1 < poisson < 0.5"
        else:
            ok = bool((x > 0).all())
            cond = f"{name} > 0"
        if not ok:
            raise ValueError(f"set_material_field: {name} violates {cond}")


def check_elasticity_field(num_tets, device, C, density=None):
    """Host validation of an elasticity-tensor field (DiffSoundObj.set_elasticity_field): C a finite fp32 / fp64
    (num_tets, 6, 6) tensor on `device`, symmetric to 1e-10 max|C| and positive definite in every tet (a Cholesky
    factorisation on the device); density None or a finite positive fp32 / fp64 (num_tets,) tensor on `device`.  Raises
    ValueError otherwise."""
    if not torch.is_tensor(C) or C.dtype not in (torch.float32, torch.float64):
        raise ValueError("set_elasticity_field: C must be a float32 or float64 tensor")
    if C.shape != (num_tets, 6, 6):
        raise ValueError(f"set_elasticity_field: C has shape {tuple(C.shape)}, expected ({num_tets}, 6, 6): one Voigt matrix "
                         "per row of tetmesh.tets")
    if C.device != torch.device(device):
        raise ValueError(f"set_elasticity_field: C is on {C.device}, the mesh on {device}")
    x = C.detach().to(torch.float64)
    if not bool(torch.isfinite(x).all()):
        raise ValueError("set_elasticity_field: C has non-finite values")
    if not bool(((x - x.transpose(1, 2)).abs().amax() <= 1e-10 * x.abs().amax())):
        raise ValueError("set_elasticity_field: C is not symmetric (to 1e-10 max|C|)")
    _, info = torch.linalg.cholesky_ex(0.5 * (x + x.transpose(1, 2)))
    bad = torch.nonzero(info).flatten()
    if bad.numel():
        raise ValueError(f"set_elasticity_field: C is not positive definite in {bad.numel()} tets (first: tet {int(bad[0])})")
    if density is not None:
        check_material_field(num_tets, device, density=density)


#: supports must hold every rigid motion: the smallest eigenvalue of the 6 x 6 R^T K_s R over the rigid fields (unit
#: translations, rotations scaled by the object's extent) must exceed this fraction of the largest.  Roundoff leaves an
#: unsupported direction near 1e-16; a genuinely soft direction (k_t = 1e-6 k_n) is far above the margin.
SUPPORT_RIGID_MARGIN = 1e-10


def check_support_stiffness(S, device, normal, tangential):
    """Host validation of support stiffnesses (DiffSoundObj.set_supports): each a Python float or a finite fp32 / fp64 (S,)
    tensor on `device`, all >= 0.  Returns (k_n, k_t) as contiguous fp64 (S,) tensors (copies).  Raises ValueError."""
    out = []
    for name, k in (("normal", normal), ("tangential", tangential)):
        if torch.is_tensor(k):
            if k.dtype not in (torch.float32, torch.float64):
                raise ValueError(f"set_supports: {name} must be a float or a float32 / float64 tensor")
            if k.shape != (S,):
                raise ValueError(f"set_supports: {name} has shape {tuple(k.shape)}, expected ({S},): one value per support "
                                 "face in ascending face order")
            if k.device != torch.device(device):
                raise ValueError(f"set_supports: {name} is on {k.device}, the mesh on {device}")
            x = k.detach().to(torch.float64).clone().contiguous()
        elif isinstance(k, (int, float)) and not isinstance(k, bool):
            x = torch.full((S,), float(k), dtype=torch.float64, device=device)
        else:
            raise ValueError(f"set_supports: {name} must be a float or a (S,) tensor")
        if not bool(torch.isfinite(x).all()):
            raise ValueError(f"set_supports: {name} has non-finite values")
        if not bool((x >= 0).all()):
            raise ValueError(f"set_supports: {name} must be >= 0")
        out.append(x)
    return out[0], out[1]


def support_rigid_matrix(p0, p1, p2, kn, kt):
    """The 6 x 6 R^T K_s R of a spring bed over the rigid fields R = [translations, rotations / L] about the centroid of
    the support corners (L their extent), from the exact edge-midpoint rule (rigid fields are linear, the integrand
    quadratic).  p0, p1, p2 (S, 3) fp64 face corners; kn, kt (S,) fp64."""
    c = torch.cat([p0, p1, p2]).mean(0)
    L = float(torch.cat([p0, p1, p2]).sub(c).norm(dim=1).max().clamp_min(1e-30))
    a = 0.5 * torch.cross(p1 - p0, p2 - p0, dim=1)
    A = a.norm(dim=1)
    n = a / A.clamp_min(1e-300)[:, None]
    Sm = (kn - kt)[:, None, None] * n[:, :, None] * n[:, None, :] + kt[:, None, None] * torch.eye(3, dtype=a.dtype,
                                                                                                    device=a.device)
    G = torch.zeros(6, 6, dtype=a.dtype, device=a.device)
    eye = torch.eye(3, dtype=a.dtype, device=a.device).expand(p0.shape[0], 3, 3)
    for x in (0.5 * (p0 + p1), 0.5 * (p1 + p2), 0.5 * (p2 + p0)):
        y = (x - c) / L
        z = torch.zeros_like(y[:, 0])
        rot = torch.stack([torch.stack([-y[:, 1], y[:, 0], z], 1), torch.stack([z, -y[:, 2], y[:, 1]], 1),
                           torch.stack([y[:, 2], z, -y[:, 0]], 1)], dim=2)          # (S, 3, 3): columns are the fields
        R = torch.cat([eye, rot], dim=2)                                             # (S, 3, 6)
        G += torch.einsum("s,sci,scd,sdj->ij", A / 3, R, Sm, R)
    return G


def material_field_from_regions(labels, materials):
    """(youngs, poisson, density), each (T,) fp64 on the device of `labels`: the material `materials[labels[t]]` (MatSet
    tuples) of every tet, for DiffSoundObj.set_material_field."""
    if not torch.is_tensor(labels) or labels.dtype not in (torch.int32, torch.int64) or labels.dim() != 1:
        raise ValueError("material_field_from_regions: labels must be a 1-D integer tensor")
    if len(materials) == 0:
        raise ValueError("material_field_from_regions: no materials")
    if labels.numel() and (int(labels.min()) < 0 or int(labels.max()) >= len(materials)):
        raise ValueError(f"material_field_from_regions: labels must lie in [0, {len(materials)})")
    tab = torch.tensor([[float(m[1]), float(m[2]), float(m[0])] for m in materials], dtype=torch.float64,
                       device=labels.device)
    per_tet = tab[labels.long()]
    return per_tet[:, 0].contiguous(), per_tet[:, 1].contiguous(), per_tet[:, 2].contiguous()


def _gram_diag(X, Y):
    """diag(X^T Y) for (n, k) fp64 blocks, in chunks the Gram kernel accepts (<= 64 columns, multiples of 8)."""
    k = X.shape[1]
    out = []
    for c0 in range(0, k, 48):
        c1 = min(k, c0 + 48)
        out.append(torch.diagonal(native.gram(X[:, c0:c1], Y[:, c0:c1])))
    return torch.cat(out)


def _vals_forward(obj):
    """lambda + (u^T K u - lambda u^T M u) of the wanted modes, (mode_num,) fp32: the value of get_vals()."""
    X, lam = obj._Xpad, obj.eigenvalues          # all wanted columns, padded to a multiple of 16
    KX, MX = native.spmm_k_and_m(obj.deform.pattern, obj._Kval, obj._Mblk, X)
    lo = obj._n_rigid
    hi = lo + obj.mode_num
    uku = _gram_diag(X, KX)[lo:hi]
    umu = _gram_diag(X, MX)[lo:hi]
    predict = torch.zeros(obj.mode_num, dtype=torch.float32, device=X.device)
    predict += lam
    predict += uku - lam * umu
    return predict


class _EigvalShape(torch.autograd.Function):
    """get_vals(): value lambda + (u^T K u - lambda u^T M u), gradient u^T (dK - lambda dM) u w.r.t.
    the (promoted) vertex positions.  Everything the backward pass needs is pinned in ctx at forward
    time (eigenvectors, eigenvalues, geometry, material), as autograd does for the reference
    (diff_model.py:390-399): a later eigen_decomposition() / update_*_matrix() on the same object
    does not change the gradient of an earlier get_vals()."""

    @staticmethod
    def forward(ctx, vertices, obj):
        lam = obj.eigenvalues
        d = obj.deform
        predict = _vals_forward(obj)
        ctx.order = obj.tetmesh.order
        ctx.lame = obj._lame_used
        ctx.vdtype = obj.tetmesh.vertices.dtype
        inc_ptr, inc = d.incidence
        ctx.U = obj.U_hat                        # a view of storage that is never written again (see _start_block)
        ctx.save_for_backward(obj._verts32, d.tets_i32, d.ctab, d.mtab(obj._density_used), lam, inc_ptr, inc)
        return predict.unsqueeze(1)

    @staticmethod
    def backward(ctx, g):
        verts32, tets, ctab, mtab, lam, inc_ptr, inc = ctx.saved_tensors
        mu, lam_l = ctx.lame
        gv = g.reshape(-1).to(torch.float64).contiguous()
        grad = native.eigval_grad_shape(verts32, tets, ctx.order, mu, lam_l, ctab, mtab, ctx.U, lam, gv, inc_ptr, inc)
        return grad.to(ctx.vdtype), None


class _EigvalField(torch.autograd.Function):
    """get_vals() of an object with a material field: the value of _EigvalShape, gradients u^T (dK - lambda dM) u to the
    vertices (native.eigval_grad_shape_field) and to the per-tet (E, nu, rho) (native.material_field_grad for (mu_t, lam_t,
    rho_t), then the chain rule of _lame elementwise).  The field values, eigenpairs and geometry the assembly used are
    pinned at forward time, as in _EigvalShape."""

    @staticmethod
    def forward(ctx, vertices, youngs, poisson, density, obj):
        lam = obj.eigenvalues
        d = obj.deform
        predict = _vals_forward(obj)
        f = obj._field_used
        ctx.order, ctx.wsum = obj.tetmesh.order, d.wsum
        ctx.vdtype = obj.tetmesh.vertices.dtype
        ctx.dtypes = tuple(None if t is None else t.dtype for t in (youngs, poisson, density))
        ctx.U = obj.U_hat
        inc_ptr, inc = d.incidence
        ctx.save_for_backward(obj._verts32, d.tets_i32, d.ctab, d.mtab(1.0), d.m32(), lam, inc_ptr, inc, f["mu"], f["lam"],
                              f["rho"], f["youngs"], f["poisson"])
        return predict.unsqueeze(1)

    @staticmethod
    def backward(ctx, g):
        verts32, tets, ctab, mtab1, m32, lam, inc_ptr, inc, mu_t, lam_t, rho_t, E, nu = ctx.saved_tensors
        gv = g.reshape(-1).to(torch.float64).contiguous()
        gverts = gE = gnu = grho = None
        if ctx.needs_input_grad[0]:
            gverts = native.eigval_grad_shape_field(verts32, tets, ctx.order, (mu_t, lam_t, rho_t), ctab, mtab1, ctx.U, lam,
                                                    gv, inc_ptr, inc).to(ctx.vdtype)
        if any(ctx.needs_input_grad[1:4]):
            G = native.material_field_grad(verts32, tets, ctx.order, m32, ctx.wsum, ctx.U, lam, gv)
            if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
                with torch.enable_grad():
                    E_, nu_ = E.detach().requires_grad_(True), nu.detach().requires_grad_(True)
                    mu_, la_ = _lame(E_, nu_)
                    gE, gnu = torch.autograd.grad((mu_ * G[:, 0] + la_ * G[:, 1]).sum(), (E_, nu_))
                gE = gE.to(ctx.dtypes[0]) if ctx.needs_input_grad[1] else None
                gnu = gnu.to(ctx.dtypes[1]) if ctx.needs_input_grad[2] else None
            if ctx.needs_input_grad[3]:
                grho = G[:, 2].to(ctx.dtypes[2])
        return gverts, gE, gnu, grho, None


class _EigvalTensor(torch.autograd.Function):
    """get_vals() of an object with an elasticity-tensor field: the value of _EigvalShape, gradients u^T (dK - lambda dM) u
    to the vertices (native.eigval_grad_shape_tensor, C fixed in world axes), to C (the symmetric strain Gram
    sum_i g_i E_t,i of native.elasticity_field_grad, unpacked to (T, 6, 6)) and to the density.  The tensors, eigenpairs
    and geometry the assembly used are pinned at forward time, as in _EigvalShape."""

    @staticmethod
    def forward(ctx, vertices, C, density, obj):
        lam = obj.eigenvalues
        d = obj.deform
        predict = _vals_forward(obj)
        f = obj._tensor_used
        ctx.order, ctx.wsum = obj.tetmesh.order, d.wsum
        ctx.vdtype = obj.tetmesh.vertices.dtype
        ctx.dtypes = (C.dtype, None if density is None else density.dtype)
        ctx.U = obj.U_hat
        inc_ptr, inc = d.incidence
        ctx.save_for_backward(obj._verts32, d.tets_i32, d.ctab, d.mtab(1.0), d.m32(), lam, inc_ptr, inc, f["C21"], f["rho"])
        return predict.unsqueeze(1)

    @staticmethod
    def backward(ctx, g):
        verts32, tets, ctab, mtab1, m32, lam, inc_ptr, inc, C21, rho_t = ctx.saved_tensors
        gv = g.reshape(-1).to(torch.float64).contiguous()
        gverts = gC = grho = None
        if ctx.needs_input_grad[0]:
            gverts = native.eigval_grad_shape_tensor(verts32, tets, ctx.order, (C21, rho_t), ctab, mtab1, ctx.U, lam, gv,
                                                     inc_ptr, inc).to(ctx.vdtype)
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            G21, G_rho = native.elasticity_field_grad(verts32, tets, ctx.order, m32, ctx.wsum, ctx.U, lam, gv)
            if ctx.needs_input_grad[1]:
                gC = G21[:, _VOIGT_UNPACK].to(ctx.dtypes[0])
            if ctx.needs_input_grad[2]:
                grho = G_rho.to(ctx.dtypes[1])
        return gverts, gC, grho, None


class _SupportTerm(torch.autograd.Function):
    """Zero-valued term of get_vals() for an object on elastic supports: the eigenvalues already include K_s (the value is
    read from Kval), and the backward adds the support part sum_i g_i u_i^T dK_s u_i of the gradient, to the vertices
    (through the area vectors of the support faces) and to the per-face normal / tangential stiffnesses
    (native.support_grad).  The stiffnesses, eigenvectors and geometry the assembly used are pinned at forward time."""

    @staticmethod
    def forward(ctx, vertices, normal, tangential, obj):
        sup = obj._sup_used
        ctx.vdtype = obj.tetmesh.vertices.dtype
        ctx.dtypes = tuple(k.dtype if torch.is_tensor(k) else None for k in (normal, tangential))
        ctx.faces, ctx.U = obj._sup["fine"], obj.U_hat
        ctx.save_for_backward(obj._verts32, obj.deform.tets_i32, sup["kn"], sup["kt"])
        return torch.zeros(obj.mode_num, 1, dtype=torch.float32, device=obj.deform.device)

    @staticmethod
    def backward(ctx, g):
        verts32, tets, kn, kt = ctx.saved_tensors
        gv = g.reshape(-1).to(torch.float64).contiguous()
        gk, gverts = native.support_grad(verts32, tets, ctx.faces, kn, kt, ctx.U, gv, want_verts=ctx.needs_input_grad[0])
        gn = gk[:, 0].to(ctx.dtypes[0]) if ctx.needs_input_grad[1] else None
        gt = gk[:, 1].to(ctx.dtypes[1]) if ctx.needs_input_grad[2] else None
        return (None if gverts is None else gverts.to(ctx.vdtype)), gn, gt, None


class _StiffFunc(torch.autograd.Function):
    """y = (mu K_mu + lam K_lam) x with gradients to x (K is symmetric: K^T g) and to the two Lame
    scalars (<g, K_mu x>, <g, K_lam x>) -- stiff_func of the reference is differentiable in both
    (diff_model.py:314-328 through deform.py:70-165)."""

    @staticmethod
    def forward(ctx, x, mu, lam, obj):
        Kmu, Kla = obj._unit_stiffness()
        pat = obj.deform.pattern
        cols = x.shape[1]
        ys = []
        for c0 in range(0, cols, 128):
            c1 = min(cols, c0 + 128)
            cp = (c1 - c0 + 15) // 16 * 16
            xp = torch.zeros(x.shape[0], cp, dtype=torch.float64, device=x.device)
            xp[:, :c1 - c0] = x[:, c0:c1]
            ys.append((native.spmm(pat, Kmu, None, xp)[:, :c1 - c0], native.spmm(pat, Kla, None, xp)[:, :c1 - c0]))
        ymu = torch.cat([a for a, _ in ys], dim=1)
        yla = torch.cat([b for _, b in ys], dim=1)
        ctx.obj = obj
        ctx.save_for_backward(ymu, yla, mu, lam)
        ctx.xdtype = x.dtype
        return (mu.double() * ymu + lam.double() * yla).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        ymu, yla, mu, lam = ctx.saved_tensors
        g64 = g.to(torch.float64)
        gx = gmu = gla = None
        if ctx.needs_input_grad[0]:
            gx = _StiffFunc.apply(g.contiguous(), mu.detach(), lam.detach(), ctx.obj).to(ctx.xdtype)
        if ctx.needs_input_grad[1]:
            gmu = (g64 * ymu).sum().to(mu.dtype)
        if ctx.needs_input_grad[2]:
            gla = (g64 * yla).sum().to(lam.dtype)
        return gx, gmu, gla, None


class _ModalGains(torch.autograd.Function):
    """g[p, m] = d_p . u_m(closest(p)) on the boundary face `face[p]` (native.modal_gains).  Differentiable in the points
    and the directions only: the mode shapes and the mesh are constants here."""

    @staticmethod
    def forward(ctx, points, directions, obj, face):
        d = obj.deform
        pts = points.detach().to(torch.float32).contiguous()
        dirs = None if directions is None else directions.detach().to(torch.float32).contiguous()
        g, closest = native.modal_gains(obj._verts32, d.tets_i32, obj.tetmesh.order, obj._boundary(), pts,
                                        face, dirs, obj.U_hat)
        obj.last_strike_points = closest
        ctx.obj, ctx.U = obj, obj.U_hat
        ctx.save_for_backward(pts, face, dirs)
        ctx.dtypes = (points.dtype, None if directions is None else directions.dtype)
        return g

    @staticmethod
    def backward(ctx, grad):
        pts, face, dirs = ctx.saved_tensors
        obj = ctx.obj
        gp, gd = native.modal_gains_backward(obj._verts32, obj.deform.tets_i32, obj.tetmesh.order,
                                             obj._boundary(), pts, face, dirs, ctx.U,
                                             grad.to(torch.float32).contiguous())
        return gp.to(ctx.dtypes[0]), (None if gd is None else gd.to(ctx.dtypes[1])), None, None


class DiffSoundObj:
    #: options of the eigensolver (see ds_lobpcg_opts in include/diffsound_sm100.h)
    # relative residual ||K u - lam M u|| / (lam ||M u||).  Eigenvalue error ~ tol^2, eigenvector (and
    # therefore d(lambda)/d(theta)) error ~ tol * lam / gap: 1e-5 keeps the gradient inside 1e-5.
    eig_tol = 1e-5
    two_level = True        # quadratic meshes: p-multigrid preconditioner (P1 coarse level) in the eigensolver
    nested_start = True     # ... and a P1 eigen-solve for the start block (skipped on a warm start)
    nested_tol = 3e-2
    nested_degree = 0       # 0: automatic
    smooth_steps = 3        # Chebyshev-Jacobi smoothing steps on the P2 operator before / after the coarse correction
    smooth_ratio = 8.0      # ... damping the upper [lmax / ratio, lmax] of the spectrum
    coarse_degree = 0       # Chebyshev steps of the P1 coarse solve (0: automatic, ~ n_coarse^(1/3) / 1.2)
    coarse_ratio = 0.0      # 0: automatic, 0.4 * degree^2
    cheb_degree = 0         # one-level Chebyshev preconditioner (linear meshes): polynomial degree, 0 = automatic
    morton = True           # the FP32 preconditioner keeps its operator in a Morton node numbering (SpMM locality)
    eig_maxit = 400
    # Sliver elements (marching-tets meshes) put stiff components into the residuals that exceed their smooth part by more than
    # FP32 resolves; the FP32 cycle then stalls (DESIGN.md section 5.2).  Policy: meshes whose worst element is `sliver_ratio`
    # times flatter than the median go straight to the FP64 Chebyshev preconditioner (ds_lobpcg_opts.precond_fp64); others try
    # the FP32 cycle for at most `eig_fast_maxit` iterations and fall back to FP64 from the block reached so far.
    fp64_fallback = True
    eig_fast_maxit = 80
    sliver_ratio = 2e-3

    def __init__(self, vertices=None, tets=None, mode_num=16, mat=MatSet.Ceramic, order=1, mat_model=FixedLinear,
                 task=None, mesh_dir=None):
        if mesh_dir:
            self.mesh_dir = mesh_dir
            self.tetmesh = TetMesh.from_triangle_mesh(mesh_dir).to_high_order(order)
        else:
            if not vertices.is_cuda:
                raise RuntimeError("diffsound_b200: vertices/tets must be CUDA tensors (there is no CPU path)")
            self.tetmesh = TetMesh(vertices, tets).to_high_order(order)
        self.deform = Deform(self.tetmesh)
        if task == "mat_baseline":
            self.material_model = mat_model(Material(mat), baseline=True)
        else:
            self.material_model = mat_model(Material(mat))
        self.mode_num = mode_num
        self.U_hat_full = None
        self.task = task
        self._Kval = self._Mblk = None
        self._density_used = None
        self._lame_used = None
        self._X = None
        self._Xpad = None
        self._warm = []
        self._q = None
        self.eig_stats = None
        self.last_strike_points = None
        self.fixed_nodes = None
        self._fixed_u8 = None
        self.material_field = None      # (youngs, poisson, density) of set_material_field, None: one material
        self._field_used = None
        self.elasticity_field = None    # (C, density) of set_elasticity_field, None: isotropic
        self._tensor_used = None
        self.supports = None            # (faces mask, normal, tangential) of set_supports, None: no supports
        self._sup = None                # native.SupportFaces of the fine (and coarse) level
        self._sup_used = None           # the (k_n, k_t) fp64 (S,) the last assembly used

    # ------------------------------------------------------------------ parameters
    def parameters(self):
        if self.task == "material":
            return self.material_model.parameters()
        elif self.task == "mat_baseline":
            return self.material_model.youngs.parameters()
        return None

    def init_material_coeffs(self, steps=5000, verbose=True):
        """Pre-train the (E, nu) logits towards the material table (diff_model.py:154-182)."""
        mm = self.material_model
        optimizer = torch.optim.Adam(mm.parameters(), lr=5e-3)
        gt_youngs, gt_poisson = mm.mat.youngs, mm.mat.poisson
        for _ in range(steps):
            optimizer.zero_grad()
            loss = (mm.youngs() - gt_youngs) ** 2 / gt_youngs ** 2 + (mm.poisson() - gt_poisson) ** 2 / gt_poisson ** 2
            loss.backward()
            optimizer.step()
        if verbose:
            print("(net) youngs: ", mm.youngs(), "poisson: ", mm.poisson())
            print("(material table) youngs: ", mm.mat.youngs, "poisson: ", mm.mat.poisson)
        self.scale = torch.eye(3, dtype=torch.float64, device=self.tetmesh.device)

    # ------------------------------------------------------------------ assembly
    def _field_snapshot(self, density):
        """The field the next assembly uses, validated again (optimisers change the tensors in place): fp64 E, nu and the
        Lame parameters of _lame, fp32 rho; a part left None is the material's scalar (density: `density`)."""
        youngs, poisson, dens = self.material_field
        d = self.deform
        check_material_field(d.num_tets, d.device, youngs, poisson, dens)
        mat = self.material_model.mat
        f64 = dict(dtype=torch.float64, device=d.device)

        def part(t, scalar):
            return torch.full((d.num_tets,), float(scalar), **f64) if t is None else t.detach().to(torch.float64).clone()

        E, nu = part(youngs, mat.youngs), part(poisson, mat.poisson)
        mu_t, lam_t = _lame(E, nu)
        rho = (torch.full((d.num_tets,), float(density), dtype=torch.float32, device=d.device) if dens is None
               else dens.detach().to(torch.float32).clone())
        return dict(youngs=E, poisson=nu, mu=mu_t.contiguous(), lam=lam_t.contiguous(), rho=rho.contiguous())

    def _tensor_snapshot(self, density):
        """The elasticity-tensor field the next assembly uses, validated again: C symmetrised in fp64 (T, 6, 6), its packed
        upper triangle C21 (T, 21) and fp32 rho (density None: `density`)."""
        C, dens = self.elasticity_field
        d = self.deform
        check_elasticity_field(d.num_tets, d.device, C, dens)
        x = C.detach().to(torch.float64)
        Cs = 0.5 * (x + x.transpose(1, 2))
        rho = (torch.full((d.num_tets,), float(density), dtype=torch.float32, device=d.device) if dens is None
               else dens.detach().to(torch.float32).clone())
        return dict(C=Cs, C21=Cs[:, _IU[0], _IU[1]].contiguous(), rho=rho.contiguous())

    def _assemble(self, density):
        d = self.deform
        mu, lam = self.material_model.lame()
        mu, lam = float(mu), float(lam)
        self._verts32 = d.verts_f32()
        pat = d.pattern
        if "_geom" not in self.__dict__:
            self._geom = torch.empty(d.num_tets * 14, dtype=torch.float64, device=d.device)
        self._tensor_used = None
        if self.elasticity_field is not None:
            self._field_used = None
            t = self._tensor_snapshot(density)
            self._tensor_used = t
            self._Kval, self._Mblk = native.assemble_km(self._verts32, d.tets_i32, self.tetmesh.order, pat, 0.0, 0.0, d.ctab,
                                                        d.m32(), Kval=self._Kval, Mblk=self._Mblk, geom=self._geom,
                                                        tensor=(t["C21"], t["rho"]))
        elif self.material_field is None:
            self._field_used = None
            self._Kval, self._Mblk = native.assemble_km(self._verts32, d.tets_i32, self.tetmesh.order, pat, mu, lam, d.ctab,
                                                        d.mtab(density), Kval=self._Kval, Mblk=self._Mblk, geom=self._geom)
        else:
            f = self._field_snapshot(density)
            self._field_used = f
            self._Kval, self._Mblk = native.assemble_km(self._verts32, d.tets_i32, self.tetmesh.order, pat, 0.0, 0.0, d.ctab,
                                                        d.m32(), Kval=self._Kval, Mblk=self._Mblk, geom=self._geom,
                                                        field=(f["mu"], f["lam"], f["rho"]))
        self._sup_used = None
        if self.supports is not None:
            kn, kt = self._support_snapshot()
            self._sup_used = dict(kn=kn, kt=kt)
            native.support_km(self._verts32, d.tets_i32, pat, self._sup["fine"], kn, kt, self._Kval)
        if self._fixed_u8 is not None:
            native.fix_nodes_km(pat, self._fixed_u8, self._Kval, self._Mblk)
        self._density_used = float(density)
        self._lame_used = (mu, lam)
        self.__dict__.pop("_stiff_coo", None)
        self.__dict__.pop("_mass_coo", None)

    def update_stiff_matrix(self, assemble_batch_size=20000):
        """K into the fixed pattern.  `assemble_batch_size` only bounded the reference's memory
        (diff_model.py:192-199); it is accepted and ignored."""
        dens = self._density_used if self._density_used is not None else self.material_model.mat.density
        self._assemble(dens)

    def update_mass_matrix(self, density):
        self._assemble(density)

    def _coo(self, values):
        idx = self.deform.pattern.coo_indices()
        n = self.deform.pattern.n
        return torch.sparse_coo_tensor(idx, values, (n, n), is_coalesced=True, check_invariants=False)

    @property
    def stiff_matrix(self):
        """torch sparse COO (n, n) fp64, coalesced, indices sorted by (row, col) -- what the reference
        keeps after `.coalesce()` (diff_model.py:216-220).  Materialised only when asked for."""
        if "_stiff_coo" not in self.__dict__:
            self._stiff_coo = self._coo(self._Kval)
        return self._stiff_coo

    @property
    def mass_matrix(self):
        if "_mass_coo" not in self.__dict__:
            self._mass_coo = self._coo(native.mass_expand(self.deform.pattern, self._Mblk))
        return self._mass_coo

    # ------------------------------------------------------------------ operators
    def stiff_func(self, x_in: torch.Tensor):
        """K(theta) x, differentiable in (E, nu) and in x: K = mu K_mu + lam K_lam (diff_model.py:314-328).
        Accepts (n,) or (n, k) like the reference, any number of columns."""
        if self.material_field is not None:
            raise NotImplementedError("stiff_func: K = mu K_mu + lam K_lam with one (mu, lam) for the whole object; it is not "
                                      "defined for a material field (set_material_field(None) first)")
        if self.elasticity_field is not None:
            raise NotImplementedError("stiff_func: K = mu K_mu + lam K_lam with one (mu, lam) for the whole object; it is not "
                                      "defined for an elasticity-tensor field (set_elasticity_field(None) first)")
        if self.supports is not None:
            raise NotImplementedError("stiff_func: K = mu K_mu + lam K_lam has no support term; it is not defined for an "
                                      "object on elastic supports (set_supports(None) first)")
        x = x_in.unsqueeze(1) if x_in.dim() == 1 else x_in
        mu, lam = self.material_model.lame()
        mu = torch.as_tensor(mu, dtype=torch.float32).to(x.device)
        lam = torch.as_tensor(lam, dtype=torch.float32).to(x.device)
        force = _StiffFunc.apply(x, mu, lam, self)
        return force.squeeze(1) if x_in.dim() == 1 else force

    def _unit_stiffness(self):
        if "_Kunit" not in self.__dict__:
            d = self.deform
            v32 = d.verts_f32()
            mt = d.mtab(self.material_model.mat.density)
            Kmu, _ = native.assemble_km(v32, d.tets_i32, self.tetmesh.order, d.pattern, 1.0, 0.0, d.ctab, mt)
            Kla, _ = native.assemble_km(v32, d.tets_i32, self.tetmesh.order, d.pattern, 0.0, 1.0, d.ctab, mt)
            if self._fixed_u8 is not None:
                native.fix_nodes_km(d.pattern, self._fixed_u8, Kmu)
                native.fix_nodes_km(d.pattern, self._fixed_u8, Kla)
            self._Kunit = (Kmu, Kla)
        return self._Kunit

    # ------------------------------------------------------------------ boundary conditions
    def fix_nodes(self, mask):
        """Clamp the object: every node of the boolean (n_nodes,) CUDA mask over `tetmesh.vertices` (the promoted nodes,
        so the caller chooses the P2 mid-edge nodes too) has all three displacement components fixed to zero.  K and M
        are constrained on their pattern (native.fix_nodes_km) after every assembly, the eigensolver keeps the rows of
        the fixed nodes at zero, and `eigenvalues` / `U_hat` are the lowest `mode_num` pairs of the clamped object (it
        has no rigid modes).  The fixed nodes must contain three non-collinear points, so that no rigid motion remains.
        `fix_nodes(None)` frees the object again.  Either way the warm start and the cached operators are dropped."""
        if mask is not None:
            if torch.is_tensor(mask) and mask.device != self.tetmesh.vertices.device:
                raise ValueError(f"fix_nodes: mask is on {mask.device}, the mesh on {self.tetmesh.vertices.device}")
            check_fixed_mask(self.tetmesh.vertices, mask)
        self.fixed_nodes = mask
        self._fixed_u8 = None if mask is None else mask.to(torch.uint8).contiguous()
        self._n_fixed = 0 if mask is None else int(mask.sum())
        self._warm = []
        self._q = None
        for key in ("_Kunit", "_stiff_coo", "_mass_coo"):
            self.__dict__.pop(key, None)
        if self._Kval is not None:
            self._assemble(self._density_used)

    # ------------------------------------------------------------------ material fields
    def set_material_field(self, youngs=None, poisson=None, density=None):
        """Give every tet its own material: (T,) fp32 / fp64 CUDA tensors on the mesh's device, indexed by the rows of
        `tetmesh.tets` (the input tets, in order), of Young's modulus, Poisson's ratio and density.  A part left None is
        the material's scalar; all three None clears the field (one material again).  The tensors are kept by reference
        and read (and validated) at every assembly, so an optimiser may update them in place; set the field again each
        step otherwise.  With a field, K = sum_t (mu_t K_mu,t + lam_t K_lam,t) with (mu_t, lam_t) = _lame(E_t, nu_t) in
        fp64, and the mass entry of tet t is double(float32(m_ab) * float32(rho_t)): a constant field gives K and M
        bitwise equal to the homogeneous object.  get_vals() is then differentiable in the three tensors too.  Rayleigh
        damping stays global (impulse_response's alpha, beta).

        The warm start is kept: a new field on the same mesh is a small perturbation of the previous solve.  Raises
        ValueError on a TrainableLinear material model (its global E, nu logits and a field would both define E)."""
        if youngs is None and poisson is None and density is None:
            self.material_field = None
        else:
            if isinstance(self.material_model, TrainableLinear):
                raise ValueError("set_material_field: the material model is TrainableLinear, whose global (E, nu) logits "
                                 "would compete with a per-tet field; build the object with FixedLinear")
            if self.elasticity_field is not None:
                raise ValueError("set_material_field: an elasticity-tensor field is set and both define the stiffness; "
                                 "clear it first (set_elasticity_field(None))")
            check_material_field(self.deform.num_tets, self.deform.device, youngs, poisson, density)
            self.material_field = (youngs, poisson, density)
        self._q = None
        for key in ("_stiff_coo", "_mass_coo"):
            self.__dict__.pop(key, None)
        if self._Kval is not None:
            self._assemble(self._density_used)

    def set_elasticity_field(self, C, density=None):
        """Give every tet its own anisotropic material: C (T, 6, 6) fp32 / fp64 CUDA tensor of elasticity matrices over the
        rows of `tetmesh.tets`, and optionally density (T,) (None: the material's scalar).  Voigt order (11, 22, 33, 23, 13,
        12) with engineering shear strains, eps_V = (e11, e22, e33, 2 e23, 2 e13, 2 e12), sigma_V = C eps_V, strain energy
        1/2 int eps_V^T C_t eps_V dV; C is in the global (mesh) frame and does not turn with the vertices.  One material
        everywhere is C0.expand(T, 6, 6); diffelastic.anisotropic builds isotropic, orthotropic and rotated tensors.
        `set_elasticity_field(None)` clears the field (and drops the warm start, so the object then solves exactly as the
        isotropic one).

        The tensors are kept by reference and validated at every assembly (shape, dtype, device, finite, symmetric to
        1e-10 max|C|, positive definite per tet); C is symmetrised before use.  get_vals() is then differentiable in the
        vertices, C (d lambda_i / dC_t is the symmetric strain Gram int_t eps_V eps_V^T of mode i) and density.  The mass
        entries round as with set_material_field.  Raises ValueError on a TrainableLinear material model or while a
        set_material_field field is set: both would define the stiffness."""
        if C is None:
            self.elasticity_field = None
            self._warm = []
        else:
            if isinstance(self.material_model, TrainableLinear):
                raise ValueError("set_elasticity_field: the material model is TrainableLinear, whose global (E, nu) logits "
                                 "would compete with a per-tet tensor; build the object with FixedLinear")
            if self.material_field is not None:
                raise ValueError("set_elasticity_field: a material field is set and both define the stiffness; clear it "
                                 "first (set_material_field(None))")
            check_elasticity_field(self.deform.num_tets, self.deform.device, C, density)
            self.elasticity_field = (C, density)
        self._q = None
        for key in ("_stiff_coo", "_mass_coo"):
            self.__dict__.pop(key, None)
        if self._Kval is not None:
            self._assemble(self._density_used)

    # ------------------------------------------------------------------ elastic supports
    def set_supports(self, faces, normal=None, tangential=None):
        """Rest the object on elastic supports: a Winkler spring bed on the boundary faces of the boolean mask `faces` over
        the rows of surface(), with normal and tangential stiffness per unit area (N/m^3; see supports.pad_stiffness for a
        pad of given material and thickness).  normal / tangential are floats or (S,) fp32 / fp64 CUDA tensors, one value
        per support face in ascending face order; tensors are kept by reference and validated again at every assembly
        (shape, device, finite, >= 0), so an optimiser may update them in place.  Face f adds int_f N_a N_b dA ((k_n - k_t)
        n n^T + k_t I) to K (native.support_km, fine and coarse level); M is unchanged.

        The object then has no rigid modes: `eigenvalues` / `U_hat` are the lowest mode_num pairs, the support's bounce and
        rock modes included, and get_vals() is differentiable in the two stiffness tensors as well.  Unless nodes are also
        clamped, the supports must hold every rigid motion (R^T K_s R positive definite, SUPPORT_RIGID_MARGIN); a flat face
        with k_t = 0, for instance, leaves the object free to slide and raises ValueError.  `set_supports(None)` removes
        them.  Either way the warm start and the cached operators are dropped."""
        if faces is None:
            self.supports = None
            self._sup = None
        else:
            srf, owner, local = self.surface()
            if not torch.is_tensor(faces) or faces.dtype != torch.bool or faces.shape != (srf.shape[0],):
                raise ValueError(f"set_supports: faces must be a boolean ({srf.shape[0]},) mask over the rows of surface()")
            if faces.device != srf.device:
                raise ValueError(f"set_supports: faces is on {faces.device}, the mesh on {srf.device}")
            sel = torch.nonzero(faces).squeeze(1)
            if sel.numel() == 0:
                raise ValueError("set_supports: no face selected; pass None to remove the supports")
            if normal is None or tangential is None:
                raise ValueError("set_supports: normal and tangential stiffnesses are required")
            prev = (self.supports, self._sup)
            self.supports = (faces, normal, tangential)
            self._sup = dict(fine=native.SupportFaces(self.deform.tets_i32, self.tetmesh.order, owner[sel], local[sel]),
                             corners=srf[sel])
            try:
                self._support_snapshot()
            except ValueError:
                self.supports, self._sup = prev
                raise
        self._warm = []
        self._q = None
        for key in ("_Kunit", "_stiff_coo", "_mass_coo"):
            self.__dict__.pop(key, None)
        if self._Kval is not None:
            self._assemble(self._density_used)

    def _support_faces_coarse(self):
        if "coarse" not in self._sup:
            fine = self._sup["fine"]
            self._sup["coarse"] = native.SupportFaces(self.deform.coarse.tets, 1, fine.owner, fine.local)
        return self._sup["coarse"]

    def _support_snapshot(self):
        """(k_n, k_t) fp64 (S,) of the supports, validated again; unless clamps are set, the rigid-motion check too."""
        _, normal, tangential = self.supports
        kn, kt = check_support_stiffness(self._sup["fine"].S, self.deform.device, normal, tangential)
        if self._fixed_u8 is None:
            p = self.tetmesh.vertices.detach().to(torch.float64)[self._sup["corners"]]
            ev = torch.linalg.eigvalsh(support_rigid_matrix(p[:, 0], p[:, 1], p[:, 2], kn, kt))
            if not bool(ev[0] > SUPPORT_RIGID_MARGIN * ev[-1]):
                raise ValueError("set_supports: the supports do not hold every rigid motion (the smallest eigenvalue of "
                                 f"R^T K_s R is {float(ev[0]):.3e}, the largest {float(ev[-1]):.3e}); support more faces, "
                                 "give them tangential stiffness, or clamp nodes")
        return kn, kt

    def support_energies(self):
        """(S, mode_num) fp64, no gradient: u_i^T K_s,f u_i of every support face f (ascending) and solved mode i for the
        stiffnesses of the last assembly; with element_energies()'s strain they sum to lambda_i."""
        if getattr(self, "U_hat", None) is None:
            raise RuntimeError("support_energies: run eigen_decomposition() first")
        if self._sup_used is None:
            raise RuntimeError("support_energies: the object has no supports (set_supports)")
        return native.support_energies(self._verts32, self.deform.tets_i32, self._sup["fine"], self._sup_used["kn"],
                                       self._sup_used["kt"], self.U_hat)

    def element_energies(self):
        """(strain, kinetic), each (T, mode_num) fp64, no gradient: u_i^T K_t u_i and u_i^T M_t u_i of every tet t and
        solved mode i (U_hat, M-normalised), for the material of the last assembly (field or not).  Summed over the tets
        they give u_i^T K u_i = lambda_i and u_i^T M u_i = 1."""
        if getattr(self, "U_hat", None) is None:
            raise RuntimeError("element_energies: run eigen_decomposition() first")
        d = self.deform
        if self._tensor_used is not None:
            t = self._tensor_used
            return native.element_energies_tensor(self._verts32, d.tets_i32, self.tetmesh.order, d.m32(), d.wsum, self.U_hat,
                                                  (t["C21"], t["rho"]))
        f = self._field_used
        if f is None:
            mu, lam = self._lame_used
            T = d.num_tets
            f = dict(mu=torch.full((T,), mu, dtype=torch.float64, device=d.device),
                     lam=torch.full((T,), lam, dtype=torch.float64, device=d.device),
                     rho=torch.full((T,), self._density_used, dtype=torch.float32, device=d.device))
        return native.element_energies(self._verts32, d.tets_i32, self.tetmesh.order, d.m32(), d.wsum, self.U_hat,
                                       (f["mu"], f["lam"], f["rho"]))

    @property
    def _n_rigid(self):
        """Rigid-body modes at the bottom of the spectrum: six free-free, none when clamped or on supports."""
        return 6 if self._fixed_u8 is None and self.supports is None else 0

    # ------------------------------------------------------------------ eigen-solve
    def eigen_decomposition(self):
        self._assemble(self.material_model.mat.density)
        self.eigen_decomposition_arpack()

    def _start_block(self, m, batch=0):
        """Start block of batch `batch` (n, m): the previous decomposition's Ritz block of this mesh when there is
        one (warm start; COPIED -- ds_lobpcg overwrites its block in place and earlier U_hat views / pending
        backward passes keep the old storage), else the six analytic rigid-body fields (unclamped objects) + seeded random
        columns."""
        n = self.deform.pattern.n
        dev = self.deform.device
        prev = self._warm[batch] if batch < len(self._warm) else None
        if prev is not None and prev.shape == (n, m):
            return prev.clone(), True
        g = torch.Generator(device=dev).manual_seed(batch)
        X = torch.randn(n, m, dtype=torch.float64, device=dev, generator=g)
        if batch == 0 and self._fixed_u8 is None:      # free or on supports: the rigid fields start the lowest modes
            p = self._verts32.double()
            p = p - p.mean(0, keepdim=True)
            X[:, :6] = 0
            for c in range(3):
                X[c::3, c] = 1
            X[0::3, 3], X[1::3, 3] = -p[:, 1], p[:, 0]
            X[1::3, 4], X[2::3, 4] = -p[:, 2], p[:, 1]
            X[2::3, 5], X[0::3, 5] = -p[:, 0], p[:, 2]
        return X, False

    def _has_slivers(self):
        """True when the flattest element of the mesh (smallest height over longest edge, from the corner nodes) is
        `sliver_ratio` times flatter than the median element."""
        if "_sliver" not in self.__dict__:
            with torch.no_grad():
                t = self.tetmesh.tets
                c = t[:, [0, 2, 4, 9]] if self.tetmesh.order == 2 else t
                p = self.tetmesh.vertices.detach()[c].double()
                e = p[:, [1, 2, 3, 2, 3, 3]] - p[:, [0, 0, 0, 1, 1, 2]]
                lmax = e.norm(dim=2).max(dim=1).values
                vol = torch.einsum("ij,ij->i", e[:, 0], torch.cross(e[:, 1], e[:, 2], dim=1)).abs() / 6
                q = vol / lmax ** 3
                self._sliver = bool(q.min() < self.sliver_ratio * q.median())
        return self._sliver

    #: pairs one eigensolver call has to converge at most (block 48 = 40 wanted + 8 guard columns); larger
    #: requests (geometry_train.py:147: mode_num = 64) are solved in batches with the converged vectors locked
    max_batch = 40

    @staticmethod
    def _block_for(need):
        return next((c for c in (16, 32, 48) if c >= need + min(4, c // 8)), None)

    def eigen_decomposition_arpack(self):
        """Lowest mode_num + 6 eigenpairs of K u = lambda M u, rigid six dropped (a clamped object or one on supports: the
        lowest mode_num pairs, see fix_nodes and set_supports).  The name is the
        reference's (diff_model.py:335-369: SciPy ARPACK shift-invert on the CPU); the solver is the
        device-resident LOBPCG of csrc/lobpcg.cu.  More pairs than one 48-column block holds are found in
        batches: every batch runs M-orthogonal to the pairs already converged (ds_lobpcg_opts.locked) and
        starts from the previous batch's guard columns."""
        k = self.mode_num
        nr = self._n_rigid
        need = k + nr
        pat = self.deform.pattern
        n_dof = pat.n if self._fixed_u8 is None else pat.n - 3 * self._n_fixed   # a block spans free dofs only
        if n_dof < 3 * 16 or n_dof < need + 16:
            raise ValueError(f"mesh too small for {k} modes (n={n_dof} free dofs)")
        deg = int(self.cheb_degree) or int(min(40, max(8, round(pat.n ** (1.0 / 3.0) / 3.0))))
        kw = {}
        coarse = self.deform.coarse if self.two_level else None
        if coarse is not None and 3 * coarse.n_nodes >= 3 * 48:
            # two-level p-multigrid preconditioner: P1 operator of the same mesh, same material
            mu, la = self._lame_used
            coarse.fixed = None if self._fixed_u8 is None else self._fixed_u8[coarse.corner_nodes].contiguous()
            sup = None if self._sup_used is None else (self._support_faces_coarse(), self._sup_used["kn"],
                                                       self._sup_used["kt"])
            if self._tensor_used is not None:       # coarse tet t is fine tet t: the same per-tet arrays
                t = self._tensor_used
                coarse.assemble(self._verts32, 0.0, 0.0, coarse.ctab, self.deform.m32(1), tensor=(t["C21"], t["rho"]),
                                supports=sup)
            elif self._field_used is None:
                coarse.assemble(self._verts32, mu, la, coarse.ctab, self.deform.coarse_mtab(self._density_used), supports=sup)
            else:       # coarse tet t is fine tet t: the same per-tet arrays
                f = self._field_used
                coarse.assemble(self._verts32, 0.0, 0.0, coarse.ctab, self.deform.m32(1), field=(f["mu"], f["lam"], f["rho"]),
                                supports=sup)
            # n_c^(1/3) scaling fits compact bodies; thin shells (the bowl fixture) need the floor: 37 -> 28 outer iterations
            cdeg = int(self.coarse_degree) or int(min(64, max(32, round((3 * coarse.n_nodes) ** (1.0 / 3.0) / 1.2))))
            cratio = float(self.coarse_ratio) or 0.4 * cdeg * cdeg
            kw = dict(coarse=coarse, smooth_steps=int(self.smooth_steps), smooth_ratio=float(self.smooth_ratio),
                      coarse_degree=cdeg, coarse_ratio=cratio, nested_tol=self.nested_tol, nested_degree=self.nested_degree)
        found_X, found_lam, warm, all_stats = [], [], [], []
        done, batch, guard = 0, 0, None
        while done < need:
            want = min(need - done, self.max_batch)
            m = self._block_for(want)
            while n_dof < 3 * m and m > 16:
                m -= 16
            if m < want:
                raise ValueError(f"mesh too small for {k} modes (n={n_dof} free dofs)")
            X, is_warm = self._start_block(m, batch)
            if guard is not None and not is_warm:
                gcols = min(guard.shape[1], m)
                X[:, :gcols] = guard[:, :gcols]            # approximate next modes left over from the previous batch
            locked = None
            if done:
                q = (done + 15) // 16 * 16
                locked = torch.zeros(pat.n, q, dtype=torch.float64, device=X.device)
                locked[:, :done] = torch.cat(found_X, dim=1)
            if kw:
                kw["nested"] = self.nested_start and not is_warm and batch == 0
            common = dict(nev=want, tol=self.eig_tol, n_rigid=nr if batch == 0 else 0,
                          coords=self._verts32 if self.morton else None, locked=locked, fixed=self._fixed_u8)
            stats = None
            if not (self.fp64_fallback and self._has_slivers()):
                try:
                    lam, res, stats = native.lobpcg(pat, self._Kval, self._Mblk, X, cheb_degree=deg, cheb_ratio=0.4 * deg * deg,
                                                    maxit=min(self.eig_maxit, self.eig_fast_maxit) if self.fp64_fallback
                                                    else self.eig_maxit, **common, **kw)
                except RuntimeError:
                    if not self.fp64_fallback:
                        raise
                    stats = None
                if stats is not None and stats["status"] != 0 and self.fp64_fallback:
                    fast_stats, stats = stats, None
                    if not bool(torch.isfinite(X).all()):
                        X, _ = self._start_block(m, batch)
            if stats is None:
                deg64 = int(self.cheb_degree) or int(min(40, max(12, round(pat.n ** (1.0 / 3.0) / 1.5))))
                lam, res, stats = native.lobpcg(pat, self._Kval, self._Mblk, X, cheb_degree=deg64, cheb_ratio=0.4 * deg64 * deg64,
                                                maxit=self.eig_maxit, precond_fp64=True, **common)
                stats["precond"] = "fp64"
            if stats["status"] != 0:
                raise RuntimeError(f"eigensolver did not converge (batch {batch}): {stats}, "
                                   f"max residual {float(res[:want].max()):.3e}")
            all_stats.append(stats)
            warm.append(X)
            found_X.append(X[:, :want])
            found_lam.append(lam[:want])
            guard = X[:, want:]
            if batch == 0:
                self.ritz_values = lam          # all block columns of the first batch (rigid modes, modes, guard columns)
            done += want
            batch += 1
        self._warm = warm
        self.eig_stats = all_stats[0] if len(all_stats) == 1 else dict(
            all_stats[0], batches=len(all_stats), iterations=sum(s["iterations"] for s in all_stats),
            spmm=sum(s["spmm"] for s in all_stats), per_batch=all_stats)
        if len(found_X) == 1:
            self._X = warm[0]                    # (n, m): wanted columns + guard columns
            self.U_hat_full = self._X[:, :need]
            lam_all = found_lam[0]
        else:
            lam_all, order = torch.sort(torch.cat(found_lam))
            self.U_hat_full = torch.cat(found_X, dim=1)[:, order].contiguous()
            self._X = self.U_hat_full
        self.eigenvalues = lam_all[nr:need].clone()
        self.U_hat = self.U_hat_full[:, nr:need]
        # all wanted columns zero-padded to a multiple of 16 for the SpMM of get_vals()
        if self._X.shape[1] % 16 == 0:
            self._Xpad = self._X
        else:
            self._Xpad = torch.zeros(pat.n, (need + 15) // 16 * 16, dtype=torch.float64, device=self._X.device)
            self._Xpad[:, :need] = self.U_hat_full
        self._q = None

    # ------------------------------------------------------------------ differentiable outputs
    def _material_forms(self):
        if self._q is None:
            d = self.deform
            self._q = native.eigval_quadforms_material(self._verts32, d.tets_i32, self.tetmesh.order,
                                                       d.mtab(self._density_used), d.wsum, self.U_hat)
        return self._q

    def get_undamped_freqs(self):
        """(mode_num, 1) fp32 undamped frequencies with gradient to the (E, nu) logits
        (diff_model.py:371-388)."""
        dev = self.deform.device
        predict = torch.zeros(self.mode_num, dtype=torch.float32, device=dev)
        predict += self.eigenvalues
        # with a material or tensor field the global (E, nu) are not parameters of K (and TrainableLinear is refused): no
        # term to add
        if self.task != "gt" and self._field_used is None and self._tensor_used is None:
            q_mu, q_la, q_m = self._material_forms()
            mu, lam = self.material_model.lame()
            mu, lam = torch.as_tensor(mu).to(dev), torch.as_tensor(lam).to(dev)
            # fp64 until the final cast (the reference does this sum in fp32, diff_model.py:382-386)
            add_term = (mu.double() * q_mu + lam.double() * q_la) - self.eigenvalues * q_m
            if self._sup_used is not None:      # lambda = u^T K u includes the spring bed
                add_term = add_term + self.support_energies().sum(0)
            predict = predict + add_term.float()
        return (torch.sqrt(predict) / 2 / np.pi).unsqueeze(1)

    def get_vals(self):
        """(mode_num, 1) fp32 eigenvalues, differentiable w.r.t. the vertex positions
        (diff_model.py:390-399), with a material or elasticity-tensor field w.r.t. its tensors, and on supports w.r.t. the
        normal and tangential stiffness tensors of set_supports."""
        vals = self._get_vals_volume()
        if self._sup_used is None:
            return vals
        _, normal, tangential = self.supports if self.supports is not None else (None, None, None)
        normal = normal if torch.is_tensor(normal) else None
        tangential = tangential if torch.is_tensor(tangential) else None
        return vals + _SupportTerm.apply(self.tetmesh.vertices, normal, tangential, self)

    def _get_vals_volume(self):
        if self._tensor_used is not None:
            C, density = self.elasticity_field if self.elasticity_field is not None else (self._tensor_used["C"], None)
            return _EigvalTensor.apply(self.tetmesh.vertices, C, density, self)
        if self._field_used is not None:
            youngs, poisson, density = self.material_field if self.material_field is not None else (None, None, None)
            return _EigvalField.apply(self.tetmesh.vertices, youngs, poisson, density, self)
        return _EigvalShape.apply(self.tetmesh.vertices, self)

    # ------------------------------------------------------------------ striking the object
    def _boundary(self):
        """(faces, owner, local) int32 of native.tet_boundary, cached per object."""
        if "_bnd" not in self.__dict__:
            d = self.deform
            self._bnd = native.tet_boundary(d.verts_f32(), d.tets_i32, self.tetmesh.order)
        return self._bnd

    def surface(self):
        """Boundary triangles of the tet mesh, cached: (faces (F, 3) int64 corner node ids into tetmesh.vertices, oriented
        outward; owner (F,) int64 tet; local (F,) int64 the tet corner opposite the face), in ascending order of the sorted
        corner triple (native.tet_boundary)."""
        if "_surface" not in self.__dict__:
            self._surface = tuple(x.long() for x in self._boundary())
        return self._surface

    def modal_gains(self, points, directions=None):
        """(P, mode_num) fp32 gains g[p, m] = d_p . u_m(x_p) of the mode_num modes of U_hat (the rigid six excluded): what
        a unit impulse at surface point x_p in direction d_p puts into each mass-normalised mode.  points (P, 3) are put
        on the surface first: x_p is the closest point of the nearest boundary face (native.mesh_sdf_nearest over the
        corner-node boundary faces; of faces at the same distance the lowest index) and is kept in
        `last_strike_points`.  directions (P, 3) default to the outward unit normal of that face; they are used as
        given (not normalised).

        Differentiable in `points` (along the surface: the normal component of the gradient is 0) and `directions`.
        The mode shapes and the mesh are constants here: no gradient reaches the vertices or the material through a
        gain.  Raises if eigen_decomposition() has not run."""
        if getattr(self, "U_hat", None) is None:
            raise RuntimeError("modal_gains: run eigen_decomposition() first")
        dev = self.deform.device
        points = points.reshape(-1, 3)
        if directions is not None:
            directions = directions.reshape(-1, 3)
        pts = points.detach().to(device=dev, dtype=torch.float32).contiguous()
        _, face = native.mesh_sdf_nearest(self._verts32, self.surface()[0], pts, want_face=True)
        return _ModalGains.apply(points, directions, self, face)

    def impulse_response(self, strike, sample_num, sr, pickup=None, strike_dir=None, pickup_dir=None, alpha=None,
                         beta=None):
        """(P, sample_num) fp32 displacement in metres per N s of impulse at the pickup point along pickup_dir, for a unit
        impulse at the strike point along strike_dir (directions default to the outward surface normal):

            y(t) = sum_m g_m(strike) g_m(pickup) / w_m exp(-c_m t) sin(w_m t),  c_m = (alpha + beta lambda_m) / 2,
            w_m = sqrt(lambda_m - c_m^2),

        sampled at t = (n + 1) / sr for n < sample_num (modal_synth's convention), with lambda = self.eigenvalues
        (detached) and Rayleigh damping alpha, beta (default: the material's).  pickup
        defaults to the strike point and direction (the driving-point response).  A mode with lambda_m <= c_m^2 is not
        oscillatory (over-damped) and gets amplitude 0.  Rendered by modal_synth; differentiable in the points, the
        directions, alpha and beta.  The product g_strike g_pickup makes the result independent of the sign of each
        eigenvector, and strike and pickup swap exactly."""
        dev = self.deform.device
        mat = self.material_model.mat

        def coef(x, default):
            x = default if x is None else x
            return (x if torch.is_tensor(x) else torch.tensor(float(x))).to(device=dev, dtype=torch.float64)

        a, b = coef(alpha, mat.alpha), coef(beta, mat.beta)
        lam = self.eigenvalues.detach()
        c = 0.5 * (a + b * lam)
        w2 = lam - c * c
        osc = w2 > 0
        omega = torch.sqrt(torch.where(osc, w2, torch.ones_like(w2)))
        if pickup is None:
            g_pick = g_strike = self.modal_gains(strike, strike_dir)
        else:
            g_pick = self.modal_gains(pickup, pickup_dir)
            g_strike = self.modal_gains(strike, strike_dir)
        amp = torch.where(osc, g_strike * g_pick / omega.float(), torch.zeros((), device=dev))
        return modal_synth(amp, c.float(), (omega / (2 * np.pi)).float(), int(sample_num), float(sr))
