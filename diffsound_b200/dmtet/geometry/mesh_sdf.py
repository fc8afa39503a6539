"""Differentiable signed distance from query points to a triangle mesh: `native.mesh_sdf_nearest` forward,
`native.mesh_sdf_backward` backward (csrc/sdf.cu).

For sdf(p) = s d with c = sum_k b_k v_k the closest point of the nearest face, u = (p - c) / d: d sdf / d p = s u and
d sdf / d v_k = -s b_k u for the corners of that face (the envelope theorem: the same formula in the face, edge and vertex
regions).  The sign (ray parity or winding number, `sign=`) is piecewise constant and has no gradient; where sdf == 0
both gradients are 0.  Where several faces are at exactly the same distance the lowest-index face is used: where their
closest points coincide (a shared edge or vertex) the gradient does not depend on the choice; on the medial axis, where
they differ, this is the subgradient of that face.
"""
import torch
from torch.autograd.function import once_differentiable

from ... import native


class _MeshSdf(torch.autograd.Function):
    @staticmethod
    def forward(ctx, verts, faces, points, brute_force, sign):
        v = verts.detach().to(torch.float32).contiguous()
        f = faces.detach().to(torch.int64).contiguous()
        p = points.detach().to(torch.float32).contiguous()
        sdf, face = native.mesh_sdf_nearest(v, f, p, brute_force=brute_force, sign=sign)
        ctx.save_for_backward(v, f, p, face, sdf)
        ctx.dtypes = (verts.dtype, points.dtype)
        ctx.mark_non_differentiable(face)
        return sdf, face

    @staticmethod
    @once_differentiable
    def backward(ctx, g, _g_face):
        v, f, p, face, sdf = ctx.saved_tensors
        want_v, _, want_p, _, _ = ctx.needs_input_grad
        if g is None or not (want_v or want_p):
            return None, None, None, None, None
        gv, gp = native.mesh_sdf_backward(v, f, p, face, sdf, g.to(torch.float32).contiguous(), want_verts=want_v,
                                          want_points=want_p)
        return (gv.to(ctx.dtypes[0]) if want_v else None), None, (gp.to(ctx.dtypes[1]) if want_p else None), None, None


def mesh_sdf(verts, faces, points, brute_force=False, sign="parity"):
    """Signed distance (P,) fp32 from points (P, 3) to the triangle mesh (verts (V, 3), faces (F, 3)), positive inside,
    differentiable with respect to `verts` and `points` (once); gradients come back in the inputs' dtypes.  All tensors
    on one CUDA device.  brute_force: every point against every face instead of the BVH (bitwise equal results).
    sign: "parity" (ray-crossing parity, for closed meshes that do not cross themselves) or "winding" (inside where the
    generalised winding number |w| >= 1/2, for open or self-intersecting meshes with consistently oriented faces); the
    distance, the nearest face and so the backward are the same for both."""
    native._sdf_sign(sign)
    sdf, _ = _MeshSdf.apply(verts, faces, points, bool(brute_force), sign)
    return sdf


def winding_number(verts, faces, points, brute_force=False):
    """Generalised winding number (P,) fp32 of the triangle mesh at points (native.mesh_winding_number; no gradient)."""
    return native.mesh_winding_number(verts.detach().to(torch.float32).contiguous(),
                                      faces.detach().to(torch.int64).contiguous(),
                                      points.detach().to(torch.float32).contiguous(), brute_force=brute_force)
