"""Thin torch-tensor wrappers over the C-ABI (include/diffsound_sm100.h).

torch is used only for device memory and streams; every function here ends in
exactly one call into libdiffsound_sm100.so on the current CUDA stream.  There
is no CPU path: CPU tensors raise.
"""
import ctypes as C

import torch

from . import _lib


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("diffsound_b200: expected a CUDA tensor (there is no CPU path)")
    if not t.is_contiguous():
        raise RuntimeError("diffsound_b200: tensor must be contiguous")
    return C.c_void_p(t.data_ptr())


def _pv(t):
    """pointer of a possibly strided 2-D row-major view (last stride 1)."""
    if not t.is_cuda:
        raise RuntimeError("diffsound_b200: expected a CUDA tensor (there is no CPU path)")
    if t.dim() != 2 or t.stride(1) != 1:
        raise RuntimeError("diffsound_b200: block must be a row-major 2-D view")
    return C.c_void_p(t.data_ptr()), t.stride(0)


class Workspace:
    """Owns a ds_workspace (device scratch arena)."""

    def __init__(self):
        lib = _lib.load()
        h = C.c_void_p()
        _lib.check(lib.ds_workspace_create(C.byref(h)), "ds_workspace_create")
        self._h = h

    @property
    def handle(self):
        return self._h

    def nbytes(self):
        return _lib.load().ds_workspace_bytes(self._h)

    def __del__(self):
        try:
            if self._h:
                _lib.load().ds_workspace_destroy(self._h)
                self._h = None
        except Exception:
            pass


_ws_cache = {}


def workspace(device=None):
    dev = torch.cuda.current_device() if device is None else torch.device(device).index
    if dev not in _ws_cache:
        with torch.cuda.device(dev):
            _ws_cache[dev] = Workspace()
    return _ws_cache[dev]


def unique_rows3(rows_f32):
    """(inverse, first) of the distinct rows of an (N, 3) fp32 array in ascending lexicographic order
    (ds_unique_rows3_*): what torch.unique(dim=0, return_inverse=True) + scatter(min) give the reference."""
    lib = _lib.load()
    assert rows_f32.dtype == torch.float32 and rows_f32.dim() == 2 and rows_f32.shape[1] == 3
    dev = rows_f32.device
    ws = workspace(dev)
    N = rows_f32.shape[0]
    if N == 0:
        e = torch.empty(0, dtype=torch.int64, device=dev)
        return e, e.clone()
    nu = C.c_int64(0)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_unique_rows3_count(ws.handle, _p(rows_f32), N, C.byref(nu), _stream()), "ds_unique_rows3_count")
        inverse = torch.empty(N, dtype=torch.int64, device=dev)
        first = torch.empty(int(nu.value), dtype=torch.int64, device=dev)
        _lib.check(lib.ds_unique_rows3_fill(ws.handle, _p(inverse), _p(first), _stream()), "ds_unique_rows3_fill")
    return inverse, first


class Pattern:
    """Block-CSR sparsity pattern of K and M plus per-slot contributor lists.  want_slot: also keep the element -> slot map
    (int32 per (tet, a, b)) that the tet-sequential assembly of quadratic meshes reads (default: quadratic meshes)."""

    def __init__(self, tets_i32, n_nodes, want_slot=None):
        lib = _lib.load()
        assert tets_i32.dtype == torch.int32 and tets_i32.is_cuda and tets_i32.is_contiguous()
        T, npe = tets_i32.shape
        dev = tets_i32.device
        self.device = dev
        self.T, self.npe, self.n_nodes = T, npe, int(n_nodes)
        ws = workspace(dev)
        nnzb = C.c_int64(0)
        with torch.cuda.device(dev):
            _lib.check(lib.ds_pattern_count(ws.handle, _p(tets_i32), T, npe, self.n_nodes, C.byref(nnzb), _stream()),
                       "ds_pattern_count")
            self.nnzb = int(nnzb.value)
            i32 = dict(dtype=torch.int32, device=dev)
            self.brow = torch.empty(self.n_nodes + 1, **i32)
            self.bcol = torch.empty(self.nnzb, **i32)
            self.contrib_ptr = torch.empty(self.nnzb + 1, **i32)
            self.contrib = torch.empty(T * npe * npe, **i32)
            if want_slot is None:
                want_slot = npe == 10
            self.slot = torch.empty(T * npe * npe, **i32) if want_slot else None
            _lib.check(lib.ds_pattern_fill(ws.handle, self.n_nodes, _p(self.brow), _p(self.bcol), _p(self.contrib_ptr),
                                           _p(self.contrib), _p(self.slot), _stream()), "ds_pattern_fill")
            # longest block row: sizes the shared-memory row image of the tet-sequential assembly
            self.max_deg = int((self.brow[1:] - self.brow[:-1]).max()) if want_slot else 0
        self._csr = None

    @property
    def nnz(self):
        return 9 * self.nnzb

    @property
    def n(self):
        return 3 * self.n_nodes

    def csr(self):
        """(crow, col) int64 -- the reference's coalesced (row, col) order."""
        if self._csr is None:
            lib = _lib.load()
            crow = torch.empty(self.n + 1, dtype=torch.int64, device=self.device)
            col = torch.empty(self.nnz, dtype=torch.int64, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(lib.ds_pattern_expand_csr(_p(self.brow), _p(self.bcol), self.n_nodes, self.nnzb, _p(crow),
                                                     _p(col), _stream()), "ds_pattern_expand_csr")
            self._csr = (crow, col)
        return self._csr

    def coo_indices(self):
        """(2, nnz) int64 like `stiff_matrix.indices()` of the reference."""
        crow, col = self.csr()
        rows = torch.repeat_interleave(torch.arange(self.n, device=self.device), crow[1:] - crow[:-1])
        return torch.stack([rows, col], dim=0)


def _check_field(field, T, dev):
    mu_t, lam_t, rho_t = field
    for name, t, dt in (("mu", mu_t, torch.float64), ("lam", lam_t, torch.float64), ("rho", rho_t, torch.float32)):
        if t.dtype != dt or t.shape != (T,) or t.device != dev or not t.is_contiguous():
            raise ValueError(f"material field: {name} must be a contiguous ({T},) {dt} tensor on {dev}")
    return _p(mu_t), _p(lam_t), _p(rho_t)


def _check_tensor(tensor, T, dev):
    C21, rho_t = tensor
    for name, t, shape, dt in (("C21", C21, (T, 21), torch.float64), ("rho", rho_t, (T,), torch.float32)):
        if t.dtype != dt or t.shape != shape or t.device != dev or not t.is_contiguous():
            raise ValueError(f"elasticity field: {name} must be a contiguous {shape} {dt} tensor on {dev}")
    return _p(C21), _p(rho_t)


def assemble_km(verts_f32, tets_i32, order, pattern, mu, lam, ctab, mtab, Kval=None, Mblk=None, geom=None, kernel=None,
                field=None, tensor=None):
    """K (scalar-CSR value order of the reference) and M (one scalar per block) into the fixed pattern.  kernel: 'tets'
    (tet-sequential rows: quadratic meshes whose pattern carries the slot map and whose rows have <= 256 blocks), 'rows'
    (balanced contributor lists: everything else) or None = pick.
    field: (mu_t (T,) fp64, lam_t (T,) fp64, rho_t (T,) fp32) one material per tet (ds_assemble_km_field /
    ds_assemble_km_tets_field); mu and lam are then ignored and mtab is the fp32 unit-density mass table (npe, npe).
    tensor: (C21 (T, 21) fp64 packed Voigt elasticity matrices, rho_t (T,) fp32) one anisotropic material per tet
    (ds_assemble_km_tensor / ds_assemble_km_tets_tensor); mu, lam and mtab as for `field`."""
    lib = _lib.load()
    dev = verts_f32.device
    assert verts_f32.dtype == torch.float32 and tets_i32.dtype == torch.int32
    T = tets_i32.shape[0]
    f64 = dict(dtype=torch.float64, device=dev)
    if Kval is None:
        Kval = torch.empty(pattern.nnz, **f64)
    if Mblk is None:
        Mblk = torch.empty(pattern.nnzb, **f64)
    if geom is None:
        geom = torch.empty(T * 14, **f64)
    can_tets = order == 2 and getattr(pattern, "slot", None) is not None and 1 <= pattern.max_deg <= 256
    if kernel is None:
        kernel = "tets" if can_tets else "rows"
    if kernel == "tets":
        if not can_tets:
            raise ValueError("assemble_km(kernel='tets') needs a quadratic mesh, Pattern(want_slot=True) and rows of <= 256 blocks")
    if tensor is not None:
        assert field is None and mtab.dtype == torch.float32
        tp = _check_tensor(tensor, T, dev)
        with torch.cuda.device(dev):
            if kernel == "tets":
                _lib.check(lib.ds_assemble_km_tets_tensor(_p(verts_f32), _p(tets_i32), T, order, pattern.n_nodes, *tp, _p(ctab),
                                                          _p(mtab), _p(pattern.brow), _p(pattern.bcol), _p(pattern.contrib_ptr),
                                                          _p(pattern.contrib), _p(pattern.slot), pattern.max_deg, pattern.nnzb,
                                                          _p(geom), _p(Kval), _p(Mblk), _stream()), "ds_assemble_km_tets_tensor")
            else:
                _lib.check(lib.ds_assemble_km_tensor(_p(verts_f32), _p(tets_i32), T, order, pattern.n_nodes, *tp, _p(ctab),
                                                     _p(mtab), _p(pattern.brow), _p(pattern.bcol), _p(pattern.contrib_ptr),
                                                     _p(pattern.contrib), pattern.nnzb, _p(geom), _p(Kval), _p(Mblk),
                                                     _stream()), "ds_assemble_km_tensor")
        return Kval, Mblk
    if field is not None:
        assert mtab.dtype == torch.float32
        fp = _check_field(field, T, dev)
        with torch.cuda.device(dev):
            if kernel == "tets":
                _lib.check(lib.ds_assemble_km_tets_field(_p(verts_f32), _p(tets_i32), T, order, pattern.n_nodes, *fp, _p(ctab),
                                                         _p(mtab), _p(pattern.brow), _p(pattern.bcol), _p(pattern.contrib_ptr),
                                                         _p(pattern.contrib), _p(pattern.slot), pattern.max_deg, pattern.nnzb,
                                                         _p(geom), _p(Kval), _p(Mblk), _stream()), "ds_assemble_km_tets_field")
            else:
                _lib.check(lib.ds_assemble_km_field(_p(verts_f32), _p(tets_i32), T, order, pattern.n_nodes, *fp, _p(ctab),
                                                    _p(mtab), _p(pattern.brow), _p(pattern.bcol), _p(pattern.contrib_ptr),
                                                    _p(pattern.contrib), pattern.nnzb, _p(geom), _p(Kval), _p(Mblk),
                                                    _stream()), "ds_assemble_km_field")
        return Kval, Mblk
    if kernel == "tets":
        with torch.cuda.device(dev):
            _lib.check(lib.ds_assemble_km_tets(_p(verts_f32), _p(tets_i32), T, order, pattern.n_nodes, float(mu), float(lam),
                                               _p(ctab), _p(mtab), _p(pattern.brow), _p(pattern.bcol), _p(pattern.contrib_ptr),
                                               _p(pattern.contrib), _p(pattern.slot), pattern.max_deg, pattern.nnzb, _p(geom),
                                               _p(Kval), _p(Mblk), _stream()), "ds_assemble_km_tets")
        return Kval, Mblk
    with torch.cuda.device(dev):
        _lib.check(lib.ds_assemble_km(_p(verts_f32), _p(tets_i32), T, order, pattern.n_nodes, float(mu), float(lam),
                                      _p(ctab), _p(mtab), _p(pattern.brow), _p(pattern.bcol), _p(pattern.contrib_ptr),
                                      _p(pattern.contrib), pattern.nnzb, _p(geom), _p(Kval), _p(Mblk), _stream()),
                   "ds_assemble_km")
    return Kval, Mblk


def fix_nodes_km(pattern, fixed, Kval, Mblk=None):
    """Clamp the nodes of the uint8 (n_nodes,) CUDA mask `fixed` in K (and M) in place (ds_fix_nodes_km): every
    off-diagonal block that touches a fixed node becomes zero; the diagonal blocks and the pattern are kept."""
    lib = _lib.load()
    assert fixed.dtype == torch.uint8 and fixed.shape == (pattern.n_nodes,)
    assert Kval.numel() == pattern.nnz and (Mblk is None or Mblk.numel() == pattern.nnzb)
    with torch.cuda.device(Kval.device):
        _lib.check(lib.ds_fix_nodes_km(_p(pattern.brow), _p(pattern.bcol), pattern.n_nodes, pattern.nnzb, _p(fixed),
                                       _p(Kval), _p(Mblk), _stream()), "ds_fix_nodes_km")
    return Kval, Mblk


class SupportFaces:
    """Support faces of one mesh level for the ds_support_* kernels: owner / local int32 (S,) (the face opposite corner
    local[s] of tet owner[s]) and the node -> (face, face-local node) incidence of ds_support_km, built from `tets_i32`."""

    def __init__(self, tets_i32, order, owner, local):
        from .diffelastic.shape_func import CORNER_LOCAL, P2_NODES
        dev = tets_i32.device
        self.order = int(order)
        self.owner = owner.to(device=dev, dtype=torch.int32).contiguous()
        self.local = local.to(device=dev, dtype=torch.int32).contiguous()
        self.S = int(self.owner.numel())
        # face-local nodes of the face opposite corner f: corners j != f, then (P2) the mid-edge nodes off corner f
        rows = []
        for f in range(4):
            r = [CORNER_LOCAL[self.order][j] for j in range(4) if j != f]
            if self.order == 2:
                r += [a for a, (l, m) in enumerate(P2_NODES) if l != m and f not in (l, m)]
            rows.append(r)
        tab = torch.tensor(rows, dtype=torch.int64, device=dev)
        nodes = tets_i32.long()[self.owner.long()[:, None], tab[self.local.long()]]          # (S, nf)
        nf = nodes.shape[1]
        ent = torch.arange(self.S * nf, device=dev)
        code = (ent // nf) * 8 + ent % nf
        order_ = torch.argsort(nodes.reshape(-1) * (8 * self.S) + code)
        flat = nodes.reshape(-1)[order_]
        self.inc_node, counts = torch.unique_consecutive(flat, return_counts=True)
        self.inc_node = self.inc_node.to(torch.int32).contiguous()
        self.inc_ptr = torch.zeros(counts.numel() + 1, dtype=torch.int32, device=dev)
        self.inc_ptr[1:] = torch.cumsum(counts, 0).to(torch.int32)
        self.inc = code[order_].to(torch.int32).contiguous()
        self.R = int(self.inc_node.numel())
        self.nodes = nodes


def _check_stiffness(k, S, dev):
    if k.dtype != torch.float64 or k.shape != (S,) or k.device != dev or not k.is_contiguous():
        raise ValueError(f"supports: stiffness must be a contiguous ({S},) float64 tensor on {dev}")
    return _p(k)


def support_km(verts_f32, tets_i32, pattern, faces, kn, kt, Kval):
    """Add the spring bed of SupportFaces `faces` with per-face stiffnesses kn, kt (S,) fp64 to Kval in place
    (ds_support_km)."""
    lib = _lib.load()
    dev = Kval.device
    assert Kval.numel() == pattern.nnz and faces.order in (1, 2)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_support_km(_p(verts_f32), _p(tets_i32), tets_i32.shape[0], faces.order, pattern.n_nodes,
                                     _p(faces.owner), _p(faces.local), faces.S, _check_stiffness(kn, faces.S, dev),
                                     _check_stiffness(kt, faces.S, dev), _p(faces.inc_node), _p(faces.inc_ptr),
                                     _p(faces.inc), faces.R, _p(pattern.brow), _p(pattern.bcol),
                                     _p(getattr(pattern, "slot", None)), pattern.nnzb, _p(Kval), _stream()), "ds_support_km")
    return Kval


def support_grad(verts_f32, tets_i32, faces, kn, kt, U, g, want_verts=True):
    """Gradient of sum_i g_i u_i^T K_s u_i (ds_support_grad): ((S, 2) fp64 to (kn, kt), (n_nodes, 3) fp64 to the node
    positions or None).  U (n, k) fp64 row-major view; g (k,) fp64."""
    lib = _lib.load()
    dev = verts_f32.device
    up, ldu = _pv(U)
    k = U.shape[1]
    assert g.dtype == torch.float64 and g.numel() == k
    n_nodes = verts_f32.shape[0]
    scratch = torch.empty(faces.S * 9, dtype=torch.float64, device=dev)
    gk = torch.empty(faces.S, 2, dtype=torch.float64, device=dev)
    gv = torch.empty(n_nodes, 3, dtype=torch.float64, device=dev) if want_verts else None
    with torch.cuda.device(dev):
        _lib.check(lib.ds_support_grad(_p(verts_f32), _p(tets_i32), tets_i32.shape[0], faces.order, n_nodes, _p(faces.owner),
                                       _p(faces.local), faces.S, _check_stiffness(kn, faces.S, dev),
                                       _check_stiffness(kt, faces.S, dev), up, ldu, k, _p(g.contiguous()),
                                       _p(faces.inc_node), _p(faces.inc_ptr), _p(faces.inc), faces.R, _p(scratch), _p(gk),
                                       _p(gv), _stream()), "ds_support_grad")
    return gk, gv


def support_energies(verts_f32, tets_i32, faces, kn, kt, U):
    """(S, k) fp64 u_i^T K_s,f u_i of every support face and mode (ds_support_energies)."""
    lib = _lib.load()
    dev = verts_f32.device
    up, ldu = _pv(U)
    k = U.shape[1]
    out = torch.empty(faces.S, k, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_support_energies(_p(verts_f32), _p(tets_i32), tets_i32.shape[0], faces.order, verts_f32.shape[0],
                                           _p(faces.owner), _p(faces.local), faces.S, _check_stiffness(kn, faces.S, dev),
                                           _check_stiffness(kt, faces.S, dev), up, ldu, k, _p(out), _stream()),
                   "ds_support_energies")
    return out


def mass_expand(pattern, Mblk):
    lib = _lib.load()
    Mval = torch.empty(pattern.nnz, dtype=torch.float64, device=Mblk.device)
    with torch.cuda.device(Mblk.device):
        _lib.check(lib.ds_mass_expand(_p(pattern.brow), pattern.n_nodes, pattern.nnzb, _p(Mblk), _p(Mval), _stream()),
                   "ds_mass_expand")
    return Mval


def assemble_mass_coo(vertices, tets, values, rows, cols, element_mm, density, order):
    """Same argument order as the reference's `assemble_mass_matrix` export."""
    lib = _lib.load()
    vnum = {1: 4, 2: 10, 3: 20}.get(order, 4)   # an invalid order is rejected by the library
    T = tets.numel() // vnum
    with torch.cuda.device(vertices.device):
        _lib.check(lib.ds_assemble_mass_coo(_p(vertices), _p(tets), T, order, _p(element_mm), float(density),
                                            _p(values), _p(rows), _p(cols), _stream()), "ds_assemble_mass_coo")


def spmm(pattern, Kval, Mblk, X, shift=0.0, alpha=1.0, beta=0.0, Y0=None, out=None):
    """out = alpha (K + shift M) X + beta Y0  (X: (n, ncols) fp64 row-major view)."""
    lib = _lib.load()
    xp, ldx = _pv(X)
    ncols = X.shape[1]
    if out is None:
        out = torch.empty(X.shape[0], ncols, dtype=torch.float64, device=X.device)
    yp, ldy = _pv(out)
    y0p, ldy0 = (None, 0) if Y0 is None else _pv(Y0)
    with torch.cuda.device(X.device):
        _lib.check(lib.ds_spmm_km(_p(pattern.brow), _p(pattern.bcol), pattern.n_nodes, _p(Kval), _p(Mblk), float(shift),
                                  xp, ldx, ncols, float(alpha), float(beta), y0p, ldy0, yp, ldy, _stream()),
                   "ds_spmm_km")
    return out


def spmm_k_and_m(pattern, Kval, Mblk, X, YK=None, YM=None):
    lib = _lib.load()
    xp, ldx = _pv(X)
    ncols = X.shape[1]
    if YK is None:
        YK = torch.empty_like(X, memory_format=torch.contiguous_format)
    if YM is None:
        YM = torch.empty_like(X, memory_format=torch.contiguous_format)
    kp, ldk = _pv(YK)
    mp, ldm = _pv(YM)
    with torch.cuda.device(X.device):
        _lib.check(lib.ds_spmm_k_and_m(_p(pattern.brow), _p(pattern.bcol), pattern.n_nodes, _p(Kval), _p(Mblk), xp, ldx,
                                       ncols, kp, ldk, mp, ldm, _stream()), "ds_spmm_k_and_m")
    return YK, YM


def gram(A, B, out=None):
    """A^T B for row-major (n, p), (n, q) fp64 blocks."""
    lib = _lib.load()
    ap, lda = _pv(A)
    bp, ldb = _pv(B)
    p, q = A.shape[1], B.shape[1]
    if out is None:
        out = torch.empty(p, q, dtype=torch.float64, device=A.device)
    gp, ldg = _pv(out)
    scratch = torch.empty(lib.ds_gram_scratch_elems(p, q), dtype=torch.float64, device=A.device)
    with torch.cuda.device(A.device):
        _lib.check(lib.ds_gram_f64(ap, lda, p, bp, ldb, q, A.shape[0], gp, ldg, _p(scratch), _stream()), "ds_gram_f64")
    return out


def gram_sym2(S, KS, MS, tiles, GK, GM):
    """GK = S^T KS, GM = S^T MS over the 8-column tiles `tiles` (ascending) of three (n, ld) fp64 blocks, ld <= 144,
    in one pass (ds_gram_sym2_f64).  Only the upper-triangle tiles of GK / GM (row-major, common stride) are written."""
    lib = _lib.load()
    assert S.shape == KS.shape == MS.shape and S.is_contiguous() and KS.is_contiguous() and MS.is_contiguous()
    assert GK.stride(0) == GM.stride(0) and GK.stride(1) == 1
    n, ld = S.shape
    scratch = torch.empty(lib.ds_gram_sym2_scratch_elems(), dtype=torch.float64, device=S.device)
    arr = (C.c_int * len(tiles))(*[int(t) for t in tiles])
    with torch.cuda.device(S.device):
        _lib.check(lib.ds_gram_sym2_f64(_p(S), _p(KS), _p(MS), ld, n, arr, len(tiles), C.c_void_p(GK.data_ptr()),
                                        C.c_void_p(GM.data_ptr()), GK.stride(0), _p(scratch), _stream()), "ds_gram_sym2_f64")


def rr_update(bufs, prow, m, C1, C2, q2):
    """Fused LOBPCG basis update (ds_rr_update_f64): for each wide buffer A (n x 3m, fp64) returns A_out with
    A_out[:, :m] = A[:, :prow] C1 and A_out[:, 2m:2m+q2] = A[:, m:prow] C2 (other columns zero)."""
    lib = _lib.load()
    outs = [torch.zeros_like(b) for b in bufs]
    ld = bufs[0].shape[1]
    assert C1.stride(0) == C2.stride(0) and C1.stride(1) == 1 and C2.stride(1) == 1
    with torch.cuda.device(bufs[0].device):
        _lib.check(lib.ds_rr_update_f64(_p(bufs[0]), _p(bufs[1]), _p(bufs[2]), ld, int(prow), int(m),
                                        C.c_void_p(C1.data_ptr()), C.c_void_p(C2.data_ptr()), int(q2), C1.stride(0),
                                        bufs[0].shape[0], _p(outs[0]), _p(outs[1]), _p(outs[2]), ld, _stream()),
                   "ds_rr_update_f64")
    return outs


def block_gemm(A, Cm, beta=0.0, out=None):
    """out = beta*out + A Cm, A (n, p), Cm (p, q)."""
    lib = _lib.load()
    ap, lda = _pv(A)
    cp, ldc = _pv(Cm)
    p, q = Cm.shape
    if out is None:
        out = torch.empty(A.shape[0], q, dtype=torch.float64, device=A.device)
        beta = 0.0
    yp, ldy = _pv(out)
    with torch.cuda.device(A.device):
        _lib.check(lib.ds_block_gemm_f64(ap, lda, p, cp, ldc, q, A.shape[0], float(beta), yp, ldy, _stream()),
                   "ds_block_gemm_f64")
    return out


def eigh_generalized(GK, GM, sigma):
    lib = _lib.load()
    N = GK.shape[0]
    dev = GK.device
    kp, ldg = _pv(GK)
    mp, ldg2 = _pv(GM)
    assert ldg == ldg2
    theta = torch.empty(N, dtype=torch.float64, device=dev)
    Cm = torch.empty(N, N, dtype=torch.float64, device=dev)
    scratch = torch.empty(lib.ds_eigh_scratch_elems(N), dtype=torch.float64, device=dev)
    info = torch.zeros(2, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_eigh_generalized_f64(kp, mp, N, ldg, float(sigma), _p(theta), _p(Cm), N, _p(scratch),
                                               _p(info), _stream()), "ds_eigh_generalized_f64")
    return theta, Cm, info


class CoarseLevel:
    """P1 level of a quadratic mesh for the two-level preconditioner (csrc/pmg.cu): corner numbering,
    coarse tets / vertices, prolongation parents and the gather lists of its transpose, plus the
    block pattern of the P1 operator.  Topology only; values come from `assemble_km(order=1)`."""

    def __init__(self, verts_f32, tets_i32):
        lib = _lib.load()
        assert tets_i32.dtype == torch.int32 and tets_i32.shape[1] == 10 and tets_i32.is_contiguous()
        dev = tets_i32.device
        T = tets_i32.shape[0]
        n_nodes = verts_f32.shape[0]
        i32 = dict(dtype=torch.int32, device=dev)
        ws = workspace(dev)
        self.cid = torch.empty(n_nodes, **i32)
        nc = C.c_int64(0)
        with torch.cuda.device(dev):
            _lib.check(lib.ds_pmg_coarse_count(ws.handle, _p(tets_i32), T, n_nodes, _p(self.cid), C.byref(nc), _stream()),
                       "ds_pmg_coarse_count")
            self.n_nodes = int(nc.value)
            self.tets = torch.empty(T, 4, **i32)
            self.verts = torch.empty(self.n_nodes, 3, dtype=torch.float32, device=dev)
            self.parents = torch.empty(2 * n_nodes, **i32)
            self.rptr = torch.empty(self.n_nodes + 1, **i32)
            self.rlist = torch.empty(2 * n_nodes, **i32)
            _lib.check(lib.ds_pmg_coarse_fill(ws.handle, _p(verts_f32), _p(tets_i32), T, n_nodes, _p(self.cid),
                                              self.n_nodes, _p(self.tets), _p(self.verts), _p(self.parents),
                                              _p(self.rptr), _p(self.rlist), _stream()), "ds_pmg_coarse_fill")
        self.n_fine_nodes = n_nodes
        self.pattern = Pattern(self.tets, self.n_nodes)
        self.corner_nodes = torch.nonzero(self.cid >= 0).squeeze(1)     # fine id of coarse node c, ascending
        self.Kval = self.Mblk = self.geom = None
        self.use_coords = True
        self.fixed = None           # uint8 (n_nodes,) clamped corner nodes, applied after every assemble()

    def assemble(self, verts_f32, mu, lam, ctab1, mtab1, field=None, tensor=None, supports=None):
        """P1 stiffness (and mass) on the corner nodes at the current vertex positions, clamped at `fixed` when set.
        field / tensor: the fine level's (mu_t, lam_t, rho_t) / (C21, rho_t) unchanged (coarse tet t is fine tet t; mtab1
        then the fp32 unit table), see assemble_km.  supports: (SupportFaces over self.tets, kn, kt), the spring bed added
        before the clamps (coarse tet t is fine tet t, so the fine level's owner / local name the same faces)."""
        self.verts = verts_f32[self.corner_nodes].contiguous()
        if self.geom is None:
            self.geom = torch.empty(self.tets.shape[0] * 14, dtype=torch.float64, device=self.tets.device)
        self.Kval, self.Mblk = assemble_km(self.verts, self.tets, 1, self.pattern, mu, lam, ctab1, mtab1,
                                           Kval=self.Kval, Mblk=self.Mblk, geom=self.geom, field=field, tensor=tensor)
        if supports is not None:
            faces, kn, kt = supports
            support_km(self.verts, self.tets, self.pattern, faces, kn, kt, self.Kval)
        if self.fixed is not None:
            fix_nodes_km(self.pattern, self.fixed, self.Kval, self.Mblk)

    def struct(self):
        assert self.Kval is not None, "CoarseLevel: assemble the P1 operator first"
        return _lib.PmgLevel(brow=self.pattern.brow.data_ptr(), bcol=self.pattern.bcol.data_ptr(),
                             n_nodes=self.n_nodes, nnzb=self.pattern.nnzb, Kval=self.Kval.data_ptr(),
                             Mblk=self.Mblk.data_ptr() if self.Mblk is not None else None,
                             parents=self.parents.data_ptr(), rptr=self.rptr.data_ptr(), rlist=self.rlist.data_ptr(),
                             coords=self.verts.data_ptr() if self.use_coords else None,
                             fixed=self.fixed.data_ptr() if self.fixed is not None else None)


def k32_pack(pattern, Kval, Mblk=None, shift=0.0):
    """FP32 block records + block-Jacobi inverses of K + shift M (ds_k32_pack)."""
    lib = _lib.load()
    dev = Kval.device
    rec = torch.empty((lib.ds_k32_record_bytes(pattern.nnzb) + 15) // 16 * 4, dtype=torch.int32, device=dev)
    invD = torch.empty(pattern.n_nodes * 9, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_k32_pack(_p(pattern.brow), _p(pattern.bcol), pattern.n_nodes, pattern.nnzb, _p(Kval),
                                   _p(Mblk), float(shift), _p(rec), _p(invD), _stream()), "ds_k32_pack")
    return rec, invD


def spmm32_chunks(pattern):
    """Row chunks of the SpMM grid (ds_spmm32_chunks), cached on the pattern."""
    ch = getattr(pattern, "_chunks32", None)
    if ch is None:
        lib = _lib.load()
        dev = pattern.brow.device
        with torch.cuda.device(dev):
            ch = torch.empty(lib.ds_spmm32_chunk_count(pattern.n_nodes) + 1, dtype=torch.int32, device=dev)
            _lib.check(lib.ds_spmm32_chunks(_p(pattern.brow), pattern.n_nodes, _p(ch), _stream()), "ds_spmm32_chunks")
        pattern._chunks32 = ch
    return ch


def spmm32(pattern, rec, X, mode=0, R=None, invD=None, Zprev=None, ab=0.0, cc=0.0, out=None):
    """mode 0: A X; 1: R - A X; 2: X + ab (X - Zprev) + cc invD (R - A X).  fp32 (n, ncols) contiguous."""
    lib = _lib.load()
    assert X.dtype == torch.float32 and X.is_contiguous()
    if out is None:
        out = torch.empty_like(X)
    with torch.cuda.device(X.device):
        _lib.check(lib.ds_spmm32(int(mode), _p(pattern.brow), _p(rec), pattern.n_nodes, X.shape[1], _p(X), _p(R),
                                 _p(invD), _p(Zprev), _p(out), float(ab), float(cc), _p(spmm32_chunks(pattern)),
                                 _stream()), "ds_spmm32")
    return out


def cheb32_solve(pattern, rec, invD, R, degree, lmax, ratio, persistent=True):
    """`degree` block-Jacobi Chebyshev steps towards A^-1 R from zero (ds_cheb32_solve); fp32 (n, ncols)."""
    lib = _lib.load()
    assert R.dtype == torch.float32 and R.is_contiguous()
    Za, Zb = torch.empty_like(R), torch.empty_like(R)
    which = C.c_int(0)
    with torch.cuda.device(R.device):
        _lib.check(lib.ds_cheb32_solve(_p(pattern.brow), _p(rec), _p(invD), pattern.n_nodes, pattern.nnzb, _p(R), R.shape[1],
                                       int(degree), float(lmax), float(ratio), int(bool(persistent)), _p(Za), _p(Zb),
                                       C.byref(which), _stream()), "ds_cheb32_solve")
    return Zb if which.value else Za


def pmg_restrict32(coarse, res):
    lib = _lib.load()
    rc = torch.empty(3 * coarse.n_nodes, res.shape[1], dtype=torch.float32, device=res.device)
    with torch.cuda.device(res.device):
        _lib.check(lib.ds_pmg_restrict32(_p(coarse.rptr), _p(coarse.rlist), coarse.n_nodes, _p(res), res.shape[1],
                                         _p(rc), _stream()), "ds_pmg_restrict32")
    return rc


def pmg_prolong_add32(coarse, zc, z):
    lib = _lib.load()
    with torch.cuda.device(z.device):
        _lib.check(lib.ds_pmg_prolong_add32(_p(coarse.parents), coarse.n_fine_nodes, _p(zc), z.shape[1], _p(z),
                                            _stream()), "ds_pmg_prolong_add32")
    return z


def lobpcg(pattern, Kval, Mblk, X, nev, tol=1e-4, maxit=200, cheb_degree=8, sigma=0.0, cheb_ratio=30.0, n_rigid=6,
           verbose=0, coarse=None, smooth_steps=3, smooth_ratio=8.0, coarse_degree=20, coarse_ratio=160.0, nested=True,
           nested_tol=3e-2, nested_degree=0, coords=None, locked=None, ortho_w=False, precond_fp64=False, fixed=None):
    """Lowest `nev` pairs of K u = lam M u from the start block X (n, m) fp64 (overwritten with the
    M-orthonormal Ritz vectors).  `coarse`: a CoarseLevel with assembled Kval -> two-level
    preconditioner.  `locked`: (n, q) fp64 contiguous, q a multiple of 16 -- M-orthonormal eigenvectors
    found by earlier calls; the iteration stays M-orthogonal to them and returns the next lowest pairs.
    `fixed`: uint8 (n_nodes,) clamped nodes (K, M constrained by fix_nodes_km, n_rigid = 0); the Ritz vectors are
    exactly zero on their rows.  The coarse level's own mask is `coarse.fixed`.
    Returns (lam (m,), resid (m,), stats dict)."""
    lib = _lib.load()
    assert X.dtype == torch.float64 and X.is_contiguous()
    n, m = X.shape
    dev = X.device
    lam = torch.empty(m, dtype=torch.float64, device=dev)
    res = torch.empty(m, dtype=torch.float64, device=dev)
    opts = _lib.LobpcgOpts(nev=int(nev), maxit=int(maxit), cheb_degree=int(cheb_degree), tol=float(tol),
                           sigma=float(sigma), cheb_ratio=float(cheb_ratio), n_rigid=int(n_rigid), verbose=int(verbose),
                           smooth_steps=int(smooth_steps), coarse_degree=int(coarse_degree),
                           smooth_ratio=float(smooth_ratio), coarse_ratio=float(coarse_ratio),
                           nested=int(bool(nested) and coarse is not None), nested_tol=float(nested_tol),
                           nested_degree=int(nested_degree), coords=None, locked=None, n_locked=0,
                           ortho_w=int(bool(ortho_w)), precond_fp64=int(bool(precond_fp64)))
    if locked is not None:
        assert locked.dtype == torch.float64 and locked.is_contiguous() and locked.shape[0] == n
        assert locked.shape[1] % 16 == 0 and locked.is_cuda
        opts.locked = locked.data_ptr()
        opts.n_locked = locked.shape[1]
    if coords is not None:
        assert coords.dtype == torch.float32 and coords.is_contiguous() and coords.shape == (pattern.n_nodes, 3)
        opts.coords = coords.data_ptr()
    if fixed is not None:
        assert fixed.dtype == torch.uint8 and fixed.is_cuda and fixed.shape == (pattern.n_nodes,)
        opts.fixed = fixed.data_ptr()
    stats = (C.c_int64 * 12)()
    ws = workspace(dev)
    if coarse is not None:
        coarse.use_coords = coords is not None
    lvl = coarse.struct() if coarse is not None else None
    with torch.cuda.device(dev):
        _lib.check(lib.ds_lobpcg(ws.handle, _p(pattern.brow), _p(pattern.bcol), pattern.n_nodes, _p(Kval), _p(Mblk),
                                 C.byref(lvl) if lvl is not None else None, _p(X), m, C.byref(opts), _p(lam), _p(res),
                                 stats, _stream()), "ds_lobpcg")
    return lam, res, dict(iterations=int(stats[0]), converged=int(stats[1]), spmm=int(stats[2]), status=int(stats[3]),
                          cheb_steps=int(stats[4]), cheb_cols_avg=(stats[5] / stats[4] if stats[4] else 0.0),
                          coarse_steps=int(stats[6]), coarse_cols_avg=(stats[7] / stats[6] if stats[6] else 0.0),
                          two_level=coarse is not None, nested_iterations=int(stats[8]), nested_status=int(stats[9]),
                          lmax_fine=stats[10] * 1e-9, lmax_coarse=stats[11] * 1e-9)


def corner_incidence(tets_i32, order, n_nodes):
    """node -> (tet*4 + corner) incidence lists (inc_ptr (n_nodes+1,), inc (4T,)) int32."""
    lib = _lib.load()
    T, npe = tets_i32.shape
    dev = tets_i32.device
    inc_ptr = torch.empty(n_nodes + 1, dtype=torch.int32, device=dev)
    inc = torch.empty(4 * T, dtype=torch.int32, device=dev)
    ws = workspace(dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_corner_incidence(ws.handle, _p(tets_i32), T, npe, order, n_nodes, _p(inc_ptr), _p(inc),
                                           _stream()), "ds_corner_incidence")
    return inc_ptr, inc


def eigval_grad_shape(verts_f32, tets_i32, order, mu, lam_lame, ctab, mtab, U, lam, g, inc_ptr, inc, tet_grad=None):
    """d/d(verts) sum_i g_i (u_i^T K u_i - lam_i u_i^T M u_i) -> (n_nodes, 3) fp32.
    U: (n, k) fp64 row-major view; lam, g: (k,) fp64."""
    lib = _lib.load()
    dev = verts_f32.device
    T = tets_i32.shape[0]
    n_nodes = verts_f32.shape[0]
    up, ldu = _pv(U)
    k = U.shape[1]
    assert lam.dtype == torch.float64 and g.dtype == torch.float64 and lam.numel() == k and g.numel() == k
    if tet_grad is None:
        tet_grad = torch.empty(T * 12, dtype=torch.float64, device=dev)
    out = torch.empty(n_nodes, 3, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_eigval_grad_shape(_p(verts_f32), _p(tets_i32), T, order, n_nodes, float(mu), float(lam_lame),
                                            _p(ctab), _p(mtab), up, ldu, k, _p(lam.contiguous()), _p(g.contiguous()),
                                            _p(inc_ptr), _p(inc), _p(tet_grad), _p(out), _stream()),
                   "ds_eigval_grad_shape")
    return out


def eigval_grad_shape_field(verts_f32, tets_i32, order, field, ctab, mtab1, U, lam, g, inc_ptr, inc, tet_grad=None):
    """eigval_grad_shape with one material per tet (ds_eigval_grad_shape_field): field = (mu_t, lam_t, rho_t) as in
    assemble_km, mtab1 the unit-density table promoted to fp64.  -> (n_nodes, 3) fp32."""
    lib = _lib.load()
    dev = verts_f32.device
    T = tets_i32.shape[0]
    n_nodes = verts_f32.shape[0]
    up, ldu = _pv(U)
    k = U.shape[1]
    assert lam.dtype == torch.float64 and g.dtype == torch.float64 and lam.numel() == k and g.numel() == k
    fp = _check_field(field, T, dev)
    if tet_grad is None:
        tet_grad = torch.empty(T * 12, dtype=torch.float64, device=dev)
    out = torch.empty(n_nodes, 3, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_eigval_grad_shape_field(_p(verts_f32), _p(tets_i32), T, order, n_nodes, *fp, _p(ctab), _p(mtab1),
                                                  up, ldu, k, _p(lam.contiguous()), _p(g.contiguous()), _p(inc_ptr), _p(inc),
                                                  _p(tet_grad), _p(out), _stream()), "ds_eigval_grad_shape_field")
    return out


def material_field_grad(verts_f32, tets_i32, order, m32, wsum, U, lam, g):
    """(T, 3) fp64 per-tet (sum_i g_i u_i^T K_mu,t u_i, sum_i g_i u_i^T K_lam,t u_i, -sum_i g_i lam_i u_i^T Mhat_t u_i)
    (ds_material_field_grad): the gradient of sum_i g_i lambda_i w.r.t. (mu_t, lam_t, rho_t).  m32: fp32 unit-density
    mass table; U (n, k) fp64 row-major view, read in place; lam, g (k,) fp64."""
    lib = _lib.load()
    dev = verts_f32.device
    T = tets_i32.shape[0]
    up, ldu = _pv(U)
    k = U.shape[1]
    assert m32.dtype == torch.float32 and lam.dtype == torch.float64 and g.dtype == torch.float64
    assert lam.numel() == k and g.numel() == k
    out = torch.empty(T, 3, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_material_field_grad(_p(verts_f32), _p(tets_i32), T, order, _p(m32), float(wsum), up, ldu, k,
                                              _p(lam.contiguous()), _p(g.contiguous()), _p(out), _stream()),
                   "ds_material_field_grad")
    return out


def element_energies(verts_f32, tets_i32, order, m32, wsum, U, field):
    """(strain, kinetic), each (T, k) fp64: u_i^T K_t u_i and u_i^T M_t u_i of every tet t and mode i (ds_element_energies);
    field = (mu_t, lam_t, rho_t) as in assemble_km."""
    lib = _lib.load()
    dev = verts_f32.device
    T = tets_i32.shape[0]
    up, ldu = _pv(U)
    k = U.shape[1]
    assert m32.dtype == torch.float32
    fp = _check_field(field, T, dev)
    strain = torch.empty(T, k, dtype=torch.float64, device=dev)
    kinetic = torch.empty(T, k, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_element_energies(_p(verts_f32), _p(tets_i32), T, order, _p(m32), float(wsum), up, ldu, k, *fp,
                                           _p(strain), _p(kinetic), _stream()), "ds_element_energies")
    return strain, kinetic


def eigval_grad_shape_tensor(verts_f32, tets_i32, order, tensor, ctab, mtab1, U, lam, g, inc_ptr, inc, tet_grad=None):
    """eigval_grad_shape with one elasticity tensor per tet (ds_eigval_grad_shape_tensor): tensor = (C21, rho_t) as in
    assemble_km, mtab1 the unit-density table promoted to fp64.  -> (n_nodes, 3) fp32."""
    lib = _lib.load()
    dev = verts_f32.device
    T = tets_i32.shape[0]
    n_nodes = verts_f32.shape[0]
    up, ldu = _pv(U)
    k = U.shape[1]
    assert lam.dtype == torch.float64 and g.dtype == torch.float64 and lam.numel() == k and g.numel() == k
    tp = _check_tensor(tensor, T, dev)
    if tet_grad is None:
        tet_grad = torch.empty(T * 12, dtype=torch.float64, device=dev)
    out = torch.empty(n_nodes, 3, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_eigval_grad_shape_tensor(_p(verts_f32), _p(tets_i32), T, order, n_nodes, *tp, _p(ctab), _p(mtab1),
                                                   up, ldu, k, _p(lam.contiguous()), _p(g.contiguous()), _p(inc_ptr), _p(inc),
                                                   _p(tet_grad), _p(out), _stream()), "ds_eigval_grad_shape_tensor")
    return out


def elasticity_field_grad(verts_f32, tets_i32, order, m32, wsum, U, lam, g):
    """(gC (T, 21), grho (T,)) fp64 (ds_elasticity_field_grad): gC the packed upper triangle of sum_i g_i E_t,i, with
    E_t,i = int_t eps_V(u_i) eps_V(u_i)^T dV the strain Gram of mode i on tet t (d lambda_i / dC_t for a symmetric C), and
    grho = -sum_i g_i lam_i u_i^T Mhat_t u_i.  m32, U, lam, g as in material_field_grad."""
    lib = _lib.load()
    dev = verts_f32.device
    T = tets_i32.shape[0]
    up, ldu = _pv(U)
    k = U.shape[1]
    assert m32.dtype == torch.float32 and lam.dtype == torch.float64 and g.dtype == torch.float64
    assert lam.numel() == k and g.numel() == k
    gC = torch.empty(T, 21, dtype=torch.float64, device=dev)
    grho = torch.empty(T, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_elasticity_field_grad(_p(verts_f32), _p(tets_i32), T, order, _p(m32), float(wsum), up, ldu, k,
                                                _p(lam.contiguous()), _p(g.contiguous()), _p(gC), _p(grho), _stream()),
                   "ds_elasticity_field_grad")
    return gC, grho


def element_energies_tensor(verts_f32, tets_i32, order, m32, wsum, U, tensor):
    """(strain, kinetic), each (T, k) fp64 (ds_element_energies_tensor): <C_t, E_t,i> and u_i^T M_t u_i; tensor = (C21,
    rho_t) as in assemble_km."""
    lib = _lib.load()
    dev = verts_f32.device
    T = tets_i32.shape[0]
    up, ldu = _pv(U)
    k = U.shape[1]
    assert m32.dtype == torch.float32
    tp = _check_tensor(tensor, T, dev)
    strain = torch.empty(T, k, dtype=torch.float64, device=dev)
    kinetic = torch.empty(T, k, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_element_energies_tensor(_p(verts_f32), _p(tets_i32), T, order, _p(m32), float(wsum), up, ldu, k, *tp,
                                                  _p(strain), _p(kinetic), _stream()), "ds_element_energies_tensor")
    return strain, kinetic


def eigval_quadforms_material(verts_f32, tets_i32, order, mtab, wsum, U):
    """(q_mu, q_lam, q_m), each (k,) fp64: u_i^T K(1,0) u_i, u_i^T K(0,1) u_i, u_i^T M u_i."""
    lib = _lib.load()
    dev = verts_f32.device
    T = tets_i32.shape[0]
    up, ldu = _pv(U)
    k = U.shape[1]
    partial = torch.empty(lib.ds_quadform_scratch_elems(k), dtype=torch.float64, device=dev)
    out = torch.empty(3, k, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_eigval_quadforms_material(_p(verts_f32), _p(tets_i32), T, order, _p(mtab), float(wsum), up,
                                                    ldu, k, _p(partial), _p(out), _stream()),
                   "ds_eigval_quadforms_material")
    return out[0], out[1], out[2]


def modal_synth_fwd(amp, damp, freq, T, sr):
    """y (B, T) fp32 = sum_m amp[b,m] exp(-damp[m] tau) sin(2 pi freq[m] tau), tau = (t+1)/sr."""
    lib = _lib.load()
    B, k = amp.shape
    assert amp.dtype == damp.dtype == freq.dtype == torch.float32 and damp.numel() == k and freq.numel() == k
    y = torch.empty(B, T, dtype=torch.float32, device=amp.device)
    with torch.cuda.device(amp.device):
        _lib.check(lib.ds_modal_synth_fwd(_p(amp), _p(damp), _p(freq), B, k, T, float(sr), _p(y), None, _stream()),
                   "ds_modal_synth_fwd")
    return y


def modal_synth_bwd(amp, damp, freq, gy, sr):
    lib = _lib.load()
    B, k = amp.shape
    T = gy.shape[1]
    assert gy.dtype == torch.float32 and gy.shape[0] == B
    dev = amp.device
    gamp = torch.empty(B, k, dtype=torch.float32, device=dev)
    gdamp = torch.empty(k, dtype=torch.float32, device=dev)
    gfreq = torch.empty(k, dtype=torch.float32, device=dev)
    scratch = torch.empty(lib.ds_synth_scratch_elems(B, k, T), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_modal_synth_bwd(_p(amp), _p(damp), _p(freq), _p(gy), B, k, T, float(sr), _p(gamp), _p(gdamp),
                                          _p(gfreq), _p(scratch), _stream()), "ds_modal_synth_bwd")
    return gamp, gdamp, gfreq


def force_fir(x, force, reverse=False):
    """Causal FIR out[b,t] = sum_i force[b,i] x[b,t-i] (reverse: the adjoint sum_i force[b,i] x[b,t+i]); fp32 (B, T)."""
    lib = _lib.load()
    assert x.dtype == torch.float32 and force.dtype == torch.float32 and x.is_contiguous() and force.is_contiguous()
    B, T = x.shape
    assert force.shape[0] == B
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(lib.ds_force_fir(_p(x), _p(force), B, T, force.shape[1], int(bool(reverse)), _p(out), _stream()),
                   "ds_force_fir")
    return out


def filtered_noise_fwd(coeff, noise, T, gain=1.0):
    """DDSP filtered noise (ds_filtered_noise_fwd): coeff (B, F, C) raw parameters, noise (B, F, L) uniform(-1, 1)
    frames -> (B, T) fp32."""
    lib = _lib.load()
    assert coeff.dtype == noise.dtype == torch.float32 and coeff.is_contiguous() and noise.is_contiguous()
    B, F, Cn = coeff.shape
    L = noise.shape[2]
    assert noise.shape[:2] == (B, F)
    y = torch.empty(B, T, dtype=torch.float32, device=coeff.device)
    with torch.cuda.device(coeff.device):
        _lib.check(lib.ds_filtered_noise_fwd(_p(coeff), _p(noise), B, F, Cn, L, int(T), float(gain), _p(y), _stream()),
                   "ds_filtered_noise_fwd")
    return y


def filtered_noise_bwd(coeff, noise, gy, gain=1.0):
    lib = _lib.load()
    B, F, Cn = coeff.shape
    L = noise.shape[2]
    g = torch.empty_like(coeff)
    gy = gy.to(torch.float32).contiguous()
    with torch.cuda.device(coeff.device):
        _lib.check(lib.ds_filtered_noise_bwd(_p(coeff), _p(noise), _p(gy), B, F, Cn, L, gy.shape[1], float(gain), _p(g),
                                             _stream()), "ds_filtered_noise_bwd")
    return g


def stft_power(x, n_fft, hop):
    """Power spectrogram (B, n_fft/2+1, frames) fp32 of x (B, T): torchaudio Spectrogram(n_fft, hop) defaults."""
    lib = _lib.load()
    assert x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 2
    B, T = x.shape
    frames = lib.ds_stft_frames(T, int(hop))
    S = torch.empty(B, n_fft // 2 + 1, frames, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.ds_stft_power(_p(x), B, T, int(n_fft), int(hop), _p(S), _stream()), "ds_stft_power")
    return S


def mss_loss_fwd(x_pred, x_true, n_fft, hop, mode, alpha, eps):
    """One scale of the spectral loss (ds_mss_loss_fwd): returns (loss 0-dim fp64 device tensor, scratch)."""
    lib = _lib.load()
    assert x_pred.dtype == x_true.dtype == torch.float32 and x_pred.is_contiguous() and x_true.is_contiguous()
    assert x_pred.shape == x_true.shape and x_pred.dim() == 2
    B, T = x_pred.shape
    scratch = torch.empty(lib.ds_mss_scratch_elems(B, T, int(n_fft), int(hop)) + 2, dtype=torch.float32, device=x_pred.device)
    if scratch.data_ptr() % 8:
        scratch = scratch[1:]
    loss = torch.empty((), dtype=torch.float64, device=x_pred.device)
    with torch.cuda.device(x_pred.device):
        _lib.check(lib.ds_mss_loss_fwd(_p(x_pred), _p(x_true), B, T, int(n_fft), int(hop), int(mode), float(alpha),
                                       float(eps), C.c_void_p(scratch.data_ptr()), _p(loss), _stream()), "ds_mss_loss_fwd")
    return loss, scratch


def mss_loss_bwd(x_pred, x_true, n_fft, hop, mode, alpha, eps, loss, upstream, scratch, gx, accumulate):
    lib = _lib.load()
    B, T = x_pred.shape
    with torch.cuda.device(x_pred.device):
        _lib.check(lib.ds_mss_loss_bwd(_p(x_pred), _p(x_true), B, T, int(n_fft), int(hop), int(mode), float(alpha),
                                       float(eps), _p(loss), float(upstream), C.c_void_p(scratch.data_ptr()), _p(gx),
                                       int(bool(accumulate)), _stream()), "ds_mss_loss_bwd")
    return gx


class prof:
    """Per-kernel-class device timing (ds_prof_*): `with native.prof() as p: ...; p.read()`.
    classes: names of the classes to time (None: all) -- a short list keeps the event overhead out of a
    timed region."""

    def __init__(self, classes=None):
        self.classes = classes

    def __enter__(self):
        lib = _lib.load()
        lib.ds_prof_reset()
        if self.classes is None:
            lib.ds_prof_enable(1)
        else:
            names = [lib.ds_prof_class_name(c).decode() for c in range(lib.ds_prof_num_classes())]
            mask = 0
            for n in self.classes:
                mask |= 1 << names.index(n)
            lib.ds_prof_enable_classes(mask)
        return self

    def __exit__(self, *exc):
        _lib.load().ds_prof_enable(0)
        return False

    @staticmethod
    def read():
        lib = _lib.load()
        out = {}
        for c in range(lib.ds_prof_num_classes()):
            ms, cnt = C.c_double(0), C.c_int64(0)
            _lib.check(lib.ds_prof_read(c, C.byref(ms), C.byref(cnt)), "ds_prof_read")
            if cnt.value:
                by, fl = C.c_double(0), C.c_double(0)
                _lib.check(lib.ds_prof_read_work(c, C.byref(by), C.byref(fl)), "ds_prof_read_work")
                out[lib.ds_prof_class_name(c).decode()] = {"ms": ms.value, "count": cnt.value, "bytes": by.value,
                                                           "flops": fl.value}
        return out


def gram_strip(KW, MW, S):
    """(GsK, GsM) = (KW^T S, MW^T S): KW, MW (n, wa) row-major views, S (n, ncol <= 144) (ds_gram_strip_f64)."""
    lib = _lib.load()
    kp, ldw = _pv(KW)
    mp, ldw2 = _pv(MW)
    sp, lds = _pv(S)
    assert ldw == ldw2
    wa, ncol = KW.shape[1], S.shape[1]
    GsK = torch.zeros(wa, ncol, dtype=torch.float64, device=S.device)
    GsM = torch.zeros(wa, ncol, dtype=torch.float64, device=S.device)
    part = torch.empty(lib.ds_gram_strip_scratch_elems(), dtype=torch.float64, device=S.device)
    with torch.cuda.device(S.device):
        _lib.check(lib.ds_gram_strip_f64(kp, mp, ldw, wa, sp, lds, ncol, S.shape[0], _p(GsK), _p(GsM), ncol, _p(part), _stream()),
                   "ds_gram_strip_f64")
    return GsK, GsM


def rr_update2(bufs, m, wa, use_p, Cm):
    """Lean LOBPCG basis update (ds_rr_update2_f64) of the three (n, 3m) buffers; returns the new buffers (W slots zero)."""
    lib = _lib.load()
    outs = [torch.zeros_like(b) for b in bufs]
    ld = bufs[0].shape[1]
    assert Cm.stride(1) == 1
    with torch.cuda.device(bufs[0].device):
        _lib.check(lib.ds_rr_update2_f64(_p(bufs[0]), _p(bufs[1]), _p(bufs[2]), ld, int(m), int(wa), int(bool(use_p)),
                                         C.c_void_p(Cm.data_ptr()), Cm.stride(0), bufs[0].shape[0], _p(outs[0]), _p(outs[1]),
                                         _p(outs[2]), ld, _stream()), "ds_rr_update2_f64")
    return outs


def gram_algebra(GK, GM, Cm, theta, m):
    """Gram pair of [X' | - | P'] from the full symmetric Gram pair of [X | W | P] (ds_gram_algebra_f64)."""
    lib = _lib.load()
    assert GK.is_contiguous() and GM.is_contiguous() and Cm.stride(1) == 1
    GKn, GMn = torch.empty_like(GK), torch.empty_like(GM)
    scratch = torch.empty(lib.ds_gram_algebra_scratch_elems(), dtype=torch.float64, device=GK.device)
    with torch.cuda.device(GK.device):
        _lib.check(lib.ds_gram_algebra_f64(_p(GK), _p(GM), _p(GKn), _p(GMn), GK.shape[1], C.c_void_p(Cm.data_ptr()),
                                           Cm.stride(0), _p(theta), int(m), _p(scratch), _stream()), "ds_gram_algebra_f64")
    return GKn, GMn


def fp64_peak(mode, iters=4096, ctas_per_sm=2):
    """Register-resident FP64 throughput in TFLOP/s: mode 0 = DFMA, 1 = DMMA m8n8k4 (ds_fp64_peak)."""
    lib = _lib.load()
    scratch = torch.zeros(8, dtype=torch.float64, device="cuda")
    out = C.c_double(0)
    _lib.check(lib.ds_fp64_peak(int(mode), int(iters), int(ctas_per_sm), _p(scratch), C.byref(out), _stream()), "ds_fp64_peak")
    return out.value


def marching_tets(sdf, thickness, tets):
    """Topology of the hollow-shell tet mesh (ds_mtet_*): returns (interp_v (E, 2) int64, tets_out (Tn, 4) int64 over ids in
    [0, n_verts + E), faces (Nf, 3) int64 over edge-vertex ids)."""
    lib = _lib.load()
    assert sdf.dtype == torch.float32 and sdf.is_contiguous() and tets.dtype == torch.int64 and tets.is_contiguous()
    dev = sdf.device
    ws = workspace(dev)
    F, nv = tets.shape[0], sdf.shape[0]
    counts = (C.c_int64 * 7)()
    with torch.cuda.device(dev):
        _lib.check(lib.ds_mtet_count(ws.handle, _p(sdf), float(thickness), _p(tets), F, nv, counts, _stream()), "ds_mtet_count")
        n_int, n1, n3, n_in, n_tri = int(counts[2]), int(counts[3]), int(counts[4]), int(counts[5]), int(counts[6])
        interp_v = torch.empty(n_int, 2, dtype=torch.int64, device=dev)
        tets_out = torch.empty(n1 + 3 * n3 + n_in, 4, dtype=torch.int64, device=dev)
        faces = torch.empty(n_tri, 3, dtype=torch.int64, device=dev)
        _lib.check(lib.ds_mtet_fill(ws.handle, _p(tets), _p(interp_v), _p(tets_out), _p(faces), _stream()), "ds_mtet_fill")
    return interp_v, tets_out, faces


def compact_ids(ids, id_range):
    """(unique ascending, inverse) of an int64 id array with values in [0, id_range) (ds_compact_ids_*)."""
    lib = _lib.load()
    flat = ids.reshape(-1).contiguous()
    dev = ids.device
    ws = workspace(dev)
    nu = C.c_int64(0)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_compact_ids_count(ws.handle, _p(flat), flat.numel(), int(id_range), C.byref(nu), _stream()),
                   "ds_compact_ids_count")
        uniq = torch.empty(int(nu.value), dtype=torch.int64, device=dev)
        inv = torch.empty_like(flat)
        _lib.check(lib.ds_compact_ids_fill(ws.handle, _p(flat), _p(uniq), _p(inv), _stream()), "ds_compact_ids_fill")
    return uniq, inv.reshape(ids.shape)


def largest_tet_component(tets, n_verts):
    """Connected components of a tet mesh on the device (ds_tet_components_*): returns (n_components, kept_verts (old ids,
    ascending) int64, tets of the largest component renumbered (order kept) int64, labels int32 (n_verts,))."""
    lib = _lib.load()
    assert tets.dtype == torch.int64 and tets.is_contiguous()
    dev = tets.device
    ws = workspace(dev)
    labels = torch.empty(n_verts, dtype=torch.int32, device=dev)
    counts = (C.c_int64 * 3)()
    with torch.cuda.device(dev):
        _lib.check(lib.ds_tet_components_count(ws.handle, _p(tets), tets.shape[0], int(n_verts), _p(labels), counts, _stream()),
                   "ds_tet_components_count")
        kept = torch.empty(int(counts[1]), dtype=torch.int64, device=dev)
        tout = torch.empty(int(counts[2]), 4, dtype=torch.int64, device=dev)
        _lib.check(lib.ds_tet_components_fill(ws.handle, _p(tets), _p(kept), _p(tout), _stream()), "ds_tet_components_fill")
    return int(counts[0]), kept, tout, labels


def _sdf_sign(sign):
    if sign not in ("parity", "winding"):
        raise ValueError(f"sign must be 'parity' or 'winding', not {sign!r}")
    return sign == "winding"


def mesh_sdf(tri_verts, faces, points, brute_force=False, sign="parity"):
    """Signed distance from each query point to a triangle mesh (ds_mesh_sdf): positive inside, negative outside, 0 on the
    surface; the mesh is used in its own coordinates.  tri_verts (V, 3) fp32, faces (F, 3) int64, points (P, 3) fp32, all
    on one device; returns (P,) fp32.  brute_force: every point against every face instead of the BVH (the test
    reference; the outputs are bitwise equal).  sign: "parity" (ray-crossing parity: closed meshes that do not cross
    themselves, any face orientation) or "winding" (ds_mesh_sdf_winding: inside where the generalised winding number
    |w| >= 1/2; open, cracked and self-intersecting meshes whose faces are consistently oriented; same distances)."""
    lib = _lib.load()
    assert tri_verts.dtype == torch.float32 and faces.dtype == torch.int64 and points.dtype == torch.float32
    assert tri_verts.dim() == 2 and tri_verts.shape[1] == 3 and faces.dim() == 2 and faces.shape[1] == 3
    assert points.dim() == 2 and points.shape[1] == 3
    if _sdf_sign(sign):
        return mesh_sdf_nearest(tri_verts, faces, points, brute_force, sign, want_face=False)[0]
    dev = points.device
    ws = workspace(dev)
    out = torch.empty(points.shape[0], dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_mesh_sdf(ws.handle, _p(tri_verts), tri_verts.shape[0], _p(faces), faces.shape[0], _p(points),
                                   points.shape[0], int(bool(brute_force)), _p(out), _stream()), "ds_mesh_sdf")
    return out


def mesh_winding_number(tri_verts, faces, points, brute_force=False):
    """Generalised winding number of a triangle mesh at each query point (ds_mesh_winding_number): 1 inside and 0 outside
    a closed, outward-oriented surface, 2 where two overlap, smooth across holes.  Arguments as `mesh_sdf`; returns (P,)
    fp32.  brute_force: the exact fp64 sum over all faces; otherwise the BVH with far-field expansions, whose error is
    measured, not bounded (at most 0.024 on the test meshes; it grows with the face area packed inside a subtree)."""
    lib = _lib.load()
    _check_mesh(tri_verts, faces, points)
    dev = points.device
    ws = workspace(dev)
    out = torch.empty(points.shape[0], dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_mesh_winding_number(ws.handle, _p(tri_verts), tri_verts.shape[0], _p(faces), faces.shape[0],
                                              _p(points), points.shape[0], int(bool(brute_force)), _p(out), _stream()),
                   "ds_mesh_winding_number")
    return out


def _check_mesh(tri_verts, faces, points):
    assert tri_verts.dtype == torch.float32 and faces.dtype == torch.int64 and points.dtype == torch.float32
    assert tri_verts.dim() == 2 and tri_verts.shape[1] == 3 and faces.dim() == 2 and faces.shape[1] == 3
    assert points.dim() == 2 and points.shape[1] == 3


def mesh_sdf_nearest(tri_verts, faces, points, brute_force=False, sign="parity", want_face=True):
    """`mesh_sdf` and the nearest face of each point (ds_mesh_sdf_nearest, or ds_mesh_sdf_winding for sign="winding"):
    returns (sdf (P,) fp32, face (P,) int32, None when not want_face).  sdf is bitwise equal to `mesh_sdf` with the same
    sign; of faces at exactly the same distance, the lowest index (both modes and both signs)."""
    lib = _lib.load()
    _check_mesh(tri_verts, faces, points)
    winding = _sdf_sign(sign)
    dev = points.device
    ws = workspace(dev)
    out = torch.empty(points.shape[0], dtype=torch.float32, device=dev)
    face = torch.empty(points.shape[0], dtype=torch.int32, device=dev) if want_face or not winding else None
    fn = lib.ds_mesh_sdf_winding if winding else lib.ds_mesh_sdf_nearest
    name = "ds_mesh_sdf_winding" if winding else "ds_mesh_sdf_nearest"
    with torch.cuda.device(dev):
        _lib.check(fn(ws.handle, _p(tri_verts), tri_verts.shape[0], _p(faces), faces.shape[0], _p(points), points.shape[0],
                      int(bool(brute_force)), _p(out), _p(face), _stream()), name)
    return out, (face if want_face else None)


def mesh_sdf_backward(tri_verts, faces, points, face, sdf, grad_sdf, want_verts=True, want_points=True):
    """Gradient of `mesh_sdf` (ds_mesh_sdf_backward) given the (sdf, face) of `mesh_sdf_nearest` and the upstream
    gradient grad_sdf (P,) fp32: returns (grad_verts (V, 3) or None, grad_points (P, 3) or None), fp32, bitwise
    reproducible."""
    lib = _lib.load()
    _check_mesh(tri_verts, faces, points)
    assert face.dtype == torch.int32 and sdf.dtype == torch.float32 and grad_sdf.dtype == torch.float32
    dev = points.device
    ws = workspace(dev)
    gv = torch.empty(tri_verts.shape[0], 3, dtype=torch.float32, device=dev) if want_verts else None
    gp = torch.empty(points.shape[0], 3, dtype=torch.float32, device=dev) if want_points else None
    with torch.cuda.device(dev):
        _lib.check(lib.ds_mesh_sdf_backward(ws.handle, _p(tri_verts), tri_verts.shape[0], _p(faces), faces.shape[0],
                                            _p(points), points.shape[0], _p(face), _p(sdf), _p(grad_sdf), _p(gv), _p(gp),
                                            _stream()), "ds_mesh_sdf_backward")
    return gv, gp


def stuff_edges(signs, dims):
    """Crossing edges of a sign field on the body-centred cubic lattice of `dims` = (nx, ny, nz) cells
    (ds_stuff_edges_*; numbering in include/diffsound_sm100.h): returns (edge ids (C,) int64 ascending, end points
    (C, 2) int64, the cut parameter running from the first to the second).  signs (NV,) int8 in {-1, 0, 1}."""
    lib = _lib.load()
    assert signs.dtype == torch.int8 and signs.dim() == 1
    dev = signs.device
    ws = workspace(dev)
    nx, ny, nz = (int(d) for d in dims)
    n = C.c_int64(0)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_stuff_edges_count(ws.handle, _p(signs), nx, ny, nz, C.byref(n), _stream()), "ds_stuff_edges_count")
        edges = torch.empty(int(n.value), dtype=torch.int64, device=dev)
        ends = torch.empty(int(n.value), 2, dtype=torch.int64, device=dev)
        _lib.check(lib.ds_stuff_edges_fill(ws.handle, _p(signs), _p(edges), _p(ends), _stream()), "ds_stuff_edges_fill")
    return edges, ends


def stuff(signs, dims, origin, h, edges, t):
    """Isosurface stuffing (ds_stuff_*): warp the lattice onto the cut points t (C,) fp64 of the crossing edges (C,)
    int64 and emit the stencils.  Returns (tets (T, 4) int64 over global ids: lattice vertices, then cut point i as
    NV + i; positions (NV + C, 3) fp32 after warping; number of warped vertices)."""
    lib = _lib.load()
    assert signs.dtype == torch.int8 and edges.dtype == torch.int64 and t.dtype == torch.float64
    dev = signs.device
    ws = workspace(dev)
    nx, ny, nz = (int(d) for d in dims)
    o = (C.c_double * 3)(*(float(x) for x in origin))
    counts = (C.c_int64 * 2)()
    nv = (nx + 1) * (ny + 1) * (nz + 1) + nx * ny * nz
    with torch.cuda.device(dev):
        _lib.check(lib.ds_stuff_count(ws.handle, _p(signs), nx, ny, nz, o, float(h), _p(edges), _p(t), edges.shape[0],
                                      counts, _stream()), "ds_stuff_count")
        tets = torch.empty(int(counts[0]), 4, dtype=torch.int64, device=dev)
        pos = torch.empty(nv + edges.shape[0], 3, dtype=torch.float32, device=dev)
        _lib.check(lib.ds_stuff_fill(ws.handle, _p(signs), _p(edges), _p(t), _p(tets), _p(pos), _stream()), "ds_stuff_fill")
    return tets, pos, int(counts[1])


def tet_boundary(verts_f32, tets_i32, order):
    """Boundary triangles of a tet mesh (ds_tet_boundary_*): the faces that belong to exactly one tet, in ascending order
    of their sorted corner triple.  verts (n, 3) fp32, tets (T, npe) int32 (corner local nodes of shape_func.CORNER_LOCAL).
    Returns (faces (F, 3) int32 corner node ids oriented outward, owner (F,) int32 tet, local (F,) int32 the tet corner
    opposite the face); bitwise reproducible, independent of tet order and corner rotation."""
    lib = _lib.load()
    assert verts_f32.dtype == torch.float32 and tets_i32.dtype == torch.int32 and tets_i32.dim() == 2
    dev = verts_f32.device
    ws = workspace(dev)
    n = C.c_int64(0)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_tet_boundary_count(ws.handle, _p(verts_f32), verts_f32.shape[0], _p(tets_i32), tets_i32.shape[0],
                                             int(order), C.byref(n), _stream()), "ds_tet_boundary_count")
        F = int(n.value)
        faces = torch.empty(F, 3, dtype=torch.int32, device=dev)
        owner = torch.empty(F, dtype=torch.int32, device=dev)
        local = torch.empty(F, dtype=torch.int32, device=dev)
        _lib.check(lib.ds_tet_boundary_fill(ws.handle, _p(faces), _p(owner), _p(local), _stream()), "ds_tet_boundary_fill")
    return faces, owner, local


def _gains_args(verts_f32, tets_i32, order, boundary, points, face, dirs, U):
    faces, owner, local = boundary
    assert verts_f32.dtype == torch.float32 and tets_i32.dtype == torch.int32 and points.dtype == torch.float32
    assert faces.dtype == torch.int32 and owner.dtype == torch.int32 and local.dtype == torch.int32
    assert face.dtype == torch.int32 and U.dtype == torch.float64 and points.dim() == 2 and points.shape[1] == 3
    assert dirs is None or (dirs.dtype == torch.float32 and dirs.shape == points.shape)
    up, ldu = _pv(U)
    return (_p(verts_f32), verts_f32.shape[0], _p(tets_i32), tets_i32.shape[0], int(order), _p(faces), _p(owner), _p(local),
            faces.shape[0], _p(points), _p(face), _p(dirs), points.shape[0], up, ldu, U.shape[1])


def modal_gains(verts_f32, tets_i32, order, boundary, points, face, dirs, U):
    """Gains of the modes U (n_dofs, k) fp64 row-major view (read in place) at points (P, 3) fp32 put on their boundary
    faces face (P,) int32 of boundary = tet_boundary(...) (ds_modal_gains): g[p, m] = d_p . u_m(closest point), d_p =
    dirs[p] (P, 3) fp32 or, for dirs None, the outward unit normal of the face.  Returns (gains (P, k) fp32, closest
    points (P, 3) fp32)."""
    lib = _lib.load()
    args = _gains_args(verts_f32, tets_i32, order, boundary, points, face, dirs, U)
    dev = points.device
    ws = workspace(dev)
    g = torch.empty(points.shape[0], U.shape[1], dtype=torch.float32, device=dev)
    cp = torch.empty(points.shape[0], 3, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ds_modal_gains(ws.handle, *args, _p(g), _p(cp), _stream()), "ds_modal_gains")
    return g, cp


def modal_gains_backward(verts_f32, tets_i32, order, boundary, points, face, dirs, U, grad):
    """Gradient of `modal_gains` (ds_modal_gains_backward) given the upstream gradient (P, k) fp32: returns
    (grad_points (P, 3), grad_dirs (P, 3) or None when dirs is None), fp32, bitwise reproducible."""
    lib = _lib.load()
    args = _gains_args(verts_f32, tets_i32, order, boundary, points, face, dirs, U)
    assert grad.dtype == torch.float32 and grad.shape == (points.shape[0], U.shape[1])
    dev = points.device
    ws = workspace(dev)
    gp = torch.empty(points.shape[0], 3, dtype=torch.float32, device=dev)
    gd = torch.empty(points.shape[0], 3, dtype=torch.float32, device=dev) if dirs is not None else None
    with torch.cuda.device(dev):
        _lib.check(lib.ds_modal_gains_backward(ws.handle, *args, _p(grad), _p(gp), _p(gd), _stream()),
                   "ds_modal_gains_backward")
    return gp, gd
