"""LOBPCG for ONE large mesh on the GPUs of a node: row-partitioned K, M and iterate blocks (SURVEY.md section 8e row 2;
BASELINE.json configs[2] "row-partitioned SpMM at 1/2/4/8 GPUs").

Reference behaviour replaced: none one-to-one -- the reference is single-GPU and solves on the CPU
(src/diffelastic/diff_model.py:335-369); its own LOBPCG (src/lobpcg/_lobpcg.py:344-477) is the host-driven loop this module
mirrors.  The step is the one of the single-GPU driver csrc/lobpcg.cu (same kernels through the C-ABI, same recurrences for
the Gram pair, same two-level FP32 preconditioner), with rank r owning the contiguous slab of node rows
[bounds[r], bounds[r+1]) and these exchanges per iteration -- the only ones the path has:

  * residual sums                 all-reduce of 2 m doubles
  * fine smoothing (6 SpMMs + 1)  halo rows of the fp32 iterate are read from the neighbours' memory over NVLink inside the
                                  SpMM kernel (ds_spmm32_rowpart, CUDA IPC); one stream-ordered barrier per step
  * coarse residual               every rank restricts ITS fine rows (ds_pmg_restrict32_range), all-reduce of the partial
                                  coarse vectors (n_coarse x w fp32, 20 MB at config 3); the P1 coarse solve (one cooperative
                                  Chebyshev launch) is replicated -- it is 15x smaller than the fine level
  * new search block              all-gather of the fp32 preconditioner output (n x w x 4 B), then K W, M W for the own rows
  * Gram strips                   all-reduce of 2 x w x 3m doubles; the small eigen-solve and the Gram recurrences are
                                  replicated (identical inputs on every rank, deterministic kernels)

The nested P1 eigen-solve for the start block is replicated as well.  What does NOT shrink with the number of GPUs is
therefore: nested solve + coarse solves + small eigen-solves (see DESIGN.md section 6 for the measured split).
"""
import ctypes as C
import types
import math
from typing import List, Optional

import torch
import torch.distributed as dist

from .. import _lib, native
from .rowpart import owner_of, packed_column_map, slab_bounds

_p = native._p


class _SlabPattern:
    """brow / bcol of a slab of node rows (column ids global): what native.spmm* need of a pattern."""

    def __init__(self, brow, bcol, n_rows):
        self.brow, self.bcol, self.n_nodes = brow, bcol, int(n_rows)
        self.nnzb = int(bcol.numel())


class _Peers:
    """`nbuf` fp32 blocks of (3 max_local) x 48 in peer-visible memory, opened on every rank (CUDA IPC)."""

    def __init__(self, rank, world, max_local, nbuf, device, group):
        lib = _lib.load()
        self.rank, self.world, self.group = rank, world, group
        self.elems = 3 * max_local * 48
        ptr = C.c_void_p()
        handle = (C.c_ubyte * 64)()
        with torch.cuda.device(device):
            _lib.check(lib.ds_peer_alloc(4 * self.elems * nbuf, C.byref(ptr), handle), "ds_peer_alloc")
        self.own = ptr.value
        handles = [None] * world
        if world > 1:
            dist.all_gather_object(handles, bytes(handle), group=group)
        else:
            handles[0] = bytes(handle)
        self.ptrs = []
        for r, h in enumerate(handles):
            if r == rank:
                self.ptrs.append(self.own)
            else:
                p = C.c_void_p()
                _lib.check(lib.ds_peer_open((C.c_ubyte * 64).from_buffer_copy(h), C.byref(p)), "ds_peer_open")
                self.ptrs.append(p.value)
        self.device = device

    def block(self, k, rows, cols):
        class _A:
            pass
        a = _A()
        a.__cuda_array_interface__ = {"shape": (rows, cols), "typestr": "<f4", "data": (self.own + 4 * self.elems * k, False),
                                      "version": 3, "strides": None}
        return torch.as_tensor(a, device=self.device)

    def parts(self, k):
        return (C.c_void_p * self.world)(*[p + 4 * self.elems * k for p in self.ptrs])

    def close(self):
        lib = _lib.load()
        if self.ptrs is None:
            return
        torch.cuda.synchronize(self.device)
        if self.world > 1:
            dist.barrier(group=self.group)
        for r, p in enumerate(self.ptrs):
            if r != self.rank:
                lib.ds_peer_close(C.c_void_p(p))
        if self.world > 1:
            dist.barrier(group=self.group)
        lib.ds_peer_free(C.c_void_p(self.own))
        self.ptrs = None


def _cheb_coefs(lmax, ratio, degree):
    """(cc0, [(ab_k, cc_k) for k = 1 .. degree-1]) of the block-Jacobi Chebyshev recurrence (Level32::cheb, csrc/precond32.cu)."""
    lmin = lmax / ratio
    theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
    sig = theta / delta
    rho = 1.0 / sig
    out = []
    for _ in range(1, degree):
        rho_new = 1.0 / (2.0 * sig - rho)
        out.append((rho_new * rho, 2.0 * rho_new / delta))
        rho = rho_new
    return 1.0 / theta, out


def coarse_column_slice(rc, w, rank, world):
    """Columns [rank * per, rank * per + per) of the first w columns of rc, per = ceil(w / world), zero-padded to the
    16-column granularity of the Chebyshev kernels: what rank `rank` solves of a column-sharded coarse solve."""
    per = -(-w // world)
    per16 = -(-per // 16) * 16
    c0 = min(rank * per, w)
    c1 = min(c0 + per, w)
    loc = torch.zeros(rc.shape[0], per16, dtype=rc.dtype, device=rc.device)
    if c1 > c0:
        loc[:, :c1 - c0] = rc[:, c0:c1]
    return loc


def coarse_column_merge(allz, w):
    """Inverse of coarse_column_slice over all ranks: allz [world, rows, per16] (rank-major, as all_gather_into_tensor
    delivers it) -> [rows, w]."""
    world, rows, _ = allz.shape
    per = -(-w // world)
    return allz[:, :, :per].permute(1, 0, 2).reshape(rows, world * per)[:, :w].contiguous()


class RowPartLOBPCG:
    """Lowest pairs of K u = lam M u with the rows of K, M, X split over the ranks of `group`.

    pattern / Kval / Mblk / coarse: the FULL operators (every rank assembles them: duplicated compute instead of a distributed
    assembly; 1 ms at config 3).  X0: (n, m) fp64 start block, identical on every rank."""

    def __init__(self, pattern, Kval, Mblk, coarse, group=None, smooth_steps=3, smooth_ratio=8.0, coarse_degree=40,
                 coarse_ratio=None, nested_tol=3e-2, verbose=False, coords=None):
        self.lib = _lib.load()
        # coords (fp32 [n_nodes, 3], optional): the solver works in a private Morton numbering of the nodes -- the slabs are
        # contiguous ranges of the space-filling curve (compact sub-domains: shorter halos) and consecutive rows of a slab
        # gather overlapping sets of X rows, the locality the L1-resident SpMM kernels are built for (single-GPU level:
        # 0.31 ms per smoothing step against 0.46 ms in lexicographic order).  X0 / the returned block stay in the caller's
        # numbering.
        self.perm = None
        if coords is not None:
            pattern = self._setup_morton(pattern, coords)
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.verbose = verbose and self.rank == 0
        self.pat = pattern
        dev = Kval.device
        self.dev = dev
        self.nu, self.sratio = int(smooth_steps), float(smooth_ratio)
        self.cdeg = int(coarse_degree)
        self.cratio = float(coarse_ratio) if coarse_ratio else 0.4 * self.cdeg * self.cdeg
        self.nested_tol = nested_tol
        self.profile, self.phase_ms, self._t_last, self._t_name = False, {}, None, None
        lib = self.lib
        # ---- slab of this rank (topology only: kept for every solve on this pattern)
        self.bounds = slab_bounds(pattern.n_nodes, self.world)
        r0, r1 = self.bounds[self.rank], self.bounds[self.rank + 1]
        self.r0, self.r1, self.nl = r0, r1, r1 - r0
        self.max_local = max(b - a for a, b in zip(self.bounds[:-1], self.bounds[1:]))
        brow = pattern.brow
        b0, b1 = int(brow[r0]), int(brow[r1])
        self.b0, self.b1 = b0, b1
        self.brow_l = (brow[r0:r1 + 1] - b0).contiguous()
        self.bcol_l = pattern.bcol[b0:b1].contiguous()
        self.slab = _SlabPattern(self.brow_l, self.bcol_l, self.nl)
        # column ids as row indices of the all-gathered (padded) fp32 block: owner * max_local + local
        own = owner_of(self.bcol_l.long(), self.bounds)
        start = torch.as_tensor(self.bounds, dtype=torch.int64, device=dev)[own]
        self.bcolP_l = (own * self.max_local + (self.bcol_l.long() - start)).to(torch.int32).contiguous()
        with torch.cuda.device(dev):
            self.chunk_l = torch.empty(lib.ds_spmm32_chunk_count(self.nl) + 1, dtype=torch.int32, device=dev)
            _lib.check(lib.ds_spmm32_chunks(_p(self.brow_l), self.nl, _p(self.chunk_l), native._stream()), "ds_spmm32_chunks")
        self.colmap = packed_column_map(pattern.n_nodes, self.bounds, dev)
        self.rec_l = torch.empty((lib.ds_k32_record_bytes(b1 - b0) + 15) // 16 * 4, dtype=torch.int32, device=dev)
        self.invD_l = torch.empty(self.nl * 9, dtype=torch.float32, device=dev)
        self.peers = _Peers(self.rank, self.world, self.max_local, 2, dev, group)
        self._tok = torch.zeros(1, device=dev)
        self.set_operators(Kval, Mblk, coarse)

    def _setup_morton(self, pattern, coords):
        """perm (new node -> old node) along a 30-bit Morton curve, the permuted block pattern and the gather indices that
        carry K / M values, the fine-node tables of the coarse level and the iterate blocks into that numbering."""
        dev = coords.device
        n = pattern.n_nodes
        c = coords.detach().to(torch.float32)
        lo, hi = c.min(0).values, c.max(0).values
        q = ((c - lo) / (hi - lo).clamp_min(1e-30) * 1023.0).long().clamp_(0, 1023)
        code = torch.zeros(n, dtype=torch.int64, device=dev)
        for b in range(10):
            for d in range(3):
                code |= ((q[:, d] >> b) & 1) << (3 * b + d)
        perm = torch.argsort(code, stable=True)
        inv = torch.empty_like(perm)
        inv[perm] = torch.arange(n, device=dev)
        brow = pattern.brow.long()
        deg_p = (brow[1:] - brow[:-1])[perm]
        brow_p = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        brow_p[1:] = torch.cumsum(deg_p, 0)
        shift = brow[:-1][perm] - brow_p[:-1]                          # old start - new start of every (new) row
        nnzb = int(brow_p[-1])
        midx = torch.repeat_interleave(shift, deg_p) + torch.arange(nnzb, device=dev)
        kidx = torch.repeat_interleave(9 * shift, 9 * deg_p) + torch.arange(9 * nnzb, device=dev)
        self.perm, self.inv = perm, inv
        self._midx, self._kidx = midx.to(torch.int32), kidx.to(torch.int32)
        ar3 = torch.arange(3, device=dev)[None, :]
        self._perm3 = (3 * perm[:, None] + ar3).reshape(-1)
        self._inv3 = (3 * inv[:, None] + ar3).reshape(-1)
        return types.SimpleNamespace(n_nodes=n, n=3 * n, nnzb=nnzb, nnz=9 * nnzb, brow=brow_p.to(torch.int32).contiguous(),
                                     bcol=inv[pattern.bcol.long()[midx]].to(torch.int32).contiguous())

    def _coarse_view(self, coarse):
        """the coarse level with its fine-node tables (parents per fine node, gather lists of fine ids, corner ids) relabelled"""
        v = types.SimpleNamespace(**vars(coarse))
        v.parents = coarse.parents.view(-1, 2)[self.perm].reshape(-1).contiguous()
        v.rlist = self.inv[coarse.rlist.long()].to(torch.int32).contiguous()
        v.corner_nodes = self.inv[coarse.corner_nodes]
        return v

    def set_operators(self, Kval, Mblk, coarse):
        """New values on the same pattern (a shape / material step): slab views of K, M, the FP32 records of the slab with
        packed (owner, local) column ids for the peer-gather SpMM, and the replicated coarse level."""
        if self.perm is not None:
            Kval, Mblk, coarse = torch.index_select(Kval, 0, self._kidx), torch.index_select(Mblk, 0, self._midx), self._coarse_view(coarse)
        self.Kval, self.Mblk, self.coarse = Kval, Mblk, coarse
        b0, b1 = self.b0, self.b1
        self.K_l = Kval[9 * b0:9 * b1]
        self.M_l = Mblk[b0:b1]
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.ds_k32_pack_slab(_p(self.brow_l), _p(self.bcol_l), self.nl, b1 - b0, self.r0, _p(self.K_l.contiguous()),
                                                 None, 0.0, _p(self.colmap), _p(self.rec_l), _p(self.invD_l), native._stream()),
                       "ds_k32_pack_slab")
        self.rec_c, self.invD_c = native.k32_pack(coarse.pattern, coarse.Kval)

    # ------------------------------------------------------------------ diagnostics
    def _tick(self, name):
        """profile=True: wall time per phase with a device synchronize at every phase boundary (diagnostic runs only)."""
        if not self.profile:
            return
        import time
        torch.cuda.synchronize(self.dev)
        now = time.perf_counter()
        if self._t_last is not None:
            self.phase_ms[self._t_name] = self.phase_ms.get(self._t_name, 0.0) + (now - self._t_last) * 1e3
        self._t_last, self._t_name = now, name

    # ------------------------------------------------------------------ collectives (stream ordered)
    def _barrier(self):
        if self.world > 1:
            dist.all_reduce(self._tok, group=self.group)

    def _allreduce(self, t):
        if self.world > 1:
            dist.all_reduce(t, group=self.group)
        return t

    # ------------------------------------------------------------------ FP32 operators on the slab
    def _spmm32(self, mode, src_k, w, out, R=None, Zprev=None, ab=0.0, cc=0.0):
        """out = op(K_slab, block src_k of every rank (halo rows over NVLink)); mode as ds_spmm32."""
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.ds_spmm32_rowpart(int(mode), _p(self.brow_l), _p(self.rec_l), self.nl, int(w), self.peers.parts(src_k),
                                                  self.world, self.rank, _p(R), _p(self.invD_l) if mode == 2 else None, _p(Zprev),
                                                  _p(out), float(ab), float(cc), native._stream()), "ds_spmm32_rowpart")

    def _fine_cheb(self, r32, w, cur, from_zero):
        """`nu` Chebyshev-Jacobi steps on the slab; the iterate ping-pongs between the two peer blocks; returns the index of
        the block that holds the result."""
        Z = [self.peers.block(k, 3 * self.nl, w) for k in (0, 1)]
        cc0, steps = _cheb_coefs(self.lmax_f, self.sratio, self.nu)
        lib = self.lib
        if from_zero:
            with torch.cuda.device(self.dev):
                _lib.check(lib.ds_jacobi32(_p(self.invD_l), _p(r32), self.nl, w, cc0, _p(Z[cur]), native._stream()), "ds_jacobi32")
            Z[cur ^ 1].zero_()
        else:
            self._barrier()
            self._spmm32(2, cur, w, Z[cur ^ 1], R=r32, Zprev=Z[cur], ab=0.0, cc=cc0)
            cur ^= 1
        for ab, cc in steps:
            self._barrier()
            self._spmm32(2, cur, w, Z[cur ^ 1], R=r32, Zprev=Z[cur ^ 1], ab=ab, cc=cc)
            cur ^= 1
        return cur

    def _estimate_lmax(self):
        """largest eigenvalue of invD K by power iteration on 16 columns through the slab SpMM (norms all-reduced)."""
        w = 16
        Z = [self.peers.block(k, 3 * self.nl, w) for k in (0, 1)]
        g = torch.Generator(device=self.dev).manual_seed(1234 + self.rank)
        Z[0].copy_(torch.rand(3 * self.nl, w, device=self.dev, generator=g) * 2 - 1)
        zero = torch.zeros(3 * self.nl, w, dtype=torch.float32, device=self.dev)
        # The first 12 steps and their three samples are queued without a host synchronisation (the ratios stay on the
        # device); the usual case reads them back once.  Same acceptance rule as before, applied in sample order.
        cur, est, prev = 0, 0.0, None
        ratios = []

        def step(sample):
            nonlocal cur
            n0 = self._allreduce((Z[cur].double() ** 2).sum(0)) if sample else None
            self._barrier()
            self._spmm32(2, cur, w, Z[cur ^ 1], R=zero, Zprev=zero, ab=-1.0, cc=-1.0)        # invD K z
            cur ^= 1
            if sample:
                n1 = self._allreduce((Z[cur].double() ** 2).sum(0))
                return torch.sqrt(n1 / n0).max()
            return None

        for it in range(12):
            r = step(it % 4 == 3)
            if r is not None:
                ratios.append(r)
        for it, e in zip((3, 7, 11), torch.stack(ratios).tolist()):      # one device -> host copy
            est = e
            done = prev is not None and est <= 1.01 * prev and it >= 11
            prev = est
        for it in range(12, 24):
            if done:
                break
            r = step(it % 4 == 3)
            if r is not None:
                est = float(r)
                done = est <= 1.01 * prev
                prev = est
        return 1.1 * est

    def _coarse_solve(self, rc, w):
        """Chebyshev solve on the (replicated) P1 operator.  Its columns are independent, so with several ranks each rank
        solves ceil(w / world) of them (padded to the kernel's 16-column granularity) and the slices are all-gathered:
        the persistent kernel costs 0.62 ms at 16 columns against 1.34 ms at 48, the all-gather of 20 MB ~0.1 ms."""
        co = self.coarse
        if self.world == 1 or w < 32:
            return native.cheb32_solve(co.pattern, self.rec_c, self.invD_c, rc, self.cdeg, self.lmax_c, self.cratio)
        loc = coarse_column_slice(rc, w, self.rank, self.world)
        zloc = native.cheb32_solve(co.pattern, self.rec_c, self.invD_c, loc, self.cdeg, self.lmax_c, self.cratio)
        allz = torch.empty(self.world, rc.shape[0], loc.shape[1], dtype=torch.float32, device=self.dev)
        dist.all_gather_into_tensor(allz, zloc.contiguous(), group=self.group)
        return coarse_column_merge(allz, w)

    def _vcycle(self, r32, w):
        """two-level V(nu, nu) cycle on the slab; returns the peer-block index holding z (rows of this rank)."""
        lib = self.lib
        cur = self._fine_cheb(r32, w, 0, True)
        res = torch.empty(3 * self.nl, w, dtype=torch.float32, device=self.dev)
        self._barrier()
        self._spmm32(1, cur, w, res, R=r32)                                                    # r - K z
        co = self.coarse
        rc = torch.empty(3 * co.n_nodes, w, dtype=torch.float32, device=self.dev)
        with torch.cuda.device(self.dev):
            _lib.check(lib.ds_pmg_restrict32_range(_p(co.rptr), _p(co.rlist), co.n_nodes, _p(res), w, self.r0, self.r1, _p(rc),
                                                   native._stream()), "ds_pmg_restrict32_range")
        self._allreduce(rc)
        zc = self._coarse_solve(rc, w)
        z = self.peers.block(cur, 3 * self.nl, w)
        with torch.cuda.device(self.dev):
            par = C.c_void_p(co.parents.data_ptr() + 8 * self.r0)
            _lib.check(lib.ds_pmg_prolong_add32(par, self.nl, _p(zc), w, _p(z), native._stream()), "ds_pmg_prolong_add32")
        return self._fine_cheb(r32, w, cur, False)

    # ------------------------------------------------------------------ the solve
    def solve(self, X0, nev, tol=1e-5, maxit=200, n_rigid=6, nested=True):
        lib, dev, m = self.lib, self.dev, X0.shape[1]
        assert X0.dtype == torch.float64 and X0.shape[0] == self.pat.n and m in (16, 32, 48)
        if self.perm is not None:
            X0 = X0[self._perm3]
        nl3, ld = 3 * self.nl, 3 * m
        co = self.coarse
        f64 = dict(dtype=torch.float64, device=dev)
        stream = native._stream
        # ---- nested iteration: the P1 eigen-problem, replicated, then prolonged (every rank prolongs all rows: the initial
        #      K X, M X products need the whole block as gather source).  It runs first: its fine level IS this solve's
        #      coarse level, so the spectral-radius estimate of the coarse Chebyshev interval is taken over from it.
        X = X0
        nested_its = 0
        self.lmax_c = None
        self._tick("nested")
        if nested and co.Mblk is not None:
            rows = (3 * co.corner_nodes[:, None] + torch.arange(3, device=dev)[None, :]).reshape(-1)
            Xc = X0[rows].contiguous()
            nc = 3 * co.n_nodes
            deg = int(min(48, max(24, round(nc ** (1.0 / 3.0) / 1.2))))
            _, _, st = native.lobpcg(co.pattern, co.Kval, co.Mblk, Xc, nev=nev, tol=self.nested_tol, maxit=40, cheb_degree=deg,
                                     cheb_ratio=0.4 * deg * deg, n_rigid=n_rigid, coords=co.verts)
            nested_its = st["iterations"]
            if st.get("lmax_fine", 0.0) > 0.0:
                self.lmax_c = st["lmax_fine"]
            X = torch.empty_like(X0)
            with torch.cuda.device(dev):
                _lib.check(lib.ds_pmg_prolong64(_p(co.parents), self.pat.n_nodes, _p(Xc), m, m, _p(X), m, stream()), "ds_pmg_prolong64")
        self._tick("lmax")
        # ---- spectral bounds (coarse: replicated, local kernel, only without a nested solve; fine: through the slab SpMM)
        if self.lmax_c is None:
            zc0 = torch.zeros(3 * co.n_nodes, 16, dtype=torch.float32, device=dev)
            g = torch.Generator(device=dev).manual_seed(99)
            a = torch.rand(3 * co.n_nodes, 16, device=dev, generator=g) * 2 - 1
            est = None
            for it in range(16):
                b = native.spmm32(co.pattern, self.rec_c, a, mode=2, R=zc0, invD=self.invD_c, Zprev=zc0, ab=-1.0, cc=-1.0)
                if it >= 11:      # the ratio grows monotonically towards lmax; kept on the device, read back once
                    r = torch.sqrt((b.double() ** 2).sum(0) / (a.double() ** 2).sum(0)).max()
                    est = r if est is None else torch.maximum(est, r)
                a = b
            self.lmax_c = 1.1 * float(est)
        self.lmax_f = self._estimate_lmax()
        self._tick("alloc")
        # ---- local buffers
        S = [torch.zeros(nl3, ld, **f64) for _ in range(2)]
        KS = [torch.zeros(nl3, ld, **f64) for _ in range(2)]
        MS = [torch.zeros(nl3, ld, **f64) for _ in range(2)]
        R = torch.empty(nl3, m, **f64)
        G = torch.zeros(2, 144, 144, **f64)           # GK | GM (one buffer: one all-reduce)
        Gn = torch.zeros(2, 144, 144, **f64)
        Gs = torch.zeros(2, 144, 144, **f64)          # strips
        Cm = torch.zeros(144, 144, **f64)
        theta = torch.zeros(144, **f64)
        lam_d = torch.zeros(m, **f64)
        sums = torch.zeros(2 * m, **f64)
        res_partial = torch.empty(296 * 2 * m, **f64)
        eig_scratch = torch.empty(lib.ds_eigh_scratch_elems(144), **f64)
        info = torch.zeros(16, dtype=torch.int32, device=dev)
        strip_partial = torch.empty(lib.ds_gram_strip_scratch_elems(), **f64)
        sym_partial = torch.empty(lib.ds_gram_sym2_scratch_elems(), **f64)
        alg_scratch = torch.empty(lib.ds_gram_algebra_scratch_elems(), **f64)
        Zfull = torch.zeros(self.world * self.max_local * 3, 48, dtype=torch.float32, device=dev)
        Zsend = torch.zeros(self.max_local * 3, 48, dtype=torch.float32, device=dev)

        def eig(slots):
            Cm.zero_()
            arr = (C.c_int * len(slots))(*slots)
            with torch.cuda.device(dev):
                _lib.check(lib.ds_eigh_generalized_idx_f64(_p(G[0]), _p(G[1]), len(slots), 144, arr, -1e-6, _p(theta), _p(Cm), 144,
                                                           _p(eig_scratch), _p(info), stream()), "ds_eigh_generalized_idx_f64")
            return int(info[0].item())

        def full_gram(w, nw, with_p):
            G.zero_()
            tiles = list(range(m // 8)) + [m // 8 + t for t in range((nw + 7) // 8)]
            if with_p:
                tiles += [2 * m // 8 + t for t in range(m // 8)]
            arr = (C.c_int * len(tiles))(*tiles)
            with torch.cuda.device(dev):
                _lib.check(lib.ds_gram_sym2_f64(_p(S[w]), _p(KS[w]), _p(MS[w]), ld, nl3, arr, len(tiles), _p(G[0]), _p(G[1]), 144,
                                                _p(sym_partial), stream()), "ds_gram_sym2_f64")
            self._allreduce(G)
            with torch.cuda.device(dev):
                _lib.check(lib.ds_sym_upper_f64(_p(G[0]), _p(G[1]), 144, 3 * m, stream()), "ds_sym_upper_f64")

        def algebra():
            nonlocal G, Gn
            with torch.cuda.device(dev):
                _lib.check(lib.ds_gram_algebra_f64(_p(G[0]), _p(G[1]), _p(Gn[0]), _p(Gn[1]), 144, _p(Cm), 144, _p(theta), m,
                                                   _p(alg_scratch), stream()), "ds_gram_algebra_f64")
            G, Gn = Gn, G

        self._tick("initial_rr")
        # ---- initial Rayleigh-Ritz on X
        S[0][:, :m] = X[3 * self.r0:3 * self.r1]
        native.spmm_k_and_m(self.slab, self.K_l, self.M_l, X, KS[0][:, :m], MS[0][:, :m])
        full_gram(0, 0, False)
        if eig(list(range(m))) != 0:
            raise RuntimeError("rowpart lobpcg: initial block is not M-independent")
        for A, B in ((S, S), (KS, KS), (MS, MS)):
            native.block_gemm(A[0][:, :m], Cm[:m, :m], out=B[1][:, :m])
        cur = 1
        lam_d.copy_(theta[:m])
        algebra()
        have_p, since_refresh, it, nconv, status = False, 0, 0, 0, 1
        rel = [1.0] * m
        for it in range(maxit + 1):
            self._tick("residual")
            with torch.cuda.device(dev):
                _lib.check(lib.ds_lobpcg_residual(_p(KS[cur]), _p(MS[cur]), ld, m, nl3, _p(lam_d), _p(R), m, _p(sums), _p(res_partial),
                                                  stream()), "ds_lobpcg_residual")
            self._allreduce(sums)
            hn = sums.cpu().tolist()
            lam = lam_d.cpu().tolist()
            nr = n_rigid
            lref = abs(lam[min(nr, m - 1)])
            act, nconv = [], 0
            for j in range(m):
                rn, mn = math.sqrt(hn[j]), math.sqrt(hn[m + j])
                scale = (lref if j < nr else abs(lam[j])) * mn
                rel[j] = rn / scale if scale > 0 else rn
                if rel[j] >= tol:
                    act.append(j)
                elif j < nev:
                    nconv += 1
            if self.verbose:
                print(f"[rowpart lobpcg] it {it:3d} conv {nconv}/{nev} active {len(act)} max rel res {max(rel[nr:nev]):.3e}", flush=True)
            if nconv >= nev:
                status = 0
                break
            if it == maxit:
                break
            na = len(act)
            w = (na + 15) & ~15
            r32 = torch.empty(nl3, w, dtype=torch.float32, device=dev)
            arr = (C.c_int * na)(*act)
            with torch.cuda.device(dev):
                _lib.check(lib.ds_gather_cols_f32(_p(R), m, arr, na, w, nl3, _p(r32), stream()), "ds_gather_cols_f32")
            self._tick("vcycle")
            zk = self._vcycle(r32, w)
            self._tick("allgather_kw_mw")
            z = self.peers.block(zk, nl3, w)
            Wv = S[cur][:, m:m + w]
            with torch.cuda.device(dev):
                _lib.check(lib.ds_widen_f32(_p(z), w, nl3, C.c_void_p(Wv.data_ptr()), ld, stream()), "ds_widen_f32")
            # ---- all-gather of the new fp32 search block, then K W, M W for the own rows
            if self.world > 1:
                send = Zsend.view(-1)[:self.max_local * 3 * w].view(self.max_local * 3, w)
                send[:nl3].copy_(z)
                full = Zfull.view(-1)[:self.world * self.max_local * 3 * w].view(self.world * self.max_local * 3, w)
                dist.all_gather_into_tensor(full, send, group=self.group)
            else:
                full = z
            with torch.cuda.device(dev):
                _lib.check(lib.ds_spmm_dual_z32(_p(self.brow_l), _p(self.bcolP_l), self.nl, self.b1 - self.b0, _p(self.chunk_l),
                                                _p(self.K_l), _p(self.M_l), _p(full), w, C.c_void_p(KS[cur][:, m:].data_ptr()), ld,
                                                C.c_void_p(MS[cur][:, m:].data_ptr()), ld, stream()), "ds_spmm_dual_z32")
            self._tick("gram")
            # ---- Gram pair: strips of the new W on top of the recurrences, or everything afresh
            use_p, fresh = have_p, since_refresh >= 8
            if fresh:
                full_gram(cur, w, have_p)
                since_refresh = 0
            else:
                with torch.cuda.device(dev):
                    _lib.check(lib.ds_gram_strip_f64(C.c_void_p(KS[cur][:, m:].data_ptr()), C.c_void_p(MS[cur][:, m:].data_ptr()), ld, w,
                                                     _p(S[cur]), ld, ld, nl3, _p(Gs[0]), _p(Gs[1]), 144, _p(strip_partial), stream()),
                               "ds_gram_strip_f64")
                self._allreduce(Gs)
                with torch.cuda.device(dev):
                    _lib.check(lib.ds_gram_insert_f64(_p(G[0]), _p(G[1]), 144, _p(Gs[0]), _p(Gs[1]), 144, m, w, stream()),
                               "ds_gram_insert_f64")
            self._tick("eigh")
            code = 1
            for attempt in range(3):
                slots = list(range(m)) + [m + s for s in range(na)] + ([2 * m + j for j in act] if use_p else [])
                code = eig(slots)
                if code == 0:
                    break
                if not fresh:
                    full_gram(cur, w, have_p)
                    fresh, since_refresh = True, 0
                    continue
                if not use_p:
                    break
                use_p = False
            if code != 0:
                raise RuntimeError(f"rowpart lobpcg: Rayleigh-Ritz breakdown at iteration {it} (info {code})")
            nxt = cur ^ 1
            self._tick("rr_update")
            with torch.cuda.device(dev):
                _lib.check(lib.ds_rr_update2_f64(_p(S[cur]), _p(KS[cur]), _p(MS[cur]), ld, m, w, int(use_p), _p(Cm), 144, nl3,
                                                 _p(S[nxt]), _p(KS[nxt]), _p(MS[nxt]), ld, stream()), "ds_rr_update2_f64")
            algebra()
            have_p = True
            since_refresh += 1
            lam_d.copy_(theta[:m])
            cur = nxt
        self._tick("gather_x")
        # ---- gather the eigenvector block (n x m) on every rank
        Xl = S[cur][:, :m].contiguous()
        if self.world > 1:
            pad = torch.zeros(3 * self.max_local, m, **f64)
            pad[:nl3] = Xl
            allx = torch.empty(self.world * 3 * self.max_local, m, **f64)
            dist.all_gather_into_tensor(allx, pad, group=self.group)
            Xfull = torch.cat([allx[3 * self.max_local * r: 3 * self.max_local * r + 3 * (self.bounds[r + 1] - self.bounds[r])]
                               for r in range(self.world)], dim=0)
        else:
            Xfull = Xl
        if self.perm is not None:
            Xfull = Xfull[self._inv3]
        self._tick("end")
        self._t_last = None
        stats = dict(iterations=it, converged=nconv, status=status, nested_iterations=nested_its, world=self.world,
                     rows_local=self.nl, two_level=True)
        return lam_d.clone(), Xfull, torch.tensor(rel, dtype=torch.float64), stats

    def close(self):
        self.peers.close()


def eigen_decomposition_rowpart(obj, group=None, verbose=False, solver=None, keep=False):
    """`DiffSoundObj.eigen_decomposition()` with the eigen-solve row-partitioned over the ranks of `group` (quadratic meshes).
    Assembly is replicated; on return `obj` holds the same attributes as after the single-GPU call, on every rank.
    `solver`: a RowPartLOBPCG of an earlier call on the same topology (partition and peer buffers are reused, only the values
    are refreshed); `keep=True` returns (stats, solver) and leaves the solver open for the next call."""
    if obj.fixed_nodes is not None:
        raise NotImplementedError("row-partitioned eigen-solve: clamped objects (DiffSoundObj.fix_nodes) are not supported; "
                                  "use eigen_decomposition() on one GPU")
    if obj.material_field is not None:
        raise NotImplementedError("row-partitioned eigen-solve: material fields (DiffSoundObj.set_material_field) are not "
                                  "supported; use eigen_decomposition() on one GPU")
    if obj.elasticity_field is not None:
        raise NotImplementedError("row-partitioned eigen-solve: elasticity-tensor fields (DiffSoundObj.set_elasticity_field) "
                                  "are not supported; use eigen_decomposition() on one GPU")
    if obj.supports is not None:
        raise NotImplementedError("row-partitioned eigen-solve: elastic supports (DiffSoundObj.set_supports) are not "
                                  "supported; use eigen_decomposition() on one GPU")
    obj._assemble(obj.material_model.mat.density)
    if obj.tetmesh.order != 2 or obj.deform.coarse is None:
        raise NotImplementedError("row-partitioned eigen-solve: quadratic meshes only (two-level preconditioner)")
    need = obj.mode_num + 6
    m = obj._block_for(need)
    if m is None:
        raise NotImplementedError("row-partitioned eigen-solve: at most 44 pairs (one block)")
    coarse = obj.deform.coarse
    mu, la = obj._lame_used
    coarse.assemble(obj._verts32, mu, la, coarse.ctab, obj.deform.coarse_mtab(obj._density_used))
    cdeg = int(obj.coarse_degree) or int(min(64, max(32, round((3 * coarse.n_nodes) ** (1.0 / 3.0) / 1.2))))
    if solver is None:
        solver = RowPartLOBPCG(obj.deform.pattern, obj._Kval, obj._Mblk, coarse, group=group, smooth_steps=obj.smooth_steps,
                               smooth_ratio=obj.smooth_ratio, coarse_degree=cdeg, coarse_ratio=float(obj.coarse_ratio) or None,
                               nested_tol=obj.nested_tol, verbose=verbose, coords=obj._verts32 if obj.morton else None)
    else:
        solver.set_operators(obj._Kval, obj._Mblk, coarse)
    try:
        X0, _ = obj._start_block(m, 0)
        lam, X, res, stats = solver.solve(X0, need, tol=obj.eig_tol, maxit=obj.eig_maxit, n_rigid=6, nested=obj.nested_start)
    finally:
        if not keep:
            solver.close()
    if stats["status"] != 0:
        raise RuntimeError(f"row-partitioned eigensolver did not converge: {stats}")
    obj.eig_stats = stats
    obj._warm = [X]
    obj._X = X
    obj.U_hat_full = X[:, :need]
    obj.eigenvalues = lam[6:need].clone()
    obj.ritz_values = lam
    obj.U_hat = X[:, 6:need]
    obj._Xpad = X
    obj._q = None
    return (stats, solver) if keep else stats
