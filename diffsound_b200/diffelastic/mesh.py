"""Tetrahedral mesh container: linear -> quadratic promotion, gmsh I/O, OBJ triangle-mesh input.

API mirror of src/diffelastic/mesh.py:12-223 (`TetMesh`).  Node numbering of a
promoted mesh is part of the parity contract (SURVEY.md A.3): quadratic node ids
are the lexicographic rank of the fp32 coordinates, exactly what
`torch.unique(dim=0)` produces in the reference (mesh.py:174-179), and the
vertex tensor keeps its autograd link to the input vertices through an index
select, so d(lambda)/d(vertices) flows back to the caller's leaf tensor.

The per-tet geometry (transform matrix, inverse, determinant) is NOT
materialised here: the assembly and gradient kernels recompute it from the four
corner nodes (csrc/assemble.cu, csrc/grad.cu).  `transform_matrix` is kept as a
lazily evaluated property for API parity.
"""
import os
import struct

import numpy as np
import torch

from .. import native

CORNER_LOCAL = {1: (0, 1, 2, 3), 2: (0, 2, 4, 9), 3: (0, 3, 6, 16)}


def _default_device():
    if not torch.cuda.is_available():
        raise RuntimeError("diffsound_b200 needs a CUDA device (there is no CPU path)")
    return torch.device("cuda", torch.cuda.current_device())


def read_msh(filename):
    """Minimal gmsh 2.2 reader (ascii or binary): returns (points float64 (V,3), {type: int64 cells}).
    Replaces the reference's `meshio.read` (mesh.py:48, :188) for the formats it ships
    (data/mesh/**/*.msh); element types: 1 line, 2 triangle, 4 tetra, 11 tetra10, 15 vertex."""
    types = {1: ("line", 2), 2: ("triangle", 3), 4: ("tetra", 4), 11: ("tetra10", 10), 15: ("vertex", 1)}
    with open(filename, "rb") as f:
        buf = f.read()
    pos = 0

    def line():
        nonlocal pos
        e = buf.index(b"\n", pos)
        s = buf[pos:e].decode()
        pos = e + 1
        return s.strip()

    if line() != "$MeshFormat":
        raise ValueError(f"{filename}: not a gmsh .msh file")
    ver, ftype, _ = line().split()
    if not ver.startswith("2"):
        raise ValueError(f"{filename}: only gmsh format 2.x is supported (got {ver})")
    binary = int(ftype) == 1
    if binary:
        if struct.unpack("i", buf[pos:pos + 4])[0] != 1:
            raise ValueError(f"{filename}: big-endian gmsh files are not supported")
        pos += 4
        if buf[pos:pos + 1] == b"\n":
            pos += 1
    if line() != "$EndMeshFormat":
        raise ValueError(f"{filename}: malformed header")
    points, cells = None, {}
    while pos < len(buf):
        tag = line()
        if tag == "$Nodes":
            n = int(line())
            if binary:
                rec = np.dtype([("id", "<i4"), ("x", "<f8", (3,))])
                arr = np.frombuffer(buf, dtype=rec, count=n, offset=pos)
                pos += n * rec.itemsize
                if buf[pos:pos + 1] == b"\n":
                    pos += 1
                ids, pts = arr["id"].astype(np.int64), arr["x"].copy()
            else:
                rows = [line().split() for _ in range(n)]
                ids = np.array([int(r[0]) for r in rows], dtype=np.int64)
                pts = np.array([[float(v) for v in r[1:4]] for r in rows])
            order = np.argsort(ids, kind="stable")
            if not np.array_equal(ids[order], np.arange(1, n + 1)):
                raise ValueError(f"{filename}: node ids must be 1..N")
            points = pts[order]
            line()
        elif tag == "$Elements":
            total, got = int(line()), 0
            if binary:
                while got < total:
                    etype, cnt, ntags = struct.unpack("<3i", buf[pos:pos + 12])
                    pos += 12
                    name, nn = types[etype]
                    w = 1 + ntags + nn
                    arr = np.frombuffer(buf, dtype="<i4", count=cnt * w, offset=pos).reshape(cnt, w)
                    pos += cnt * w * 4
                    cells.setdefault(name, []).append(arr[:, 1 + ntags:].astype(np.int64) - 1)
                    got += cnt
                if buf[pos:pos + 1] == b"\n":
                    pos += 1
            else:
                for _ in range(total):
                    r = [int(v) for v in line().split()]
                    name, nn = types[r[1]]
                    cells.setdefault(name, []).append(np.array([r[3 + r[2]:]], dtype=np.int64) - 1)
            line()
        else:
            end = ("$End" + tag[1:]).encode()
            at = buf.find(end, pos)
            if at < 0:
                break
            pos = at + len(end) + 1
    if points is None:
        raise ValueError(f"{filename}: no $Nodes section")
    return points, {k: np.concatenate(v, axis=0) for k, v in cells.items()}


def read_obj(filename):
    """Wavefront OBJ triangle mesh: returns (verts float32 (V,3), faces int64 (F,3)), the form the reference's `.obj`
    targets (data/mesh/*.obj) take in `apply_sdf(path)`.  Reads `v` and `f` records only; face corners may be written
    `i`, `i/j`, `i//k` or `i/j/k`, with 1-based or negative (relative to the vertices read so far) indices; polygons are
    split into a triangle fan.  A missing file raises FileNotFoundError, a file without faces or with an index out of
    range ValueError."""
    verts, faces = [], []
    with open(filename, "r") as f:
        for lineno, raw in enumerate(f, 1):
            rec = raw.split("#", 1)[0].split()
            if not rec:
                continue
            if rec[0] == "v":
                if len(rec) < 4:
                    raise ValueError(f"{filename}:{lineno}: vertex with fewer than 3 coordinates")
                verts.append((float(rec[1]), float(rec[2]), float(rec[3])))
            elif rec[0] == "f":
                if len(rec) < 4:
                    raise ValueError(f"{filename}:{lineno}: face with fewer than 3 corners")
                ids = []
                for c in rec[1:]:
                    i = int(c.split("/", 1)[0])
                    j = i - 1 if i > 0 else len(verts) + i      # positive indices are checked once all vertices are read
                    if i == 0 or j < 0:
                        raise ValueError(f"{filename}:{lineno}: vertex index {i} out of range")
                    ids.append(j)
                faces.extend((ids[0], ids[k], ids[k + 1]) for k in range(1, len(ids) - 1))
    if not faces:
        raise ValueError(f"{filename}: no faces")
    faces = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    if faces.max() >= len(verts):
        raise ValueError(f"{filename}: vertex index {int(faces.max()) + 1} out of range (1..{len(verts)})")
    return np.asarray(verts, dtype=np.float32).reshape(-1, 3), faces


def write_msh(filename, points, cells, cell_type):
    """gmsh 2.2 ascii writer for one block of tetra / tetra10 cells."""
    code = {"tetra": 4, "tetra10": 11}[cell_type]
    with open(filename, "w") as f:
        f.write("$MeshFormat\n2.2 0 8\n$EndMeshFormat\n$Nodes\n%d\n" % len(points))
        for i, p in enumerate(points):
            f.write("%d %.17g %.17g %.17g\n" % (i + 1, p[0], p[1], p[2]))
        f.write("$EndNodes\n$Elements\n%d\n" % len(cells))
        for i, c in enumerate(cells):
            f.write("%d %d 2 0 0 %s\n" % (i + 1, code, " ".join(str(int(v) + 1) for v in c)))
        f.write("$EndElements\n")


class TetMesh:
    """Tetrahedral mesh: `vertices` (V,3) fp32, `tets` (T,4|10) int64, `order` 1|2."""

    def __init__(self, vertices=None, tets=None, order=1):
        self.vertices = vertices
        self.tets = tets
        if vertices is not None:
            self.device = vertices.device
        self.order = order

    def __repr__(self):
        return "TetMesh(vertices={}, tets={}, order={})".format(self.vertices.shape, self.tets.shape, self.order)

    @staticmethod
    def from_triangle_mesh(filename, log=False):
        """Load `<filename>_.msh` (the tetrahedralisation fTetWild leaves next to a surface mesh,
        mesh.py:33-56).  Running fTetWild itself is outside the hot path: a missing file raises."""
        path = filename + "_.msh"
        if not os.path.exists(path):
            raise FileNotFoundError(
                f"{path} not found: tetrahedralise {filename} with FloatTetwild_bin first (mesh.py:44-46)")
        points, cells = read_msh(path)
        dev = _default_device()
        vertices = torch.tensor(points, dtype=torch.float32, device=dev)
        tets = torch.tensor(cells["tetra"], dtype=torch.int64, device=dev)
        if log:
            print("Load tetramesh with ", len(vertices), " vertices & ", len(tets), " tets")
        return TetMesh(vertices, tets)

    @property
    def transform_matrix(self):
        """(T,3,3) fp32, columns x1-x4, x2-x4, x3-x4 of the corner nodes (mesh.py:69-99)."""
        if not hasattr(self, "_transform_matrix"):
            c = CORNER_LOCAL[self.order]
            v1, v2, v3, v4 = (self.vertices[self.tets[:, i]] for i in c)
            self._transform_matrix = torch.stack([v1 - v4, v2 - v4, v3 - v4], dim=2).to(torch.float32)
        return self._transform_matrix

    def to_high_order(self, order):
        """Order-1 mesh -> order `order` (1 or 2).  Local node order of a quadratic tet:
        [v0, m01, v1, m12, v2, m02, m03, m13, m23, v3] (mesh.py:139-154)."""
        assert self.order == 1
        if order == 1:
            return TetMesh(self.vertices, self.tets, order=1)
        if order != 2:
            raise NotImplementedError("only orders 1 and 2 can be built (the reference's order 3 is unreachable, "
                                      "mesh.py:116-160)")
        T, V = self.tets.shape[0], self.vertices.shape[0]
        vf = self.vertices[self.tets]
        a, b, c, d = vf[:, 0], vf[:, 1], vf[:, 2], vf[:, 3]
        mids = torch.cat([(a + b) / 2, (b + c) / 2, (a + c) / 2, (a + d) / 2, (b + d) / 2, (c + d) / 2], dim=0)
        allv = torch.cat([self.vertices, mids], dim=0)
        ar = torch.arange(T, dtype=self.tets.dtype, device=self.tets.device)
        t = self.tets
        new_tets = torch.stack([t[:, 0], V + ar, t[:, 1], V + T + ar, t[:, 2], V + 2 * T + ar, V + 3 * T + ar,
                                V + 4 * T + ar, V + 5 * T + ar, t[:, 3]], dim=1)
        mesh = TetMesh(allv, new_tets, order=2)
        mesh.remove_duplicate_vertices()
        return mesh

    def remove_duplicate_vertices(self):
        """Renumber nodes by lexicographic coordinate order; representative = smallest original
        index (mesh.py:162-179: torch.unique(dim=0) + scatter-min).  The sort runs in csrc/mesh.cu."""
        if not self.vertices.is_cuda:
            raise RuntimeError("diffsound_b200: mesh tensors must live on a CUDA device (there is no CPU path)")
        inv, first = native.unique_rows3(self.vertices.detach().to(torch.float32).contiguous())
        self.tets = inv[self.tets]
        self.vertices = self.vertices[first]
        if hasattr(self, "_transform_matrix"):
            del self._transform_matrix

    def import_from_file(self, filename):
        points, cells = read_msh(filename)
        dev = _default_device()
        self.vertices = torch.from_numpy(points).float().to(dev)
        self.tets = torch.from_numpy(cells["tetra"]).long().to(dev)
        self.device = self.vertices.device
        self.order = 1
        self.remove_duplicate_vertices()
        print(f"Mesh loaded from file {filename}")
        return self

    def export(self, filename):
        if self.order not in (1, 2):
            raise NotImplementedError("export supports orders 1 and 2")
        write_msh(filename, self.vertices.detach().cpu().numpy(), self.tets.detach().cpu().numpy(),
                  "tetra" if self.order == 1 else "tetra10")
        print(f"Mesh saved to file {filename}")
