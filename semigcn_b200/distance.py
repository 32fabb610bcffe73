"""Point-to-surface distance and the two-sided mesh distance: the accuracy metric of the inpainting evaluation.

SeMIGCN reports the mean distance from the inpainted mesh to the ground-truth surface over the bounding-box diagonal,
overall and in the hole region (sgcn.py:183,193 through check/dist_check.py).  ``mesh_distance`` computes that family of
statistics with vertices as the samples: for every vertex of one mesh the exact distance to the closed triangles of the
other (csrc/surface_dist.cu, an exact nearest-triangle search over a uniform grid), reduced in fp64.

Coordinates are rounded to fp32 (the library's storage type) and every distance is evaluated in fp64 on those values.
``dist[i]`` is the minimum over all faces of the distance from point i to the closed triangle, ``face[i]`` the smallest
face id attaining it.  Zero-area faces, duplicate faces and non-manifold soup are valid targets, and the target need
not be closed.  A query with a non-finite coordinate gets ``dist = NaN``, ``face = -1``.  Parity with pymeshlab's
distance filters is not pinned (DESIGN.md §3).
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import numpy as np
import torch
from torch import Tensor

from . import _lib as L
from ._lib import SgbError, check, ptr, require_cuda, stream_ptr
from .losses import _dev_tensor

# at most this many grid cells per face, and (cell, face) pairs per face before the grid is coarsened
_CELLS_PER_FACE = 4
_PAIRS_PER_FACE = 32
_PAIRS_FLOOR = 1 << 20
# faces are binned with their bounding box widened by this fraction of a cell, so that rounding at a cell border cannot
# drop a face from a cell its box touches
_BIN_EPS = 1e-6


def _device_of(*xs) -> torch.device:
    for x in xs:
        if isinstance(x, Tensor):
            require_cuda(x)
            return x.device
    return torch.device("cuda", torch.cuda.current_device())


class SurfaceIndex:
    """Uniform-grid index of a target triangle mesh for exact point-to-surface queries.

    ``vs`` [nv, 3] and ``faces`` [nf, 3] are CUDA tensors or numpy arrays (``Mesh.vs`` / ``Mesh.faces``); CPU tensors are
    refused.  The grid is built once, with torch ops on the device: cells of edge ``cell_size`` (default: the mean edge
    length, enlarged until there are at most 4 cells per face), every face listed in each cell its bounding box
    overlaps.  When a few large faces would list more than ~32 (cell, face) pairs per face, the cell size doubles until
    they fit.  The result of a query does not depend on the grid.  Building synchronises with the host (the validation
    and the sizing of the grid read device values); ``query`` and ``stats`` do not.

    Raises ``SgbError`` for a non-finite vertex, a face id outside ``[0, nv)`` or an empty face list.
    """

    def __init__(self, vs, faces, cell_size: Optional[float] = None):
        dev = _device_of(vs, faces)
        v = _dev_tensor(vs, dev, torch.float32)
        f = _dev_tensor(faces, dev, torch.int64)
        if v.dim() != 2 or v.shape[1] != 3 or f.dim() != 2 or f.shape[1] != 3:
            raise SgbError("SurfaceIndex: vs must be [nv, 3] and faces [nf, 3]")
        nv, nf = int(v.shape[0]), int(f.shape[0])
        if nf == 0 or nf >= 2 ** 31:
            raise SgbError(f"SurfaceIndex: the target needs between 1 and 2^31 - 1 faces, got {nf}")
        if not bool(torch.isfinite(v).all()):
            raise SgbError("SurfaceIndex: the target has a non-finite vertex")
        if bool(((f < 0) | (f >= nv)).any()):
            raise SgbError(f"SurfaceIndex: a face id lies outside [0, {nv})")
        self.device, self.nf = dev, nf
        tri = v[f]                                                       # [nf, 3 corners, 3]
        self.tris = torch.zeros((nf, 12), dtype=torch.float32, device=dev)
        self.tris[:, :9] = tri.reshape(nf, 9)
        lo, hi = v.min(0).values, v.max(0).values
        origin = lo.double()
        ext = (hi.double() - origin).cpu()
        if cell_size is None:
            e = torch.linalg.norm(tri - tri.roll(1, dims=1), dim=2)
            h = float(e.double().mean())
            diag = float(torch.linalg.norm(ext))
            if not h > 0.0:
                h = diag if diag > 0.0 else 1.0
            cells = float(torch.prod(torch.floor(ext / h) + 1))
            if cells > _CELLS_PER_FACE * nf:
                h *= (cells / (_CELLS_PER_FACE * nf)) ** (1.0 / 3.0)
        else:
            h = float(cell_size)
            if not h > 0.0:
                raise SgbError("SurfaceIndex: cell_size must be positive")
        bmin, bmax = tri.min(1).values.double(), tri.max(1).values.double()
        budget = max(_PAIRS_PER_FACE * nf, _PAIRS_FLOOR)
        while True:
            h = float(np.float32(h))                                     # the kernel receives h as a float
            dims = (torch.floor(ext / h) + 1).to(torch.int64)
            while int(torch.prod(dims)) >= 2 ** 31:
                h = float(np.float32(h * 2.0))
                dims = (torch.floor(ext / h) + 1).to(torch.int64)
            g = dims.to(dev)
            c0 = torch.minimum(torch.floor((bmin - origin) / h - _BIN_EPS).clamp_min(0).to(torch.int64), g - 1)
            c1 = torch.minimum(torch.floor((bmax - origin) / h + _BIN_EPS).clamp_min(0).to(torch.int64), g - 1)
            span = c1 - c0 + 1                                           # [nf, 3] cells per axis
            per_face = span.prod(1)
            total = int(per_face.sum())
            if total <= budget or int(torch.prod(dims)) == 1:
                break
            h *= 2.0
        gx, gy, gz = (int(d) for d in dims)
        face_id = torch.repeat_interleave(torch.arange(nf, device=dev), per_face, output_size=total)
        first = torch.cumsum(per_face, 0) - per_face
        k = torch.arange(total, device=dev) - first[face_id]
        sx, sy = span[face_id, 0], span[face_id, 1]
        cx = c0[face_id, 0] + k % sx
        cy = c0[face_id, 1] + (k // sx) % sy
        cz = c0[face_id, 2] + k // (sx * sy)
        cell = (cz * gy + cy) * gx + cx
        cell, order = torch.sort(cell, stable=True)                      # faces ascend inside a cell
        self.cell_faces = face_id[order].to(torch.int32)
        self.cell_start = torch.zeros(gx * gy * gz + 1, dtype=torch.int32, device=dev)
        self.cell_start[1:] = torch.cumsum(torch.bincount(cell, minlength=gx * gy * gz), 0).to(torch.int32)
        self.origin = tuple(float(x) for x in origin.cpu())
        self.cell_size, self.dims, self.pairs = h, (gx, gy, gz), total

    def query(self, points) -> Tuple[Tensor, Tensor]:
        """``(dist float32 [n], face int32 [n])`` of ``points`` [n, 3] against the surface; stream-ordered, no host sync."""
        if isinstance(points, Tensor):
            require_cuda(points)
        p = _dev_tensor(points, self.device, torch.float32)
        if p.dim() != 2 or p.shape[1] != 3:
            raise SgbError("SurfaceIndex.query: points must be [n, 3]")
        if p.stride(1) != 1:
            p = p.contiguous()
        n = int(p.shape[0])
        dist = torch.empty(n, dtype=torch.float32, device=self.device)
        face = torch.empty(n, dtype=torch.int32, device=self.device)
        lib = L.load()
        with torch.cuda.device(self.device):
            check(lib.sgb_point_surface_distance(ptr(p), p.stride(0), n, ptr(self.tris), self.nf, ptr(self.cell_start),
                                                 ptr(self.cell_faces), *self.origin, self.cell_size, *self.dims,
                                                 ptr(dist), ptr(face), stream_ptr(self.device)), "sgb_point_surface_distance")
        L.count(1)
        return dist, face

    def stats(self, points, mask=None) -> Dict[str, Tensor]:
        """fp64 device scalars ``mean``, ``rms``, ``max`` and ``count`` of the distances of ``points`` (those where the
        optional boolean ``mask`` [n] is set) to the surface.  A non-finite distance propagates into mean, rms and max; an
        empty selection gives NaN.  No host sync."""
        d = self.query(points)[0].double()
        if mask is None:
            m = torch.ones_like(d, dtype=torch.bool)
        else:
            if isinstance(mask, Tensor):
                require_cuda(mask)
            m = _dev_tensor(mask, self.device).reshape(-1)
            if m.numel() != d.numel():
                raise SgbError(f"mask has {m.numel()} entries, expected {d.numel()}")
            m = m.bool()
        count = m.sum(dtype=torch.float64)
        w = torch.where(m, d, 0.0)
        mx = torch.where(m, d, float("-inf")).max()
        return {"mean": w.sum(dtype=torch.float64) / count, "rms": torch.sqrt((w * w).sum(dtype=torch.float64) / count),
                "max": torch.where(count > 0, mx, float("nan")), "count": count}


def mesh_distance(a_vs, a_faces, b_vs, b_faces, mask_a=None, mask_b=None) -> dict:
    """Vertex-sampled distances between meshes A (e.g. the network output) and B (e.g. the ground truth), as fp64
    device scalars:

    - ``a_to_b`` / ``b_to_a``: ``mean``, ``rms``, ``max`` (and ``count``) of A's vertices to surface B and of B's vertices
      to surface A;
    - ``a_to_b_mask`` / ``b_to_a_mask`` (when ``mask_a`` / ``mask_b`` is given): the same over the masked vertices only,
      e.g. the hole region ``~v_mask`` of the output; an empty mask gives NaN;
    - ``mean``: the two-sided mean, (a_to_b mean + b_to_a mean) / 2; ``hausdorff``: the larger of the two maxima;
    - ``diag``: the diagonal of B's bounding box (the reference's accuracy is ``mean / diag``).
    """
    ia, ib = SurfaceIndex(a_vs, a_faces), SurfaceIndex(b_vs, b_faces)
    out = {"a_to_b": ib.stats(a_vs), "b_to_a": ia.stats(b_vs)}
    if mask_a is not None:
        out["a_to_b_mask"] = ib.stats(a_vs, mask_a)
    if mask_b is not None:
        out["b_to_a_mask"] = ia.stats(b_vs, mask_b)
    out["mean"] = (out["a_to_b"]["mean"] + out["b_to_a"]["mean"]) * 0.5
    out["hausdorff"] = torch.maximum(out["a_to_b"]["max"], out["b_to_a"]["max"])
    bv = _dev_tensor(b_vs, ib.device, torch.float64)
    out["diag"] = torch.linalg.norm(bv.max(0).values - bv.min(0).values)
    return out
