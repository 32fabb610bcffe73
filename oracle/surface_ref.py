"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Never imported by ``semigcn_b200`` (the product).

Brute-force fp64 point-to-surface distance, the yardstick of ``semigcn_b200.distance`` (csrc/surface_dist.cu).  It tests
every query against every face and shares no method with the kernel: the point is projected onto the face's plane and the
plane distance is taken when the projection lies inside the face (edge-function signs); otherwise, and for zero-area
faces, the distance is the minimum of the three point-to-segment distances.  Unpinned against pymeshlab, which is not
available here (DESIGN.md §3); the tests hold this file to hand-derived answers (tests/test_oracle_surface.py).
"""
from __future__ import annotations

import torch
from torch import Tensor


def _seg_dist(p: Tensor, a: Tensor, b: Tensor) -> Tensor:
    """|p - closest point of segment [a, b]|; p [P, 1, 3], a / b [1, F, 3] -> [P, F]."""
    ab = b - a
    l2 = (ab * ab).sum(-1)
    t = ((p - a) * ab).sum(-1) / torch.where(l2 > 0, l2, torch.ones_like(l2))
    t = torch.where(l2 > 0, t.clamp(0.0, 1.0), torch.zeros_like(t))
    return torch.linalg.norm(p - (a + t.unsqueeze(-1) * ab), dim=-1)


def point_triangle_distances(points: Tensor, vs: Tensor, faces: Tensor) -> Tensor:
    """[P, F] fp64 distances from every point to every closed triangle."""
    p = points.double().unsqueeze(1)
    tri = vs.double()[faces.long()]
    a, b, c = (tri[:, k].unsqueeze(0) for k in range(3))
    n = torch.linalg.cross(b - a, c - a)
    nn = (n * n).sum(-1)
    seg = torch.minimum(torch.minimum(_seg_dist(p, a, b), _seg_dist(p, b, c)), _seg_dist(p, c, a))
    safe = torch.where(nn > 0, nn, torch.ones_like(nn))
    h = ((p - a) * n).sum(-1) / safe                                   # signed height over |n|^2
    proj = p - h.unsqueeze(-1) * n
    inside = nn > 0
    for u, v in ((a, b), (b, c), (c, a)):
        inside = inside & ((torch.linalg.cross(v - u, proj - u) * n).sum(-1) >= 0)
    plane = h.abs() * torch.sqrt(safe)
    return torch.where(inside, plane, seg)


def point_surface_distance(points: Tensor, vs: Tensor, faces: Tensor, chunk: int = 256):
    """(dist [P] fp64, face [P] int64 = the smallest face id attaining dist, second [P] fp64 = the second-smallest
    distance over the other faces, +inf with a single face)."""
    dist, face, second = [], [], []
    for s in range(0, points.shape[0], chunk):
        d = point_triangle_distances(points[s:s + chunk], vs, faces)
        best, idx = d.min(1)                                            # first minimal index = smallest face id
        dist.append(best)
        face.append(idx)
        rest = d.scatter(1, idx.unsqueeze(1), float("inf"))
        second.append(rest.min(1).values)
    return torch.cat(dist), torch.cat(face), torch.cat(second)
