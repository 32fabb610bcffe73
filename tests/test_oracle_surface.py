"""The brute-force fp64 point-to-surface oracle (oracle/surface_ref.py) against hand-derived answers (CPU)."""
import math

import torch

from oracle import surface_ref as S

D = torch.float64
# one triangle in the plane z = 0: corners (0,0,0), (4,0,0), (0,4,0)
TRI_V = torch.tensor([[0.0, 0.0, 0.0], [4.0, 0.0, 0.0], [0.0, 4.0, 0.0]], dtype=D)
TRI_F = torch.tensor([[0, 1, 2]])


def one(p, vs=TRI_V, faces=TRI_F):
    d, f, _ = S.point_surface_distance(torch.tensor([p], dtype=D), vs, faces)
    return float(d[0]), int(f[0])


def test_above_the_interior_is_the_height():
    assert one([1.0, 1.0, 2.5]) == (2.5, 0)
    assert one([1.0, 1.0, -0.75]) == (0.75, 0)
    assert one([1.0, 1.0, 0.0]) == (0.0, 0)


def test_beyond_an_edge_is_the_segment_distance():
    assert one([2.0, -3.0, 4.0])[0] == 5.0                              # edge on y = 0, foot (2, 0, 0)
    # hypotenuse x + y = 4: (3, 3, 0) is sqrt(2) from its foot (2, 2, 0)
    assert math.isclose(one([3.0, 3.0, 0.0])[0], math.sqrt(2.0), rel_tol=1e-15)


def test_beyond_a_corner_is_the_vertex_distance():
    assert one([-3.0, -4.0, 0.0])[0] == 5.0
    assert math.isclose(one([6.0, -1.0, 2.0])[0], 3.0, rel_tol=1e-15)  # corner (4, 0, 0)
    assert one([0.0, 4.0, 0.0])[0] == 0.0


def test_degenerate_faces():
    vs = torch.tensor([[0.0, 0.0, 0.0], [2.0, 0.0, 0.0], [5.0, 0.0, 0.0], [1.0, 1.0, 1.0]], dtype=D)
    collinear = torch.tensor([[0, 1, 2]])
    assert one([3.0, 4.0, 0.0], vs, collinear)[0] == 4.0                 # the segment [0, 5] on the x axis
    assert one([8.0, 0.0, 4.0], vs, collinear)[0] == 5.0                 # beyond its far end
    coincident = torch.tensor([[3, 3, 3]])
    assert math.isclose(one([1.0, 4.0, 5.0], vs, coincident)[0], 5.0, rel_tol=1e-15)
    two_equal = torch.tensor([[0, 0, 2]])
    assert one([1.0, -2.0, 0.0], vs, two_equal)[0] == 2.0
    # a duplicated face ties exactly: the smaller id wins, and the second-best distance equals the best
    dup = torch.tensor([[0, 1, 3], [0, 2, 3], [0, 1, 3]])
    d, f, second = S.point_surface_distance(torch.tensor([[1.0, -1.0, 0.0]], dtype=D), vs, dup)
    assert int(f[0]) == 0 and float(second[0]) == float(d[0]) == 1.0


def test_inside_a_closed_convex_mesh_is_the_nearest_face_plane():
    # the cube [-1, 2] x [-1, 1] x [-1, 1], two triangles per side
    c = torch.tensor([[x, y, z] for x in (-1.0, 2.0) for y in (-1.0, 1.0) for z in (-1.0, 1.0)], dtype=D)
    quads = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
    faces = torch.tensor([t for a, b, cc, d in quads for t in ((a, b, cc), (a, cc, d))])
    g = torch.Generator().manual_seed(1)
    p = torch.rand(200, 3, generator=g, dtype=D) * torch.tensor([2.8, 1.8, 1.8], dtype=D) - torch.tensor([0.9, 0.9, 0.9], dtype=D)
    d, _, _ = S.point_surface_distance(p, c, faces)
    planes = torch.stack([p[:, 0] + 1, 2 - p[:, 0], p[:, 1] + 1, 1 - p[:, 1], p[:, 2] + 1, 1 - p[:, 2]], 1).min(1).values
    assert torch.allclose(d, planes, rtol=0, atol=1e-14)
