"""Point-to-surface distance (csrc/surface_dist.cu through semigcn_b200/distance.py) against the brute-force fp64 oracle
(oracle/surface_ref.py), against exact answers on the 998 562-vertex icosphere, and the two-sided mesh distance."""
import math

import pytest
import torch

from oracle import surface_ref as S
from semigcn_b200 import SgbError, meshgen
from semigcn_b200.distance import SurfaceIndex, mesh_distance

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _diag(vs):
    return float(torch.linalg.norm(vs.max(0).values - vs.min(0).values))


def _sphere(freq, noisy):
    m = meshgen.icosphere(freq, dtype=torch.float64)
    vs = m.vs
    if noisy:
        g = torch.Generator().manual_seed(freq)
        vs = vs * (1.0 + 0.02 * torch.randn(vs.shape[0], 1, generator=g, dtype=torch.float64))
    return vs.float(), m.faces


def _flat_grid(k=24):
    """An open k x k grid of unit squares in the plane z = 0, two triangles each."""
    ii, jj = torch.meshgrid(torch.arange(k + 1), torch.arange(k + 1), indexing="ij")
    vs = torch.stack([ii.reshape(-1), jj.reshape(-1), torch.zeros((k + 1) ** 2, dtype=torch.int64)], 1).float() * 0.1
    a = (ii[:k, :k] * (k + 1) + jj[:k, :k]).reshape(-1)
    faces = torch.cat([torch.stack([a, a + k + 1, a + 1], 1), torch.stack([a + 1, a + k + 1, a + k + 2], 1)])
    return vs, faces


def _soup():
    """Non-manifold soup: random small triangles, zero-area faces (collinear, two equal and three equal corners),
    duplicated faces and a few faces a hundred times larger than the rest."""
    g = torch.Generator().manual_seed(5)
    c = torch.rand(300, 1, 3, generator=g) * 2 - 1
    small = (c + 0.08 * (torch.rand(300, 3, 3, generator=g) - 0.5)).reshape(-1, 3)
    vs = [small]
    faces = [torch.arange(900).reshape(300, 3)]
    base = 900
    p0, p1 = torch.rand(40, 3, generator=g) * 2 - 1, torch.rand(40, 3, generator=g) * 2 - 1
    t = torch.rand(40, 1, generator=g)
    vs.append(torch.stack([p0, p1, p0 + t * (p1 - p0)], 1).reshape(-1, 3))     # collinear: the third corner on the segment
    faces.append(base + torch.arange(120).reshape(40, 3))
    base += 120
    faces.append(torch.stack([base + torch.arange(40), base + torch.arange(40), base + 40 + torch.arange(40)], 1))
    faces.append(torch.stack([base + torch.arange(40)] * 3, 1))                # coincident corners
    vs.append(torch.rand(80, 3, generator=g) * 2 - 1)
    base += 80
    faces.append(torch.tensor([[0, 1, 2], [base, base + 1, base + 2], [base, base + 2, base + 3]]))
    vs.append(torch.tensor([[-60.0, -60.0, 0.3], [60.0, -60.0, 0.3], [60.0, 60.0, 0.3], [-60.0, 60.0, -40.0]]))
    f = torch.cat(faces)
    dup = f[torch.randperm(f.shape[0], generator=g)[:60]]
    f = torch.cat([f, dup, f[:30]])                                             # duplicates, also of the first faces
    return torch.cat(vs), f


MESHES = {
    "sphere642": lambda: _sphere(8, False),
    "sphere642_noisy": lambda: _sphere(8, True),
    "sphere2562": lambda: _sphere(16, False),
    "sphere2562_noisy": lambda: _sphere(16, True),
    "flat_grid": _flat_grid,
    "soup": _soup,
}


def _queries(vs, faces, seed=0):
    """Points on the surface, within +-1e-4 of the diagonal off it, at ten diagonals away and near the box centre."""
    g = torch.Generator().manual_seed(seed)
    v = vs.double()
    diag = _diag(v)
    tri = v[faces]
    nrm = torch.linalg.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    ok = torch.linalg.norm(nrm, dim=1) > 0
    tri, nrm = tri[ok], nrm[ok]
    nrm = nrm / torch.linalg.norm(nrm, dim=1, keepdim=True)
    pick = torch.randint(0, tri.shape[0], (600,), generator=g)
    w = torch.rand(600, 3, generator=g, dtype=torch.float64)
    w = w / w.sum(1, keepdim=True)
    on = (w.unsqueeze(2) * tri[pick]).sum(1)
    near = on + (torch.rand(600, 1, generator=g, dtype=torch.float64) * 2 - 1) * 1e-4 * diag * nrm[pick]
    u = torch.randn(100, 3, generator=g, dtype=torch.float64)
    centre = (v.max(0).values + v.min(0).values) / 2
    far = centre + 10 * diag * u / torch.linalg.norm(u, dim=1, keepdim=True)
    mid = centre + 0.02 * diag * torch.randn(100, 3, generator=g, dtype=torch.float64)
    return torch.cat([on, near, far, mid]).float()


def _check_against_oracle(vs, faces, pts, dist, face):
    d_ref, f_ref, second = S.point_surface_distance(pts.double(), vs.double(), faces)
    diag = _diag(vs.double())
    err = (dist.double().cpu() - d_ref).abs().max().item()
    assert err <= 1e-6 * diag, f"max |dist - oracle| = {err:.3e} (diag {diag:.3e})"
    clear = (second - d_ref) > 1e-9 * diag
    assert clear.sum() > 0.5 * len(clear)
    bad = (face.cpu().long() != f_ref) & clear
    assert not bool(bad.any()), f"{int(bad.sum())} faces differ from the oracle's, e.g. query {int(bad.nonzero()[0])}"


@pytest.mark.parametrize("name", sorted(MESHES))
def test_matches_fp64_oracle(name):
    vs, faces = MESHES[name]()
    pts = _queries(vs, faces)
    idx = SurfaceIndex(vs.to(DEV), faces.to(DEV))
    dist, face = idx.query(pts.to(DEV))
    assert dist.dtype == torch.float32 and face.dtype == torch.int32
    _check_against_oracle(vs, faces, pts, dist, face)


@pytest.mark.parametrize("name", ["sphere2562_noisy", "flat_grid"])
def test_self_distance_is_zero_on_an_incident_face(name):
    vs, faces = MESHES[name]()
    dist, face = SurfaceIndex(vs.to(DEV), faces.to(DEV)).query(vs.to(DEV))
    assert bool((dist == 0).all())
    n = vs.shape[0]
    first = torch.full((n,), faces.shape[0], dtype=torch.int64)
    first.scatter_reduce_(0, faces.reshape(-1), torch.arange(faces.shape[0]).repeat_interleave(3), reduce="amin")
    assert torch.equal(face.cpu().long(), first)             # the smallest incident face: all of them tie at 0


def _tie_mesh():
    """Six triangles at distance exactly 1 from the origin (one per side of the cube [-1, 1]^3, the origin's foot in each
    interior, every quantity a power of two).  Face 0 is on the +x side, which a ring search reaches last."""
    base = torch.tensor([[1.0, -1.0, -1.0], [1.0, 3.0, -1.0], [1.0, -1.0, 3.0]])
    tris = []
    for axis, sign in ((0, 1.0), (0, -1.0), (1, -1.0), (1, 1.0), (2, -1.0), (2, 1.0)):
        t = base.roll(axis, dims=1)
        t[:, axis] *= sign
        tris.append(t)
    return torch.cat(tris), torch.arange(18).reshape(6, 3)


@pytest.mark.parametrize("name", ["sphere2562_noisy", "flat_grid", "soup", "ties"])
def test_grid_independent_bit_identical(name):
    vs, faces = _tie_mesh() if name == "ties" else MESHES[name]()
    pts = torch.zeros(1, 3) if name == "ties" else _queries(vs, faces, seed=1)
    diag = _diag(vs.double())
    out = []
    for cell in (4 * diag, None, diag / 200):
        idx = SurfaceIndex(vs.to(DEV), faces.to(DEV), cell_size=cell)
        out.append((idx.dims, *idx.query(pts.to(DEV))))
    assert out[0][0] == (1, 1, 1) and out[2][0] != out[1][0]
    for dims, d, f in out[1:]:
        assert torch.equal(d, out[0][1]) and torch.equal(f, out[0][2]), dims
    if name == "ties":
        assert out[0][1].item() == 1.0 and out[0][2].item() == 0


def test_fullsize_icosphere_exact_answers():
    vs, faces = _sphere(316, False)
    assert vs.shape[0] == 998562
    vs, faces = vs.to(DEV), faces.to(DEV)
    diag = _diag(vs.double())
    idx = SurfaceIndex(vs, faces)
    # above face centroids: distance h, nearest face f
    g = torch.Generator(device=DEV).manual_seed(3)
    f = torch.randint(0, faces.shape[0], (30000,), device=DEV, generator=g)
    tri = vs.double()[faces[f]]
    nrm = torch.linalg.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    nrm = nrm / torch.linalg.norm(nrm, dim=1, keepdim=True)
    h = torch.tensor([1e-5, 1e-3, 0.05], dtype=torch.float64, device=DEV).repeat(10000)
    pts = (tri.mean(1) + h.unsqueeze(1) * nrm).float()
    dist, face = idx.query(pts)
    assert (dist.double() - h).abs().max().item() <= 1e-6 * diag
    assert torch.equal(face.long(), f)
    # inside points: the distance to the surface of a convex body is the smallest distance to a face plane
    u = torch.randn(4096, 3, device=DEV, generator=g, dtype=torch.float64)
    inside = (u / torch.linalg.norm(u, dim=1, keepdim=True) * 0.99 * torch.rand(4096, 1, device=DEV, generator=g,
                                                                                 dtype=torch.float64)).float()
    dist, _ = idx.query(inside)
    p = inside.double()
    tri = vs.double()[faces]
    nrm = torch.linalg.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    nrm = nrm / torch.linalg.norm(nrm, dim=1, keepdim=True)
    off = (nrm * tri[:, 0]).sum(1)
    ref = torch.full((4096,), math.inf, dtype=torch.float64, device=DEV)
    for s in range(0, faces.shape[0], 16384):
        ref = torch.minimum(ref, (off[s:s + 16384] - p @ nrm[s:s + 16384].T).min(1).values)
    assert (dist.double() - ref).abs().max().item() <= 1e-6 * diag


def test_non_finite_and_invalid_input():
    vs, faces = MESHES["sphere642_noisy"]()
    idx = SurfaceIndex(vs.to(DEV), faces.to(DEV))
    pts = _queries(vs, faces)[:64].to(DEV)
    d0, f0 = idx.query(pts)
    bad = pts.clone()
    bad[3, 0], bad[10, 2], bad[20, 1] = float("nan"), float("inf"), float("-inf")
    d1, f1 = idx.query(bad)
    rows = torch.tensor([3, 10, 20], device=DEV)
    assert bool(d1[rows].isnan().all()) and bool((f1[rows] == -1).all())
    keep = torch.ones(64, dtype=torch.bool, device=DEV)
    keep[rows] = False
    assert torch.equal(d1[keep], d0[keep]) and torch.equal(f1[keep], f0[keep])
    v_nan = vs.clone()
    v_nan[5, 1] = float("nan")
    with pytest.raises(SgbError):
        SurfaceIndex(v_nan.to(DEV), faces.to(DEV))
    f_bad = faces.clone()
    f_bad[7, 2] = vs.shape[0]
    with pytest.raises(SgbError):
        SurfaceIndex(vs.to(DEV), f_bad.to(DEV))
    with pytest.raises(SgbError):
        SurfaceIndex(vs.to(DEV), (-f_bad).to(DEV))
    with pytest.raises(SgbError):
        SurfaceIndex(vs, faces)
    with pytest.raises(SgbError):
        idx.query(pts.cpu())


def test_deterministic_no_sync_and_graph_capturable():
    vs, faces = MESHES["sphere2562_noisy"]()
    idx = SurfaceIndex(vs.to(DEV), faces.to(DEV))
    pts = _queries(vs, faces).to(DEV)
    mask = torch.arange(pts.shape[0], device=DEV) % 3 == 0
    a, b = idx.query(pts), idx.query(pts)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        idx.query(pts)
        idx.stats(pts)
        idx.stats(pts, mask)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    static = pts.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        idx.query(static)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gd, gf = idx.query(static)
    fresh = _queries(vs, faces, seed=7).to(DEV)
    static.copy_(fresh)
    graph.replay()
    ed, ef = idx.query(fresh)
    torch.cuda.synchronize()
    assert torch.equal(gd, ed) and torch.equal(gf, ef)


def _ref_stats(d, m):
    d = d[m]
    if d.numel() == 0:
        return {"mean": math.nan, "rms": math.nan, "max": math.nan}
    return {"mean": d.mean().item(), "rms": d.square().mean().sqrt().item(), "max": d.max().item()}


def test_mesh_distance_metric_on_the_synthetic_problem():
    prob = meshgen.synth_inpainting_problem(8, n_dummy=1)
    mesh, hole = prob["mesh"], ~prob["v_mask"]
    a_vs, b_vs, faces = prob["ini_vs"], mesh.vs, mesh.faces
    assert 0 < int(hole.sum()) < hole.numel()
    out = mesh_distance(a_vs.numpy(), faces.numpy(), b_vs.to(DEV), faces.to(DEV), mask_a=hole.numpy(), mask_b=hole.to(DEV))
    assert all(v.dtype == torch.float64 and v.is_cuda for k in ("a_to_b", "b_to_a") for v in out[k].values())
    # fp64 reductions of the kernel's own per-point distances
    d_ab = SurfaceIndex(b_vs.to(DEV), faces.to(DEV)).query(a_vs.to(DEV))[0].double().cpu()
    d_ba = SurfaceIndex(a_vs.to(DEV), faces.to(DEV)).query(b_vs.to(DEV))[0].double().cpu()
    every = torch.ones_like(hole)
    want = {"a_to_b": _ref_stats(d_ab, every), "b_to_a": _ref_stats(d_ba, every),
            "a_to_b_mask": _ref_stats(d_ab, hole), "b_to_a_mask": _ref_stats(d_ba, hole)}
    for key, stats in want.items():
        for s, v in stats.items():
            assert math.isclose(out[key][s].item(), v, rel_tol=1e-12), (key, s)
    assert math.isclose(out["mean"].item(), (want["a_to_b"]["mean"] + want["b_to_a"]["mean"]) / 2, rel_tol=1e-12)
    assert out["hausdorff"].item() == max(want["a_to_b"]["max"], want["b_to_a"]["max"])
    assert math.isclose(out["diag"].item(), _diag(b_vs), rel_tol=1e-12)
    assert out["a_to_b_mask"]["count"].item() == int(hole.sum())
    # the same statistics from the oracle's distances
    diag = _diag(b_vs)
    o_ab = S.point_surface_distance(a_vs.float().double(), b_vs.float().double(), faces)[0]
    o_ba = S.point_surface_distance(b_vs.float().double(), a_vs.float().double(), faces)[0]
    for key, d, m in (("a_to_b", o_ab, every), ("b_to_a", o_ba, every), ("a_to_b_mask", o_ab, hole), ("b_to_a_mask", o_ba, hole)):
        for s, v in _ref_stats(d, m).items():
            assert abs(out[key][s].item() - v) <= 1e-6 * diag, (key, s)
    # an empty mask gives NaN
    empty = mesh_distance(a_vs.to(DEV), faces.to(DEV), b_vs.to(DEV), faces.to(DEV), mask_a=torch.zeros_like(hole).to(DEV))
    assert all(math.isnan(empty["a_to_b_mask"][s].item()) for s in ("mean", "rms", "max"))
    assert empty["a_to_b_mask"]["count"].item() == 0
