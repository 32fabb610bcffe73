"""GPU parity tests of the individual C-ABI entry points against the CPU oracle.
Bars (SURVEY.md §8(d)): graph builder and aggregation BIT-EXACT; dense transform / BatchNorm
within 1e-5 norm-relative of an fp64 evaluation."""
import numpy as np
import pytest
import torch

from helpers import (assert_bit_equal, assert_close, load_golden, random_graph, rel_err, stable_csr_from_edges)
from oracle import pyg_ref as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _ops():
    from semigcn_b200 import ops
    return ops


GRAPHS = [
    dict(n=50, nnz=200, seed=0),
    dict(n=64, nnz=300, seed=1, self_loops=9),
    dict(n=64, nnz=300, seed=2, duplicates=40),
    dict(n=70, nnz=200, seed=3, isolated=11),
    dict(n=300, nnz=4000, seed=4, self_loops=5, duplicates=50, isolated=3, symmetric=True),
    dict(n=5000, nnz=60000, seed=5),
    dict(n=20, nnz=4000, seed=6, duplicates=500),          # very long rows (rank kernel, multi-batch gather)
]


def check_moments(partials, y64, tol=2e-6):
    """(count, mean, M2) partial rows merge (Chan) to the exact column count / mean / sum of squared deviations."""
    p = partials.double().cpu()
    n, mean, m2 = p[:, 0], p[:, 1], p[:, 2]
    N = n.sum(0)
    assert torch.all(N == y64.shape[0])
    tot_mean = (n * mean).sum(0) / N
    tot_m2 = m2.sum(0) + (n * (mean - tot_mean) ** 2).sum(0)
    assert_close(tot_mean, y64.mean(0), tol, "mean")
    assert_close(tot_m2, ((y64 - y64.mean(0)) ** 2).sum(0), 10 * tol, "M2")


def _graph(kw):
    kw = dict(kw)
    n = kw.pop("n")
    return n, random_graph(n, **kw)


# ------------------------------------------------------------------ 1. graph builder
@pytest.mark.parametrize("kw", GRAPHS)
@pytest.mark.parametrize("mode", [0, 1])
def test_graph_build_bit_exact(kw, mode):
    ops = _ops()
    n, ei = _graph(kw)
    g = ops.MeshGraph(ei.to(DEV), n, mode, with_perm=True)
    for by_source, (rowptr, colidx, perm) in ((False, (g.rowptr, g.colidx, g.perm)), (True, (g.rowptr_t, g.colidx_t, g.perm_t))):
        rp, ci, pm = stable_csr_from_edges(ei, n, by_source)
        assert_bit_equal(rowptr, rp, "rowptr")
        m = int(rp[-1])
        assert_bit_equal(colidx[:m], ci, "colidx")
        assert_bit_equal(perm, pm, "perm")
    # dis against the oracle's deg.pow_(-0.5) (degree over targets +1 for GCN, over sources for Cheb)
    row, col = ei
    keep = row != col
    if mode == 0:
        deg = torch.bincount(col[keep], minlength=n).float() + 1
    else:
        deg = torch.bincount(row[keep], minlength=n).float()
    dis = deg.pow_(-0.5)
    dis[dis == float("inf")] = 0
    assert_bit_equal(g.dis, dis, "dis")
    # packed (col, weight) stream == the oracle's per-edge norm (gcn_norm / ChebConv.__norm__), slot by slot
    ei2, w = (O.gcn_norm if mode == 0 else O.cheb_norm)(ei, n)
    m = int(keep.sum())
    assert torch.equal(ei2[:, :m], ei[:, keep])                 # the oracle keeps non-loop edges first, in order
    for by_source, edges, perm in ((False, g.edges, g.perm), (True, g.edges_t, g.perm_t)):
        slots, edges = perm.cpu().long()[keep], edges.cpu()
        assert_bit_equal(edges[:, 0][slots], (ei[0] if not by_source else ei[1])[keep].to(torch.int32), "edges.col")
        assert_bit_equal(edges[:, 1].view(torch.float32)[slots], w[:m], "edges.w")


def test_graph_build_all_degrees_bit_exact():
    """dis for every degree 1..4096 (star-like rows) == torch-CPU pow(-0.5) (A.5)."""
    ops = _ops()
    degs = torch.arange(1, 1025)
    n = int(degs.numel()) + 1100
    tgt = torch.repeat_interleave(torch.arange(degs.numel()), degs)
    src = torch.cat([torch.arange(d) + 1024 for d in degs.tolist()])         # sources never equal targets
    ei = torch.stack([src, tgt])
    g = ops.MeshGraph(ei.to(DEV), n, 0)
    want = (degs.float() + 1).pow_(-0.5)
    assert_bit_equal(g.dis[:degs.numel()], want, "dis(deg+1)")


def test_graph_build_errors_and_empty():
    ops = _ops()
    from semigcn_b200 import SgbError
    with pytest.raises(SgbError):
        ops.MeshGraph(torch.tensor([[0, 5], [1, 0]], device=DEV), 3, 0)
    g = ops.MeshGraph(torch.zeros((2, 0), dtype=torch.int64, device=DEV), 4, 0)
    assert g.rowptr.tolist() == [0, 0, 0, 0, 0] and torch.all(g.dis == 1.0)


@pytest.mark.parametrize("n", [4, 8])
def test_graph_build_golden_mesh(n):
    ops = _ops()
    gold = load_golden(n)
    ei = torch.from_numpy(gold["edge_index"])
    nv = gold["vs"].shape[0]
    g = ops.MeshGraph(ei.to(DEV), nv, 1)
    deg = (g.rowptr[1:] - g.rowptr[:-1]).float().cpu()
    assert np.array_equal(deg.numpy(), gold["v_dims"])          # reference util/mesh.py:267
    assert torch.equal(g.rowptr.cpu(), g.rowptr_t.cpu())        # mesh graph is symmetric


# ------------------------------------------------------------------ 2. SpMM
WIDTHS = [1, 3, 4, 8, 16, 32, 60, 64, 128, 130, 256, 512, 640]


@pytest.mark.parametrize("c", WIDTHS)
@pytest.mark.parametrize("mode", [0, 1])
def test_spmm_bit_exact_vs_oracle_propagate(c, mode):
    ops = _ops()
    n, ei = _graph(GRAPHS[4])
    torch.manual_seed(c)
    x = torch.randn(n, c)
    ei2, w = (O.gcn_norm if mode == 0 else O.cheb_norm)(ei, n)
    want = O.propagate(ei2, w, x)
    g = ops.MeshGraph(ei.to(DEV), n, mode)
    got = ops.spmm(g, x.to(DEV))
    assert_bit_equal(got, want, f"spmm mode={mode} c={c}")


@pytest.mark.parametrize("kw", GRAPHS)
def test_spmm_graph_zoo_and_transpose(kw):
    ops = _ops()
    n, ei = _graph(kw)
    torch.manual_seed(1)
    x = torch.randn(n, 32)
    for mode, norm in ((0, O.gcn_norm), (1, O.cheb_norm)):
        g = ops.MeshGraph(ei.to(DEV), n, mode)
        ei2, w = norm(ei, n)
        assert_bit_equal(ops.spmm(g, x.to(DEV)), O.propagate(ei2, w, x), "forward")
        # backward aggregation = autograd of the oracle (index_select backward = index_add over row)
        xr = x.clone().requires_grad_(True)
        O.propagate(ei2, w, xr).backward(torch.ones(n, 32) * x)
        got = ops.spmm(g, x.to(DEV), transpose=True)
        assert_close(got, xr.grad, 2e-6, "transpose")


def test_spmm_epilogue_cheb_recurrence_bias_and_prologue():
    ops = _ops()
    n, ei = _graph(GRAPHS[5])
    torch.manual_seed(2)
    c = 64
    x, t0, bias = torch.randn(n, c), torch.randn(n, c), torch.randn(c)
    ei2, w = O.cheb_norm(ei, n)
    g = ops.MeshGraph(ei.to(DEV), n, 1)
    want = 2.0 * O.propagate(ei2, w, x) - t0
    got = ops.spmm(g, x.to(DEV), alpha=2.0, addend=t0.to(DEV), beta=-1.0)
    assert_bit_equal(got, want, "T2 = 2 L^ T1 - T0")
    g0 = ops.MeshGraph(ei.to(DEV), n, 0)
    ei3, w3 = O.gcn_norm(ei, n)
    want = O.propagate(ei3, w3, x) + bias
    assert_bit_equal(ops.spmm(g0, x.to(DEV), bias=bias.to(DEV)), want, "+bias")
    # fused BN-affine + LeakyReLU on the gathered operand
    mu, sc, sh = torch.randn(c), torch.rand(c) + 0.5, torch.randn(c)
    z = torch.nn.functional.leaky_relu((x - mu) * sc + sh, 0.01)
    want = O.propagate(ei3, w3, z)
    got = ops.spmm(g0, x.to(DEV), in_affine=(mu.to(DEV), sc.to(DEV), sh.to(DEV), 0.01))
    assert_close(got, want, 2e-6, "prologue")


@pytest.mark.parametrize("c", [4, 16, 64, 256, 512])
def test_spmm_stats_epilogue(c):
    ops = _ops()
    n, ei = _graph(GRAPHS[5])
    torch.manual_seed(3)
    x = torch.randn(n, c) + 0.3
    g = ops.MeshGraph(ei.to(DEV), n, 0)
    y, partials = ops.spmm(g, x.to(DEV), want_stats=True)
    check_moments(partials, y.double().cpu())


def test_spmm_deterministic():
    ops = _ops()
    n, ei = _graph(GRAPHS[5])
    x = torch.randn(n, 128, device=DEV)
    g = ops.MeshGraph(ei.to(DEV), n, 0)
    a = ops.spmm(g, x)
    for _ in range(3):
        assert torch.equal(a, ops.spmm(g, x))


# ------------------------------------------------------------------ 3. dense transform
SHAPES = [(1000, 16, 4), (1000, 3, 16), (777, 32, 16), (1030, 64, 32), (515, 128, 64), (2049, 256, 128), (1200, 512, 256),
          (640, 256, 512), (130, 130, 70), (128, 48, 200)]


@pytest.mark.parametrize("m,n,k", SHAPES)
@pytest.mark.parametrize("transb", [True, False])
def test_gemm_vs_fp64(m, n, k, transb):
    ops = _ops()
    torch.manual_seed(m + n + k)
    a = torch.randn(m, k)
    b = torch.randn(n, k) if transb else torch.randn(k, n)
    bias = torch.randn(n)
    want = a.double() @ (b.double().t() if transb else b.double()) + bias.double()
    got, partials = ops.gemm(a.to(DEV), b.to(DEV), transb=transb, bias=bias.to(DEV), want_stats=True)
    assert_close(got, want, 2e-6, "gemm")
    check_moments(partials, got.double().cpu())
    # accumulate
    c0 = torch.randn(m, n)
    got2 = ops.gemm(a.to(DEV), b.to(DEV), transb=transb, out=c0.to(DEV).clone(), accumulate=True)
    assert_close(got2, want - bias.double() + c0.double(), 2e-6, "accumulate")


def test_gemm_unknown_engine_is_refused():
    """sgb_gemm takes engines 0, 1 and 3, sgb_gemm_tn 0, 1, 3 and 4: engine 2 is an error, not a fallback."""
    ops = _ops()
    from semigcn_b200._lib import SgbError
    a = torch.randn(3000, 128, device=DEV)
    with pytest.raises(SgbError, match="bad engine 2"):
        ops.gemm(a, torch.randn(256, 128, device=DEV), engine=2)
    with pytest.raises(SgbError, match="bad engine 2"):
        ops.gemm_tn(torch.randn(3000, 256, device=DEV), a, engine=2)


@pytest.mark.parametrize("m,n,k", [(5000, 16, 4), (4097, 64, 32), (3000, 256, 128), (2500, 130, 70), (100000, 32, 16), (300, 512, 256)])
def test_gemm_tn_and_colsum(m, n, k):
    ops = _ops()
    torch.manual_seed(m)
    g, a = torch.randn(m, n), torch.randn(m, k)
    got = ops.gemm_tn(g.to(DEV), a.to(DEV))
    assert_close(got, g.double().t() @ a.double(), 5e-6, "gemm_tn")
    again = ops.gemm_tn(g.to(DEV), a.to(DEV))
    assert torch.equal(got, again), "split-m reduction must be deterministic"
    acc = ops.gemm_tn(g.to(DEV), a.to(DEV), out=got.clone(), accumulate=True)
    assert_close(acc, 2 * (g.double().t() @ a.double()), 5e-6, "gemm_tn accumulate")
    assert_close(ops.gemm_tn(g.to(DEV), a.to(DEV), engine=1), g.double().t() @ a.double(), 2e-6, "gemm_tn fp32 tiles")
    assert_close(ops.colsum(g.to(DEV)), g.double().sum(0), 2e-6, "colsum")


# ------------------------------------------------------------------ 4. BatchNorm + LeakyReLU
@pytest.mark.parametrize("m,c", [(1000, 4), (5000, 16), (3001, 3), (2000, 130), (4000, 256), (777, 512)])
@pytest.mark.parametrize("slope", [0.01, 0.0, 1.0])
def test_bn_act_forward_backward_vs_torch(m, c, slope):
    ops = _ops()
    torch.manual_seed(c)
    y = torch.randn(m, c) * 2 + 0.7
    bn_ref = torch.nn.BatchNorm1d(c).double()
    bn_ref.weight.data.uniform_(0.5, 1.5)
    bn_ref.bias.data.normal_()
    bn = torch.nn.BatchNorm1d(c).to(DEV)
    bn.load_state_dict({k: v.float() if v.dtype.is_floating_point else v for k, v in bn_ref.state_dict().items()})
    yr = y.double().requires_grad_(True)
    zr = torch.nn.functional.leaky_relu(bn_ref(yr), slope)
    dz = torch.randn(m, c)
    zr.backward(dz.double())
    yg = y.to(DEV).requires_grad_(True)
    z = ops.bn_act(yg, bn, slope)
    z.backward(dz.to(DEV))
    assert_close(z, zr, 2e-6, "z")
    assert_close(yg.grad, yr.grad, 1e-5, "dy")
    assert_close(bn.weight.grad, bn_ref.weight.grad, 1e-5, "dgamma")
    assert_close(bn.bias.grad, bn_ref.bias.grad, 1e-5, "dbeta")
    assert_close(bn.running_mean, bn_ref.running_mean, 1e-6, "running_mean")
    assert_close(bn.running_var, bn_ref.running_var, 1e-6, "running_var")
    assert int(bn.num_batches_tracked) == 1
    # eval mode uses the running statistics
    bn.eval(); bn_ref.eval()
    assert_close(ops.bn_act(y.to(DEV), bn, slope), torch.nn.functional.leaky_relu(bn_ref(y.double()), slope), 2e-6, "eval")


# ------------------------------------------------------------------ 5. tcgen05 fp16-split engine
TC_SHAPES = [(1000, 64, 64), (129, 16, 8), (5000, 256, 256), (4100, 512, 256), (3000, 128, 64), (2500, 256, 512), (1000, 48, 36),
             (20000, 256, 128), (777, 80, 200),
             # many tiles per CTA (the kernels are persistent, one CTA per SM): the ring positions / phases of every role wrap
             # dozens of times and the converter groups drift apart -- the regime of the 1 M-vertex bench (a parity-aliasing
             # hang of the two-group converter only showed there, never on the one-tile-per-CTA shapes above)
             (150001, 256, 256), (120000, 512, 96), (90000, 64, 352)]


@pytest.mark.parametrize("m,n,k", TC_SHAPES)
@pytest.mark.parametrize("transb", [True, False])
@pytest.mark.parametrize("engine", [3])
def test_gemm_tensor_core_engine_vs_fp64(m, n, k, transb, engine):
    """engine=3 (tcgen05, error-compensated 2xFP16 split) must hold the same fp32-level bar as the CUDA-core tiles."""
    ops = _ops()
    torch.manual_seed(m + n + k)
    a = torch.randn(m, k)
    b = torch.randn(n, k) if transb else torch.randn(k, n)
    bias = torch.randn(n)
    want = a.double() @ (b.double().t() if transb else b.double()) + bias.double()
    got, partials = ops.gemm(a.to(DEV), b.to(DEV), transb=transb, bias=bias.to(DEV), want_stats=True, engine=engine)
    assert_close(got, want, 5e-6, "gemm tc")   # tensor-core accumulation truncates: a few e-6, bar is 1e-5
    check_moments(partials, got.double().cpu())
    c0 = torch.randn(m, n)
    got2 = ops.gemm(a.to(DEV), b.to(DEV), transb=transb, out=c0.to(DEV).clone(), accumulate=True, engine=engine)
    assert_close(got2, want - bias.double() + c0.double(), 5e-6, "accumulate")
    again = ops.gemm(a.to(DEV), b.to(DEV), transb=transb, bias=bias.to(DEV), engine=engine)
    assert torch.equal(got, again), "tensor-core path must be deterministic"
    # a caller-supplied max|A| (any power-of-two bracket of the true one) gives the same bits
    amax = a.abs().max().reshape(1).to(DEV)
    assert torch.equal(got, ops.gemm(a.to(DEV), b.to(DEV), transb=transb, bias=bias.to(DEV), engine=engine, a_amax=amax))


@pytest.mark.parametrize("scale_a,scale_b", [(1e-9, 1.0), (3e4, 1e-3), (1e-20, 1e12), (1.0, 1e-30)])
def test_gemm_f16_split_engine_scales(scale_a, scale_b):
    """engine=3 rescales both operands by a per-tensor power of two: tiny gradients / large activations keep
    fp32-level (norm-relative) accuracy, and elements six orders of magnitude below the maximum keep row accuracy."""
    ops = _ops()
    torch.manual_seed(11)
    m, n, k = 3000, 128, 256
    a, b = torch.randn(m, k) * scale_a, torch.randn(n, k) * scale_b
    got = ops.gemm(a.to(DEV), b.to(DEV), engine=3)
    assert_close(got, a.double() @ b.double().t(), 5e-6, "scaled operands")
    rows = torch.logspace(-6, 0, m).reshape(-1, 1)
    a2 = a * rows
    got = ops.gemm(a2.to(DEV), b.to(DEV), engine=3)
    want = a2.double() @ b.double().t()
    row_err = ((got.cpu().double() - want).abs().max(1)[0] / want.abs().max(1)[0]).max().item()
    assert row_err <= 1e-5, f"row-relative error {row_err:.2e}"
    g = torch.randn(m, n) * scale_b
    got = ops.gemm_tn(g.to(DEV), a.to(DEV), engine=3)
    assert_close(got, g.double().t() @ a.double(), 5e-6, "scaled operands (tn)")


@pytest.mark.parametrize("m,n,k", [(5000, 128, 64), (4097, 64, 32), (30000, 256, 256), (2500, 132, 72), (100000, 512, 256),
                                   (70000, 256, 512), (300, 16, 4), (9000, 64, 128),
                                   # narrow shapes, hundreds of stages per CTA: the two alternating converter groups
                                   (400000, 32, 64), (300001, 64, 32), (250000, 16, 16), (199999, 48, 36), (350000, 64, 128)])
@pytest.mark.parametrize("engine", [3])
def test_gemm_tn_tensor_core_engine(m, n, k, engine):
    """Weight gradient on tcgen05 (split over vertices, fixed-order reduce), 2xFP16-split engine."""
    ops = _ops()
    torch.manual_seed(m + k)
    g, a = torch.randn(m, n), torch.randn(m, k)
    want = g.double().t() @ a.double()
    got = ops.gemm_tn(g.to(DEV), a.to(DEV), engine=engine)
    assert_close(got, want, 5e-6, "gemm_tn tc")
    assert torch.equal(got, ops.gemm_tn(g.to(DEV), a.to(DEV), engine=engine)), "must be deterministic"
    acc = ops.gemm_tn(g.to(DEV), a.to(DEV), out=got.clone(), accumulate=True, engine=engine)
    assert_close(acc, 2 * want, 5e-6, "accumulate")


def test_bn_near_constant_channels():
    """Channels with |mean| >> std (e.g. the mask channel of the SGCN input, util/networks.py:79):
    the centred affine and the (count, mean, M2) partials must keep fp32-level accuracy where
    sum / sum-of-squares statistics and x*scale + shift' lose it."""
    ops = _ops()
    torch.manual_seed(11)
    m, c = 20000, 16
    y = 300.0 + 1e-2 * torch.randn(m, c)
    y[:, 3] = 1.0 + 1e-4 * torch.randn(m)
    bn_ref = torch.nn.BatchNorm1d(c).double()
    bn = torch.nn.BatchNorm1d(c).to(DEV)
    yr = y.double().requires_grad_(True)
    zr = torch.nn.functional.leaky_relu(bn_ref(yr), 0.01)
    dz = torch.randn(m, c)
    zr.backward(dz.double())
    yg = y.to(DEV).requires_grad_(True)
    z = ops.bn_act(yg, bn, 0.01)
    z.backward(dz.to(DEV))
    bn32 = torch.nn.BatchNorm1d(c)
    z32 = torch.nn.functional.leaky_relu(bn32(y), 0.01)
    e_ours, e_t32 = rel_err(z, zr), rel_err(z32, zr)
    assert e_ours <= max(2.0 * e_t32, 1e-5), f"ours {e_ours:.2e} vs torch-fp32 {e_t32:.2e}"
    assert_close(bn.running_var, bn_ref.running_var, 1e-4, "running_var")


# ------------------------------------------------------------------------------------------------------------------
# mask generation on the aggregation kernel, boolean semiring (SURVEY.md §8(f)-3)
# ------------------------------------------------------------------------------------------------------------------
def test_mask_dilation_on_the_spmm_kernel():
    """semigcn_b200.data.make_dummy_mask / dilate_mask / vmask_to_fmask on the GPU (k-ring dilation = SpMM in SGB_MODE_ADJ
    with the identity in the epilogue, then > 0) against the masks the REFERENCE's own util/datamaker.py:110-159 produced
    under its numpy seed (tests/golden/make_golden_masks.py): bit-identical."""
    import numpy as np
    from oracle import mask_ref
    from semigcn_b200 import SgbError, data as sdata, meshgen
    gold = load_golden("ref_masks_n4.npz")
    ei = torch.from_numpy(gold["edge_index"]).to(DEV)
    faces = torch.from_numpy(gold["faces"]).long().to(DEV)
    n = int(ei.max()) + 1
    rng = np.random.RandomState(int(gold["seed"]))
    vmask, fmask = sdata.make_dummy_mask(ei, faces, n, dm_size=int(gold["dm_size"]), kn=[int(k) for k in gold["kn"]], rng=rng)
    assert torch.equal(vmask.cpu(), torch.from_numpy(gold["vmask_dummy"]))
    assert torch.equal(fmask.cpu(), torch.from_numpy(gold["fmask_dummy"]))
    f_real = sdata.vmask_to_fmask(faces, torch.from_numpy(gold["v_real"]).to(DEV))
    assert f_real.dtype == torch.bool and torch.equal(f_real.cpu(), torch.from_numpy(gold["f_real"]))
    # a larger mesh, the reference's default sizes (40 masks per ring count, 3 / 4 / 5 rings), against the CPU restatement
    m = meshgen.icosphere(20)
    g = torch.Generator().manual_seed(3)
    seeds = (torch.rand(m.num_vertices, 40, generator=g) < 0.014).float()
    for rings in (0, 1, 4):
        got = sdata.dilate_mask(m.edge_index.to(DEV), seeds.to(DEV), rings)
        assert torch.equal(got.cpu(), mask_ref.dilate_mask(m.edge_index, seeds, rings)), rings
    with pytest.raises(SgbError):
        sdata.dilate_mask(m.edge_index, seeds, 1)              # CPU tensors are refused: no fallback


# ------------------------------------------------------------------------------------------------------------------
# Mesh drop-in (topology tables + CG refinement) on the GPU (SURVEY.md §8(f)-4)
# ------------------------------------------------------------------------------------------------------------------
def test_mesh_dropin_on_gpu(tmp_path):
    """The same tensor code as tests/test_mesh_topology.py with device="cuda": identical tables on the reference fixture, and a
    100 002-vertex mesh (the reference's dense N x N construction would need 40 GB there) whose refinement solve converges."""
    import os
    from semigcn_b200 import meshgen
    from semigcn_b200.mesh import Mesh
    from test_mesh_topology import check_against_fixture
    gold = load_golden("ref_meshtopo_n8.npz")
    path = os.path.join(str(tmp_path), "m.obj")
    meshgen.write_obj(path, torch.from_numpy(gold["obj_vs"]), torch.from_numpy(gold["faces"]))
    m = Mesh(path, device=DEV)
    assert m.Lap.is_cuda
    check_against_fixture(m, gold)
    out = Mesh.mesh_merge(m.Lap, m, torch.from_numpy(gold["merge_new_pos"]), torch.from_numpy(gold["merge_preserve"]), w=1.0)
    assert out.is_cuda and np.abs(out.cpu().numpy() - gold["merge_f64"]).max() <= 1e-6 * np.abs(gold["merge_f64"]).max()
    ico = meshgen.icosphere(100, dtype=torch.float64)
    big = Mesh(vs=ico.vs.numpy(), faces=ico.faces.numpy(), device=DEV)
    assert len(big.edges) == 300000 and big.edge_index.shape == (2, 600000)
    g = torch.Generator().manual_seed(1)
    new_pos = torch.from_numpy(big.vs).float() + 0.01 * torch.randn(len(big.vs), 3, generator=g)
    preserve = torch.from_numpy(big.vs[:, 2] < 0.9)
    ref, info = Mesh.mesh_merge(big.Lap, big, new_pos, preserve, w=1.0, return_info=True)
    assert info["relative_residual"] <= 1e-8, info
    keep = preserve.numpy()
    assert np.abs(ref.cpu().numpy()[keep] - big.vs[keep].astype(np.float32)).max() <= 0.05


def test_input_prep_bit_identical_to_the_reference_ops():
    """util/networks.py:67-79 (bounding-box normalise, mask multiply, concatenate) as two kernels: bit-identical to the torch ops."""
    from semigcn_b200 import ops
    g = torch.Generator().manual_seed(9)
    for n in (1, 37, 10242, 300001):
        z1 = (torch.randn(n, 3, generator=g) * torch.tensor([0.3, 2.0, 0.01]) + torch.tensor([-1.0, 0.5, 3.0]))
        dm = (torch.rand(n, 1, generator=g) > 0.2).float()
        z_min, z_max = torch.min(z1, dim=0, keepdim=True)[0], torch.max(z1, dim=0, keepdim=True)[0]
        z_sc = torch.max(z_max - z_min)
        zc = (z_min + z_max) * 0.5
        want = torch.cat([dm * ((z1 - zc) / z_sc), dm], dim=1)
        if n == 1:
            continue                       # z_sc = 0: the reference divides by zero (NaN); nothing to pin
        got = ops.input_prep(z1.to(DEV), dm.to(DEV))
        assert_bit_equal(got, want, f"input_prep n={n}")
        ones = ops.input_prep(z1.to(DEV), None)
        assert_bit_equal(ones, torch.cat([(z1 - zc) / z_sc, torch.ones(n, 1)], dim=1), f"input_prep (no mask) n={n}")


PAIR_SHAPES = [(100000, 256, 256), (65537, 512, 256), (40000, 256, 512), (20011, 256, 128), (9000, 256, 32), (33000, 512, 96)]


@pytest.mark.parametrize("m,n,k", PAIR_SHAPES)
def test_gemm_tn_pair_engine(m, n, k):
    """Weight gradient on CTA pairs (cta_group::2, engine=4): same accuracy / determinism bar as the single-CTA engines."""
    ops = _ops()
    gen = torch.Generator().manual_seed(m + n + k)
    g = torch.randn(m, n, generator=gen) * 1e-3
    a = torch.randn(m, k, generator=gen)
    want = g.double().t() @ a.double()
    got = ops.gemm_tn(g.to(DEV), a.to(DEV), engine=4)
    assert_close(got, want, 1e-5, f"gemm_tn pair engine {m}x{n}x{k}")
    assert torch.equal(got, ops.gemm_tn(g.to(DEV), a.to(DEV), engine=4)), "must be deterministic"
    acc = ops.gemm_tn(g.to(DEV), a.to(DEV), out=got.clone(), accumulate=True, engine=4)
    assert_close(acc, 2 * want, 1e-5, "accumulate")


F16_PAIR_SHAPES = [(100000, 256, 256), (65537, 512, 256), (40001, 256, 512), (33000, 128, 64), (50000, 352, 96), (70001, 32, 16),
                   (129, 256, 64), (300, 512, 32)]


@pytest.mark.parametrize("m,n,k", F16_PAIR_SHAPES)
@pytest.mark.parametrize("transb", [True, False])
def test_gemm_f16_split_engine_on_cta_pairs(m, n, k, transb, monkeypatch):
    """The fp16-split transform on CTA pairs (cta_group::2, UMMA M = 256): forced on with SGB_F16_PAIR=1 for every shape whose
    n-tiles split into two halves of whole core-matrix rows, compared with fp64 and with the single-CTA kernel (SGB_F16_PAIR=0);
    odd numbers of m-tiles (the second CTA of the last pair has no rows), partial n-tiles, one tile pair in all."""
    ops = _ops()
    torch.manual_seed(m + n + k)
    a = torch.randn(m, k)
    b = torch.randn(n, k) if transb else torch.randn(k, n)
    bias = torch.randn(n)
    want = a.double() @ (b.double().t() if transb else b.double()) + bias.double()
    monkeypatch.setenv("SGB_F16_PAIR", "1")
    got, partials = ops.gemm(a.to(DEV), b.to(DEV), transb=transb, bias=bias.to(DEV), want_stats=True, engine=3)
    assert_close(got, want, 5e-6, "gemm on CTA pairs")
    check_moments(partials, got.double().cpu())
    c0 = torch.randn(m, n)
    got2 = ops.gemm(a.to(DEV), b.to(DEV), transb=transb, out=c0.to(DEV).clone(), accumulate=True, engine=3)
    assert_close(got2, want - bias.double() + c0.double(), 5e-6, "accumulate")
    assert torch.equal(got, ops.gemm(a.to(DEV), b.to(DEV), transb=transb, bias=bias.to(DEV), engine=3)), "must be deterministic"
    monkeypatch.setenv("SGB_F16_PAIR", "0")
    single = ops.gemm(a.to(DEV), b.to(DEV), transb=transb, bias=bias.to(DEV), engine=3)
    assert_close(got, single.double(), 1e-6, "pair vs single CTA")
