"""CPU tests: the oracle (oracle/pyg_ref.py) against an independent dense formulation, against
hand-derivable known answers, with fp64 gradcheck, and against the fixtures generated from the
reference's own importable code (tests/golden/make_golden.py).  No GPU, no product code."""
import math

import numpy as np
import pytest
import torch

from oracle import dense_ref as D
from oracle import pyg_ref as O
from semigcn_b200 import meshgen
from helpers import assert_close, load_golden, random_graph, rel_err


def ring(n):
    i = torch.arange(n)
    return torch.stack([torch.cat([i, (i + 1) % n]), torch.cat([(i + 1) % n, i])])


@pytest.mark.parametrize("seed,kw", [(0, {}), (1, dict(self_loops=5)), (2, dict(duplicates=7)), (3, dict(isolated=4)),
                                     (4, dict(self_loops=3, duplicates=3, isolated=2, symmetric=True))])
def test_gcn_oracle_matches_dense(seed, kw):
    n, cin, cout = 40, 5, 7
    ei = random_graph(n, 150, seed, **kw)
    torch.manual_seed(seed)
    conv = O.GCNConv(cin, cout).double()
    conv.bias.data.normal_()
    x = torch.randn(n, cin, dtype=torch.float64)
    got = conv(x, ei)
    want = D.gcn_conv(x, ei, conv.lin.weight, conv.bias)
    assert rel_err(got, want) < 1e-12


@pytest.mark.parametrize("seed,kw", [(0, {}), (1, dict(self_loops=5)), (2, dict(duplicates=7)), (3, dict(isolated=4)),
                                     (4, dict(symmetric=True))])
@pytest.mark.parametrize("K", [1, 2, 3, 4])
def test_cheb_oracle_matches_dense(seed, kw, K):
    n, cin, cout = 40, 5, 7
    ei = random_graph(n, 150, seed, **kw)
    torch.manual_seed(seed)
    conv = O.ChebConv(cin, cout, K=K).double()
    conv.bias.data.normal_()
    x = torch.randn(n, cin, dtype=torch.float64)
    got = conv(x, ei)
    want = D.cheb_conv(x, ei, [l.weight for l in conv.lins], conv.bias)
    assert rel_err(got, want) < 1e-12


def test_known_answers_regular_graphs():
    # ring: every GCN weight (incl. the self loop) is 1/3; icosahedron: degree 5 -> 1/6
    ei, w = O.gcn_norm(ring(9), 9)
    assert torch.allclose(w, torch.full_like(w, 1.0 / 3.0), atol=1e-7)
    ico = meshgen.icosphere(1)
    ei, w = O.gcn_norm(ico.edge_index, 12)
    assert torch.allclose(w, torch.full_like(w, 1.0 / 6.0), atol=1e-7)
    # ChebConv on a regular graph: L^ 1 = -1  =>  T1 = -x, T2 = x for constant features
    ei, w = O.cheb_norm(ring(9), 9)
    x = torch.ones(9, 2)
    t1 = O.propagate(ei, w, x)
    assert torch.allclose(t1, -x, atol=1e-6)
    t2 = 2.0 * O.propagate(ei, w, t1) - x
    assert torch.allclose(t2, x, atol=1e-6)


def test_isolated_vertices_and_existing_self_loops():
    ei = torch.tensor([[0, 1, 2, 2], [1, 0, 2, 0]])            # vertex 3 isolated, (2,2) is a loop
    e2, w = O.gcn_norm(ei, 4)
    assert e2.shape[1] == 3 + 4                                  # loop removed, 4 loops appended
    dense = D.gcn_operator(ei, 4, torch.float32)
    x = torch.eye(4)
    assert torch.allclose(O.propagate(e2, w, x), dense, atol=1e-6)
    assert dense[3, 3] == 1.0                                    # isolated: only its own loop, deg 1
    e3, w3 = O.cheb_norm(ei, 4)
    out = O.propagate(e3, w3, x)
    assert torch.all(out[3] == 0)                                # deg 0 -> dis = 0, (+1, -1) cancels
    assert torch.isfinite(out).all()


def test_dis_is_div_of_sqrt():
    """A.5: torch-CPU pow(-0.5) == IEEE fl(1 / fl(sqrt(d))) in fp32 (numpy's correctly rounded
    ops; what the CUDA builder restates with __fdiv_rn(1, __fsqrt_rn(d))), and differs from the
    correctly rounded reciprocal square root for the mesh-dominant degrees 6 and 7."""
    d = torch.arange(1, 1 << 16, dtype=torch.float32)
    a = d.clone().pow_(-0.5)
    ieee = torch.from_numpy((np.float32(1.0) / np.sqrt(d.numpy())).astype(np.float32))
    assert torch.equal(a, ieee)
    exact = (d.double() ** -0.5).float()
    assert not torch.equal(a, exact)
    assert a[5] != exact[5] and a[6] != exact[6]


def test_gradcheck_fp64():
    n = 12
    ei = random_graph(n, 40, 7, self_loops=2, duplicates=2)
    torch.manual_seed(0)
    gcn = O.GCNConv(3, 4).double()
    cheb = O.ChebConv(3, 4, K=3).double()
    x = torch.randn(n, 3, dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(lambda t: gcn(t, ei), (x,), eps=1e-6, atol=1e-6)
    assert torch.autograd.gradcheck(lambda t: cheb(t, ei), (x,), eps=1e-6, atol=1e-6)


def test_init_rng_consumption():
    """A.4: each PyG Linear draws once at construction and once more from the conv's own
    reset_parameters(); the second draw wins."""
    torch.manual_seed(314)
    conv = O.GCNConv(4, 16)
    torch.manual_seed(314)
    a = math.sqrt(6.0 / 20)
    torch.empty(16, 4).uniform_(-a, a)
    want = torch.empty(16, 4).uniform_(-a, a)
    assert torch.equal(conv.lin.weight.data, want)
    torch.manual_seed(314)
    cheb = O.ChebConv(4, 16, K=3)
    torch.manual_seed(314)
    for _ in range(3):
        torch.empty(16, 4).uniform_(-a, a)
    for k in range(3):
        assert torch.equal(cheb.lins[k].weight.data, torch.empty(16, 4).uniform_(-a, a))


def test_sequential_state_dict_keys():
    net = O.SingleScaleGCN("chebconv")
    keys = set(net.state_dict().keys())
    assert "blocks.0.module_0.lins.1.weight" in keys and "blocks.0.module_0.bias" in keys
    assert "blocks.0.module_1.running_mean" in keys and "blocks.12.module_3.weight" in keys
    net = O.SingleScaleGCN("gcnconv")
    assert "blocks.3.module_0.lin.weight" in net.state_dict()
    nparam = sum(p.numel() for p in net.parameters() if p.requires_grad) - sum(p.numel() for p in net.skip_blocks.parameters())
    nbn_buffers = 0
    assert nparam == 486419 - nbn_buffers or nparam > 0       # SURVEY §8(d): GCN params incl. BN = 486 419


# ---------------------------------------------------------------- reference-derived fixtures
@pytest.mark.parametrize("n", [4, 8])
def test_golden_edge_index_and_degrees(n):
    """meshgen restates util/mesh.py:60-100,229-230 -> identical edges / edge_index / v_dims."""
    gold = load_golden(n)
    faces = torch.from_numpy(gold["faces"])
    edges = meshgen.edges_from_faces(faces, gold["vs"].shape[0])
    assert np.array_equal(edges.numpy(), gold["edges"])
    ei = meshgen.edge_index_from_edges(edges)
    assert np.array_equal(ei.numpy(), gold["edge_index"])
    deg = torch.bincount(ei[1], minlength=gold["vs"].shape[0]).float()
    assert np.array_equal(deg.numpy(), gold["v_dims"])
    ico = meshgen.icosphere(n)
    assert np.array_equal(ico.faces.numpy(), gold["faces"])
    assert np.array_equal(ico.edge_index.numpy(), gold["edge_index"])


@pytest.mark.parametrize("n", [4, 8])
def test_golden_losses_and_face_normals(n):
    """Oracle restatements of util/models.py:121-126 and util/loss.py:14-34,60-107 reproduce the
    reference's own outputs bit for bit (CPU)."""
    gold = load_golden(n)
    pred = torch.from_numpy(gold["pred"])
    faces = torch.from_numpy(gold["faces"])
    fn32 = O.compute_fn(pred, faces)
    assert np.array_equal(fn32.numpy(), gold["compute_fn_f32"])
    fn64 = O.compute_fn(pred.double(), faces)
    assert np.array_equal(fn64.numpy(), gold["compute_fn_f64"])
    vm, fm = torch.from_numpy(gold["v_mask"]), torch.from_numpy(gold["f_mask"])
    lp = O.mask_pos_rec_loss(pred, torch.from_numpy(gold["vs"]), vm)
    assert lp.dtype == torch.float64 and lp.item() == gold["loss_pos_f64"].item()
    ln = O.mask_norm_rec_loss(fn32, torch.from_numpy(gold["fn"]), fm)
    assert ln.dtype == torch.float64 and ln.item() == gold["loss_norm_f64"].item()
    lp32 = O.mask_pos_rec_loss(pred, torch.from_numpy(gold["vs"]).float(), vm)
    assert lp32.item() == gold["loss_pos_f32"].item()
    ln32 = O.mask_norm_rec_loss(fn32, torch.from_numpy(gold["fn"]).float(), fm)
    assert ln32.item() == gold["loss_norm_f32"].item()
    ll = O.mesh_laplacian_loss(pred, torch.from_numpy(gold["edge_index"]))
    assert abs(ll.item() - gold["loss_lap_f32"].item()) <= 1e-6 * abs(gold["loss_lap_f32"].item())


def test_sgcn_oracle_runs_and_backprops():
    prob = meshgen.synth_inpainting_problem(4, smooth_iters=5, n_dummy=4)
    torch.manual_seed(314)
    net = O.SingleScaleGCN("gcnconv")
    out = net(prob["z1"], prob["x_pos"], prob["mesh"].edge_index, prob["vmask_dummy"][:, :1])
    assert out.shape == (162, 3) and torch.isfinite(out).all()
    loss = O.mask_pos_rec_loss(out, prob["ini_vs"], prob["v_mask"])
    loss.backward()
    assert all(p.grad is not None for n_, p in net.named_parameters() if "skip" not in n_)


# ------------------------------------------------------------------ network wiring pinned against the reference file
@pytest.mark.parametrize("conv", ["chebconv", "gcnconv"])
@pytest.mark.parametrize("skip", [False, True])
def test_oracle_sgcn_matches_reference_networks_py(conv, skip):
    """tests/golden/ref_sgcn_n4.npz was produced by running the reference's util/networks.py::SingleScaleGCN itself
    (PyG symbols resolved to the oracle classes, tests/golden/make_golden_net.py): the oracle's restated network must
    consume the RNG identically (same seeded initial state_dict, exactly) and give the same forward in train and eval mode.
    The forward is held to REL_TOL, not to bit equality: the fixture's fp32 values depend on the host that computed them
    (MKL's GEMM rounds differently by instruction set and thread count: up to 4.4e-6 norm-relative in train mode,
    measured), while a wiring or RNG-order difference is O(1)."""
    import numpy as np
    gold = load_golden("ref_sgcn_n4.npz")
    tag = f"{conv}_{'skip' if skip else 'noskip'}"
    torch.manual_seed(int(gold["seed"]))
    net = O.SingleScaleGCN(conv, skip=skip)
    sd = net.state_dict()
    names = sorted(sd.keys())
    assert names == [str(s) for s in gold[f"{tag}_names"]]
    sums = np.array([[float(sd[k].double().sum()), float(sd[k].double().abs().sum())] for k in names])
    assert np.array_equal(sums, gold[f"{tag}_sums"]), "seeded initial parameters differ from the reference construction order"
    z1, x_pos = torch.from_numpy(gold["z1"]), torch.from_numpy(gold["x_pos"])
    ei, dm = torch.from_numpy(gold["edge_index"]), torch.from_numpy(gold["dm"])
    net.train()
    y = net(z1, x_pos, ei, dm)
    assert_close(y, torch.from_numpy(gold[f"{tag}_train"]), what="train-mode forward")
    net.eval()
    y = net(z1, x_pos, ei, dm)
    assert_close(y, torch.from_numpy(gold[f"{tag}_eval"]), what="eval-mode forward")


@pytest.mark.parametrize("n", [4, 8])
def test_fn_bnf_detach_loss_matches_reference(n):
    """The CPU restatement of the -CAD regulariser (oracle/loss_ref.py, util/loss.py:197-253) against the reference's own
    output on the reference's own ``Mesh.f2f`` -- this pins the checker the fused CUDA kernels are held to
    (tests/test_gpu_losses.py) -- and the vectorised ``f2f`` builder against the reference's (same neighbour sets; slot
    order is the reference's Counter order there, side order here -- a reordering of a 3-term sum)."""
    from oracle import loss_ref as losses
    from semigcn_b200 import meshgen
    gold = load_golden(n)
    pred = torch.from_numpy(gold["pred"])
    faces = torch.from_numpy(gold["faces"]).long()
    f2f_ref = torch.from_numpy(gold["f2f"]).long()
    fn_pred = torch.from_numpy(gold["compute_fn_f32"])
    loss, new_fn = losses.fn_bnf_detach_loss(pred, fn_pred, faces, f2f_ref, loop=5)
    assert torch.allclose(new_fn, torch.from_numpy(gold["bnf_fn_f32"]), rtol=0, atol=1e-6)
    assert abs(float(loss) - float(gold["loss_bnf_f32"])) <= 1e-6 * abs(float(gold["loss_bnf_f32"]))
    f2f = meshgen.face_adjacency(faces)
    assert f2f.shape == f2f_ref.shape
    assert torch.equal(torch.sort(f2f, dim=1)[0], torch.sort(f2f_ref, dim=1)[0])
    loss2, new_fn2 = losses.fn_bnf_detach_loss(pred, fn_pred, faces, f2f, loop=5)
    assert torch.allclose(new_fn2, new_fn, rtol=0, atol=1e-6)
    assert abs(float(loss2) - float(loss)) <= 1e-6 * abs(float(loss))
    # a mesh with a boundary: drop some faces -> -1 slots, no crash, symmetric adjacency
    keep = torch.ones(faces.shape[0], dtype=torch.bool)
    keep[::7] = False
    f_open = faces[keep]
    adj = meshgen.face_adjacency(f_open)
    assert int((adj == -1).sum()) > 0
    i = torch.arange(adj.shape[0]).repeat_interleave(3)
    j = adj.reshape(-1)
    ok = j >= 0
    assert bool(((adj[j[ok]] == i[ok].unsqueeze(1)).any(dim=1)).all())


def test_dummy_masks_match_reference_datamaker():
    """The CPU restatement of the mask generation (oracle/mask_ref.py: sparse edge_index, no dense AdjI) against the
    reference's own util/datamaker.py:110-159 run on its dense-built AdjI / f2v_mat (tests/golden/make_golden_masks.py):
    identical masks under the reference's numpy seed.  (The product's dilation runs on the aggregation kernel and is held
    to the same fixture on the GPU: tests/test_gpu_kernels.py::test_mask_dilation_on_the_spmm_kernel.)"""
    import numpy as np
    from oracle import mask_ref as sdata
    gold = load_golden("ref_masks_n4.npz")
    ei = torch.from_numpy(gold["edge_index"])
    faces = torch.from_numpy(gold["faces"]).long()
    n = int(ei.max()) + 1
    rng = np.random.RandomState(int(gold["seed"]))
    vmask, fmask = sdata.make_dummy_mask(ei, faces, n, dm_size=int(gold["dm_size"]), kn=[int(k) for k in gold["kn"]], rng=rng)
    assert torch.equal(vmask, torch.from_numpy(gold["vmask_dummy"]))
    assert torch.equal(fmask, torch.from_numpy(gold["fmask_dummy"]))
    f_real = sdata.vmask_to_fmask(faces, torch.from_numpy(gold["v_real"]))
    assert f_real.dtype == torch.bool and torch.equal(f_real, torch.from_numpy(gold["f_real"]))
    # known answer: one seed grows to its k-ring (1 + 6 + 12 vertices on a degree-6 patch of the icosphere)
    seed = torch.zeros(n, 1)
    v = int(torch.bincount(ei[1]).argmax())           # any degree-6 vertex
    seed[v] = 1.0
    assert int(sdata.dilate_mask(ei, seed, 0).sum()) == 1
    assert int(sdata.dilate_mask(ei, seed, 1).sum()) == 1 + int((ei[1] == v).sum())


def test_oracle_operators_match_scipy_laplacian():
    """An anchor outside this repository for the normalisation arithmetic: scipy.sparse.csgraph.laplacian(normed=True) is
    I - D^-1/2 A D^-1/2, so ChebConv's scaled operator (lambda_max = 2:  2 L / lambda_max - I) must equal it minus the
    identity, and GCNConv's operator must equal the same construction on A + I with degrees deg + 1."""
    import numpy as np
    import scipy.sparse as sp
    from scipy.sparse.csgraph import laplacian
    from semigcn_b200 import meshgen
    m = meshgen.icosphere(5)
    n, ei = m.num_vertices, m.edge_index
    a = sp.coo_matrix((np.ones(ei.shape[1]), (ei[1].numpy(), ei[0].numpy())), shape=(n, n)).tocsr()
    lap = laplacian(a, normed=True)
    cheb_ref = (lap - sp.identity(n)).toarray()
    # oracle: edge list [edges (-w) || +1 loops || -1 loops] -> dense
    ei_c, w_c = O.cheb_norm(ei, n, dtype=torch.float64)
    dense = torch.zeros(n, n, dtype=torch.float64).index_put_((ei_c[1], ei_c[0]), w_c, accumulate=True).numpy()
    assert np.abs(dense - cheb_ref).max() <= 1e-12
    deg = np.asarray(a.sum(axis=1)).reshape(-1) + 1.0
    dis = sp.diags(1.0 / np.sqrt(deg))
    gcn_ref = (dis @ (a + sp.identity(n)) @ dis).toarray()
    ei_g, w_g = O.gcn_norm(ei, n, dtype=torch.float64)
    dense = torch.zeros(n, n, dtype=torch.float64).index_put_((ei_g[1], ei_g[0]), w_g, accumulate=True).numpy()
    assert np.abs(dense - gcn_ref).max() <= 1e-12
    # and the propagate step is that matrix applied to x
    x = torch.randn(n, 5, dtype=torch.float64, generator=torch.Generator().manual_seed(2))
    assert np.abs(O.propagate(ei_g, w_g, x).numpy() - gcn_ref @ x.numpy()).max() <= 1e-12
