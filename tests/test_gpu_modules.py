"""GPU parity tests at the drop-in boundary: our GCNConv / ChebConv / Sequential / SGCN against
the CPU oracle (restatement of PyG 2.2.0) on the same seeded inputs and identical state_dicts.
Tolerance: max|a-b| / max|b| <= 1e-5 for layer outputs and gradients (BASELINE.json north_star)."""
import copy

import numpy as np
import pytest
import torch
import torch.nn as nn

from helpers import REL_TOL, assert_close, load_golden, random_graph, rel_err
from oracle import pyg_ref as O
from semigcn_b200 import meshgen

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _grads_close(ours: nn.Module, ref: nn.Module, tol=REL_TOL, skip_zero_bias=True):
    ro = dict(ref.named_parameters())
    for name, p in ours.named_parameters():
        r = ro[name]
        if r.grad is None:
            assert p.grad is None or p.grad.abs().max() == 0, name
            continue
        assert p.grad is not None, name
        if skip_zero_bias and name.endswith("module_0.bias"):
            # a conv bias followed by BatchNorm has an exactly-zero true gradient: both sides hold
            # rounding noise only; compare on the scale of the weight gradient instead
            continue
        assert_close(p.grad, r.grad, tol, name)


@pytest.mark.parametrize("cin,cout", [(4, 16), (16, 32), (64, 128), (128, 64), (256, 256), (16, 3), (3, 5)])
@pytest.mark.parametrize("kind", ["gcn", "cheb"])
def test_conv_forward_backward_vs_oracle(cin, cout, kind):
    from semigcn_b200.nn import ChebConv, GCNConv
    mesh = meshgen.icosphere(6)
    n = mesh.num_vertices
    torch.manual_seed(cin * 1000 + cout)
    ref = O.GCNConv(cin, cout) if kind == "gcn" else O.ChebConv(cin, cout, K=3)
    ref.bias.data.normal_()
    ours = (GCNConv(cin, cout) if kind == "gcn" else ChebConv(cin, cout, K=3))
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(DEV)
    x = torch.randn(n, cin)
    dy = torch.randn(n, cout)
    xr = x.clone().requires_grad_(True)
    yr = ref(xr, mesh.edge_index)
    yr.backward(dy)
    xg = x.to(DEV).requires_grad_(True)
    y = ours(xg, mesh.edge_index.to(DEV))
    y.backward(dy.to(DEV))
    assert_close(y, yr, REL_TOL, "output")
    assert_close(xg.grad, xr.grad, REL_TOL, "dx")
    _grads_close(ours, ref, skip_zero_bias=False)


@pytest.mark.parametrize("kw", [dict(n=200, nnz=1500, seed=11, self_loops=7, duplicates=30, isolated=5),
                                dict(n=300, nnz=2000, seed=12, symmetric=True)])
@pytest.mark.parametrize("kind", ["gcn", "cheb"])
def test_conv_on_irregular_graphs(kw, kind):
    """Asymmetric edge lists, duplicates, existing self loops, isolated vertices."""
    from semigcn_b200.nn import ChebConv, GCNConv
    kw = dict(kw)
    n = kw.pop("n")
    ei = random_graph(n, **kw)
    torch.manual_seed(5)
    ref = O.GCNConv(8, 12) if kind == "gcn" else O.ChebConv(8, 12, K=3)
    ours = (GCNConv(8, 12) if kind == "gcn" else ChebConv(8, 12, K=3))
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(DEV)
    x = torch.randn(n, 8)
    xr = x.clone().requires_grad_(True)
    yr = ref(xr, ei)
    yr.backward(torch.ones_like(yr))
    xg = x.to(DEV).requires_grad_(True)
    y = ours(xg, ei.to(DEV))
    y.backward(torch.ones_like(y))
    assert_close(y, yr, REL_TOL, "output")
    assert_close(xg.grad, xr.grad, REL_TOL, "dx")
    _grads_close(ours, ref, skip_zero_bias=False)


@pytest.mark.parametrize("K", [1, 2, 4])
def test_chebconv_other_orders(K):
    from semigcn_b200.nn import ChebConv
    mesh = meshgen.icosphere(4)
    torch.manual_seed(K)
    ref = O.ChebConv(6, 10, K=K)
    ours = ChebConv(6, 10, K=K)
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(DEV)
    x = torch.randn(mesh.num_vertices, 6)
    xr = x.clone().requires_grad_(True)
    yr = ref(xr, mesh.edge_index)
    yr.sum().backward()
    xg = x.to(DEV).requires_grad_(True)
    y = ours(xg, mesh.edge_index.to(DEV))
    y.sum().backward()
    assert_close(y, yr, REL_TOL, "output")
    assert_close(xg.grad, xr.grad, REL_TOL, "dx")
    _grads_close(ours, ref, skip_zero_bias=False)


@pytest.mark.parametrize("cin,cout", [(4, 16), (64, 128), (128, 32), (16, 3)])
@pytest.mark.parametrize("kind", ["gcn", "cheb"])
@pytest.mark.parametrize("train", [True, False])
def test_fused_block_vs_oracle_sequential(cin, cout, kind, train):
    """conv -> BatchNorm1d -> LeakyReLU (-> Linear) exactly as util/networks.py:24-36 builds it."""
    from semigcn_b200.nn import ChebConv, GCNConv, Sequential
    mesh = meshgen.icosphere(7)
    n = mesh.num_vertices
    torch.manual_seed(cin + cout)

    def build(mod):
        conv = (mod.GCNConv(cin, cout) if kind == "gcn" else mod.ChebConv(cin, cout, K=3))
        return mod.Sequential("x, edge_index", [(conv, "x, edge_index -> x"), nn.BatchNorm1d(cout), nn.LeakyReLU(),
                                                (nn.Linear(cout, 3), "x -> x")])
    import semigcn_b200.nn as OURS
    ref = build(O)
    ref.module_1.weight.data.uniform_(0.5, 1.5)
    ref.module_1.bias.data.normal_()
    ref.module_1.running_mean.normal_()
    ref.module_1.running_var.uniform_(0.5, 2.0)
    ours = build(OURS)
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(DEV)
    ref.train(train); ours.train(train)
    x = torch.randn(n, cin)
    dy = torch.randn(n, 3)
    xr = x.clone().requires_grad_(True)
    yr = ref(xr, mesh.edge_index)
    yr.backward(dy)
    xg = x.to(DEV).requires_grad_(True)
    y = ours(xg, mesh.edge_index.to(DEV))
    y.backward(dy.to(DEV))
    assert_close(y, yr, REL_TOL, "output")
    assert_close(xg.grad, xr.grad, REL_TOL, "dx")
    _grads_close(ours, ref)
    for k in ("module_1.running_mean", "module_1.running_var", "module_1.num_batches_tracked"):
        assert_close(ours.state_dict()[k].float(), ref.state_dict()[k].float(), 1e-6, k)


def _sgcn_pair(conv, seed=314, skip=False):
    from semigcn_b200.networks import SingleScaleGCN
    torch.manual_seed(seed)
    ref = O.SingleScaleGCN(conv, skip=skip)
    ours = SingleScaleGCN(DEV, conv=conv, skip=skip)
    ours.load_state_dict(ref.state_dict())
    return ours.to(DEV), ref


# (icosphere frequency, weight seeds, skip, conv): 1 002 vertices run every transform on the CUDA-core tiles, 33 642 vertices
# run them on the tcgen05 fp16-split CTA pairs (m >= 32 768)
SGCN_CASES = ([pytest.param(10, (314, 1, 2), skip, conv, id=f"{skip}-{conv}") for skip in (False, True)
               for conv in ("gcnconv", "chebconv")]
              + [pytest.param(58, (314,), False, conv, id=f"n33642-False-{conv}") for conv in ("gcnconv", "chebconv")])


@pytest.mark.parametrize("freq,seeds,skip,conv", SGCN_CASES)
def test_sgcn_forward_backward_vs_oracle(freq, seeds, skip, conv):
    """Whole 13-block SGCN (util/networks.py) on a 1 002-vertex icosphere with three weight seeds, and on a 33 642-vertex
    one (the tensor-core path) with one.
    Positions and loss must match the fp32 CPU oracle to 1e-5 (at 33 642 vertices, where the fp32 oracle is itself further
    than that from fp64: be within max(1e-5, 2x the fp32 oracle's distance) of fp64).
    Gradients that crossed 13 BatchNorm + LeakyReLU layers are compared with an fp64 evaluation of the
    oracle.  In ANY fp32 implementation they carry amplified rounding noise plus discrete LeakyReLU
    "kink flips" (a pre-activation within rounding of zero takes the other branch than in fp64): the
    fp32 CPU oracle itself is 1e-6 .. 3e-2 away from fp64 depending on seed and depth, and where a flip
    happens ours and the oracle's deviation are often bit-identical (tools/diag_grads.py).  So the
    demand is statistical: every gradient points the same way as the fp64 one, and over all
    (seed, parameter) pairs ours is typically as close to fp64 as the fp32 oracle is.  The layer-level
    1e-5 bar is enforced per layer in the tests above."""
    from semigcn_b200.data import Data
    prob = meshgen.synth_inpainting_problem(freq, smooth_iters=10, n_dummy=4)
    mesh = prob["mesh"]
    dm = prob["vmask_dummy"][:, :1] * prob["v_mask"].float().reshape(-1, 1)
    rows = []
    for seed in seeds:
        ours, ref = _sgcn_pair(conv, seed=seed, skip=skip)
        ref64 = copy.deepcopy(ref).double()

        def run_ref(net, dtype):
            z1 = prob["z1"].to(dtype).clone().requires_grad_(True)
            out = net(z1, prob["x_pos"].to(dtype), mesh.edge_index, dm.to(dtype))
            loss = O.mask_pos_rec_loss(out, prob["ini_vs"], prob["v_mask"]) + \
                4.0 * O.mask_norm_rec_loss(O.compute_fn(out, mesh.faces), prob["fn"], prob["f_mask"])
            loss.backward()
            return out, loss, z1.grad

        out_r, loss_r, dz_r = run_ref(ref, torch.float32)
        out_64, loss_64, dz_64 = run_ref(ref64, torch.float64)
        z1g = prob["z1"].to(DEV).requires_grad_(True)
        data = Data(z1=z1g, x_pos=prob["x_pos"].to(DEV), edge_index=mesh.edge_index.to(DEV))
        out = ours(data, dm)
        loss = O.mask_pos_rec_loss(out, prob["ini_vs"].to(DEV), prob["v_mask"].to(DEV)) + \
            4.0 * O.mask_norm_rec_loss(O.compute_fn(out, mesh.faces.to(DEV)), prob["fn"].to(DEV), prob["f_mask"].to(DEV))
        loss.backward()
        e_pos, e_pos32, e_pos64 = rel_err(out, out_r), rel_err(out_r, out_64), rel_err(out, out_64)
        msg = f"positions: {e_pos:.2e} from the fp32 oracle, {e_pos64:.2e} from fp64 (the fp32 oracle: {e_pos32:.2e})"
        if freq <= 10:
            assert e_pos <= REL_TOL, msg
            assert abs(loss.item() - loss_r.item()) <= 1e-5 * abs(loss_r.item())
        else:
            # 13 blocks at 33 642 vertices: the fp32 oracle itself is 1.6e-5 .. 3.0e-5 from fp64 (measured on a B200 host,
            # ours 1.9e-5 .. 3.1e-5 from the fp32 oracle), so the truth is fp64 and the bar that of test_bn_near_constant_channels
            assert e_pos64 <= max(REL_TOL, 2.0 * e_pos32), msg
            e_loss32 = abs(loss_r.item() - loss_64.item())
            assert abs(loss.item() - loss_64.item()) <= max(1e-5 * abs(loss_64.item()), 2.0 * e_loss32), \
                f"loss {loss.item()!r}, fp32 oracle {loss_r.item()!r}, fp64 {loss_64.item()!r}"

        def check(name, g_ours, g_ref32, g_ref64):
            e_ours, e_ref = rel_err(g_ours, g_ref64), rel_err(g_ref32, g_ref64)
            cos = torch.nn.functional.cosine_similarity(g_ours.detach().double().cpu().flatten(), g_ref64.flatten(), dim=0).item()
            rows.append((f"seed {seed} {name}", e_ours, e_ref, cos))

        check("d z1", z1g.grad, dz_r, dz_64)
        r32, r64 = dict(ref.named_parameters()), dict(ref64.named_parameters())
        for name, p in ours.named_parameters():
            if r32[name].grad is None or name.endswith("module_0.bias"):
                continue
            check(name, p.grad, r32[name].grad, r64[name].grad)
    table = "\n".join(f"{n:48s} ours {eo:.2e}  fp32-oracle {er:.2e}  cos {c:.6f}" for n, eo, er, c in rows)
    ratios = torch.tensor([max(eo, 1e-7) / max(er, 1e-7) for _, eo, er, _ in rows])
    assert min(c for *_, c in rows) >= 0.99, table
    assert float(ratios.median()) <= 3.0, f"median error ratio ours / fp32-oracle = {float(ratios.median()):.2f}\n{table}"
    assert float((ratios <= 3.0).float().mean()) >= 0.6, table
    assert max(eo for _, eo, _, _ in rows) <= 0.1, table


def test_sgcn_training_100_steps_tracks_oracle():
    """BASELINE.json asks for a final vertex error <= 1e-4 of the bounding-box diagonal after 100
    steps.  MEASURED (tools/measure_training_divergence.py -> profiles/r2_training_divergence.json,
    oracle only, no product code; BASELINE.md §5): the fp32 CPU oracle is 5.6e-4 of the diagonal away
    from its own fp64 evaluation after ONE Adam step and 7.9e-2 after 100, and a 1-ulp perturbation of
    the initial weights does the same -- so that bar cannot be met by any pair of fp32 implementations.
    The replacement gate stated in BASELINE.md §5 is what this test enforces: with the fp64 oracle
    as the truth, after 1 step and after 100 identical-schedule steps our trajectory is no further
    from it than a small multiple of the fp32 oracle's own distance, and the training loss has
    dropped alike."""
    from semigcn_b200.data import Data
    prob = meshgen.synth_inpainting_problem(6, smooth_iters=10, n_dummy=8)
    mesh = prob["mesh"]
    vm = prob["v_mask"]
    bbox = (prob["ini_vs"].max(0)[0] - prob["ini_vs"].min(0)[0]).norm().item()
    ours, ref = _sgcn_pair("gcnconv")
    ref64 = copy.deepcopy(ref).double()
    nets = {"ours": ours, "ref32": ref, "ref64": ref64}
    opts = {k: torch.optim.Adam(v.parameters(), lr=0.01) for k, v in nets.items()}
    data = Data(z1=prob["z1"].to(DEV), x_pos=prob["x_pos"].to(DEV), edge_index=mesh.edge_index.to(DEV))

    def fwd(name, dm):
        if name == "ours":
            return nets[name](data, dm)
        dt = torch.float64 if name == "ref64" else torch.float32
        return nets[name](prob["z1"].to(dt), prob["x_pos"].to(dt), mesh.edge_index, dm.to(dt))

    g = torch.Generator().manual_seed(314)
    first, last, step1 = {}, {}, {}
    for step in range(100):
        j = int(torch.randint(0, 8, (1,), generator=g))
        dm = prob["vmask_dummy"][:, j:j + 1] * vm.float().reshape(-1, 1)
        for name in nets:
            opts[name].zero_grad()
            out = fwd(name, dm)
            loss = O.mask_pos_rec_loss(out, prob["ini_vs"].to(out.device), vm.to(out.device))
            loss.backward()
            opts[name].step()
            if step == 0:
                first[name] = loss.item()
            last[name] = loss.item()
        if step == 0:
            with torch.no_grad():
                step1 = {name: fwd(name, dm).detach().cpu().double() for name in nets}
    e1_ours = (step1["ours"] - step1["ref64"]).norm(dim=1).max().item() / bbox
    e1_ref = (step1["ref32"] - step1["ref64"]).norm(dim=1).max().item() / bbox
    assert e1_ours <= 3.0 * e1_ref + 1e-4, f"after 1 step: ours {e1_ours:.2e} vs fp32 oracle {e1_ref:.2e}"
    for n_ in nets.values():
        n_.eval()
    with torch.no_grad():
        fin = {name: fwd(name, vm.float().reshape(-1, 1)).cpu().double() for name in nets}
    e_ours = (fin["ours"] - fin["ref64"]).norm(dim=1).max().item() / bbox
    e_ref = (fin["ref32"] - fin["ref64"]).norm(dim=1).max().item() / bbox
    assert e_ours <= 4.0 * e_ref + 1e-4, f"after 100 steps: ours {e_ours:.2e} vs fp32 oracle {e_ref:.2e} (fp64 oracle as truth)"
    assert last["ours"] < 0.7 * first["ours"] and last["ours"] <= 2.0 * max(last["ref32"], last["ref64"]), (first, last)


def test_reference_scripts_import_surface():
    """The reference's util/networks.py pattern, written against the torch_geometric shim names."""
    import semigcn_b200.compat as compat
    compat.install(force=True)
    from torch_geometric.nn import ChebConv, Sequential
    blk = Sequential("x, edge_index", [(ChebConv(4, 16, K=3), "x, edge_index -> x"), nn.BatchNorm1d(16), nn.LeakyReLU()]).to(DEV)
    mesh = meshgen.icosphere(3)
    y = blk(torch.randn(mesh.num_vertices, 4, device=DEV), mesh.edge_index.to(DEV))
    assert y.shape == (mesh.num_vertices, 16) and torch.isfinite(y).all()


@pytest.mark.parametrize("conv", ["chebconv", "gcnconv"])
@pytest.mark.parametrize("skip", [False, True])
def test_sgcn_matches_reference_networks_py_fixture(conv, skip):
    """Drop-in network vs the fixture produced by the reference's own util/networks.py (tests/golden/make_golden_net.py):
    same seeded initial parameters (PyG's double reset_parameters RNG consumption, SURVEY.md A.4) and the same forward
    output in train and eval mode within the 1e-5 bar."""
    import numpy as np
    from helpers import load_golden
    from semigcn_b200.data import Data
    from semigcn_b200.networks import SingleScaleGCN
    gold = load_golden("ref_sgcn_n4.npz")
    tag = f"{conv}_{'skip' if skip else 'noskip'}"
    torch.manual_seed(int(gold["seed"]))
    net = SingleScaleGCN("cpu", conv=conv, skip=skip)
    sd = net.state_dict()
    names = sorted(sd.keys())
    assert names == [str(s) for s in gold[f"{tag}_names"]]
    sums = np.array([[float(sd[k].double().sum()), float(sd[k].double().abs().sum())] for k in names])
    assert np.array_equal(sums, gold[f"{tag}_sums"]), "seeded initial parameters differ from the reference"
    net = net.to(DEV)
    net.device = DEV
    data = Data(z1=torch.from_numpy(gold["z1"]).to(DEV), x_pos=torch.from_numpy(gold["x_pos"]).to(DEV),
                edge_index=torch.from_numpy(gold["edge_index"]).to(DEV))
    net.train()
    y = net(data, gold["dm"])                                  # np.ndarray mask, as sgcn.py passes it
    assert_close(y, torch.from_numpy(gold[f"{tag}_train"]), REL_TOL, "train-mode forward")
    net.eval()
    y = net(data, torch.from_numpy(gold["dm"]))
    assert_close(y, torch.from_numpy(gold[f"{tag}_eval"]), REL_TOL, "eval-mode forward")
