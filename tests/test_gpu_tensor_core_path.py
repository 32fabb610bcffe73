"""The tcgen05 fp16-split path as the conv blocks compose it, against float64.

The dense transforms go to the tensor-core engines only above fixed row counts (csrc/gemm.cu): the forward / dX GEMM from
m >= 2048 (k_gemm_f16<0>), the weight gradient from m >= 4096 (k_gemm_tn_f16), CTA pairs from m >= 32 768 (k_gemm_f16<1>,
k_gemm_tn_f16_pair).  The meshes here sit just above each threshold, and a kernel census (torch.profiler) asserts that each
one reached the kernels it is meant for, so a change of the dispatch policy fails here instead of quietly testing the
CUDA-core tiles again.

What a fused block composes on that path is checked too: the max|x| scalars that the SpMM, BatchNorm and colsum kernels
publish for the engine's per-tensor scale (bit-exact against torch), the version guard of ``ops.tag_amax``, accumulate
together with BatchNorm statistics, outputs written into strided views (sentinels around them must survive), and operands
with inf / NaN entries.  Bar: the project's 1e-5 norm-relative against an fp64 evaluation of the oracle."""
import copy
import os
import re

import pytest
import torch
import torch.nn as nn

from helpers import REL_TOL, assert_close, random_graph, rel_err
from oracle import pyg_ref as O
from test_gpu_kernels import check_moments

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

F16_SINGLE = re.compile(r"k_gemm_f16<(0|false)>")
F16_PAIR = re.compile(r"k_gemm_f16<(1|true)>")
TN_SINGLE = re.compile(r"k_gemm_tn_f16\(")
TN_PAIR = re.compile(r"k_gemm_tn_f16_pair")
AMAX = re.compile(r"\bk_amax\b")


def _ops():
    from semigcn_b200 import ops
    return ops


def _icosphere(freq, nv):
    from semigcn_b200 import meshgen
    m = meshgen.icosphere(freq)
    assert m.num_vertices == nv
    return m


@pytest.fixture(scope="module")
def mesh_2252():
    """fp16 forward on single CTAs, weight gradient on the CUDA cores (m < 4096)."""
    return _icosphere(15, 2252)


@pytest.fixture(scope="module")
def mesh_4412():
    """adds the single-CTA weight gradient k_gemm_tn_f16."""
    return _icosphere(21, 4412)


@pytest.fixture(scope="module")
def mesh_33642():
    """CTA pairs; 263 m-tiles is odd, so the second CTA of the last pair has no rows."""
    return _icosphere(58, 33642)


@pytest.fixture(scope="module", autouse=True)
def _oracle_threads():
    torch.set_num_threads(os.cpu_count() or 1)


def census(fn):
    """Run fn under torch.profiler (CUDA activities); return (fn's result, names of the device activities in launch order)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return out, names


def _count(names, pat):
    return sum(1 for n in names if pat.search(n))


def assert_census(names, want=(), absent=()):
    kernels = sorted(set(n[:80] for n in names if "k_" in n))
    for p in want:
        assert _count(names, p) > 0, f"{p.pattern} was not launched; kernels: {kernels}"
    for p in absent:
        assert _count(names, p) == 0, f"{p.pattern} was launched; kernels: {kernels}"


def expected_engines(nv, cout):
    """Tensor-core kernels a conv block with `cout` output channels must reach on an nv-vertex mesh (and must not)."""
    if nv < 4096:
        return (F16_SINGLE,), (F16_PAIR, TN_SINGLE, TN_PAIR)
    if nv < 32768:
        return (F16_SINGLE, TN_SINGLE), (F16_PAIR, TN_PAIR)
    return (F16_PAIR, TN_PAIR if cout % 256 == 0 else TN_SINGLE), ()


# ------------------------------------------------------------------------------------------------------------------
# fused conv -> BatchNorm1d -> LeakyReLU blocks against the oracle evaluated in float64
# ------------------------------------------------------------------------------------------------------------------
def _block(mod, kind, cin, cout, K, bias=True):
    conv = mod.GCNConv(cin, cout, bias=bias) if kind == "gcn" else mod.ChebConv(cin, cout, K=K, bias=bias)
    return mod.Sequential("x, edge_index", [(conv, "x, edge_index -> x"), nn.BatchNorm1d(cout), nn.LeakyReLU()])


def _randomise(seq):
    with torch.no_grad():
        seq.module_0.bias.uniform_(-0.5, 0.5)        # PyG initialises it to zero: make the bias path visible
        seq.module_1.weight.uniform_(0.5, 1.5)
        seq.module_1.bias.normal_()
        seq.module_1.running_mean.normal_()
        seq.module_1.running_var.uniform_(0.5, 2.0)


def _ours_and_ref64(blocks):
    """(our modules on the device, the same modules as the fp64 oracle) from oracle modules with randomised state."""
    import semigcn_b200.nn as N
    ours = []
    for ref, spec in blocks:
        o = _block(N, *spec)
        o.load_state_dict(ref.state_dict())
        ours.append(o.to(DEV))
    return ours, [copy.deepcopy(ref).double() for ref, _ in blocks]


def _kink_free(dz, out64):
    # no gradient through outputs within 1e-4 of the LeakyReLU kink: there an fp32-rounding-level difference of the
    # pre-activation legitimately takes the other slope than the fp64 evaluation
    return dz * (out64.detach().abs() > 1e-4).to(dz.dtype)


def _compare(errs, got, want, what, tol=REL_TOL):
    e = rel_err(got, want)
    errs[what] = e
    assert e <= tol, f"{what}: norm-relative error {e:.3e} against fp64 > {tol:.0e}"


def _compare_params(errs, ours, ref64, train, tag=""):
    r = dict(ref64.named_parameters())
    for name, p in ours.named_parameters():
        if train and name == "module_0.bias":
            # training-mode BatchNorm removes the batch mean: the true gradient of the conv bias is exactly 0 (ours is
            # exactly 0, the fp64 evaluation holds rounding noise)
            assert torch.all(p.grad == 0), name
            continue
        _compare(errs, p.grad, r[name].grad, tag + "d " + name)
    for k in ("running_mean", "running_var"):
        _compare(errs, getattr(ours.module_1, k), getattr(ref64.module_1, k), tag + k)


BLOCK_CFGS = [("gcn", 64, 128, 1), ("gcn", 256, 512, 1),          # aggregate-first
              ("gcn", 256, 64, 1), ("gcn", 512, 256, 1),          # transform-first
              ("gcn", 16, 32, 1),                                 # at the engine threshold: n = 32, k = 16
              ("cheb", 256, 256, 1), ("cheb", 256, 256, 2), ("cheb", 256, 256, 3), ("cheb", 256, 256, 4),
              ("cheb", 128, 256, 3)]


@pytest.mark.parametrize("nv", [2252, 4412, 33642])
@pytest.mark.parametrize("kind,cin,cout,K", BLOCK_CFGS)
@pytest.mark.parametrize("train", [True, False])
def test_fused_block_on_tensor_cores_vs_fp64(request, nv, kind, cin, cout, K, train):
    mesh = request.getfixturevalue(f"mesh_{nv}")
    torch.manual_seed(cin * 7 + cout + K)
    ref = _block(O, kind, cin, cout, K)
    _randomise(ref)
    (ours,), (ref64,) = _ours_and_ref64([(ref, (kind, cin, cout, K))])
    ours.train(train)
    ref64.train(train)
    gen = torch.Generator().manual_seed(nv + cin + cout)
    x = torch.randn(nv, cin, generator=gen)
    dz = torch.randn(nv, cout, generator=gen)
    xr = x.double().requires_grad_(True)
    out64 = ref64(xr, mesh.edge_index)
    dz = _kink_free(dz, out64)
    out64.backward(dz.double())
    ei = mesh.edge_index.to(DEV)
    xg = x.to(DEV).requires_grad_(True)

    def step():
        out = ours(xg, ei)
        out.backward(dz.to(DEV))
        return out

    out, names = census(step)
    want, absent = expected_engines(nv, cout)
    assert_census(names, want, absent)
    errs = {}
    _compare(errs, out, out64, "out")
    _compare(errs, xg.grad, xr.grad, "dX")
    _compare_params(errs, ours, ref64, train)
    print(f"{kind}({cin}, {cout}, K={K}) {'train' if train else 'eval'} {nv} vertices: "
          + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))


# ------------------------------------------------------------------------------------------------------------------
# max|x| handoffs between blocks, and the version guard of ops.tag_amax
# ------------------------------------------------------------------------------------------------------------------
CHAIN = [("gcn", 64, 256, 1), ("gcn", 256, 128, 1)]      # aggregate-first, then transform-first on the first block's output


@pytest.mark.parametrize("nv", [4412, 33642])
@pytest.mark.parametrize("edit", [False, True])
def test_two_block_chain_handoffs_vs_fp64(request, nv, edit):
    """Every tensor-core operand of this chain has a producer that publishes its max|.|: the SpMM (P of block 1, dH of
    block 2), bn_act_apply (block 1's output = block 2's transform input, through ops.tag_amax) and bn_act_bwd (dY).  So no
    k_amax reduction runs.  An in-place edit between the blocks (x *= 2^12) must make the published maximum unusable: a
    stale one would be 4096 x too small and overflow the fp16 split."""
    ops = _ops()
    mesh = request.getfixturevalue(f"mesh_{nv}")
    torch.manual_seed(77)
    refs = []
    for spec in CHAIN:
        r = _block(O, *spec)
        _randomise(r)
        refs.append((r, spec))
    ours, refs64 = _ours_and_ref64(refs)
    gen = torch.Generator().manual_seed(nv)
    x = torch.randn(nv, CHAIN[0][1], generator=gen)
    dz = torch.randn(nv, CHAIN[-1][2], generator=gen)

    def chain(blocks, xin, ei, check_tag=False):
        h = blocks[0](xin, ei)
        if edit:
            h.mul_(2.0 ** 12)
            if check_tag:
                assert ops.amax_of(h) is None, "an in-place edit must make the published max|x| stale"
        elif check_tag:
            assert ops.amax_of(h) is not None, "the fused block publishes max|z| of its output"
        return blocks[1](h, ei)

    xr = x.double().requires_grad_(True)
    out64 = chain(refs64, xr, mesh.edge_index)
    dz = _kink_free(dz, out64)
    out64.backward(dz.double())
    ei = mesh.edge_index.to(DEV)
    xg = x.to(DEV).requires_grad_(True)

    def step():
        out = chain(ours, xg, ei, check_tag=True)
        out.backward(dz.to(DEV))
        return out

    out, names = census(step)
    assert_census(names, (F16_PAIR if nv >= 32768 else F16_SINGLE, TN_PAIR if nv >= 32768 else TN_SINGLE))
    n_amax = _count(names, AMAX)
    if edit:
        assert n_amax > 0, "the edited activation has no valid max|x|: the engine must reduce it itself"
    else:
        assert n_amax == 0, f"{n_amax} k_amax launches although every operand's producer publishes its max"
    errs = {}
    _compare(errs, out, out64, "out")
    _compare(errs, xg.grad, xr.grad, "dX")
    for i, (o, r) in enumerate(zip(ours, refs64)):
        _compare_params(errs, o, r, True, tag=f"block {i} ")
    print(f"chain {nv} vertices edit={edit}: " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))


@pytest.mark.parametrize("kind,cin,cout", [("gcn", 128, 256), ("cheb", 256, 128)])
@pytest.mark.parametrize("bias", [True, False])
def test_bare_conv_on_cta_pairs_vs_fp64(mesh_33642, kind, cin, cout, bias):
    """A bare conv receives a dY none of our kernels produced: its max|dY| comes from colsum(amax_out=) when there is a
    bias, from one ops.amax pass otherwise, and is shared by the weight-gradient and dX GEMMs."""
    from semigcn_b200 import nn as N
    mesh = mesh_33642
    nv = mesh.num_vertices
    torch.manual_seed(cin + cout)
    ref = O.GCNConv(cin, cout, bias=bias) if kind == "gcn" else O.ChebConv(cin, cout, K=3, bias=bias)
    if bias:
        with torch.no_grad():
            ref.bias.uniform_(-0.5, 0.5)
    ours = (N.GCNConv(cin, cout, bias=bias) if kind == "gcn" else N.ChebConv(cin, cout, K=3, bias=bias))
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(DEV)
    ref64 = copy.deepcopy(ref).double()
    gen = torch.Generator().manual_seed(cin * 1000 + cout)
    x, g = torch.randn(nv, cin, generator=gen), torch.randn(nv, cout, generator=gen)
    xr = x.double().requires_grad_(True)
    out64 = ref64(xr, mesh.edge_index)
    out64.backward(g.double())
    ei = mesh.edge_index.to(DEV)
    xg = x.to(DEV).requires_grad_(True)

    def step():
        out = ours(xg, ei)
        out.backward(g.to(DEV))
        return out

    out, names = census(step)
    assert_census(names, expected_engines(nv, cout)[0])
    if kind == "gcn":      # aggregate-first: the forward operand comes from the SpMM; dY from colsum or ONE ops.amax
        assert _count(names, AMAX) == (0 if bias else 1), [n for n in names if AMAX.search(n)]
    errs = {}
    _compare(errs, out, out64, "out")
    _compare(errs, xg.grad, xr.grad, "dX")
    r = dict(ref64.named_parameters())
    for name, p in ours.named_parameters():
        _compare(errs, p.grad, r[name].grad, "d " + name)
    print(f"bare {kind}({cin}, {cout}) bias={bias}: " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))


# ------------------------------------------------------------------------------------------------------------------
# kernel contracts: published max|x| bit-exact, accumulate + statistics, views and canaries, non-finite operands
# ------------------------------------------------------------------------------------------------------------------
def _amax_ref(t):
    t = t.detach()
    fin = t[torch.isfinite(t)]
    return fin.abs().max().reshape(1) if fin.numel() else torch.zeros(1, device=t.device)


def _assert_slot(slot, t, what):
    want = _amax_ref(t)
    assert torch.equal(slot.view(torch.int32), want.to(slot.device).view(torch.int32)), \
        f"{what}: published max {slot.item()!r}, max over the finite |entries| {want.item()!r}"


def _prefilled_slots(ops, t_want):
    """A zeroed slot, one holding 2x the true maximum (must stay) and one holding half of it (must be raised)."""
    true = _amax_ref(t_want).item()
    s0, big, small = ops.new_amax(DEV), ops.new_amax(DEV), ops.new_amax(DEV)
    big.fill_(2.0 * true)
    small.fill_(0.5 * true)
    return s0, big, small


def _check_prefilled(slots, t, what):
    s0, big, small = slots
    _assert_slot(s0, t, what)
    _assert_slot(small, t, what + " (slot held less)")
    assert big.item() == 2.0 * _amax_ref(t).item(), f"{what}: a slot holding more must keep its value (max(old, new))"


@pytest.fixture(scope="module")
def mesh_graphs(mesh_2252):
    ops = _ops()
    ei = mesh_2252.edge_index.to(DEV)
    return {mode: ops.MeshGraph(ei, mesh_2252.num_vertices, mode) for mode in (0, 1)}


SPMM_VARIANTS = ["plain", "transpose", "recurrence", "bias", "prologue", "stats"]


@pytest.mark.parametrize("variant", SPMM_VARIANTS)
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("c", [64, 30])           # vectorised (c % 4 == 0) and scalar configuration
@pytest.mark.parametrize("nonfinite", [False, True])
def test_spmm_amax_out_bit_exact(mesh_graphs, variant, mode, c, nonfinite):
    ops = _ops()
    g = mesh_graphs[mode]
    n = g.n
    gen = torch.Generator(device=DEV).manual_seed(c + mode)
    x = torch.randn(n, c, device=DEV, generator=gen) * 3.0
    addend = torch.randn(n, c, device=DEV, generator=gen)
    bias = torch.randn(c, device=DEV, generator=gen)
    mu, sc, sh = (torch.randn(c, device=DEV, generator=gen), torch.rand(c, device=DEV, generator=gen) + 0.5,
                  torch.randn(c, device=DEV, generator=gen))
    if nonfinite:
        x[17, 3] = float("inf")
        x[900, 5] = float("nan")
    kw = dict(transpose=variant == "transpose")
    if variant == "recurrence":
        kw.update(alpha=2.0, addend=addend, beta=-1.0)
    elif variant == "bias":
        kw.update(bias=bias)
    elif variant == "prologue":
        kw.update(in_affine=(mu, sc, sh, 0.01))
    elif variant == "stats":
        kw.update(want_stats=True)
    y = ops.spmm(g, x, **kw)
    y = y[0] if variant == "stats" else y
    if nonfinite:
        assert not torch.isfinite(y).all()
    slots = _prefilled_slots(ops, y)
    for s in slots:
        ops.spmm(g, x, amax_out=s, **kw)
    _check_prefilled(slots, y, f"spmm {variant}")


@pytest.mark.parametrize("c", [64, 30])
@pytest.mark.parametrize("nonfinite", [False, True])
def test_bn_and_colsum_amax_out_bit_exact(c, nonfinite):
    ops = _ops()
    m = 3001
    gen = torch.Generator(device=DEV).manual_seed(c)
    y = torch.randn(m, c, device=DEV, generator=gen) * 2.0 + 0.5
    dz = torch.randn(m, c, device=DEV, generator=gen)
    mean, invstd = y.mean(0), torch.rsqrt(y.var(0, unbiased=False) + 1e-5)
    scale = invstd * (torch.rand(c, device=DEV, generator=gen) + 0.5)
    shift = torch.randn(c, device=DEV, generator=gen)
    if nonfinite:
        y[5, 2] = float("inf")
        y[6, 1] = float("nan")
        dz[40, 0] = float("inf")
    z = ops.bn_act_apply(y, mean, scale, shift, 0.01)
    slots = _prefilled_slots(ops, z)
    for s in slots:
        ops.bn_act_apply(y, mean, scale, shift, 0.01, amax_out=s)
    _check_prefilled(slots, z, "bn_act_apply")
    for training in (True, False):
        dy = ops.bn_act_bwd(dz, y, scale, shift, mean, invstd, 0.01, training)[0]
        slots = _prefilled_slots(ops, dy)
        for s in slots:
            ops.bn_act_bwd(dz, y, scale, shift, mean, invstd, 0.01, training, amax_out=s)
        _check_prefilled(slots, dy, f"bn_act_bwd training={training}")
    # colsum zeroes its slot itself: the result is max|G| whatever the slot held
    for fill in (0.0, 1e30):
        s = torch.full((1,), fill, device=DEV)
        ops.colsum(dz, amax_out=s)
        _assert_slot(s, dz, "colsum")


def test_ops_amax_bit_exact_and_none_for_unaligned_views():
    ops = _ops()
    gen = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn(5000, 72, device=DEV, generator=gen)
    x[10, 10] = float("inf")
    x[11, 11] = -float("inf")
    x[12, 12] = float("nan")
    _assert_slot(ops.amax(x), x, "ops.amax")
    _assert_slot(ops.amax(x[:, 8:72]), x[:, 8:72], "ops.amax (aligned view)")
    assert ops.amax(x[:, 1:65]) is None, "a view off the 16-byte alignment has no vectorised max pass"
    assert ops.amax(x[:, :30]) is None, "c % 4 != 0"


ENGINES = [0, 1, 3, "3pair"]


def _engine(monkeypatch, e):
    if e == "3pair":
        monkeypatch.setenv("SGB_F16_PAIR", "1")
        return 3
    monkeypatch.delenv("SGB_F16_PAIR", raising=False)
    return e


@pytest.mark.parametrize("m,n,k,pair", [(3000, 128, 64, False), (33000, 256, 128, True), (20011, 96, 256, "env")])
def test_gemm_published_amax_gives_the_engines_bits(monkeypatch, m, n, k, pair):
    """gemm engine 3 (single CTA, and pairs by size or forced): a supplied max|A| gives the same bits as the engine's own
    reduction; gemm_tn engines 3 and 4 likewise with g_amax and a_amax."""
    ops = _ops()
    if pair == "env":
        monkeypatch.setenv("SGB_F16_PAIR", "1")
    gen = torch.Generator(device=DEV).manual_seed(m)
    a, b = torch.randn(m, k, device=DEV, generator=gen) * 7.0, torch.randn(n, k, device=DEV, generator=gen)
    g = torch.randn(m, n, device=DEV, generator=gen) * 1e-3

    def run():
        return ops.gemm(a, b, engine=3), ops.gemm(a, b, engine=3, a_amax=ops.amax(a))
    (own, given), names = census(run)
    assert_census(names, (F16_PAIR if pair else F16_SINGLE,))
    assert torch.equal(own, given)
    assert_close(own, a.double() @ b.double().t(), 5e-6, "gemm")
    for engine in (3, 4) if n % 256 == 0 else (3,):
        own = ops.gemm_tn(g, a, engine=engine)
        assert torch.equal(own, ops.gemm_tn(g, a, engine=engine, g_amax=ops.amax(g), a_amax=ops.amax(a))), f"gemm_tn engine {engine}"
        assert_close(own, g.double().t() @ a.double(), 5e-6, f"gemm_tn engine {engine}")


@pytest.mark.parametrize("engine", [1, 3, "3pair"])
@pytest.mark.parametrize("m,n,k", [(3000, 256, 128), (33000, 96, 64), (129, 80, 48)])
def test_gemm_accumulate_with_statistics(monkeypatch, engine, m, n, k):
    """C += A B^T + bias with the BatchNorm moments of the FINAL C (the ChebConv block's second transform)."""
    ops = _ops()
    e = _engine(monkeypatch, engine)
    gen = torch.Generator(device=DEV).manual_seed(m + n)
    a, b = torch.randn(m, k, device=DEV, generator=gen), torch.randn(n, k, device=DEV, generator=gen)
    bias = torch.randn(n, device=DEV, generator=gen)
    c0 = torch.randn(m, n, device=DEV, generator=gen) * 2.0 + 1.0
    want = c0.double() + a.double() @ b.double().t() + bias.double()
    got, partials = ops.gemm(a, b, bias=bias, out=c0.clone(), accumulate=True, want_stats=True, engine=e)
    assert_close(got, want, 5e-6, "accumulate")
    check_moments(partials, got.double().cpu())
    check_moments(partials, want.cpu())


SENTINEL = -559038737          # 0xDEADBEEF: the float -6.3e18, visible wherever a kernel reads or writes it by mistake


def _canary(rows, cols):
    return torch.full((rows, cols), SENTINEL, dtype=torch.int32, device=DEV).view(torch.float32)


def _assert_canary(buf, rows, cols, what):
    b = buf.view(torch.int32).clone()
    b[rows, cols] = SENTINEL
    bad = int((b != SENTINEL).sum())
    assert bad == 0, f"{what}: {bad} elements outside the output view were written"


def _strided(t, pad=8, off=4):
    """t's values in an interior view of a wider buffer (leading dimension + pad, 16-byte aligned)."""
    rows, cols = t.shape
    big = torch.randn(rows, cols + pad, device=t.device)
    big[:, off:off + cols] = t
    return big[:, off:off + cols]


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("m", [129, 33000])
@pytest.mark.parametrize("transb", [True, False])
def test_gemm_into_views_with_canaries(monkeypatch, engine, m, transb):
    ops = _ops()
    n, k = 80, 64
    e = _engine(monkeypatch, engine)
    gen = torch.Generator(device=DEV).manual_seed(m + n + k)
    a = torch.randn(m, k, device=DEV, generator=gen)
    b = torch.randn(n, k, device=DEV, generator=gen) if transb else torch.randn(k, n, device=DEV, generator=gen)
    bias = torch.randn(n, device=DEV, generator=gen)
    a_v, b_v = _strided(a), _strided(b)                 # lda = k + 8, ldb > k (transb) / > n
    assert a_v.stride(0) > k and b_v.stride(0) > b.shape[1]
    buf = _canary(m + 2, n + 24)
    c_v = buf[1:m + 1, 8:8 + n]
    ops.gemm(a_v, b_v, transb=transb, bias=bias, out=c_v, engine=e)
    _assert_canary(buf, slice(1, m + 1), slice(8, 8 + n), "gemm C")
    dense = ops.gemm(a, b, transb=transb, bias=bias, engine=e)
    assert torch.equal(c_v, dense), "the view result must be bit-identical to the contiguous call"
    assert_close(c_v, a.double() @ (b.double().t() if transb else b.double()) + bias.double(), 5e-6, "gemm")
    # accumulate into the view: reads the view's own elements only
    ops.gemm(a_v, b_v, transb=transb, out=c_v, accumulate=True, engine=e)
    _assert_canary(buf, slice(1, m + 1), slice(8, 8 + n), "gemm C (accumulate)")
    assert_close(c_v, 2.0 * (a.double() @ (b.double().t() if transb else b.double())) + bias.double(), 5e-6, "accumulate")


@pytest.mark.parametrize("engine", [0, 1, 3])
@pytest.mark.parametrize("m", [129, 33000])
def test_gemm_tn_and_colsum_into_views_with_canaries(engine, m):
    ops = _ops()
    n, k = 80, 64
    gen = torch.Generator(device=DEV).manual_seed(m + 1)
    g, a = torch.randn(m, n, device=DEV, generator=gen), torch.randn(m, k, device=DEV, generator=gen)
    buf = _canary(n + 2, k + 24)
    d_v = buf[1:n + 1, 8:8 + k]
    ops.gemm_tn(_strided(g), _strided(a), out=d_v, engine=engine)
    _assert_canary(buf, slice(1, n + 1), slice(8, 8 + k), "gemm_tn D")
    assert torch.equal(d_v, ops.gemm_tn(g, a, engine=engine)), "the view result must be bit-identical to the contiguous call"
    assert_close(d_v, g.double().t() @ a.double(), 5e-6, "gemm_tn")
    obuf = _canary(1, n + 8)
    ops.colsum(_strided(g), out=obuf[0, 4:4 + n])
    _assert_canary(obuf, slice(0, 1), slice(4, 4 + n), "colsum")
    assert torch.equal(obuf[0, 4:4 + n], ops.colsum(g))


@pytest.mark.parametrize("m", [129, 33000])
@pytest.mark.parametrize("c", [80, 30])
def test_spmm_and_bn_act_apply_into_views_with_canaries(m, c):
    ops = _ops()
    ei = random_graph(m, 6 * m, seed=m, symmetric=True).to(DEV)
    g = ops.MeshGraph(ei, m, 0)
    gen = torch.Generator(device=DEV).manual_seed(c)
    x = torch.randn(m, c, device=DEV, generator=gen)
    buf = _canary(m + 2, c + 24)
    y_v = buf[1:m + 1, 8:8 + c]
    ops.spmm(g, _strided(x), out=y_v)
    _assert_canary(buf, slice(1, m + 1), slice(8, 8 + c), "spmm y")
    assert torch.equal(y_v, ops.spmm(g, x))
    mean, scale, shift = (torch.randn(c, device=DEV, generator=gen), torch.rand(c, device=DEV, generator=gen) + 0.5,
                          torch.randn(c, device=DEV, generator=gen))
    zbuf = _canary(m + 2, c + 24)
    z_v = zbuf[1:m + 1, 8:8 + c]
    ops.bn_act_apply(_strided(x), mean, scale, shift, 0.01, out=z_v)
    _assert_canary(zbuf, slice(1, m + 1), slice(8, 8 + c), "bn_act_apply z")
    assert torch.equal(z_v, ops.bn_act_apply(x, mean, scale, shift, 0.01))


@pytest.mark.parametrize("what", ["a", "c"])
def test_gemm_misaligned_views(what):
    """Operands off the 16-byte alignment: engine 0 falls back to the CUDA-core tiles (and stays exact), an explicit
    engine 3 refuses."""
    from semigcn_b200 import SgbError
    ops = _ops()
    m, n, k = 3000, 80, 64
    gen = torch.Generator(device=DEV).manual_seed(5)
    a, b = torch.randn(m, k, device=DEV, generator=gen), torch.randn(n, k, device=DEV, generator=gen)
    a_in = _strided(a, pad=8, off=1) if what == "a" else a
    buf = _canary(m, n + 8)
    c_v = buf[:, 1:1 + n] if what == "c" else buf[:, 4:4 + n]
    ops.gemm(a_in, b, out=c_v)
    _assert_canary(buf, slice(0, m), slice(1, 1 + n) if what == "c" else slice(4, 4 + n), "gemm C")
    assert_close(c_v, a.double() @ b.double().t(), 2e-6, "misaligned fallback")
    with pytest.raises(SgbError):
        ops.gemm(a_in, b, out=c_v, engine=3)


@pytest.mark.parametrize("engine", [1, 3, "3pair"])
@pytest.mark.parametrize("bad", ["nan", "inf"])
@pytest.mark.parametrize("scale", [1.0, 1e5])
def test_gemm_nonfinite_rows(monkeypatch, engine, bad, scale):
    """A NaN or inf in one row of A: exactly the rows the fp64 product makes non-finite are non-finite, every other row
    stays within 1e-5 row-relative.  With entries above the fp16 range (1e5) the per-tensor scale must come from the finite
    maximum: a scale of 1 overflows the fp16 split of every row."""
    ops = _ops()
    e = _engine(monkeypatch, engine)
    m, n, k = 3000, 128, 64
    gen = torch.Generator(device=DEV).manual_seed(17)
    a, b = torch.randn(m, k, device=DEV, generator=gen) * scale, torch.randn(n, k, device=DEV, generator=gen)
    a[1234, 7] = float(bad)
    want = a.double() @ b.double().t()
    for a_amax in (None, ops.amax(a)):
        got = ops.gemm(a, b, engine=e, a_amax=a_amax).double()
        bad_want, bad_got = ~torch.isfinite(want).all(1), ~torch.isfinite(got).all(1)
        assert torch.equal(bad_got, bad_want), \
            f"non-finite rows {bad_got.nonzero().flatten()[:10].tolist()} (of {int(bad_got.sum())}), fp64: {bad_want.nonzero().flatten().tolist()}"
        ok = ~bad_want
        row_err = ((got[ok] - want[ok]).abs().max(1)[0] / want[ok].abs().max(1)[0]).max().item()
        assert row_err <= 1e-5, f"row-relative error {row_err:.2e} of the finite rows"
