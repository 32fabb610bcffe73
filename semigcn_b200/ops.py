"""Host-side wrappers (torch tensors in, C-ABI calls out) and the autograd Functions built on
them.  PyTorch supplies device memory, streams and the autograd tape; every kernel launched
here is ours (libsemigcn_b200.so).  No CPU path: CPU tensors raise.
"""
from __future__ import annotations

import os
import weakref
from collections import OrderedDict
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib as L
from . import profile as _prof
from ._lib import MODE_ADJ, MODE_CHEB, MODE_GCN, SgbError, check, ptr, require_cuda, stream_ptr

Affine = Optional[Tuple[Tensor, Tensor, Tensor, float]]   # (mean[c], scale[c], shift[c], slope): fused centred BN + LeakyReLU on load


def _f32c(t: Tensor, name: str) -> Tensor:
    if t.dtype != torch.float32:
        raise SgbError(f"{name}: expected float32, got {t.dtype}")
    if t.dim() == 2 and t.stride(1) != 1:
        t = t.contiguous()
    elif t.dim() != 2 and not t.is_contiguous():
        t = t.contiguous()
    return t


def _ws(nbytes: int, device) -> Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def new_amax(device, count: int = 1) -> Tensor:
    """Zeroed device floats for the ``amax_out`` of a producing kernel; the filled slot is then handed to the
    fp16-split GEMM engine as ``a_amax`` / ``g_amax`` (it spares the engine its own reduction pass)."""
    return torch.zeros(count, dtype=torch.float32, device=device)


AMAX_ATTR = "_sgb_amax"     # python attribute on an activation tensor: (device scalar max|x| published by its producer, tensor version)


def tag_amax(t: Tensor, amax_slot: Tensor) -> None:
    """Attach the producer's max|t| (over the finite entries of t: inf and NaN are skipped) to the tensor object, together
    with the tensor's version counter: any in-place edit between two blocks (``x *= k``, ``x.add_(skip)``, an in-place
    activation in user code) bumps ``_version`` and makes the tag stale -- ``amax_of`` then returns None and the GEMM
    engine reduces max|x| itself (a stale, too small maximum would overflow the fp16 split silently)."""
    setattr(t, AMAX_ATTR, (amax_slot, t._version))


def amax_of(t: Tensor) -> Optional[Tensor]:
    tag = getattr(t, AMAX_ATTR, None)
    if tag is None:
        return None
    a, version = tag
    return a if (a.device == t.device and version == t._version) else None


# ----------------------------------------------------------------------------------------
# graph: CSR by target (forward) and by source (backward) + dis, cached per edge_index
# ----------------------------------------------------------------------------------------
class MeshGraph:
    """Normalised sparse operator of one ``edge_index`` for one mode (GCN / CHEB / ADJ).

    Holds what PyG recomputes in every conv call (gcn_norm / get_laplacian, SURVEY.md §8(a3)):
    ``rowptr/colidx`` grouped by target in stable edge order, the same grouped by source for
    the backward pass, ``dis = deg^-1/2`` (bit-exact) and the normalised edge weights packed with the column ids
    (``edges``: int32 [nnz, 2] = (column, float bits of the weight), the stream the aggregation kernel reads).
    """

    def __init__(self, edge_index: Tensor, num_nodes: int, mode: int, with_perm: bool = False):
        require_cuda(edge_index)
        if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.shape[0] != 2:
            raise SgbError("edge_index must be an int64 tensor of shape [2, nnz]")
        lib = L.load()
        ei = edge_index.contiguous()
        dev = ei.device
        nnz, n = int(ei.shape[1]), int(num_nodes)
        self.n, self.nnz, self.mode, self.device = n, nnz, mode, dev
        # vertex-partitioned mode (semigcn_b200/dist.py) overrides these three
        self.halo, self.comm, self.n_global = None, None, n
        wsb = lib.sgb_graph_build_workspace_bytes(nnz, n)
        ws = _ws(wsb, dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        self.dis = torch.empty(n, dtype=torch.float32, device=dev)
        out = []
        with torch.cuda.device(dev):
            for transpose in (0, 1):
                rowptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
                colidx = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
                edges = torch.empty((max(nnz, 1), 2), dtype=torch.int32, device=dev)     # sgb_edge_t[nnz]
                perm = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev) if with_perm else None
                check(lib.sgb_graph_build(ptr(ei), nnz, n, mode, transpose, ptr(rowptr), ptr(colidx), ptr(edges),
                                          ptr(self.dis), ptr(perm), ptr(err), ptr(ws), wsb, stream_ptr(dev)), "sgb_graph_build")
                L.count(7)
                out.append((rowptr, colidx, perm, edges))
        # one host sync per (edge_index, mode), at cache-fill time only
        if int(err.item()) != 0:
            raise SgbError("edge_index contains vertex ids outside [0, num_nodes)")
        (self.rowptr, self.colidx, self.perm, self.edges), (self.rowptr_t, self.colidx_t, self.perm_t, self.edges_t) = out

    def csr(self, transpose: bool):
        """(rowptr, packed (col, weight) stream) of the forward (by target) or backward (by source) operator."""
        return (self.rowptr_t, self.edges_t) if transpose else (self.rowptr, self.edges)

    def edge_weights(self, transpose: bool = False) -> Tensor:
        """Per-slot normalised weights (float32 view of the packed stream), CSR order."""
        e = self.edges_t if transpose else self.edges
        return e[:, 1].view(torch.float32)


_GRAPH_CACHE: "OrderedDict[tuple, tuple]" = OrderedDict()   # key -> (graph, edge_index kept alive, bytes)
_GRAPH_CACHE_PINNED: set = set()         # partitioned operators registered by dist.register_partition: never evicted
_GRAPH_CACHE_MAX_BYTES = int(float(os.environ.get("SGB_GRAPH_CACHE_MB", "4096")) * 2 ** 20)
_GRAPH_BY_CONTENT: dict = {}             # (fingerprint, shape, device, mode, N) -> pointer key of the entry that holds the graph
_GRAPH_ALIAS: dict = {}                  # pointer key of ANOTHER tensor with the same content -> (weakref to that tensor, canonical pointer key)


def _graph_bytes(g: "MeshGraph", edge_index: Tensor) -> int:
    per_dir = 4 * (g.n + 1) + 4 * max(g.nnz, 1) + 8 * max(g.nnz, 1)
    return 2 * per_dir + 4 * g.n + edge_index.numel() * edge_index.element_size()


def _fingerprint(edge_index: Tensor) -> tuple:
    lib = L.load()
    ei = edge_index.contiguous()
    out = torch.empty(2, dtype=torch.int64, device=ei.device)
    with torch.cuda.device(ei.device):
        check(lib.sgb_fingerprint(ptr(ei), ei.numel(), ptr(out), stream_ptr(ei.device)), "sgb_fingerprint")
    L.count(1)
    return tuple(out.tolist())          # one host sync, only on a pointer miss


def _evict() -> None:
    total = sum(v[2] for v in _GRAPH_CACHE.values())
    while total > _GRAPH_CACHE_MAX_BYTES and len(_GRAPH_CACHE) > 1:
        victim = next((k for k in _GRAPH_CACHE if k not in _GRAPH_CACHE_PINNED), None)
        if victim is None or victim == next(reversed(_GRAPH_CACHE)):
            break
        total -= _GRAPH_CACHE[victim][2]
        del _GRAPH_CACHE[victim]
        for ck in [ck for ck, pk in _GRAPH_BY_CONTENT.items() if pk == victim]:
            del _GRAPH_BY_CONTENT[ck]


def graph_for(edge_index: Tensor, num_nodes: int, mode: int) -> MeshGraph:
    """Two-level cache.  Fast path: (storage pointer, shape, version counter, device, mode, N) -- the reference passes the
    same ``edge_index`` to every conv of a forward (util/networks.py:86) and never mutates it.  On a pointer miss the
    CONTENT decides (128-bit fingerprint, one hash pass + one host sync): ``data.edge_index.to(self.device)`` of a CPU
    dataset (util/networks.py:65) makes a fresh device tensor every forward, which must not mean a CSR rebuild per step
    nor a cache that fills with stale copies.  Bounded by bytes (``SGB_GRAPH_CACHE_MB``, default 4 GiB), LRU."""
    require_cuda(edge_index)
    key = (edge_index.data_ptr(), tuple(edge_index.shape), edge_index._version, str(edge_index.device), mode, int(num_nodes))
    hit = _GRAPH_CACHE.get(key)
    if hit is not None:
        _GRAPH_CACHE.move_to_end(key)
        return hit[0]
    alias = _GRAPH_ALIAS.get(key)
    if alias is not None:
        # a tensor whose content was fingerprinted before: valid only while that very tensor object is alive (a recycled
        # pointer under a new tensor object must be fingerprinted again), referenced weakly so the cache never pins copies
        if alias[0]() is edge_index and alias[1] in _GRAPH_CACHE:
            _GRAPH_CACHE.move_to_end(alias[1])
            return _GRAPH_CACHE[alias[1]][0]
        del _GRAPH_ALIAS[key]
    ckey = (_fingerprint(edge_index), tuple(edge_index.shape), str(edge_index.device), mode, int(num_nodes))
    pkey = _GRAPH_BY_CONTENT.get(ckey)
    if pkey is not None and pkey in _GRAPH_CACHE:
        _GRAPH_CACHE.move_to_end(pkey)
        if len(_GRAPH_ALIAS) >= 256:         # keys of dead tensors / old version counters
            for k in [k for k, (wr, _) in _GRAPH_ALIAS.items() if wr() is None or k[2] != wr()._version]:
                del _GRAPH_ALIAS[k]
        _GRAPH_ALIAS[key] = (weakref.ref(edge_index), pkey)      # the other convs of this forward hit without hashing
        return _GRAPH_CACHE[pkey][0]
    g = MeshGraph(edge_index, num_nodes, mode)
    _GRAPH_CACHE[key] = (g, edge_index, _graph_bytes(g, edge_index))      # keep the tensor alive so the pointer cannot be recycled
    _GRAPH_BY_CONTENT[ckey] = key
    _evict()
    return g


def clear_graph_cache() -> None:
    _GRAPH_CACHE.clear()
    _GRAPH_CACHE_PINNED.clear()
    _GRAPH_BY_CONTENT.clear()
    _GRAPH_ALIAS.clear()


# ----------------------------------------------------------------------------------------
# thin functional wrappers
# ----------------------------------------------------------------------------------------
def spmm(g: MeshGraph, x: Tensor, transpose: bool = False, in_affine: Affine = None, alpha: float = 1.0,
         addend: Optional[Tensor] = None, beta: float = 0.0, bias: Optional[Tensor] = None,
         want_stats: bool = False, out: Optional[Tensor] = None, amax_out: Optional[Tensor] = None):
    """``amax_out``: zero-initialised device float that receives max|y| (see ``new_amax``)."""
    lib = L.load()
    require_cuda(x, addend, bias)
    x = _f32c(x, "x")
    n, c = x.shape
    if n != g.n:
        raise SgbError(f"x has {n} rows but the graph has {g.n} vertices")
    y = out if out is not None else torch.empty((n, c), dtype=torch.float32, device=x.device)
    if addend is not None:
        addend = _f32c(addend, "addend")
    rowptr, edges = g.csr(transpose)
    mu, sc, sh, slope = (in_affine if in_affine is not None else (None, None, None, 0.0))
    nnz_eff = int(g.nnz) + (n if g.mode == MODE_GCN else 0)
    sp = _prof.span(f"spmm_c{c}", 4.0 * (2 * n * c + nnz_eff + 2 * n + 1 + (n * c if addend is not None else 0)),
                    2.0 * nnz_eff * c) if _prof.ACTIVE is not None else None
    # Vertex-partitioned mode: the ghost rows of x come from their owners (pack -> all-to-all).  With the owned vertices
    # numbered interior-first, the rows that touch no ghost are aggregated WHILE the exchange is in flight (the collective
    # runs on the communicator's stream), the boundary rows after it: two launches over disjoint row ranges of one operator.
    n_int = int(getattr(g, "n_interior", 0)) if g.halo is not None else 0
    ranges = [(0, n, True)] if not (0 < n_int < n) else [(0, n_int, False), (n_int, n - n_int, True)]
    pending = g.halo.start(x) if g.halo is not None else None
    partials, row_off = None, 0
    if want_stats:
        rows = sum(lib.sgb_spmm_stat_rows(cnt, c) for (_, cnt, _) in ranges)
        partials = torch.empty((rows, 3, c), dtype=torch.float32, device=x.device)
    xg = None
    with torch.cuda.device(x.device):
        for (r0, cnt, needs_ghosts) in ranges:
            if needs_ghosts and pending is not None:
                xg = g.halo.finish(pending)
            part = partials[row_off:] if partials is not None else None
            check(lib.sgb_spmm_range(ptr(rowptr), ptr(edges), ptr(g.dis), g.mode, ptr(x), x.stride(0), r0, cnt, c,
                                     ptr(xg) if needs_ghosts else None, xg.stride(0) if (needs_ghosts and xg is not None) else 0, n,
                                     ptr(mu), ptr(sc), ptr(sh), float(slope), float(alpha), ptr(addend),
                                     addend.stride(0) if addend is not None else 0, float(beta), ptr(bias),
                                     ptr(y), y.stride(0), ptr(part), ptr(amax_out), stream_ptr(x.device)), "sgb_spmm")
            if partials is not None:
                row_off += lib.sgb_spmm_stat_rows(cnt, c)
            L.count(1)
    if sp is not None:
        sp.close()
    return (y, partials) if want_stats else y


def gemm(a: Tensor, b: Tensor, transb: bool = True, a_affine: Affine = None, bias: Optional[Tensor] = None,
         out: Optional[Tensor] = None, accumulate: bool = False, want_stats: bool = False, engine: int = 0,
         a_amax: Optional[Tensor] = None):
    """C (+)= f(A) @ (B^T if transb else B) + bias.  ``a_amax``: optional device scalar max|A| (from the kernel
    that produced A) for the fp16-split tensor-core engine; None = the engine reduces it itself."""
    lib = L.load()
    require_cuda(a, b, bias)
    a, b = _f32c(a, "a"), _f32c(b, "b")
    m, k = a.shape
    n = b.shape[0] if transb else b.shape[1]
    if (b.shape[1] if transb else b.shape[0]) != k:
        raise SgbError(f"gemm: inner dimensions differ ({a.shape} x {b.shape}, transb={transb})")
    c = out if out is not None else torch.empty((m, n), dtype=torch.float32, device=a.device)
    partials = None
    if want_stats:
        partials = torch.empty((lib.sgb_gemm_stat_rows(m), 3, n), dtype=torch.float32, device=a.device)
    mu, sc, sh, slope = (a_affine if a_affine is not None else (None, None, None, 0.0))
    sp = _prof.span(f"gemm_n{n}_k{k}", 4.0 * (m * (k + n) + k * n + (m * n if accumulate else 0)), 2.0 * m * n * k) \
        if _prof.ACTIVE is not None else None
    wsb = lib.sgb_gemm_workspace_bytes(m, n, k, engine)
    ws = _ws(wsb, a.device) if wsb else None
    with torch.cuda.device(a.device):
        check(lib.sgb_gemm(1 if transb else 0, ptr(a), a.stride(0), ptr(b), b.stride(0), ptr(c), c.stride(0), m, n, k,
                           ptr(mu), ptr(sc), ptr(sh), float(slope), ptr(bias), 1 if accumulate else 0, ptr(partials),
                           ptr(a_amax), ptr(ws), wsb, engine, stream_ptr(a.device)), "sgb_gemm")
    if sp is not None:
        sp.close()
    L.count(1)
    return (c, partials) if want_stats else c


def gemm_tn(gmat: Tensor, a: Tensor, out: Optional[Tensor] = None, accumulate: bool = False, engine: int = 0,
            g_amax: Optional[Tensor] = None, a_amax: Optional[Tensor] = None) -> Tensor:
    """D[n,k] (+)= G[m,n]^T @ A[m,k]  (weight gradient)."""
    lib = L.load()
    require_cuda(gmat, a)
    gmat, a = _f32c(gmat, "g"), _f32c(a, "a")
    m, n = gmat.shape
    k = a.shape[1]
    if a.shape[0] != m:
        raise SgbError("gemm_tn: row counts differ")
    d = out if out is not None else torch.empty((n, k), dtype=torch.float32, device=a.device)
    wsb = lib.sgb_gemm_tn_workspace_bytes(m, n, k)
    ws = _ws(wsb, a.device)
    sp = _prof.span(f"gemm_tn_n{n}_k{k}", 4.0 * (m * (k + n) + k * n), 2.0 * m * n * k) if _prof.ACTIVE is not None else None
    with torch.cuda.device(a.device):
        check(lib.sgb_gemm_tn(ptr(gmat), gmat.stride(0), ptr(a), a.stride(0), ptr(d), d.stride(0), m, n, k,
                              1 if accumulate else 0, ptr(g_amax), ptr(a_amax), ptr(ws), wsb, engine, stream_ptr(a.device)), "sgb_gemm_tn")
    if sp is not None:
        sp.close()
    L.count(2)
    return d


def colsum(gmat: Tensor, out: Optional[Tensor] = None, accumulate: bool = False, amax_out: Optional[Tensor] = None) -> Tensor:
    """Column sums (bias gradient); ``amax_out`` (device float) additionally receives max|G| from the same pass."""
    lib = L.load()
    require_cuda(gmat)
    gmat = _f32c(gmat, "g")
    m, n = gmat.shape
    o = out if out is not None else torch.empty(n, dtype=torch.float32, device=gmat.device)
    wsb = lib.sgb_colsum_workspace_bytes(m, n)
    ws = _ws(wsb, gmat.device)
    sp = _prof.span(f"colsum_c{n}", 4.0 * m * n) if _prof.ACTIVE is not None else None
    with torch.cuda.device(gmat.device):
        check(lib.sgb_colsum(ptr(gmat), gmat.stride(0), m, n, ptr(o), 1 if accumulate else 0, ptr(amax_out), ptr(ws), wsb,
                             stream_ptr(gmat.device)), "sgb_colsum")
    if sp is not None:
        sp.close()
    L.count(2)
    return o


def tensor_core_likely(m: int, cin: int, cout: int) -> bool:
    """Mirror of the engine policy in csrc/gemm.cu (tc_worthwhile / tn_tc_worthwhile): will the dX GEMM [m, cout] x
    [cout, cin] or the dW GEMM of a layer go to the fp16-split tensor-core engine (which wants max|operand|)?"""
    return m >= 2048 and ((cin >= 32 and cout >= 16) or (cout >= 32 and cin >= 16))


def amax(x: Tensor) -> Optional[Tensor]:
    """Device scalar max|x| in one streaming pass, or None when the layout is not the vectorised one (the GEMM engine then
    reduces it itself).  Used once per operand that none of our kernels produced, then shared by all its consumers."""
    lib = L.load()
    require_cuda(x)
    x = _f32c(x, "x")
    m, c = x.shape
    if c % 4 != 0 or x.stride(0) % 4 != 0 or x.data_ptr() % 16 != 0:
        return None
    out = torch.empty(1, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        check(lib.sgb_amax(ptr(x), x.stride(0), m, c, ptr(out), stream_ptr(x.device)), "sgb_amax")
    L.count(1)
    return out


def input_prep(z1: Tensor, dm: Optional[Tensor]) -> Tensor:
    """x [N, 4] = (dm * ((z1 - zc) / z_sc), dm): the bounding-box normalisation + mask + concatenation of
    util/networks.py:67-79 as two kernels (csrc/prep.cu), bit-identical to the torch ops.  No gradient (inputs)."""
    lib = L.load()
    require_cuda(z1, dm)
    z1 = _f32c(z1.detach(), "z1")
    n = int(z1.shape[0])
    if z1.dim() != 2 or z1.shape[1] != 3:
        raise SgbError("input_prep: z1 must be [N, 3]")
    if dm is not None:
        dm = dm.detach().to(torch.float32).reshape(-1).contiguous()
        if dm.numel() != n:
            raise SgbError("input_prep: mask must have one entry per vertex")
    x = torch.empty((n, 4), dtype=torch.float32, device=z1.device)
    scratch = torch.empty(16, dtype=torch.float32, device=z1.device)
    sp = _prof.span("input_prep", 4.0 * 11 * n) if _prof.ACTIVE is not None else None
    with torch.cuda.device(z1.device):
        check(lib.sgb_input_prep(ptr(z1), z1.stride(0), n, ptr(dm), ptr(x), ptr(scratch), stream_ptr(z1.device)), "sgb_input_prep")
    if sp is not None:
        sp.close()
    L.count(3)
    return x


def col_stats(y: Tensor) -> Tensor:
    lib = L.load()
    y = _f32c(y, "y")
    m, c = y.shape
    partials = torch.empty((lib.sgb_col_stat_rows(m, c), 3, c), dtype=torch.float32, device=y.device)
    sp = _prof.span(f"col_stats_c{c}", 4.0 * m * c) if _prof.ACTIVE is not None else None
    with torch.cuda.device(y.device):
        check(lib.sgb_col_stats(ptr(y), y.stride(0), m, c, ptr(partials), stream_ptr(y.device)), "sgb_col_stats")
    if sp is not None:
        sp.close()
    L.count(1)
    return partials


def gather_rows(x: Tensor, idx: Tensor, out: Optional[Tensor] = None) -> Tensor:
    """out[k, :] = x[idx[k], :] (idx int32)."""
    lib = L.load()
    require_cuda(x, idx)
    x = _f32c(x, "x")
    count, c = int(idx.numel()), int(x.shape[1])
    o = out if out is not None else torch.empty((count, c), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        check(lib.sgb_gather_rows(ptr(x), x.stride(0), ptr(idx), count, c, ptr(o), o.stride(0), stream_ptr(x.device)), "sgb_gather_rows")
    L.count(1)
    return o


def merge_moment_rows(partials: Tensor) -> Tensor:
    """[rows, 3, c] (count, mean, M2) partial rows -> one merged [1, 3, c] float32 row (plain torch ops on the tensor's
    device, float64 inside).  n = sum n_r, mean = sum n_r mean_r / n, M2 = sum (M2_r + n_r (mean_r - mean)^2): the
    many-way form of Chan's pairwise merge; rows with count 0 drop out.  CUDA tensors go through ``sgb_moments_merge``
    (one launch, fp64 inside); the torch form below serves CPU tensors (gloo tests of the host logic)."""
    if partials.is_cuda:
        lib = L.load()
        partials = partials.contiguous()
        rows, _, c = partials.shape
        out = torch.empty((1, 3, c), dtype=torch.float32, device=partials.device)
        with torch.cuda.device(partials.device):
            check(lib.sgb_moments_merge(ptr(partials), rows, c, ptr(out), stream_ptr(partials.device)), "sgb_moments_merge")
        L.count(1)
        return out
    p = partials.to(torch.float64)
    n_r, mean_r, m2_r = p[:, 0, :], p[:, 1, :], p[:, 2, :]
    n = n_r.sum(dim=0)
    safe = torch.where(n > 0, n, torch.ones_like(n))
    mean = (n_r * mean_r).sum(dim=0) / safe
    d = mean_r - mean.unsqueeze(0)
    m2 = (m2_r + n_r * d * d).sum(dim=0)
    return torch.stack([n, mean, m2]).unsqueeze(0).to(torch.float32).contiguous()


def bn_finalize(partials: Tensor, count: int, gamma: Optional[Tensor], beta: Optional[Tensor], eps: float,
                momentum: float, running_mean: Optional[Tensor], running_var: Optional[Tensor], comm=None):
    lib = L.load()
    if comm is not None:
        # SyncBN: each rank folds its own (count, mean, M2) rows into ONE row (sgb_moments_merge), the ranks all-gather
        # those rows -- 12*c bytes per rank, the same on every rank whatever its vertex count or the kernel that produced
        # the layer -- and every rank merges the same `world` rows in the same order: identical statistics everywhere.
        # (All-gathering the raw rows needs equal row counts on all ranks, which uneven vertex ranges do not give.)
        partials = comm.all_gather_cat(merge_moment_rows(partials).contiguous())
    rows, _, c = partials.shape
    dev = partials.device
    sp = _prof.span("bn_finalize", 12.0 * rows * c) if _prof.ACTIVE is not None else None
    st = torch.empty((4, c), dtype=torch.float32, device=dev)     # mean, invstd, scale, shift
    with torch.cuda.device(dev):
        check(lib.sgb_bn_finalize(ptr(partials), rows, c, count, ptr(gamma), ptr(beta), float(eps), float(momentum),
                                  ptr(running_mean), ptr(running_var), ptr(st[0]), ptr(st[1]), ptr(st[2]), ptr(st[3]),
                                  stream_ptr(dev)), "sgb_bn_finalize")
    if sp is not None:
        sp.close()
    L.count(1)
    return st[0], st[1], st[2], st[3]


def bn_act_apply(y: Tensor, mean: Tensor, scale: Tensor, shift: Tensor, slope: float, out: Optional[Tensor] = None,
                 amax_out: Optional[Tensor] = None) -> Tensor:
    lib = L.load()
    y = _f32c(y, "y")
    m, c = y.shape
    z = out if out is not None else torch.empty_like(y)
    sp = _prof.span(f"bn_act_apply_c{c}", 8.0 * m * c) if _prof.ACTIVE is not None else None
    with torch.cuda.device(y.device):
        check(lib.sgb_bn_act_apply(ptr(y), y.stride(0), m, c, ptr(mean), ptr(scale), ptr(shift), float(slope), ptr(z), z.stride(0),
                                   ptr(amax_out), stream_ptr(y.device)), "sgb_bn_act_apply")
    if sp is not None:
        sp.close()
    L.count(1)
    return z


def bn_act_bwd(dz: Tensor, y: Tensor, scale: Tensor, shift: Tensor, mean: Optional[Tensor], invstd: Optional[Tensor],
               slope: float, training: bool, want_param_grads: bool = True, comm=None, n_global: Optional[int] = None,
               amax_out: Optional[Tensor] = None):
    """dY (and dgamma, dbeta) of Z = lrelu(BN(Y)) given dZ."""
    lib = L.load()
    dz, y = _f32c(dz, "dz"), _f32c(y, "y")
    m, c = y.shape
    dev = y.device
    dy = torch.empty_like(y)
    dgamma = dbeta = sums = None
    sp = _prof.span(f"bn_act_bwd_c{c}", 4.0 * m * c * (5 if training else 3)) if _prof.ACTIVE is not None else None
    with torch.cuda.device(dev):
        if training or want_param_grads:
            if mean is None:       # eval mode: xhat from the running statistics folded in scale/shift is not available
                raise SgbError("bn_act_bwd: mean/invstd required")
            rows = lib.sgb_col_stat_rows(m, c)
            partials = torch.empty((rows, 2, c), dtype=torch.float32, device=dev)
            check(lib.sgb_bn_act_bwd_reduce(ptr(dz), dz.stride(0), ptr(y), y.stride(0), m, c, ptr(scale), ptr(shift),
                                            ptr(mean), ptr(invstd), float(slope), ptr(partials), stream_ptr(dev)),
                  "sgb_bn_act_bwd_reduce")
            sums = torch.empty((2, c), dtype=torch.float32, device=dev)
            dgamma = torch.empty(c, dtype=torch.float32, device=dev)
            dbeta = torch.empty(c, dtype=torch.float32, device=dev)
            check(lib.sgb_bn_bwd_finalize(ptr(partials), rows, c, ptr(sums), ptr(dgamma), ptr(dbeta), 0, stream_ptr(dev)),
                  "sgb_bn_bwd_finalize")
            L.count(2)
            if comm is not None and training:
                # dgamma / dbeta stay LOCAL contributions (summed with the other parameter gradients later);
                # the apply pass needs the GLOBAL sums over all n_global vertices: the kernel divides by the
                # local row count m, hence the m / n_global factor
                sums = comm.all_reduce_sum(sums.clone()) * (float(m) / float(n_global))
        check(lib.sgb_bn_act_bwd_apply(ptr(dz), dz.stride(0), ptr(y), y.stride(0), m, c, ptr(scale), ptr(shift), ptr(mean),
                                       ptr(invstd), ptr(sums), float(slope), 1 if training else 0, ptr(dy), dy.stride(0),
                                       ptr(amax_out), stream_ptr(dev)), "sgb_bn_act_bwd_apply")
        L.count(1)
    if sp is not None:
        sp.close()
    return dy, dgamma, dbeta


# ----------------------------------------------------------------------------------------
# autograd Functions (unfused building blocks; the fused conv+BN+act block lives in nn.py)
# ----------------------------------------------------------------------------------------
class PropagateFn(torch.autograd.Function):
    """y = alpha * (S x) + beta * addend;  backward: dx = alpha * (S^T dy), daddend = beta * dy."""

    @staticmethod
    def forward(ctx, x: Tensor, graph: MeshGraph, alpha: float, addend: Optional[Tensor], beta: float):
        ctx.graph, ctx.alpha, ctx.beta = graph, alpha, beta
        ctx.has_addend = addend is not None
        return spmm(graph, x, alpha=alpha, addend=addend, beta=beta)

    @staticmethod
    def backward(ctx, dy: Tensor):
        dy = dy.contiguous()
        dx = spmm(ctx.graph, dy, transpose=True, alpha=ctx.alpha) if ctx.needs_input_grad[0] else None
        dadd = None
        if ctx.has_addend and ctx.needs_input_grad[3]:
            dadd = dy * ctx.beta
        return dx, None, None, dadd, None


def propagate(graph: MeshGraph, x: Tensor, alpha: float = 1.0, addend: Optional[Tensor] = None, beta: float = 0.0) -> Tensor:
    return PropagateFn.apply(x, graph, alpha, addend, beta)


# ----------------------------------------------------------------------------------------
# rectangular sparse operator (MeshPool / MeshUnpool, util/meshnet.py:9-27): y = S x on the SpMM kernel
# ----------------------------------------------------------------------------------------
class SparseOp:
    """A fixed sparse matrix S [n_out, n_in] as the two CSRs the SpMM kernel consumes (forward: by row; backward: by
    column), built once from a ``torch.sparse`` COO (or dense) tensor with plain torch ops on its device.  Entries of a
    row are in ascending column order = the order the CPU ``torch.sparse.mm`` of the reference sums a coalesced matrix.
    ``row_scale`` folds a per-row factor into the weights (MeshPool's division by the row sum)."""

    def __init__(self, mat: Tensor, row_scale: Optional[Tensor] = None):
        require_cuda(mat)
        m = (mat if mat.is_sparse else mat.to_sparse()).coalesce()
        if m.dim() != 2:
            raise SgbError("SparseOp: expected a 2-D matrix")
        dev = m.device
        self.n_out, self.n_in = int(m.shape[0]), int(m.shape[1])
        idx, val = m.indices(), m.values().to(torch.float32)
        rows, cols = idx[0], idx[1]
        self.nnz = int(val.numel())
        if self.n_out >= 2 ** 31 - 1 or self.n_in >= 2 ** 31 - 1 or self.nnz >= 2 ** 31 - 1:
            raise SgbError("SparseOp: dimensions exceed int32")
        if row_scale is not None:
            val = val * row_scale.to(torch.float32).reshape(-1)[rows]

        def csr(r, c, v, n_r):
            key = r * max(self.n_in, self.n_out) + c           # coalesce() already sorts (row, col); the transpose needs it
            order = torch.argsort(key, stable=True)
            r, c, v = r[order], c[order], v[order]
            rowptr = torch.zeros(n_r + 1, dtype=torch.int64, device=dev)
            rowptr[1:] = torch.cumsum(torch.bincount(r, minlength=n_r), 0)
            edges = torch.empty((max(self.nnz, 1), 2), dtype=torch.int32, device=dev)
            edges.zero_()
            edges[:self.nnz, 0] = c.to(torch.int32)
            edges[:self.nnz, 1] = v.contiguous().view(torch.int32)
            return rowptr.to(torch.int32).contiguous(), edges.contiguous()

        self.rowptr, self.edges = csr(rows, cols, val, self.n_out)
        self.rowptr_t, self.edges_t = csr(cols, rows, val, self.n_in)
        self._dis = torch.zeros(1, dtype=torch.float32, device=dev)    # not read in SGB_MODE_ADJ; the ABI wants a pointer
        self.device = dev

    def apply(self, x: Tensor, transpose: bool = False) -> Tensor:
        lib = L.load()
        require_cuda(x)
        x = _f32c(x, "x")
        n_in, n_out = (self.n_out, self.n_in) if transpose else (self.n_in, self.n_out)
        if x.dim() != 2 or x.shape[0] != n_in:
            raise SgbError(f"SparseOp: x has {tuple(x.shape)} rows/cols, expected {n_in} rows")
        c = int(x.shape[1])
        y = torch.empty((n_out, c), dtype=torch.float32, device=x.device)
        rowptr, edges = (self.rowptr_t, self.edges_t) if transpose else (self.rowptr, self.edges)
        sp = _prof.span(f"sparse_mm_c{c}", 4.0 * ((n_in + n_out) * c + 2 * self.nnz + n_out + 1), 2.0 * self.nnz * c) \
            if _prof.ACTIVE is not None else None
        with torch.cuda.device(x.device):
            check(lib.sgb_spmm(ptr(rowptr), ptr(edges), ptr(self._dis), MODE_ADJ, ptr(x), x.stride(0), n_out, c,
                               None, None, None, 0.0, 1.0, None, 0, 0.0, None, ptr(y), y.stride(0), None, None,
                               stream_ptr(x.device)), "sgb_spmm (SparseOp)")
        if sp is not None:
            sp.close()
        L.count(1)
        return y


class SparseMMFn(torch.autograd.Function):
    """y = S x;  dx = S^T dy (gather over the by-column CSR: atomic-free, deterministic)."""

    @staticmethod
    def forward(ctx, x: Tensor, op: SparseOp):
        ctx.op = op
        return op.apply(x)

    @staticmethod
    def backward(ctx, dy: Tensor):
        return (ctx.op.apply(dy.contiguous(), transpose=True) if ctx.needs_input_grad[0] else None), None


def sparse_mm(op: SparseOp, x: Tensor) -> Tensor:
    return SparseMMFn.apply(x, op)


class LinearFn(torch.autograd.Function):
    """y = x W^T (+ b) on our GEMM tiles; dX = dY W, dW = dY^T X (split-m, fixed order), db = colsum(dY)."""

    @staticmethod
    def forward(ctx, x: Tensor, weight: Tensor, bias: Optional[Tensor]):
        x = _f32c(x, "x")
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return gemm(x, weight, transb=True, bias=bias)

    @staticmethod
    def backward(ctx, dy: Tensor):
        x, weight = ctx.saved_tensors
        dy = dy.contiguous()
        dx = gemm(dy, weight, transb=False) if ctx.needs_input_grad[0] else None
        dw = gemm_tn(dy, x) if ctx.needs_input_grad[1] else None
        db = colsum(dy) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return dx, dw, db


def linear(x: Tensor, weight: Tensor, bias: Optional[Tensor] = None) -> Tensor:
    return LinearFn.apply(x, weight, bias)


def eval_affine(running_mean: Tensor, running_var: Tensor, gamma: Optional[Tensor], beta: Optional[Tensor], eps: float):
    """Eval-mode BatchNorm as the centred affine (mean, invstd, scale = gamma*invstd, shift = beta)."""
    invstd = torch.rsqrt(running_var + eps)
    scale = (invstd * gamma if gamma is not None else invstd).contiguous()
    shift = (beta if beta is not None else torch.zeros_like(invstd)).contiguous()
    return running_mean.contiguous(), invstd.contiguous(), scale, shift


class BnActFn(torch.autograd.Function):
    """Z = lrelu(BatchNorm1d(Y)); training: batch statistics (+ running-stat update), eval: running stats."""

    @staticmethod
    def forward(ctx, y, gamma, beta, running_mean, running_var, eps, momentum, slope, training, partials):
        y = _f32c(y, "y")
        m, c = y.shape
        if training:
            if partials is None:
                partials = col_stats(y)
            mean, invstd, scale, shift = bn_finalize(partials, m, gamma, beta, eps, momentum, running_mean, running_var)
        else:
            mean, invstd, scale, shift = eval_affine(running_mean, running_var, gamma, beta, eps)
        z = bn_act_apply(y, mean, scale, shift, slope)
        ctx.save_for_backward(y, scale, shift, mean, invstd)
        ctx.slope, ctx.training, ctx.has_affine = slope, training, gamma is not None
        return z

    @staticmethod
    def backward(ctx, dz):
        y, scale, shift, mean, invstd = ctx.saved_tensors
        dy, dgamma, dbeta = bn_act_bwd(dz.contiguous(), y, scale, shift, mean, invstd, ctx.slope, ctx.training)
        if not ctx.has_affine:
            dgamma = dbeta = None
        return dy, dgamma, dbeta, None, None, None, None, None, None, None


def bn_act(y: Tensor, bn: torch.nn.BatchNorm1d, slope: float, partials: Optional[Tensor] = None) -> Tensor:
    """BatchNorm1d module semantics (torch.nn.BatchNorm1d) + LeakyReLU(slope); slope=1 -> BN only, 0 -> ReLU."""
    training = bn.training or (bn.running_mean is None)
    momentum = 0.1 if bn.momentum is None else bn.momentum
    if training and bn.track_running_stats and bn.num_batches_tracked is not None:
        bn.num_batches_tracked.add_(1)
        if bn.momentum is None:
            momentum = 1.0 / float(bn.num_batches_tracked)
    rm = bn.running_mean if (training and bn.track_running_stats) or not training else None
    rv = bn.running_var if (training and bn.track_running_stats) or not training else None
    return BnActFn.apply(y, bn.weight, bn.bias, rm, rv, bn.eps, momentum, slope, training, partials)
