"""Micro-benchmarks of the individual kernels on the 1M-vertex icosphere (CUDA events, L2 flushed by size)."""
import sys, torch, json
sys.path.insert(0, '.')
from semigcn_b200 import ops, meshgen
dev = 'cuda:0'
what = sys.argv[1] if len(sys.argv) > 1 else 'spmm,gemm,gemm_tn,bn'
freq = int(sys.argv[2]) if len(sys.argv) > 2 else 316
mesh = meshgen.icosphere(freq, device=dev)
n, nnz = mesh.num_vertices, mesh.nnz
print('vertices', n, 'nnz', nnz)
def timeit(fn, reps=5, warm=2):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps
if what == 'spmm1':      # one width, GCN mode, for ncu captures:  bench_kernels.py spmm1 <freq> <c>
    c = int(sys.argv[3])
    g = ops.MeshGraph(mesh.edge_index, n, 0)
    x = torch.randn(n, c, device=dev)
    ms = timeit(lambda: ops.spmm(g, x))
    print(f'spmm c={c}: {ms:.3f} ms')
    sys.exit(0)
if 'spmm' in what.split(','):
    for mode in (0, 1):
        g = ops.MeshGraph(mesh.edge_index, n, mode)
        for c in (4, 16, 32, 64, 128, 256, 512):
            x = torch.randn(n, c, device=dev)
            ms = timeit(lambda: ops.spmm(g, x))
            by = 4.0 * (2 * n * c + nnz + (n if mode == 0 else 0) + 2 * n + 1)
            ms_s = timeit(lambda: ops.spmm(g, x, want_stats=True))
            print(f'spmm mode={mode} c={c:4d}: {ms:7.3f} ms  {by / ms / 1e6:8.1f} GB/s | +stats {ms_s:7.3f} ms')
if 'gemm' in what.split(','):
    for (k, nn) in ((64, 128), (128, 256), (256, 256), (256, 512), (512, 256), (256, 128), (128, 64)):
        a = torch.randn(n, k, device=dev); w = torch.randn(nn, k, device=dev)
        ms = timeit(lambda: ops.gemm(a, w, engine=3), reps=3, warm=1)
        print(f'gemm k={k} n={nn} engine=3: {ms:7.3f} ms  {2.0 * n * k * nn / ms / 1e9:7.1f} TFLOP/s  {4.0 * n * (k + nn) / ms / 1e6:7.1f} GB/s')
        amx = a.abs().max().reshape(1)
        ms3 = timeit(lambda: ops.gemm(a, w, engine=3, a_amax=amx), reps=3, warm=1)
        print(f'     engine 3 with a_amax supplied: {ms3:7.3f} ms  {4.0 * n * (k + nn) / ms3 / 1e6:7.1f} GB/s')
if 'gemm_tn' in what:
    for (k, nn) in ((64, 128), (128, 256), (256, 256), (256, 512), (512, 256), (256, 128), (128, 64)):
        a = torch.randn(n, k, device=dev); g_ = torch.randn(n, nn, device=dev)
        ms = timeit(lambda: ops.gemm_tn(g_, a, engine=3), reps=3, warm=1)
        print(f'gemm_tn k={k} n={nn} engine=3: {ms:7.3f} ms  {2.0 * n * k * nn / ms / 1e9:7.1f} TFLOP/s  {4.0 * n * (k + nn) / ms / 1e6:7.1f} GB/s')
        ga, aa = g_.abs().max().reshape(1), a.abs().max().reshape(1)
        ms3 = timeit(lambda: ops.gemm_tn(g_, a, engine=3, g_amax=ga, a_amax=aa), reps=3, warm=1)
        print(f'     engine 3 with amax supplied: {ms3:7.3f} ms  {4.0 * n * (k + nn) / ms3 / 1e6:7.1f} GB/s')
if 'bn' in what:
    for c in (16, 64, 256, 512):
        y = torch.randn(n, c, device=dev); dz = torch.randn(n, c, device=dev)
        bn = torch.nn.BatchNorm1d(c).to(dev)
        st = ops.bn_finalize(ops.col_stats(y), n, bn.weight, bn.bias, 1e-5, 0.1, None, None)
        ms_a = timeit(lambda: ops.bn_act_apply(y, st[0], st[2], st[3], 0.01))
        ms_b = timeit(lambda: ops.bn_act_bwd(dz, y, st[2], st[3], st[0], st[1], 0.01, True))
        ms_c = timeit(lambda: ops.col_stats(y))
        print(f'bn c={c}: apply {ms_a:.3f} ms ({8.0*n*c/ms_a/1e6:.0f} GB/s)  bwd {ms_b:.3f} ms ({20.0*n*c/ms_b/1e6:.0f} GB/s)  col_stats {ms_c:.3f} ms ({4.0*n*c/ms_c/1e6:.0f} GB/s)')
