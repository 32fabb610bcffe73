"""Point-to-surface distance on synthetic icospheres: build and query time, candidates per query, and the accuracy of the
"do nothing" baseline of the synthetic inpainting problem.  Prints one JSON line.

    python tools/bench_mesh_distance.py [--freqs 32,100,316,632] [--reps 10]

Frequencies 32 / 100 / 316 / 632 are the 10 242 / 100 002 / 998 562 / 3 994 242-vertex spheres.  Per size, the queries are
the initial (noisy) positions of `synth_inpainting_problem` against the exact sphere, and the exact sphere's vertices
against the noisy mesh.  Times are CUDA events after one warm-up; the build includes its host syncs.  Beyond 100 k vertices
the working set (48 B per face of triangles, 4 B per cell and per (cell, face) pair) exceeds the 126 MB L2, and repeated
queries are timed as they run, without flushing the L2 in between.  The candidates tested per query are counted by a
second build of csrc/surface_dist.cu with SGB_SURFACE_COUNT_CANDIDATES (the face output then holds the count), compiled
into a temporary directory.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from semigcn_b200 import _lib as L, meshgen  # noqa: E402
from semigcn_b200.distance import SurfaceIndex, mesh_distance  # noqa: E402


def counting_library(tmp):
    out = os.path.join(tmp, "libcount.so")
    src = [os.path.join(L.CSRC, f) for f in ("api.cu", "surface_dist.cu")]
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared",
                    "-DSGB_SURFACE_COUNT_CANDIDATES", *src, "-o", out, "-lcudart"], check=True, capture_output=True)
    lib = C.CDLL(out)
    fn = lib.sgb_point_surface_distance
    fn.restype, fn.argtypes = L.SIGNATURES["sgb_point_surface_distance"]
    return fn


def candidates_per_query(fn, idx, pts):
    p = pts.to(torch.float32).contiguous()
    n = p.shape[0]
    dist = torch.empty(n, dtype=torch.float32, device=p.device)
    cnt = torch.empty(n, dtype=torch.int32, device=p.device)
    L.check(fn(p.data_ptr(), 3, n, idx.tris.data_ptr(), idx.nf, idx.cell_start.data_ptr(), idx.cell_faces.data_ptr(), *idx.origin,
               idx.cell_size, *idx.dims, dist.data_ptr(), cnt.data_ptr(), L.stream_ptr(p.device)), "counting build")
    return cnt.double().mean().item()


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--freqs", default="32,100,316,632")
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_mesh_distance.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"device": torch.cuda.get_device_name(dev), "power_limit": smi.stdout.strip() or None, "sizes": []}
    with tempfile.TemporaryDirectory() as tmp:
        count_fn = counting_library(tmp)
        for freq in (int(f) for f in args.freqs.split(",")):
            prob = meshgen.synth_inpainting_problem(freq, device=dev, n_dummy=1)
            mesh, hole = prob["mesh"], ~prob["v_mask"]
            exact, noisy, faces = mesh.vs, prob["ini_vs"], mesh.faces
            row = {"vertices": mesh.num_vertices, "faces": int(faces.shape[0])}
            for name, target, queries in (("noisy_to_exact", exact, noisy), ("exact_to_noisy", noisy, exact)):
                build_ms = timed(lambda: SurfaceIndex(target, faces), max(1, args.reps // 5))
                idx = SurfaceIndex(target, faces)
                q = queries.to(torch.float32).contiguous()
                query_ms = timed(lambda: idx.query(q), args.reps)
                row[name] = {"build_ms": round(build_ms, 3), "query_ms": round(query_ms, 3),
                             "queries_per_s": round(q.shape[0] / query_ms * 1e3), "grid": list(idx.dims),
                             "cell_size": idx.cell_size, "pairs_per_face": round(idx.pairs / idx.nf, 2),
                             "candidates_per_query": round(candidates_per_query(count_fn, idx, q), 1)}
                del idx
            m = mesh_distance(noisy, faces, exact, faces, mask_a=hole, mask_b=hole)
            diag = m["diag"].item()
            row["metric_over_diag"] = {"two_sided_mean": m["mean"].item() / diag, "hausdorff": m["hausdorff"].item() / diag,
                                       "hole_a_to_b_mean": m["a_to_b_mask"]["mean"].item() / diag,
                                       "hole_b_to_a_mean": m["b_to_a_mask"]["mean"].item() / diag,
                                       "hole_vertices": int(m["a_to_b_mask"]["count"].item())}
            res["sizes"].append(row)
            del prob, mesh, m
            torch.cuda.empty_cache()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
