"""ctypes binding of ``libsemigcn_b200.so`` (the C-ABI declared in include/semigcn_b200.h).

There is NO fallback: if the library is missing or a call fails this raises.  The product
path never imports anything from ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("SGB_LIB_PATH") or os.path.join(CSRC, "libsemigcn_b200.so")   # override: A/B builds of the same ABI

MODE_GCN, MODE_CHEB, MODE_ADJ = 0, 1, 2

_i64, _i32, _f32, _vp, _sz = C.c_int64, C.c_int, C.c_float, C.c_void_p, C.c_size_t
_f64 = C.c_double

# name -> (restype, argtypes); must list every symbol of include/semigcn_b200.h
SIGNATURES = {
    "sgb_version": (_i32, []),
    "sgb_last_error": (C.c_char_p, []),
    "sgb_num_sms": (_i32, []),
    "sgb_fingerprint": (_i32, [_vp, _i64, _vp, _vp]),
    "sgb_graph_build_workspace_bytes": (_sz, [_i64, _i64]),
    "sgb_graph_build": (_i32, [_vp, _i64, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "sgb_spmm_stat_rows": (_i32, [_i64, _i32]),
    "sgb_spmm": (_i32, [_vp, _vp, _vp, _i32, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _f32, _f32, _vp, _i64, _f32,
                        _vp, _vp, _i64, _vp, _vp, _vp]),
    "sgb_spmm_halo": (_i32, [_vp, _vp, _vp, _i32, _vp, _i64, _i64, _i32, _vp, _i64, _i64, _vp, _vp, _vp, _f32, _f32, _vp, _i64, _f32,
                             _vp, _vp, _i64, _vp, _vp, _vp]),
    "sgb_spmm_range": (_i32, [_vp, _vp, _vp, _i32, _vp, _i64, _i64, _i64, _i32, _vp, _i64, _i64, _vp, _vp, _vp, _f32, _f32, _vp, _i64, _f32,
                              _vp, _vp, _i64, _vp, _vp, _vp]),
    "sgb_gather_rows": (_i32, [_vp, _i64, _vp, _i64, _i32, _vp, _i64, _vp]),
    "sgb_gemm_stat_rows": (_i32, [_i64]),
    "sgb_gemm_workspace_bytes": (_sz, [_i64, _i32, _i32, _i32]),
    "sgb_gemm": (_i32, [_i32, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _sz, _i32, _vp]),
    "sgb_gemm_tn_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "sgb_gemm_tn": (_i32, [_vp, _i64, _vp, _i64, _vp, _i64, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _sz, _i32, _vp]),
    "sgb_colsum_workspace_bytes": (_sz, [_i64, _i32]),
    "sgb_colsum": (_i32, [_vp, _i64, _i64, _i32, _vp, _i32, _vp, _vp, _sz, _vp]),
    "sgb_amax": (_i32, [_vp, _i64, _i64, _i32, _vp, _vp]),
    "sgb_moments_merge": (_i32, [_vp, _i32, _i32, _vp, _vp]),
    "sgb_col_stat_rows": (_i32, [_i64, _i32]),
    "sgb_col_stats": (_i32, [_vp, _i64, _i64, _i32, _vp, _vp]),
    "sgb_bn_finalize": (_i32, [_vp, _i32, _i32, _i64, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sgb_bn_act_apply": (_i32, [_vp, _i64, _i64, _i32, _vp, _vp, _vp, _f32, _vp, _i64, _vp, _vp]),
    "sgb_bn_act_bwd_reduce": (_i32, [_vp, _i64, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _f32, _vp, _vp]),
    "sgb_bn_bwd_finalize": (_i32, [_vp, _i32, _i32, _vp, _vp, _vp, _i32, _vp]),
    "sgb_bn_act_bwd_apply": (_i32, [_vp, _i64, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _i32,
                                    _vp, _i64, _vp, _vp]),
    "sgb_loss_partial_rows": (_i32, []),
    "sgb_incidence_build_workspace_bytes": (_sz, [_i64, _i64]),
    "sgb_incidence_build": (_i32, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "sgb_step_loss_fwd": (_i32, [_vp, _i64, _i64, _vp, _i32, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sgb_step_loss_bwd": (_i32, [_vp, _i64, _i64, _vp, _i32, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "sgb_lap_loss_fwd": (_i32, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sgb_input_prep": (_i32, [_vp, _i64, _i64, _vp, _vp, _vp, _vp]),
    "sgb_bnf_work_floats": (_sz, [_i64]),
    "sgb_bnf_partial_rows": (_i32, []),
    "sgb_bnf_loss_fwd": (_i32, [_vp, _i64, _i64, _vp, _vp, _i64, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "sgb_bnf_loss_bwd": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp]),
    "sgb_lap_loss_bwd": (_i32, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "sgb_point_surface_distance": (_i32, [_vp, _i64, _i64, _vp, _i64, _vp, _vp, _f32, _f32, _f32, _f32, _i32, _i32, _i32,
                                          _vp, _vp, _vp]),
}

_lib: Optional[C.CDLL] = None


class SgbError(RuntimeError):
    pass


def build_library(verbose: bool = False) -> str:
    """Compile the extension in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-C", CSRC, "-j", str(os.cpu_count() or 4)], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:])
        print(out.stderr[-4000:])
    if out.returncode != 0:
        raise SgbError("building libsemigcn_b200.so failed")
    return LIB_PATH


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SgbError(
            f"{LIB_PATH} not found: the CUDA extension is required (no CPU fallback). "
            "Build it with `python -c 'import __graft_entry__ as g; g.build()'` or `make -C semigcn_b200/csrc`.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().sgb_last_error().decode("utf-8", "replace")
        raise SgbError(f"{what} failed (code {rc}): {msg}")


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(*tensors: torch.Tensor) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise SgbError("semigcn_b200 runs on CUDA tensors only (sm_100a); there is no CPU fallback")


# launch accounting for bench.py's `gpu_launches` claim (kernels launched by our library)
LAUNCHES = 0


def count(n: int) -> None:
    global LAUNCHES
    LAUNCHES += n
