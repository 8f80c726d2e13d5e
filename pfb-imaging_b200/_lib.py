"""ctypes binding of the C-ABI library ``libpfbgrid.so`` (``include/pfbgrid.h``).

There is no CPU fallback: if the CUDA library is missing or fails to load, or no
B200 is visible when a compute entry point is called, the product path raises.
"""

from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB_PATH = os.environ.get("PFBG_LIB") or os.path.join(HERE, "libpfbgrid.so")  # PFBG_LIB: A/B builds
CSRC = os.path.join(HERE, "csrc")

PFBG_F32, PFBG_F64 = 0, 1
PFBG_ERR_ARG = 1
HOST_PTRS, DEVICE_PTRS, APPLY_WGT, NO_MASK_ZERO = 0, 1, 2, 4
PINNED_IN, PINNED_OUT, BEAM_CACHED = 16, 32, 64
PLAN_EXTERNAL_STACK = 1
IPC_BLOB_BYTES = 96

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-shared",
]


class PlanDesc(C.Structure):
    _fields_ = [
        ("precision", C.c_int32), ("device", C.c_int32),
        ("nx", C.c_int32), ("ny", C.c_int32), ("nu", C.c_int32), ("nv", C.c_int32),
        ("W", C.c_int32), ("nplanes", C.c_int32),
        ("do_wgridding", C.c_int32), ("divide_by_n", C.c_int32),
        ("beta", C.c_double), ("pixsize_x", C.c_double), ("pixsize_y", C.c_double),
        ("center_x", C.c_double), ("center_y", C.c_double),
        ("usign", C.c_double), ("vsign", C.c_double), ("wsign", C.c_double),
        ("w0", C.c_double), ("dw", C.c_double), ("nshift", C.c_double),
        ("corr_u", C.c_void_p), ("corr_v", C.c_void_p),
        ("gl_x", C.c_void_p), ("gl_w", C.c_void_p),
        ("n_gl", C.c_int32), ("pmirror", C.c_int32), ("fast_screen", C.c_int32), ("flags", C.c_int32),
    ]


class PlanInfo(C.Structure):
    _fields_ = [
        ("nrow", C.c_int64), ("nvis", C.c_int64), ("nactive", C.c_int64),
        ("grid_bytes", C.c_int64), ("total_bytes", C.c_int64),
        ("nchan", C.c_int32), ("nplanes", C.c_int32),
        ("nu", C.c_int32), ("nv", C.c_int32), ("W", C.c_int32), ("n_work_items", C.c_int32),
    ]


# symbol -> (restype, argtypes); must list every symbol include/pfbgrid.h declares
_vp, _i32, _i64, _u32, _dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_double
SIGNATURES = {
    "pfbg_last_error": (C.c_char_p, []),
    "pfbg_version": (C.c_int, []),
    "pfbg_device_count": (C.c_int, [C.POINTER(_i32)]),
    "pfbg_plan_create": (C.c_int, [C.POINTER(PlanDesc), C.POINTER(_vp)]),
    "pfbg_plan_destroy": (C.c_int, [_vp]),
    "pfbg_plan_get_info": (C.c_int, [_vp, C.POINTER(PlanInfo)]),
    "pfbg_plan_set_wrange": (C.c_int, [_vp, _dbl, _i32, _i32]),
    "pfbg_plan_set_stack": (C.c_int, [_vp, _vp, C.c_uint64]),
    "pfbg_bind_vis": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _u32, _vp]),
    "pfbg_bind_weights": (C.c_int, [_vp, _vp, _u32, _vp]),
    "pfbg_plan_set_batch": (C.c_int, [_vp, _i32, _vp, _vp]),
    "pfbg_bind_vis_batch": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _u32, _vp]),
    "pfbg_bin_dump": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "pfbg_grid": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _vp, _u32, _vp]),
    "pfbg_grid_psf": (C.c_int, [_vp, _dbl, _dbl, _dbl, _vp, _vp, _u32, _vp]),
    "pfbg_degrid": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _vp]),
    "pfbg_hessian": (C.c_int, [_vp, _vp, _vp, _dbl, _dbl, _vp, _u32, _vp]),
    "pfbg_host_register": (C.c_int, [_vp, C.c_uint64]),
    "pfbg_host_unregister": (C.c_int, [_vp]),
    "pfbg_set_profiling": (C.c_int, [_vp, _i32]),
    "pfbg_get_timings": (C.c_int, [_vp, C.POINTER(C.c_float), _i32, C.POINTER(_i32)]),
    "pfbg_launch_count": (_i64, []),
    "pfbg_counts": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _i32,
                              _dbl, _dbl, _dbl, _dbl, _vp, _u32, _vp]),
    "pfbg_counts_cells": (C.c_int, [_i32, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _dbl, _dbl, _dbl, _dbl, _vp]),
    "pfbg_conv_create": (C.c_int, [_i32, _i32, _i32, _i32, _i32, _i32, C.POINTER(_vp)]),
    "pfbg_conv_destroy": (C.c_int, [_vp]),
    "pfbg_conv_set_kernel": (C.c_int, [_vp, _vp, _i32, _u32, _vp]),
    "pfbg_conv_apply": (C.c_int, [_vp, _vp, _vp, _dbl, _vp, _u32, _vp]),
    "pfbg_conv_info": (C.c_int, [_vp, C.POINTER(_i32), C.POINTER(_i32)]),
    "pfbg_conv_set_gauss": (C.c_int, [_vp, C.POINTER(_dbl), C.POINTER(_dbl), _i32]),
    "pfbg_conv_apply_add": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _vp]),
    "pfbg_conv_apply_shifted": (C.c_int, [_vp, _vp, _vp, _dbl, _i32, _vp, _u32, _vp]),
    "pfbg_conv_apply_scaled": (C.c_int, [_vp, _vp, _vp, _vp, _dbl, _dbl, _vp, _u32, _vp]),
    "pfbg_debug_fft1d": (C.c_int, [_i32, _i32, _i32, _i32, _vp, _vp, _i32, _i32]),
    "pfbg_debug_es_fast64": (C.c_int, [_i32, _i64, _vp, C.c_double, _vp]),
    "pfbg_weight_data_corr": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i64, _i64, _i64, _i64,
                                        _vp, _vp, _u32, _vp]),
    "pfbg_debug_fft2": (C.c_int, [_i32, _i32, _i32, _i32, _vp, _vp, _i32, _i32]),
    "pfbg_counts_to_weights": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _i32,
                                         _dbl, _dbl, _dbl, _dbl, _dbl, _u32, _vp]),
    "pfbg_counts_to_weights_batch": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32,
                                               _dbl, _dbl, _dbl, _dbl, _dbl, _vp, _u32, _vp]),
    "pfbg_bind_weights_robust": (C.c_int, [_vp, _vp, _i32, _i32, _dbl, _dbl, _dbl, _dbl, _dbl, _u32, _vp]),
    "pfbg_l2_reweight": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _i64, _i32, _dbl, _vp, _vp, _u32, _vp]),
    "pfbg_host_hash64": (C.c_int, [_vp, C.c_uint64, C.POINTER(C.c_uint64)]),
    "pfbg_ipc_export": (C.c_int, [_vp, _vp]),
    "pfbg_ipc_open": (C.c_int, [_i32, _vp, C.POINTER(_vp)]),
    "pfbg_ipc_close_all": (C.c_int, []),
    "pfbg_split_owner_init": (C.c_int, [_vp, _i32, _vp]),
    "pfbg_split_owner_connect": (C.c_int, [_vp, _vp]),
    "pfbg_split_helper_create": (C.c_int, [C.POINTER(PlanDesc), _i32, _vp, _vp, C.POINTER(_vp), _vp]),
    "pfbg_split_helper_serve": (C.c_int, [_vp, _vp]),
    "pfbg_split_status": (C.c_int, [_vp, _vp, C.POINTER(_i32)]),
    "pfbg_split_end": (C.c_int, [_vp]),
    "pfbg_plan_get_window": (C.c_int, [_vp, _vp]),
    # include/pfbsara.h
    "pfbs_psi_create": (C.c_int, [_i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                  _vp, _vp, _i32, _i32, C.POINTER(_vp)]),
    "pfbs_psi_destroy": (C.c_int, [_vp]),
    "pfbs_psi_dot": (C.c_int, [_vp, _vp, _vp, _u32, _vp]),
    "pfbs_psi_hdot": (C.c_int, [_vp, _vp, _vp, _u32, _vp]),
    "pfbs_dual_update": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _dbl, _dbl, _i32, _i64, _vp, _i32, _vp, _vp]),
    "pfbs_prox_21m": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _dbl, _dbl, _i32, _i64, _vp]),
    "pfbs_axpby": (C.c_int, [_i32, _i32, _vp, _dbl, _vp, _dbl, _vp, _i64, _vp]),
    "pfbs_extrapolate": (C.c_int, [_i32, _i32, _vp, _vp, _i64, _vp]),
    "pfbs_primal_step": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _dbl, _i32, _i32, _i64, _vp]),
    "pfbs_dot2": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _i64, C.POINTER(_dbl), _vp]),
    "pfbs_norm_diff": (C.c_int, [_i32, _i32, _vp, _vp, _i64, C.POINTER(_dbl), _vp]),
    "pfbs_clark_create": (C.c_int, [_i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _u32, _vp, C.POINTER(_vp)]),
    "pfbs_clark_destroy": (C.c_int, [_vp]),
    "pfbs_clark_run": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _dbl, _dbl, _dbl, _i32, _dbl, _i32, C.POINTER(_i32), _vp, _vp,
                                 _vp, _vp, _i64, _vp, _u32, _vp]),
    "pfbs_tree_cg_work_bytes": (_i64, [_i32, _vp, _i64]),
    "pfbs_tree_cg": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _dbl, _i32, _i32, _vp, _i64, _vp,
                               _vp, _vp, _vp]),
}

_lib = None


# translation units of libpfbgrid.so and every file each one includes, directly or not (incremental rebuilds: the
# gridder unit takes minutes to compile, the others seconds; tests/test_build_units.py keeps the lists exact)
_UNITS = {
    "pfbgrid.cu": ["common.cuh", "fft.cuh", "fused_fft.cuh", "kernels.cuh", "runs.cuh", "runs_mma.cuh", "cols2_api.h",
                   "fused_common.cuh", "fft_host.h", "host.h", "../../include/pfbgrid.h"],
    "colsfft.cu": ["common.cuh", "fft.cuh", "fft2.cuh", "cols2.cuh", "rows2.cuh", "cols2_api.h", "fused_common.cuh",
                   "fft_host.h", "host.h", "../../include/pfbgrid.h"],
    "psfconv.cu": ["psfconv.cuh", "fft.cuh", "fft_host.h", "host.h", "../../include/pfbgrid.h"],
    "weighting.cu": ["weighting.cuh", "common.cuh", "host.h", "../../include/pfbgrid.h"],
    "pfbsara.cu": ["sara.cuh", "clean.cuh", "cg.cuh", "host.h", "../../include/pfbsara.h", "../../include/pfbgrid.h"],
}


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile ``csrc/*.cu`` for sm_100a into ``libpfbgrid.so`` (in-tree), one object per translation unit.

    Stale units compile concurrently, so a clean build takes about as long as the slowest unit."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    objs, stale = [], []
    for unit, deps in _UNITS.items():
        src = os.path.join(CSRC, unit)
        obj = os.path.join(objdir, unit.replace(".cu", ".o"))
        objs.append(obj)
        stamps = [os.path.getmtime(src)] + [os.path.getmtime(os.path.normpath(os.path.join(CSRC, d))) for d in deps]
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(stamps):
            cmd = [nvcc, *flags, "-c", src, "-o", obj]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
                print(" ".join(cmd), file=sys.stderr)
            stale.append(cmd)
    with ThreadPoolExecutor(max_workers=max(1, len(stale))) as pool:
        results = list(pool.map(lambda cmd: subprocess.run(cmd, capture_output=True, text=True), stale))
    for res in results:
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed:\n{res.stdout}\n{res.stderr}")
        if verbose:
            print(res.stderr, file=sys.stderr)
    if stale or not os.path.exists(LIB_PATH) or any(os.path.getmtime(o) > os.path.getmtime(LIB_PATH) for o in objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", *objs, "-o", LIB_PATH, "-lcufft",
               "-Xlinker", "-rpath=/usr/local/cuda/lib64"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    return LIB_PATH


def load():
    """Load the library (building it if nvcc is available and it is missing/stale)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        try:
            build()
        except Exception as e:  # no silent fallback
            raise RuntimeError(
                f"{LIB_PATH} is missing and could not be built ({e}); run `python __graft_entry__.py build`"
            ) from e
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the ABI and the header drift
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        msg = load().pfbg_last_error()
        raise RuntimeError(f"pfbgrid error {rc}: {msg.decode() if msg else '?'}")


def device_count() -> int:
    n = _i32(0)
    check(load().pfbg_device_count(C.byref(n)))
    return n.value
