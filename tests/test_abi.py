"""CPU: the C-ABI library builds, loads and exports every symbol include/pfbgrid.h declares;
compute entry points fail loudly (no CPU fallback) when no B200 is present."""
import ctypes
import os
import re

import numpy as np
import pytest

from pfb_imaging_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    syms = set()
    for h in ("pfbgrid.h", "pfbsara.h"):  # every header under include/
        src = open(os.path.join(ROOT, "include", h)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        syms |= set(re.findall(r"\b(pfb[gs]_[a-z_0-9]+)\s*\(", src))
    return sorted(syms)


def test_header_declares_symbols():
    syms = header_symbols()
    assert "pfbg_grid" in syms and "pfbg_degrid" in syms and "pfbg_hessian" in syms and "pfbg_bind_vis" in syms
    assert "pfbs_psi_dot" in syms and "pfbs_dual_update" in syms
    assert len(syms) >= 24
    assert sorted(os.listdir(os.path.join(ROOT, "include"))) == ["pfbgrid.h", "pfbsara.h"]


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(_lib.build())
    for s in header_symbols():
        assert hasattr(lib, s), f"{s} declared in include/pfbgrid.h but not exported"


def test_binding_covers_header():
    assert set(header_symbols()) == set(_lib.SIGNATURES), "ctypes SIGNATURES and the header drifted"
    lib = _lib.load()
    assert lib.pfbg_version() >= 100


def test_struct_layout_matches_header():
    # 8 int32 + 2 int32 + 11 doubles + 4 pointers + 4 int32 (n_gl, pmirror, fast_screen, flags)
    assert ctypes.sizeof(_lib.PlanDesc) == 10 * 4 + 11 * 8 + 4 * 8 + 4 * 4
    assert ctypes.sizeof(_lib.PlanInfo) == 5 * 8 + 6 * 4


@pytest.mark.parametrize("w", [9, 16])
def test_fp32_plans_stop_at_w8(w):
    """An fp32 descriptor with W > 8 (the planner's W_LIMIT) is an argument error of pfbg_plan_create and of
    pfbg_split_helper_create, named as such, before any CUDA call: so it also holds without a GPU."""
    lib = _lib.load()
    keep = [np.ones(64), np.ones(64), np.linspace(0.1, 0.9, 4), np.full(4, 0.25)]
    d = _lib.PlanDesc(precision=_lib.PFBG_F32, device=0, nx=64, ny=64, nu=96, nv=96, W=w, nplanes=16, do_wgridding=1,
                      divide_by_n=1, beta=2.3 * w, pixsize_x=1e-5, pixsize_y=1e-5, usign=1.0, vsign=1.0, wsign=1.0,
                      w0=0.0, dw=1.0, corr_u=keep[0].ctypes.data, corr_v=keep[1].ctypes.data,
                      gl_x=keep[2].ctypes.data, gl_w=keep[3].ctypes.data, n_gl=4)
    out = ctypes.c_void_p()
    assert lib.pfbg_plan_create(ctypes.byref(d), ctypes.byref(out)) == _lib.PFBG_ERR_ARG
    assert b"fp32 plans stop at W=8" in lib.pfbg_last_error()
    assert not out.value
    window = np.array([0, 96, 0, 96], dtype=np.int32)
    blobs = ctypes.create_string_buffer(4 * _lib.IPC_BLOB_BYTES)
    mailbox = ctypes.create_string_buffer(_lib.IPC_BLOB_BYTES)
    rc = lib.pfbg_split_helper_create(ctypes.byref(d), 1, window.ctypes.data, blobs, ctypes.byref(out), mailbox)
    assert rc == _lib.PFBG_ERR_ARG
    assert b"fp32 plans stop at W=8" in lib.pfbg_last_error()
    assert not out.value


def _no_gpu():
    try:
        return _lib.device_count() == 0
    except RuntimeError:
        return True


@pytest.mark.skipif(not _no_gpu(), reason="only meaningful on the GPU-less build container")
def test_no_silent_cpu_fallback():
    from pfb_imaging_b200 import wgridder

    uvw = np.zeros((4, 3))
    freq = np.array([1e9])
    with pytest.raises(RuntimeError, match="pfbgrid error"):
        wgridder.dirty2vis(uvw=uvw, freq=freq, dirty=np.ones((16, 16)), pixsize_x=1e-5, pixsize_y=1e-5, epsilon=1e-5)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "pfb-imaging_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f"{f} imports the oracle"


@pytest.mark.skipif(not _no_gpu(), reason="only meaningful on the GPU-less build container")
def test_sara_has_no_cpu_fallback():
    from pfb_imaging_b200.sara import PsiNocopyt

    with pytest.raises(RuntimeError, match="pfbgrid error"):
        PsiNocopyt(1, 64, 64, ["self", "db1"], 1, 1)


def test_host_content_hash_sees_single_element_edits():
    """The plan cache of pfb_imaging_b200.operators validates cached bindings with pfbg_host_hash64: ONE changed
    element anywhere in an array (a newly flagged sample, a re-weighted one) must change the hash."""
    from pfb_imaging_b200.wgridder import content_hash

    rng = np.random.default_rng(0)
    for n in (1, 7, 8, 31, 32, 33, 4097, 3_000_001):
        m = rng.integers(0, 2, n).astype(np.uint8)
        h0 = content_hash(m)
        assert h0 == content_hash(m.copy())
        for k in {0, n // 3, n // 2, n - 1}:
            m2 = m.copy()
            m2[k] ^= 1
            assert content_hash(m2) != h0, (n, k)
    w = rng.uniform(0.5, 1.5, (1500, 640))  # 7.7 MB: the threaded path
    h0 = content_hash(w)
    for idx in [(0, 0), (700, 333), (1499, 639), (1, 638)]:
        w2 = w.copy()
        w2[idx] = np.nextafter(w2[idx], 2.0)
        assert content_hash(w2) != h0
    assert content_hash(w[:, ::2]) == content_hash(np.ascontiguousarray(w[:, ::2]))  # strided views hash their content
    assert content_hash(w[:10]) != content_hash(w[:11])
