"""GPU: the in-shared-memory mixed-radix FFT engine (csrc/fft.cuh) against numpy, and the fused
plane transforms against the cuFFT path of the same library."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.fft as sfft

from pfb_imaging_b200 import _lib
from pfbg_testutil import rel_l2

pytestmark = pytest.mark.gpu

SIZES = [32, 64, 96, 160, 224, 256, 480, 512, 1120, 2048, 3360, 4096, 6144, 7168,
         11, 22, 121, 1331, 5632, 5775, 12672,  # radix 11 (ducc0.fft.good_size PSF grids), up to 2^7 3^2 11
         6561,  # 3^8: eight generic odd stages
         12800, 16384]  # 12800: fp64 rows at the shared-memory limit; 2^14: fp32 only
KMAX_SMEM = 232448  # 227 KB of opt-in shared memory per CTA


def fits(n, prec):
    """fft_smem_bytes(n) <= 227 KB: one pad element per 16 (fp32) / 8 (fp64) elements."""
    e = n - 1
    return (e + (e >> (4 if prec == "single" else 3)) + 1) * (8 if prec == "single" else 16) <= KMAX_SMEM


@pytest.mark.parametrize("prec", ["single", "double"])
@pytest.mark.parametrize("mode", [0, 1])
def test_fft_engine_matches_numpy(gpu, prec, mode):
    """Against a long-double scipy.fft reference of the device-precision input; the tolerance grows with log2(n)
    and never exceeds the old flat 3e-6 (fp32) / 1e-13 (fp64)."""
    lib = _lib.load()
    rng = np.random.default_rng(7)
    cdt = np.complex64 if prec == "single" else np.complex128
    checked = []
    for n in SIZES:
        if not fits(n, prec):
            continue
        tol = min(3e-6, 2e-7 * np.log2(n)) if prec == "single" else min(1e-13, 1e-14 * np.log2(n))
        x = (rng.standard_normal((3, n)) + 1j * rng.standard_normal((3, n))).astype(cdt)
        xl = x.astype(np.clongdouble)
        for inverse in (0, 1):
            out = np.empty_like(x)
            _lib.check(lib.pfbg_debug_fft1d(_lib.PFBG_F32 if prec == "single" else _lib.PFBG_F64, 0, n, 3,
                                            C.c_void_p(x.ctypes.data), C.c_void_p(out.ctypes.data), mode, inverse))
            ref = sfft.ifft(xl, axis=1) * n if inverse else sfft.fft(xl, axis=1)
            err = float(np.linalg.norm((out.astype(np.clongdouble) - ref).astype(np.complex128))
                        / np.linalg.norm(ref.astype(np.complex128)))
            assert err <= tol, (n, mode, inverse, err, tol)
        checked.append(n)
    assert (16384 in checked) == (prec == "single") and 12800 in checked and 12672 in checked


CHILD = """
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + "/tests")
from pfb_imaging_b200 import wgridder as W
from pfbg_testutil import small_problem
p = small_problem(nrow=800, nchan=3, nx=96, ny=64, seed=4)
out = {{}}
for prec, eps in (("single", 1e-4), ("double", 1e-8)):
    rdt, cdt = (np.float32, np.complex64) if prec == "single" else (np.float64, np.complex128)
    gp = W.plan_for(p["uvw"], p["freq"], npix_x=96, npix_y=64, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=eps,
                    precision=prec, mask=p["mask"], center_x=0.01, flip_v=True)
    out[prec + "_v"] = gp.degrid(p["img"].astype(rdt))
    out[prec + "_d"] = gp.grid(p["vis"].astype(cdt), p["wgt"].astype(rdt))
    gp.bind_weights(p["wgt"].astype(rdt))
    out[prec + "_h"] = gp.hessian(p["img"].astype(rdt), beam=np.full((96, 64), 0.9, rdt), wsum=3.0, eta=0.1)
    gp.close()
np.savez(sys.argv[1], **out)
"""


def test_fused_transforms_match_cufft_path(gpu, tmp_path):
    """Same inputs through PFBG_FFT=cufft (k_img2grid/k_grid2img + cuFFT) and the fused kernels."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "child.py"
    script.write_text(CHILD.format(root=root))
    res = {}
    for mode in ("cufft", "fused"):
        env = dict(os.environ, PFBG_FFT=mode)
        f = tmp_path / f"{mode}.npz"
        r = subprocess.run([sys.executable, str(script), str(f)], env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
        res[mode] = np.load(f)
    for k in res["cufft"].files:
        tol = 2e-5 if k.startswith("single") else 1e-12
        assert rel_l2(res["fused"][k], res["cufft"][k]) <= tol, k
