"""GPU: the PSF-convolution Hessian (csrc/psfconv.cuh, ``pfbg_conv_*``) at production sizes, against a long-double
``scipy.fft`` reference of the same operation,

    out = beam * crop(IRFFT2(RFFT2(pad(beam * x)) * khat)) + eta * x.

The reference starts from the inputs rounded to the device precision, so input rounding is not charged to the kernel.
Every case is checked with three metrics, ``u`` the unit roundoff of the device precision and
``bound = 4 u log2(nx_psf ny_psf)``:

* global rel-L2 <= bound;
* max|err| / max|ref| <= 4 bound;
* the worst row-wise and column-wise rel-L2 <= 8 bound (a single bad row pair, column block or Nyquist column moves
  the global rel-L2 of a 4096-row image by only ~1e-5 relative to its own error).

The sizes are chosen for the regime they select (``conv_setup_t``: column-block width C; ``factorize``: the radix
list); ``pfbg_conv_info`` reports C and the table pins it, so a change of the selection rules cannot silently drop
an arm from the suite.

Measured on a B200 (1000 W power limit), worst over the beam / eta combinations of each case, as a fraction of its
bound (global rel-L2 / max-abs / worst row / worst column, each over its own limit):

    case (nx_psf x ny_psf, image)           fp32                      fp64
    5760x5760 img 4096x4096                 0.06 / 0.02 / 0.01 / 0.01 0.06 / 0.02 / 0.01 / 0.01
    5632x5632 img 5632x4094                 0.12 / 0.04 / 0.03 / 0.02 0.08 / 0.04 / 0.02 / 0.01
    5775x5775 img 4097x4095                 0.07 / 0.03 / 0.02 / 0.01 0.08 / 0.03 / 0.02 / 0.01
    5670x5670 img 1x5670                    0.04 / 0.01 / 0.01 / -    0.04 / 0.01 / 0.01 / -
    6480x6480 img 3001x4093                 0.04 / 0.02 / 0.01 / 0.01 0.07 / 0.03 / 0.01 / 0.01
    8192x8192 img 8192x1024                 0.10 / 0.04 / 0.03 / 0.01 0.06 / 0.02 / 0.02 / 0.01
    11520x2880 img 8192x2048                0.07 / 0.03 / 0.02 / 0.01 0.07 / 0.03 / 0.01 / 0.01
    14336x720 img 10001x720                 0.08 / 0.04 / 0.03 / 0.01 rejected
    720x12800 img 512x9000                  0.07 / 0.03 / 0.01 / 0.01 0.07 / 0.02 / 0.01 / 0.01
    720x26880 img 720x20000                 0.07 / 0.02 / 0.01 / 0.01 rejected
    6561x6561 img 4097x1                    0.03 / 0.01 / -    / 0.00 0.06 / 0.02 / -    / 0.01
    2x2 img 1x1                             0.22 / 0.06 / -    / -    0.03 / 0.01 / -    / -
    2x2 img 2x2                             0.14 / 0.03 / -    / -    0.13 / 0.03 / -    / -
    3x3 img 3x3                             0.11 / 0.02 / -    / -    0.11 / 0.03 / -    / -
    5x4 img 5x3                             0.08 / 0.02 / -    / -    0.12 / 0.03 / -    / -
    11x11 img 7x11                          0.08 / 0.03 / -    / -    0.10 / 0.03 / -    / -
    99x98 img 51x77                         0.11 / 0.03 / 0.02 / 0.02 0.10 / 0.03 / 0.02 / 0.02
    96x98 img 96x98                         0.12 / 0.04 / 0.02 / 0.02 0.10 / 0.03 / 0.02 / 0.02
    99x98 img 1x50                          0.04 / 0.01 / 0.01 / -    0.03 / 0.01 / 0.00 / -
    99x98 img 60x1                          0.08 / 0.03 / -    / 0.01 0.07 / 0.02 / -    / 0.01
    full spectrum 3x3 img 3x3               0.19 / 0.06 / -    / -    0.22 / 0.06 / -    / -
    full spectrum 5x4 img 5x3               0.12 / 0.04 / -    / -    0.11 / 0.04 / -    / -
    full spectrum 11x11 img 7x11            0.09 / 0.03 / -    / -    0.12 / 0.03 / -    / -
    full spectrum 99x98 img 60x45           0.12 / 0.04 / 0.02 / 0.02 0.10 / 0.03 / 0.02 / 0.02
    full spectrum 1575x1540 img 1201x1001   0.08 / 0.02 / 0.01 / 0.01 0.09 / 0.03 / 0.01 / 0.01
    full spectrum 720x5775 img 511x4097     0.07 / 0.02 / 0.01 / 0.01 0.09 / 0.02 / 0.01 / 0.01
    HessPSF 5760x5760 img 4096x4096, 2 bands                          0.05 / 0.02 / 0.01 / 0.01

Every case sits at or below 0.22 of its bound, so the constant 4 leaves a factor of about 5 of headroom, while one
mis-indexed row pair, column block or Nyquist column gives an O(1) row or column error.  ("-": the row or
column metric needs at least 16 pixels along that axis.)
"""
import ctypes as C
import math
import os

import numpy as np
import pytest
import scipy.fft as sfft

from pfb_imaging_b200 import _lib
from pfb_imaging_b200 import psf as P

gpu = pytest.mark.gpu
LD, CLD = np.longdouble, np.clongdouble
WORKERS = os.cpu_count() or 1
KMAX_SMEM = 232448  # 227 KB of opt-in shared memory per CTA (pfbgrid.cu kMaxSmem)
UNIT = {np.float32: 2.0**-24, np.float64: 2.0**-53}


# --- the host-side selection rules of pfbgrid.cu, restated ------------------------------------------------------------
def factorize(n, fp32):
    """pfbgrid.cu factorize(): odd radices first (11, 7, 5, 3), then radix 16 (fp32) / 8 (fp64) and one last power of
    two; None when n has another prime factor or needs more than 12 stages."""
    rad, m = [], n
    for r in (11, 7, 5, 3):
        while m % r == 0:
            rad.append(r)
            m //= r
    a = 0
    while m % 2 == 0:
        m //= 2
        a += 1
    if m != 1:
        return None
    lg = 4 if fp32 else 3
    while a >= lg:
        rad.append(1 << lg)
        a -= lg
    if a:
        rad.append(1 << a)
    return rad if len(rad) <= 12 else None


def smem_bytes(nelem, fp32):
    """fft_smem_bytes(): one pad element per 16 (fp32) / 8 (fp64) elements."""
    e = nelem - 1
    return (e + (e >> (4 if fp32 else 3)) + 1) * (8 if fp32 else 16)


def col_block(nxp, nyp, fp32):
    """conv_setup_t(): C columns per CTA of the column pass, 0 when the sizes are rejected."""
    if factorize(nxp, fp32) is None or factorize(nyp, fp32) is None or smem_bytes(nyp, fp32) > KMAX_SMEM:
        return 0
    cc = 4 if fp32 else 2
    while cc > 1 and (nyp % cc or smem_bytes(nxp * cc, fp32) > KMAX_SMEM):
        cc //= 2
    return cc if smem_bytes(nxp * cc, fp32) <= KMAX_SMEM else 0


# (nx_psf, ny_psf, nx, ny, C fp32, C fp64 (0: rejected), why)
CASES = [
    (5760, 5760, 4096, 4096, 4, 2, "c3 / Clark production shape"),
    (5632, 5632, 5632, 4094, 4, 2, "radix 11; nx == nx_psf; ny % 4 == 2"),
    (5775, 5775, 4097, 4095, 1, 1, "odd: every odd radix, C = 1 from parity; odd nx"),
    (5670, 5670, 1, 5670, 2, 2, "ny_psf = 2 mod 4; nx = 1; ny == ny_psf"),
    (6480, 6480, 3001, 4093, 4, 1, "fp64 C = 1 from shared-memory size; odd nx, ny % 4 == 1"),
    (8192, 8192, 8192, 1024, 2, 1, "fp32 C = 2 from size; deepest power-of-two dispatch"),
    (11520, 2880, 8192, 2048, 2, 1, "the PSF of an 8192^2 field"),
    (14336, 720, 10001, 720, 1, 0, "fp32 C = 1 from size; odd nx"),
    (720, 12800, 512, 9000, 4, 2, "rows at the fp64 shared-memory limit"),
    (720, 26880, 720, 20000, 4, 0, "rows at the fp32 shared-memory limit"),
    (6561, 6561, 4097, 1, 1, 1, "3^8: eight generic odd stages; ny = 1"),
    (2, 2, 1, 1, 2, 2, "tiny"),
    (2, 2, 2, 2, 2, 2, "tiny, no padding"),
    (3, 3, 3, 3, 1, 1, "tiny odd"),
    (5, 4, 5, 3, 4, 2, "tiny, radix 5 and 4"),
    (11, 11, 7, 11, 1, 1, "radix 11 at n = 11"),
    (99, 98, 51, 77, 2, 2, "radix 11 along x, 7 * 7 along y at small n"),
    (96, 98, 96, 98, 2, 2, "no padding, ny_psf = 2 mod 4"),
    (99, 98, 1, 50, 2, 2, "nx = 1"),
    (99, 98, 60, 1, 2, 2, "ny = 1"),
]
# the stage lists the big cases are chosen for (pfbgrid.cu factorize)
RADICES = {
    (5760, True): [5, 3, 3, 16, 8], (5760, False): [5, 3, 3, 8, 8, 2],
    (5632, True): [11, 16, 16, 2], (5632, False): [11, 8, 8, 8],
    (5775, True): [11, 7, 5, 5, 3], (5775, False): [11, 7, 5, 5, 3],
    (5670, True): [7, 5, 3, 3, 3, 3, 2], (5670, False): [7, 5, 3, 3, 3, 3, 2],
    (6480, False): [5, 3, 3, 3, 3, 8, 2],
    (8192, False): [8, 8, 8, 8, 2],
    (14336, True): [7, 16, 16, 8],
    (6561, True): [3] * 8, (6561, False): [3] * 8,
}


def _cid(c):
    return f"{c[0]}x{c[1]}-img{c[2]}x{c[3]}"


def test_selection_rules_cover_the_table():
    """CPU: the restated rules give the table's C and radix lists, so the table still reaches every arm it claims."""
    for nxp, nyp, nx, ny, c32, c64, _ in CASES:
        assert col_block(nxp, nyp, True) == c32, (nxp, nyp)
        assert col_block(nxp, nyp, False) == c64, (nxp, nyp)
    for (n, fp32), rad in RADICES.items():
        assert factorize(n, fp32) == rad, (n, fp32)
    arms = [r for (n, fp32) in RADICES for r in factorize(n, fp32)]
    assert 11 in arms and 7 in arms
    assert any(factorize(n, f).count(3) >= 2 for n, f in RADICES)
    assert any(factorize(n, f)[-1] in (2, 4) for n, f in RADICES)
    assert {c[4] for c in CASES} >= {1, 2, 4} and {c[5] for c in CASES} >= {0, 1, 2}
    assert any(c[1] % 2 for c in CASES) and any(c[1] % 4 == 2 for c in CASES)
    assert any(c[2] % 2 and c[2] > 1 for c in CASES) and any(c[3] % 4 for c in CASES)


# --- helpers -----------------------------------------------------------------------------------------------------------
def _hermitian_edges(k, nyp):
    """Make the l = 0 (and, for even ny_psf, the Nyquist) column of a half spectrum Hermitian along the first axis, as
    the half spectrum of a real kernel is: irfft2 and the device agree only on such kernels."""
    nxp = k.shape[0]
    m = (-np.arange(nxp)) % nxp
    for col in (0, nyp // 2) if nyp % 2 == 0 else (0,):
        k[:, col] = 0.5 * (k[:, col] + np.conj(k[m, col]))
    return k


def _psf_kernel(nxp, nyp, rng, complex_kernel, support=24):
    """Half spectrum of a real, PSF-like kernel: a random block around the origin (wrapped) plus a peak.  Complex
    (``psfhat``) or its modulus (``abspsf``); both are spectra of real kernels."""
    hx, hy = min(support, nxp) // 2, min(support, nyp) // 2
    ix = np.arange(-hx, min(support, nxp) - hx) % nxp
    iy = np.arange(-hy, min(support, nyp) - hy) % nyp
    k = np.zeros((nxp, nyp))
    k[np.ix_(ix, iy)] = rng.standard_normal((ix.size, iy.size))
    k[0, 0] += 4.0
    khat = sfft.rfft2(k, workers=WORKERS)
    if not complex_kernel:
        khat = np.abs(khat).astype(np.complex128)
    return _hermitian_edges(khat, nyp)


def _reference(x, khat, nxp, nyp, beam=None, eta=0.0):
    """Long-double reference from device-precision inputs (half spectrum of a real kernel)."""
    nx, ny = x.shape
    xin = x.astype(LD)
    if beam is not None:
        xin = xin * beam.astype(LD)
    t = sfft.rfft(xin, n=nyp, axis=1, workers=WORKERS)
    t = sfft.fft(t, n=nxp, axis=0, workers=WORKERS)
    t *= khat.astype(CLD)
    t = sfft.ifft(t, axis=0, workers=WORKERS)[:nx]
    out = sfft.irfft(t, n=nyp, axis=1, workers=WORKERS)[:, :ny]
    if beam is not None:
        out *= beam.astype(LD)
    if eta:
        out += LD(eta) * x.astype(LD)
    return out


def _errors(got, ref):
    """(global rel-L2, max|err| / max|ref|, worst row rel-L2, worst column rel-L2); a row (column) metric needs rows
    (columns) of at least 16 pixels to be meaningful and is 0 otherwise."""
    e = (got.astype(LD) - ref).astype(np.float64)
    r = ref.astype(np.float64)
    g = float(np.linalg.norm(e) / np.linalg.norm(r))
    mx = float(np.abs(e).max() / np.abs(r).max())
    nx, ny = r.shape
    row = float((np.linalg.norm(e, axis=1) / np.linalg.norm(r, axis=1)).max()) if ny >= 16 else 0.0
    col = float((np.linalg.norm(e, axis=0) / np.linalg.norm(r, axis=0)).max()) if nx >= 16 else 0.0
    return g, mx, row, col


def _bound(dt, nxp, nyp):
    return 4.0 * UNIT[dt] * math.log2(max(nxp * nyp, 2))


def _check(got, ref, dt, nxp, nyp, what):
    b = _bound(dt, nxp, nyp)
    g, mx, row, col = _errors(got, ref)
    print(f"psfconv {what}: bound {b:.2e}  rel-L2 {g / b:.3f}  max {mx / (4 * b):.3f}  row {row / (8 * b):.3f}  "
          f"col {col / (8 * b):.3f}")
    assert g <= b, (what, "global rel-L2", g, b)
    assert mx <= 4 * b, (what, "max|err|/max|ref|", mx, 4 * b)
    assert row <= 8 * b, (what, "worst row rel-L2", row, 8 * b)
    assert col <= 8 * b, (what, "worst column rel-L2", col, 8 * b)


def _info(cv):
    cb, rt = C.c_int32(0), C.c_int32(0)
    _lib.check(cv._lib.pfbg_conv_info(cv._h, C.byref(cb), C.byref(rt)))
    return cb.value, rt.value


# --- against the long-double reference --------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("case", CASES, ids=[_cid(c) for c in CASES])
def test_conv_matches_long_double_reference(gpu, case, dt):
    nxp, nyp, nx, ny, c32, c64, why = case
    cexp = c32 if dt == np.float32 else c64
    if cexp == 0:  # past the shared-memory limit: the library's error, not a launch failure
        with pytest.raises(RuntimeError, match="pfbgrid error"):
            P.PsfConvolver(nx, ny, nxp, nyp, dtype=dt)
        return
    rng = np.random.default_rng(nxp * 7 + nyp + nx)
    cdt = np.complex64 if dt == np.float32 else np.complex128
    khat = _psf_kernel(nxp, nyp, rng, complex_kernel=True).astype(cdt)
    cv = P.PsfConvolver(nx, ny, nxp, nyp, dtype=dt)
    try:
        cb, rt = _info(cv)
        assert cb == cexp, (why, cb, cexp)
        assert 128 <= rt <= 256 and rt % 32 == 0
        x = rng.standard_normal((nx, ny)).astype(dt)
        # beam / eta none / 0 with the complex psfhat; set / != 0 with the real abspsf
        cv.set_kernel(khat)
        _check(cv.apply(x), _reference(x, khat, nxp, nyp), dt, nxp, nyp, f"{_cid(case)} {dt.__name__} plain")
        absk = np.abs(khat).astype(cdt)
        beam = rng.uniform(0.3, 1.0, (nx, ny)).astype(dt)
        cv.set_kernel(absk)
        _check(cv.apply(x, beam=beam, eta=0.37), _reference(x, absk, nxp, nyp, beam, 0.37), dt, nxp, nyp,
               f"{_cid(case)} {dt.__name__} beam+eta")
    finally:
        cv.close()


# --- properties that need no FFT reference ----------------------------------------------------------------------------
IMPULSE = [(2, 2, 2, 2), (3, 3, 3, 3), (11, 11, 11, 11), (5, 4, 5, 3), (99, 98, 60, 45), (98, 99, 97, 98),
           (1575, 1540, 1001, 1201), (5775, 5775, 4097, 4095)]


@gpu
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("nxp,nyp,nx,ny", IMPULSE)
def test_impulse_gives_the_shifted_psf(gpu, nxp, nyp, nx, ny, dt):
    """A delta at (a, b) convolved with psfhat = rfft2(ifftshift(psf)) is psf[(i-a+nxp//2) % nxp, (j-b+nyp//2) % nyp]
    on the image: pins the wrap-around indexing, odd sizes included."""
    rng = np.random.default_rng(nxp + 3 * nyp)
    psf = rng.standard_normal((nxp, nyp))
    cdt = np.complex64 if dt == np.float32 else np.complex128
    psfhat = _hermitian_edges(np.fft.rfft2(np.fft.ifftshift(psf)), nyp).astype(cdt)
    cv = P.PsfConvolver(nx, ny, nxp, nyp, dtype=dt).set_kernel(psfhat)
    tol = 4 * _bound(dt, nxp, nyp)
    try:
        for a, b in {(0, 0), (nx - 1, ny - 1), (nx - 1, 0), (0, ny - 1), (nx // 2, ny // 2)}:
            x = np.zeros((nx, ny), dtype=dt)
            x[a, b] = 1
            got = cv.apply(x)
            i = (np.arange(nx)[:, None] - a + nxp // 2) % nxp
            j = (np.arange(ny)[None, :] - b + nyp // 2) % nyp
            err = np.abs(got - psf[i, j]).max() / np.abs(psf).max()
            assert err <= tol, ((a, b), err, tol)
    finally:
        cv.close()


@gpu
@pytest.mark.parametrize("nxp,nyp,nx,ny", [(99, 98, 60, 45), (1575, 1540, 1001, 1201), (5775, 5775, 4097, 4095)])
def test_adjoint_with_beam_fp64(gpu, nxp, nyp, nx, ny):
    """With a real kernel and a beam the operator is self-adjoint: <Hx, y> = <x, Hy> to 1e-13."""
    rng = np.random.default_rng(nx)
    absk = np.abs(_psf_kernel(nxp, nyp, rng, complex_kernel=True))
    beam = rng.uniform(0.3, 1.0, (nx, ny))
    cv = P.PsfConvolver(nx, ny, nxp, nyp, dtype=np.float64).set_kernel(absk)
    try:
        x, y = rng.standard_normal((2, nx, ny))
        hx, hy = cv.apply(x, beam=beam, eta=0.2), cv.apply(y, beam=beam, eta=0.2)
        a, b = float(np.vdot(hx, y)), float(np.vdot(x, hy))
        scale = np.linalg.norm(hx) * np.linalg.norm(y)
        assert abs(a - b) <= 1e-13 * scale, (a, b, scale)
    finally:
        cv.close()


@gpu
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("nxp,nyp,nx,ny", [(3, 3, 3, 3), (5, 4, 5, 3), (11, 11, 7, 11), (99, 98, 60, 45),
                                           (1575, 1540, 1201, 1001), (720, 5775, 511, 4097)])
def test_full_spectrum_kernel(gpu, nxp, nyp, nx, ny, dt):
    """set_kernel(half=0) (k_hermitize) with a random non-Hermitian complex kernel: Re(ifft2(fft2(xpad) khat))."""
    rng = np.random.default_rng(nxp * nyp)
    cdt = np.complex64 if dt == np.float32 else np.complex128
    khat = (rng.standard_normal((nxp, nyp)) + 1j * rng.standard_normal((nxp, nyp))).astype(cdt)
    x = rng.standard_normal((nx, ny)).astype(dt)
    xpad = np.zeros((nxp, nyp), dtype=CLD)
    xpad[:nx, :ny] = x
    ref = sfft.ifft2(sfft.fft2(xpad, workers=WORKERS) * khat.astype(CLD), workers=WORKERS).real[:nx, :ny]
    cv = P.PsfConvolver(nx, ny, nxp, nyp, dtype=dt).set_kernel(khat)
    try:
        _check(cv.apply(x), ref, dt, nxp, nyp, f"full {nxp}x{nyp}-img{nx}x{ny} {dt.__name__}")
    finally:
        cv.close()


@gpu
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("nxp,nyp,nx,ny", [(5760, 5760, 4096, 4096), (5775, 5775, 4097, 4095), (99, 98, 51, 77)])
def test_device_pointer_path_is_bitwise_the_host_path(gpu, nxp, nyp, nx, ny, dt):
    """apply_dev on torch tensors on a non-default stream (what SARA and Clark call) equals the host-pointer path bit
    for bit, and two applies are bitwise equal."""
    import torch

    rng = np.random.default_rng(nyp)
    cdt = np.complex64 if dt == np.float32 else np.complex128
    absk = np.abs(_psf_kernel(nxp, nyp, rng, complex_kernel=True)).astype(cdt)
    x = rng.standard_normal((nx, ny)).astype(dt)
    beam = rng.uniform(0.3, 1.0, (nx, ny)).astype(dt)
    cv = P.PsfConvolver(nx, ny, nxp, nyp, dtype=dt).set_kernel(absk)
    try:
        host = cv.apply(x, beam=beam, eta=0.37)
        assert np.array_equal(host, cv.apply(x, beam=beam, eta=0.37))
        dev = torch.device("cuda", cv.device)
        xt, bt = torch.from_numpy(x).to(dev), torch.from_numpy(beam).to(dev)
        outs = [torch.full_like(xt, float("nan")) for _ in range(2)]
        torch.cuda.synchronize(dev)
        s = torch.cuda.Stream(dev)
        for o in outs:
            cv.apply_dev(xt.data_ptr(), o.data_ptr(), bt.data_ptr(), 0.37, stream=s.cuda_stream)
        s.synchronize()
        for o in outs:
            assert np.array_equal(o.cpu().numpy(), host)
    finally:
        cv.close()


@gpu
def test_hesspsf_production_shape(gpu):
    """HessPSF.dot at the c3 operator's shape: 4096^2 images, 5760^2 PSF, beam, eta (2 bands, fp64)."""
    rng = np.random.default_rng(33)
    nband, nx, ny, nxp, nyp = 2, 4096, 4096, 5760, 5760
    abspsf = np.stack([np.abs(_psf_kernel(nxp, nyp, rng, complex_kernel=True)) for _ in range(nband)])
    beam = rng.uniform(0.3, 1.0, (nband, nx, ny))
    x = rng.standard_normal((nband, nx, ny))
    H = P.HessPSF(nx, ny, abspsf, beam=beam, eta=0.37, cgverbose=0)
    try:
        hx = H.dot(x)
    finally:
        H.close()
    for b in range(nband):
        _check(hx[b], _reference(x[b], abspsf[b], nxp, nyp, beam[b], 0.37), np.float64, nxp, nyp, f"HessPSF band {b}")


# --- limits -----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dt,nxp,nyp,ok", [
    (np.float64, 720, 12800, True), (np.float64, 720, 13125, False),    # rows at the fp64 shared-memory limit
    (np.float32, 720, 26880, True), (np.float32, 720, 27648, False),    # ... and at the fp32 one
    (np.float64, 14336, 720, False), (np.float32, 14336, 720, True),    # columns: fp64 C = 1 no longer fits
    (np.float32, 208, 64, False), (np.float64, 64, 208, False),         # prime factor 13
])
def test_limits(gpu, dt, nxp, nyp, ok):
    fp32 = dt == np.float32
    assert (col_block(nxp, nyp, fp32) > 0) == ok
    if ok:
        cv = P.PsfConvolver(16, 16, nxp, nyp, dtype=dt)
        assert _info(cv)[0] == col_block(nxp, nyp, fp32)
        cv.close()
    else:
        with pytest.raises(RuntimeError, match="pfbgrid error"):
            P.PsfConvolver(16, 16, nxp, nyp, dtype=dt)


# --- kernel caches of the drop-ins ------------------------------------------------------------------------------------
def _np_conv(x, khat, nxp, nyp):
    return np.fft.irfft2(np.fft.rfft2(x, s=(nxp, nyp)) * khat, s=(nxp, nyp))[: x.shape[0], : x.shape[1]]


@gpu
def test_convolver_cache_sees_in_place_edits(gpu):
    """An in-place edit of the kernel off the old checksum's stride, or a conjugation (|k| unchanged), must reach the
    device: the next call convolves with the new kernel."""
    nx, ny, nxp, nyp = 64, 48, 96, 80  # half spectrum 96 x 41
    rng = np.random.default_rng(5)
    x = rng.standard_normal((nx, ny))
    P.clear_convolver_cache()
    try:
        absk = np.abs(_psf_kernel(nxp, nyp, rng, complex_kernel=True).real) + 0.5
        first = P.hessian_psf_slice(x, abspsf=absk, lastsize=nyp)
        assert np.abs(first - _np_conv(x, absk, nxp, nyp)).max() <= 1e-12 * np.abs(first).max()
        f = 10 * (nyp // 2 + 1) + 5  # (10, 5): 415 is not a multiple of the old stride 3, and not an edge column
        assert f % (absk.size // 1024) != 0
        absk.flat[f] += 50.0
        got = P.hessian_psf_slice(x, abspsf=absk, lastsize=nyp)
        ref = _np_conv(x, absk, nxp, nyp)
        assert np.abs(ref - first).max() > 1e-3 * np.abs(ref).max()
        assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max()

        psf = rng.standard_normal((nxp, nyp))  # no symmetry: conj(psfhat) is the spectrum of another kernel
        psfhat = np.fft.rfft2(np.fft.ifftshift(psf))
        out = np.empty((nx, ny))
        P.psf_convolve_slice(None, None, out, psfhat, nyp, x)
        first = out.copy()
        np.conjugate(psfhat, out=psfhat)
        P.psf_convolve_slice(None, None, out, psfhat, nyp, x)
        ref = _np_conv(x, psfhat, nxp, nyp)
        assert np.abs(ref - first).max() > 1e-3 * np.abs(ref).max()
        assert np.abs(out - ref).max() <= 1e-12 * np.abs(ref).max()
    finally:
        P.clear_convolver_cache()


@gpu
def test_direct_cache_sees_in_place_edits(gpu):
    nx, ny, nxp, nyp = 64, 48, 96, 80
    rng = np.random.default_rng(6)
    x = rng.standard_normal((nx, ny))
    absk = np.abs(_psf_kernel(nxp, nyp, rng, complex_kernel=True).real) + 0.5
    first = P.hess_direct_slice(x, abspsf=absk, lastsize=nyp, eta=1.0)
    absk.flat[10 * (nyp // 2 + 1) + 5] += 50.0
    got = P.hess_direct_slice(x, abspsf=absk, lastsize=nyp, eta=1.0)
    ref = _np_conv(x, absk + 1.0, nxp, nyp)
    assert np.abs(ref - first).max() > 1e-3 * np.abs(ref).max()
    assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max()


@gpu
def test_clark_cache_sees_in_place_edits(gpu):
    """clean.clark caches the uploaded PSF: editing PSF off the old checksum's stride, or conjugating PSFHAT, in place
    must give what a fresh handle gives."""
    from pfb_imaging_b200 import clean

    rng = np.random.default_rng(8)
    nxp = nyp = 48
    nx = ny = 32
    xx = np.arange(nxp)[:, None] - nxp // 2
    yy = np.arange(nyp)[None, :] - nyp // 2
    psf = np.exp(-(xx**2 + yy**2) / 8.0)[None] + 0.05 * rng.standard_normal((1, nxp, nyp))
    psf[0, nxp // 2, nyp // 2] = 1.0
    psfhat = np.fft.rfft2(np.fft.ifftshift(psf, axes=(1, 2)), axes=(1, 2))
    sky = np.zeros((1, nx, ny))
    sky[0, rng.integers(0, nx, 6), rng.integers(0, ny, 6)] = rng.uniform(1, 5, 6)
    dirty = np.fft.irfft2(np.fft.rfft2(sky, s=(nxp, nyp)) * psfhat, s=(nxp, nyp))[:, :nx, :ny]
    kw = dict(gamma=0.1, pf=0.01, maxit=5, submaxit=200)

    def fresh():
        cl = clean.Clark(psf.copy(), psfhat.copy(), nx=nx, ny=ny)
        try:
            return cl(dirty, **kw)[:2]
        finally:
            cl.close()

    clean.clear_clark_cache()
    try:
        m0, r0, _ = clean.clark(dirty, psf, psfhat, **kw)
        np.conjugate(psfhat, out=psfhat)
        m1, r1, _ = clean.clark(dirty, psf, psfhat, **kw)
        fm, fr = fresh()
        assert not np.array_equal(r1, r0)
        assert np.array_equal(m1, fm) and np.array_equal(r1, fr)
        f = (nxp // 2) * nyp + nyp // 2 + 1  # next to the peak, off the old stride 2
        assert f % (psf.size // 1024) != 0
        psf.flat[f] += 0.5
        m2, r2, _ = clean.clark(dirty, psf, psfhat, **kw)
        fm, fr = fresh()
        assert not (np.array_equal(m2, m1) and np.array_equal(r2, r1))
        assert np.array_equal(m2, fm) and np.array_equal(r2, fr)
    finally:
        clean.clear_clark_cache()
