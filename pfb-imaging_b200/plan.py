"""Host-side plan for the B200 w-stacked gridder.

A :class:`Plan` fixes everything the CUDA kernels need and nothing they can
decide themselves: oversampled grid ``nu x nv``, ES-kernel support ``W`` and
shape ``beta``, the w-plane stack ``(w0, dw, nplanes)``, the ``n-1`` shift, and
the fp64 separable grid-correction vectors.  It replaces the parameter search
ducc0.wgridder 0.41.0 (``pyproject.toml:42``, ``uv.lock:1119-1120``; source not
in the reference tree) performs internally for every ``vis2dirty`` /
``dirty2vis`` call made from ``src/pfb_imaging/operators/gridder.py:78-100``
and ``operators/hessian.py:50-89``.

Conventions (pinned by ``tests/test_hessian_approx.py:23-67`` and
``operators/gridder.py:23-34``):

    l_i = center_x + (i - nx/2) * pixsize_x       m_j likewise
    nm1 = n - 1 = -(l^2+m^2) / (sqrt(1-l^2-m^2) + 1)
    vis = sum_ij dirty_ij * exp(-2 pi i f/c (u l + v m - w nm1))   [/ n]

``flip_u`` negates ``u`` *and* ``center_x`` (same for v); ``flip_w`` negates w.
"""

from __future__ import annotations

import functools
import math
import os
from dataclasses import dataclass, field

import numpy as np
from numpy.polynomial.legendre import leggauss

from . import kernel_table as kt

LIGHTSPEED = 299792458.0  # scipy.constants.c, as used at operators/gridder.py:12

TILE = 16  # uv tile edge of the binning kernel (cells)
N_GL = 64  # Gauss-Legendre nodes for the w-correction evaluated on device
FAST_SCREEN_EPS = 3e-6  # fp32 plans at or above this accuracy take the w-screen phasors from the SFU


def good_size(n: int, primes=(2, 3, 5, 7)) -> int:
    """Smallest integer >= n whose prime factors are all in `primes`.

    Stands in for ``ducc0.fft.good_size`` (``utils/misc.py:921-951``) with the
    factor set restricted to what cuFFT handles without Bluestein.
    """
    n = int(n)
    if n <= 1:
        return 1
    best = 1 << (n - 1).bit_length()
    p7 = 1
    while p7 < best:
        p57 = p7
        while p57 < best:
            p357 = p57
            while p357 < best:
                x = p357
                while x < n:
                    x *= 2
                if x < best:
                    best = x
                if 3 not in primes:
                    break
                p357 *= 3
            if 5 not in primes:
                break
            p57 *= 5
        if 7 not in primes:
            break
        p7 *= 7
    return best


def padded_size(n: int, sigma: float, W: int, mult: int = 2 * TILE) -> int:
    """Oversampled grid length: a 7-smooth multiple of `mult`, >= sigma*n and >= n+W."""
    need = max(int(math.ceil(sigma * n - 1e-9)), n + W + 1)
    return good_size((need + mult - 1) // mult) * mult


def nm1_of_r2(r2):
    r2 = np.asarray(r2, dtype=np.float64)
    return -r2 / (np.sqrt(1.0 - r2) + 1.0)


def _axis_range2(c, n, d):
    """min and max of l^2 over the pixel centres l = c + (i - n/2) d, i in [0, n)."""
    lo = c - (n // 2) * d
    hi = c + (n - 1 - n // 2) * d
    a, b = min(lo, hi), max(lo, hi)
    mx = max(a * a, b * b)
    mn = 0.0 if a <= 0.0 <= b else min(a * a, b * b)
    return mn, mx


@dataclass
class Plan:
    precision: str  # "single" | "double"
    nx: int
    ny: int
    nu: int
    nv: int
    W: int
    beta: float
    sigma: float
    nplanes: int
    w0: float
    dw: float
    nshift: float
    pixsize_x: float
    pixsize_y: float
    center_x: float  # after the flip rule
    center_y: float
    usign: float
    vsign: float
    wsign: float
    do_wgridding: bool
    divide_by_n: bool
    epsilon: float
    kernel_err: float
    corr_u: np.ndarray = field(repr=False)  # (nx,) fp64: 1/psihat(i'/nu)
    corr_v: np.ndarray = field(repr=False)
    gl_x: np.ndarray = field(repr=False)  # nodes on [0,1] for psihat_w on device
    gl_w: np.ndarray = field(repr=False)
    est_cost: float = 0.0
    pmirror: int = 0  # virtual planes below plane 0 served by Hermitian mirroring (then w0 == dw/2)
    nplanes_std: int = 0  # planes a stack without mirroring would need for the same |w| range (reporting only)
    fast_screen: int = 0  # fp32, epsilon >= 3e-6: w-screen phasors from the SFU (abs. error ~5e-7)

    @property
    def real_bytes(self) -> int:
        return 4 if self.precision == "single" else 8

    def info(self) -> dict:
        return dict(
            precision=self.precision, nx=self.nx, ny=self.ny, nu=self.nu, nv=self.nv,
            W=self.W, beta=self.beta, sigma=self.sigma, nplanes=self.nplanes,
            w0=self.w0, dw=self.dw, nshift=self.nshift, kernel_err=self.kernel_err,
            pmirror=self.pmirror, nplanes_std=self.nplanes_std, fast_screen=self.fast_screen,
        )


def _mirror_planes(wmax, dw, W):
    """Planes needed when they sit at (p + 1/2) dw and the ones below zero are mirrored: the highest sample's
    first plane is floor(wmax/dw - 1/2 - W/2) + 1 (one plane of slack for rounding in the fp64 division)."""
    top = int(math.floor(wmax / dw - 0.5 - 0.5 * W)) + 1
    return max(top + W + 1, W, (W + 2) // 2)


def w_range(uvw, freq, wsign=1.0):
    """min/max of |w|*f/c over all rows and channels (wavelengths).

    The kernels fold samples with w < 0 onto -(u,v,w) with the conjugate visibility (the image is
    real), so the plane stack only has to cover |w|; `wsign` is therefore irrelevant and kept for
    the call signature only.
    """
    w = np.abs(np.asarray(uvw)[:, 2].astype(np.float64))
    f = np.asarray(freq, dtype=np.float64)
    if w.size == 0 or f.size == 0:
        return 0.0, 0.0
    return float(w.min()) * float(f.min()) / LIGHTSPEED, float(w.max()) * float(f.max()) / LIGHTSPEED


@functools.lru_cache(maxsize=64)
def _correction(n, nbig, W, beta):
    ip = np.arange(n) - n // 2
    out = 1.0 / kt.kernel_ft(ip / float(nbig), W, beta)
    out.setflags(write=False)
    return out


@functools.lru_cache(maxsize=4)
def _gl_half(n):
    gx, gw = leggauss(2 * n)
    gx, gw = gx[n:].copy(), gw[n:].copy()  # positive half; the integrand is even
    gx.setflags(write=False)
    gw.setflags(write=False)
    return gx, gw


# Cost model (seconds, one direction), calibrated on B200 (DESIGN.md "plan cost model"):
#   * run kernels (W <= 8): issue-bound, ~constant per sample whatever W is;
#   * direct kernels (W > 8): one atomic / gather per footprint cell;
#   * plane work (zero / FFT / screen): per complex cell of the oversampled stack.
COST_VIS_RUNS = {"single": 1.35e-10, "double": 4.0e-10}
COST_CELL_UPDATE = {"single": 7.0e-13, "double": 5.0e-12}
COST_GRID_CELL = {"single": 8.0e-12, "double": 2.0e-11}
RUNS_MAX_W = 8


def fft_cost_factor(n, precision):
    """Relative cost per cell of the fused shared-memory transforms for an axis of n = 2^a 3^b 5^c 7^d 11^e cells: one
    pass over the data per radix stage (powers of two go three (fp64, radix 8) or four (fp32, radix 16) at a time),
    odd radices cost more per pass.  Measured on the C2 geometry in fp64 (12 / 11 / 10 planes, ms per forward + inverse
    pair): 5760 -> 13.5, 6144 -> 10.3, 6048 -> 15.2, 6720 -> 19.0, 7168 -> 15.6, i.e. 0.73 / 1.02 / 1.13 / 0.90 of the
    per-cell cost at 5760; this model gives 0.78 / 1.13 / 1.03 / 0.97.  Normalised to the sizes COST_GRID_CELL was
    measured at (fp32: 6144, fp64: 5760)."""
    stage = {3: 1.0, 5: 1.4, 7: 2.2, 11: 3.5}
    k = 3 if precision == "double" else 4
    m, cost, a = int(n), 0.0, 0
    while m % 2 == 0:
        m //= 2
        a += 1
    cost += -(-a // k)
    for pr, c in stage.items():
        while m % pr == 0:
            m //= pr
            cost += c
    if m != 1:
        cost += 5.0 * math.log2(m)  # not a size the plan produces
    return cost / (6.4 if precision == "double" else 4.0)


def vis_cost(precision, W, ndim, nvis=0):
    """Run kernels: one warp per run for W <= 8; fp64 9 <= W <= 12: a team of 3 warps on the DMMA path
    (csrc/runs_mma.cuh; measured 5.1e-10 s per sample and direction on the C2 band of 25 M samples, whatever W is in
    that range, and 1.15e-9 on the 1 M samples of C1, which do not fill the GPU);
    fp64 13 <= W <= 16: scalar teams of 8 warps.  Single precision stops at W_LIMIT = 8."""
    if W <= RUNS_MAX_W:
        # W < 8 with w-gridding leaves the constant-stride / cyclic-column flush and fetch of the one-warp kernels for
        # their general path (C1 in fp64, W = 7 against W = 8: degrid 1.18 against 0.40 ms, grid 0.74 against 0.47 ms)
        return COST_VIS_RUNS[precision] * (2.0 if (W < RUNS_MAX_W and ndim == 3) else 1.0)
    if W <= 12:
        return COST_VIS_RUNS[precision] * (1.3 if nvis >= 4_000_000 else 3.0)
    return COST_VIS_RUNS[precision] * 9.0


# Largest kernel support per precision.  In single precision the grid
# correction 1/psihat amplifies the fp32 round-off of the FFT by
# psihat(0)/psihat(1/(2 sigma)) ~ exp(beta - sqrt(beta^2 - (pi W / (2 sigma))^2)),
# which explodes for wide kernels at low oversampling; ducc0 applies the same
# cap (W <= 8 for float).
W_LIMIT = {"single": 8, "double": kt.W_MAX}


def make_plan(
    *, nx, ny, pixsize_x, pixsize_y, center_x=0.0, center_y=0.0, epsilon,
    flip_u=False, flip_v=False, flip_w=False, do_wgridding=True, divide_by_n=True,
    sigma_min=1.1, sigma_max=2.6, precision="double", wmin=0.0, wmax=0.0, nvis=0,
    force_sigma=None, force_W=None, safety=None, mirror=True, max_stack_bytes=None,
) -> Plan:
    """Choose (sigma, W, beta, nu, nv, planes) for one gridder geometry."""
    nx, ny = int(nx), int(ny)
    if nx <= 0 or ny <= 0 or nx % 2 or ny % 2:
        raise ValueError("image dimensions must be positive and even (utils/misc.py:930-932)")
    if not (pixsize_x > 0 and pixsize_y > 0):
        raise ValueError("pixel sizes must be positive")
    if not (epsilon > 0):
        raise ValueError("epsilon must be positive")
    if precision not in ("single", "double"):
        raise ValueError("precision must be 'single' or 'double'")
    if precision == "single" and epsilon < 1e-7 * 3:
        raise ValueError("epsilon too small for single precision (needs >= 3e-7)")
    if epsilon < 1e-13:
        raise ValueError("epsilon too small for double precision")

    if wmin < 0.0 or wmax < wmin:  # the kernels fold w < 0 onto w > 0: the planes cover |w|
        wmin, wmax = (0.0 if wmin * wmax <= 0.0 else min(abs(wmin), abs(wmax))), max(abs(wmin), abs(wmax))
    cx = -center_x if flip_u else center_x
    cy = -center_y if flip_v else center_y
    usign = -1.0 if flip_u else 1.0
    vsign = -1.0 if flip_v else 1.0
    wsign = -1.0 if flip_w else 1.0

    l2min, l2max = _axis_range2(cx, nx, pixsize_x)
    m2min, m2max = _axis_range2(cy, ny, pixsize_y)
    if l2max + m2max >= 1.0:
        raise ValueError("image extends beyond the unit sphere (l^2+m^2 >= 1)")
    nm1_lo = float(nm1_of_r2(l2max + m2max))  # most negative
    nm1_hi = float(nm1_of_r2(l2min + m2min))
    if do_wgridding:
        nshift = -0.5 * (nm1_lo + nm1_hi)
        numax = max(0.5 * (nm1_hi - nm1_lo), 1e-300)
    else:
        nshift, numax = 0.0, 0.0

    # Error budget: the 1-D kernel error must stay below epsilon / safety.  Double precision
    # splits epsilon linearly over the interpolated axes (worst-case sum; this is what keeps the
    # max-abs bound of /root/reference/tests/test_hessian_approx.py:188-231 at epsilon=1e-10),
    # single precision splits it in quadrature (the contract there is the relative L2 norm and
    # fp32 round-off, not the kernel, sets the max-abs floor).
    ndim = 3 if do_wgridding else 2
    if safety is None:
        safety = float(ndim) if precision == "double" else math.sqrt(ndim)
    target = epsilon / safety

    sig_lo = max(float(sigma_min), kt.SIGMAS[0])
    sig_hi = max(min(float(sigma_max), kt.SIGMAS[-1]), sig_lo)
    if force_sigma is not None:
        cand_sig = [float(force_sigma)]
    else:
        cand_sig = [s for s in kt.SIGMAS if sig_lo - 1e-9 <= s <= sig_hi + 1e-9] or [sig_lo]

    best = None
    for s in cand_sig:
        W = None
        for Wc in range(kt.W_MIN, W_LIMIT[precision] + 1):
            if force_W is not None and Wc != force_W:
                continue
            beta, err = kt.lookup(s, Wc)
            if err <= target or force_W is not None:
                W = Wc
                break
        if W is None:
            continue
        # smallest admissible W for this sigma (a larger W never helps at fixed sigma)
        nu = padded_size(nx, s, W)
        nv = padded_size(ny, s, W)
        sig_eff = min(nu / nx, nv / ny)
        if do_wgridding and wmax > wmin:
            dw = 1.0 / (2.0 * s * numax)
            npl = int(math.ceil((wmax - wmin) / dw)) + W
            if mirror:
                npl = min(npl, _mirror_planes(wmax, dw, W))
        elif do_wgridding:
            dw = 1.0 / (2.0 * s * numax)
            npl = W
        else:
            dw, npl = 1.0, 1
        cost = (
            2.0 * nvis * vis_cost(precision, W, ndim, nvis)
            + 2.0 * npl * nu * nv * COST_GRID_CELL[precision]
            * 0.5 * (fft_cost_factor(nu, precision) + fft_cost_factor(nv, precision))
        )
        # `max_stack_bytes`: what the caller can spare for the plane stack (e.g. the bands of a GPU that share one
        # stack next to everything else that is resident): candidates beyond it only win when nothing fits
        stack = npl * nu * nv * (8 if precision == "single" else 16)
        if max_stack_bytes is not None and stack > max_stack_bytes:
            cost += 1e6 * (1.0 + stack / max_stack_bytes)
        if best is None or cost < best[0]:
            best = (cost, s, W, beta, err, nu, nv, dw, npl, sig_eff)
    if best is None:
        raise ValueError(
            f"no (sigma, W) in [{sig_lo}, {sig_hi}] x [{kt.W_MIN}, {W_LIMIT[precision]}] reaches "
            f"epsilon={epsilon} in {precision} precision"
        )
    cost, s, W, beta, err, nu, nv, dw, npl, sig_eff = best

    pmirror = 0
    if do_wgridding:
        npl_std = (int(math.ceil((wmax - wmin) / dw)) + W) if wmax > wmin else W
        if mirror and wmax > wmin and _mirror_planes(wmax, dw, W) < npl_std:
            # |w| reaches down to ~0: put the planes at (p + 1/2) dw and serve the W/2 planes below zero through
            # the Hermitian mirror of planes 0..W/2-1 instead of storing and transforming them
            w0 = 0.5 * dw
            npl = _mirror_planes(wmax, dw, W)
            pmirror = (W + 2) // 2
        else:
            # plane p sits at w0 + p*dw; the lowest sample's support starts at plane 0
            npl = npl_std
            w0 = 0.5 * (wmin + wmax) - 0.5 * (npl - 1) * dw
    else:
        w0 = 0.0

    gl_x, gl_w = _gl_half(N_GL)

    return Plan(
        precision=precision, nx=nx, ny=ny, nu=nu, nv=nv, W=W, beta=float(beta), sigma=float(s),
        nplanes=int(npl), w0=float(w0), dw=float(dw), nshift=float(nshift),
        pixsize_x=float(pixsize_x), pixsize_y=float(pixsize_y), center_x=float(cx), center_y=float(cy),
        usign=usign, vsign=vsign, wsign=wsign, do_wgridding=bool(do_wgridding),
        divide_by_n=bool(divide_by_n), epsilon=float(epsilon), kernel_err=float(err),
        corr_u=_correction(nx, nu, W, beta), corr_v=_correction(ny, nv, W, beta),
        gl_x=gl_x, gl_w=gl_w, est_cost=float(cost), pmirror=int(pmirror),
        nplanes_std=int(npl_std if do_wgridding else 1),
        fast_screen=int(precision == "single" and do_wgridding and epsilon >= FAST_SCREEN_EPS
                        and os.environ.get("PFBG_FAST_SCREEN", "1") != "0"),
    )


def make_batch_plan(wranges, *, nvis_per_snapshot=0, **kw):
    """Plan shared by a batch of snapshots of ONE image geometry (pfb hci, utils/stokes2im.py:635-683).

    `wranges`: per snapshot ``(wmin, wmax)`` of ``|w| f / c`` (see :func:`w_range`).  sigma, W, beta and the plane
    spacing come from :func:`make_plan` for the widest snapshot; every snapshot then gets its own block of planes,
    placed like the planes of a single plan without mirroring: ``ceil((wmax - wmin) / dw) + W`` planes centred on
    its w-range.  Returns ``(plan, snap_w0, snap_np)``; ``plan.nplanes`` is the total."""
    wr = np.asarray(wranges, dtype=np.float64).reshape(-1, 2)
    if wr.shape[0] == 0:
        raise ValueError("a batch needs at least one snapshot")
    span = wr[:, 1] - wr[:, 0]
    k = int(np.argmax(span))
    kw = dict(kw)
    kw["mirror"] = False
    plan = make_plan(wmin=float(wr[k, 0]), wmax=float(wr[k, 1]), nvis=int(nvis_per_snapshot), **kw)
    W, dw = plan.W, plan.dw
    if plan.do_wgridding:
        npl = np.where(span > 0, np.ceil(span / dw).astype(np.int64) + W, W).astype(np.int32)
        w0 = 0.5 * (wr[:, 0] + wr[:, 1]) - 0.5 * (npl - 1) * dw
    else:
        npl = np.ones(wr.shape[0], dtype=np.int32)
        w0 = np.zeros(wr.shape[0])
    plan.nplanes_std = int(npl.sum())
    return plan, np.ascontiguousarray(w0, dtype=np.float64), np.ascontiguousarray(npl, dtype=np.int32)
