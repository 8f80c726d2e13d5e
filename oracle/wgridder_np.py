"""TEST INFRASTRUCTURE ONLY — numpy restatement of the w-stacked gridder.

The algorithm on the hot path lives in the third-party dependency
``ducc0.wgridder`` (``/root/reference/pyproject.toml:42`` ``ducc0>=0.35.0``,
locked 0.41.0 at ``uv.lock:1119-1120``), which is absent from
``/root/reference`` and cannot be installed here.  This module restates its
*published* algorithm (Arras, Reinecke, Westermann & Ensslin 2021, A&A 646 A58:
"improved w-stacking" with an exponential-of-semicircle kernel — the kernel
definition is also in-tree at ``src/pfb_imaging/utils/weighting.py:25-35``) in
plain fp64 numpy, anchored on the reference's own call sites
(``operators/gridder.py:78-100,128-143``, ``operators/hessian.py:50-89``).

It serves two purposes:
  * the **bit-exact binning/index oracle** for CUDA kernel 1 (`bin_indices`):
    every fp64 operation is a single correctly-rounded IEEE op in a fixed
    order, so numpy and the device agree bit for bit;
  * an end-to-end CPU restatement (`vis2dirty_np`, `dirty2vis_np`) that is
    itself pinned against the explicit DFT (``oracle/dft.py``) and the golden
    vectors under ``tests/golden/``.

Parity with ducc0 0.41.0's own outputs is **unpinned** (no ducc0 binary or
stored ducc0 arrays exist); the enforced contract is rel-L2 <= epsilon against
the DFT the reference's tests use as truth.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU baseline may
import this module.
"""

from __future__ import annotations

import numpy as np
from numpy.polynomial.legendre import leggauss

LIGHTSPEED = 299792458.0
TILE = 16


def es_kernel(x, beta):
    arg = (1.0 - x) * (1.0 + x)
    inside = arg >= 0.0
    return np.where(inside, np.exp(beta * (np.sqrt(np.where(inside, arg, 0.0)) - 1.0)), 0.0)


_GX, _GW = leggauss(200)


def kernel_ft(xi, W, beta):
    xi = np.atleast_1d(np.asarray(xi, dtype=np.float64))
    return 0.5 * W * (np.cos(np.pi * W * np.outer(xi, _GX)) @ (es_kernel(_GX, beta) * _GW))


# --------------------------------------------------------------------------
# kernel 1 oracle: bit-exact coordinates, first-cell indices, sort keys
# --------------------------------------------------------------------------
def bin_indices(plan, uvw, freq, mask=None, row_offsets=None, snap_w0=None, snap_np=None):
    """Per-visibility grid coordinates and the sorted bucket order.

    Returns a dict with, for the *active* samples (mask != 0) in row-major
    (row, chan) order: flat index `idx`, `iu0, iv0, ip0` (int32; first touched
    cell per axis, iu0/iv0 may be negative = periodic wrap), `key` (uint64) and
    `order` (stable argsort of key), plus `gu, gv, gw` (fp64 grid coordinates).

    Batched snapshots (`row_offsets`, `snap_w0`, `snap_np`, as given to
    ``pfbg_plan_set_batch`` / ``pfbg_bind_vis_batch``; ``plan.nplanes`` is the
    total): rows [row_offsets[s], row_offsets[s+1]) take their plane from
    snapshot s's own w0, are clamped to its own snap_np[s] planes and are
    shifted by its plane base (the sum of the plane counts before it);
    `snap` holds each sample's snapshot.
    """
    uvw = np.asarray(uvw, dtype=np.float64)
    freq = np.asarray(freq, dtype=np.float64)
    nrow, nchan = uvw.shape[0], freq.size
    W = plan.W
    s = freq / LIGHTSPEED  # (nchan,)
    ut = (plan.usign * uvw[:, 0])[:, None] * s[None, :]
    vt = (plan.vsign * uvw[:, 1])[:, None] * s[None, :]
    wt = (plan.wsign * uvw[:, 2])[:, None] * s[None, :]
    # Hermitian fold: samples with w < 0 are handled at -(u,v,w) with the conjugate visibility
    # (valid because the image is real); the w-planes then only cover |w|.  ducc0 does the same.
    fold = (wt < 0.0) if plan.do_wgridding else np.zeros(wt.shape, dtype=bool)
    ut = np.where(fold, -ut, ut)
    vt = np.where(fold, -vt, vt)
    wt = np.where(fold, -wt, wt)

    def coord(t, pix, n):
        x = t * pix
        f = x - np.floor(x)
        g = f * float(n) + 0.5 * n
        g = np.where(g >= n, g - n, g)
        i0 = np.floor(g - 0.5 * W).astype(np.int64) + 1
        return g, i0

    gu, iu0 = coord(ut, plan.pixsize_x, plan.nu)
    gv, iv0 = coord(vt, plan.pixsize_y, plan.nv)
    if row_offsets is None:
        w0 = plan.w0
        hi = plan.nplanes - W
        pbase = 0
        snap = np.zeros((nrow, 1), dtype=np.int64)
    else:
        ro = np.asarray(row_offsets, dtype=np.int64)
        npl = np.asarray(snap_np, dtype=np.int64)
        snap = np.repeat(np.arange(ro.size - 1), np.diff(ro))[:, None]
        w0 = np.asarray(snap_w0, dtype=np.float64)[snap]
        hi = npl[snap] - W
        pbase = np.concatenate([[0], np.cumsum(npl)[:-1]])[snap]
    if plan.do_wgridding:
        gw = (wt - w0) / plan.dw
        ip0 = np.floor(gw - 0.5 * W).astype(np.int64) + 1
        ip0 = np.clip(ip0, -int(getattr(plan, "pmirror", 0)), hi)
    else:
        gw = np.zeros_like(wt)
        ip0 = np.zeros(wt.shape, dtype=np.int64)
    gw = gw + pbase  # absolute plane units (exact: small integers), as the device adds them
    ip0 = ip0 + pbase

    if mask is None:
        active = np.ones((nrow, nchan), dtype=bool)
    else:
        active = np.asarray(mask) != 0
    idx = np.flatnonzero(active.ravel())
    gu, gv, gw = gu.ravel()[idx], gv.ravel()[idx], gw.ravel()[idx]
    iu0, iv0, ip0 = iu0.ravel()[idx], iv0.ravel()[idx], ip0.ravel()[idx]

    iuw = np.mod(iu0, plan.nu)
    ivw = np.mod(iv0, plan.nv)
    ntv = plan.nv // TILE
    tile = (iuw // TILE) * ntv + (ivw // TILE)
    fine = (iuw % TILE) * TILE + (ivw % TILE)
    pm = int(getattr(plan, "pmirror", 0))
    key = ((tile * (plan.nplanes + pm) + (ip0 + pm)) * (TILE * TILE) + fine).astype(np.uint64)
    order = np.argsort(key, kind="stable")
    return dict(
        idx=idx.astype(np.int64), iu0=iu0.astype(np.int32), iv0=iv0.astype(np.int32),
        ip0=ip0.astype(np.int32), key=key, order=order.astype(np.int64), gu=gu, gv=gv, gw=gw,
        ut=ut.ravel()[idx], vt=vt.ravel()[idx], wt=wt.ravel()[idx], conj=fold.ravel()[idx],
        snap=np.broadcast_to(snap, (nrow, nchan)).ravel()[idx],
    )


def _weights(g, i0, W, beta):
    """ES weights of the W cells i0..i0+W-1 for coordinate g: (n, W)."""
    x = (i0[:, None] + np.arange(W)[None, :]) - g[:, None]
    return es_kernel(2.0 * x / W, beta)


def _mirror(plan, pidx, iu, iv):
    """Planes below zero (mirror planes, plan.pmirror > 0: w_p = (p + 1/2) dw) are the Hermitian mirror of
    plane -p-1: cell (iu, iv) -> ((-iu) mod nu, (-iv) mod nv), value conjugated.  Returns the stored
    (plane, iu, iv) and the mask of conjugated entries."""
    neg = pidx < 0
    return (np.where(neg, -pidx - 1, pidx), np.where(neg, np.mod(-iu, plan.nu), iu), np.where(neg, np.mod(-iv, plan.nv), iv), neg)


def _vis_phase(plan, b):
    """Per-sample phase (in turns) of the centre shift and the n-1 shift."""
    t = b["ut"] * plan.center_x + b["vt"] * plan.center_y
    if plan.do_wgridding:
        t = t + b["wt"] * plan.nshift
    return t - np.rint(t)


_FACTOR_CACHE = {}


def _kernel_ft_many(xi, W, beta):
    """psihat at many points: exact quadrature for small inputs, otherwise a cubic spline through
    4097 exact samples (psihat is entire and even; spline error ~1e-12 relative)."""
    xi = np.asarray(xi, dtype=np.float64)
    if xi.size <= (1 << 18):
        return kernel_ft(xi.ravel(), W, beta).reshape(xi.shape)
    from scipy.interpolate import CubicSpline

    lo, hi = float(xi.min()), float(xi.max())
    pad = 1e-3 * max(hi - lo, 1e-12)
    t = np.linspace(lo - pad, hi + pad, 4097)
    return CubicSpline(t, kernel_ft(t, W, beta))(xi)


def _image_factors(plan):
    """Plan-level constants (cached per plan object: they are set-up work, not part of an apply)."""
    hit = _FACTOR_CACHE.get(id(plan))
    if hit is not None and hit[0] is plan:
        return hit[1]
    res = _image_factors_uncached(plan)
    _FACTOR_CACHE.clear()
    _FACTOR_CACHE[id(plan)] = (plan, res)
    return res


def _image_factors_uncached(plan):
    nx, ny, W = plan.nx, plan.ny, plan.W
    ipx = np.arange(nx) - nx // 2
    ipy = np.arange(ny) - ny // 2
    l = plan.center_x + ipx * plan.pixsize_x
    m = plan.center_y + ipy * plan.pixsize_y
    r2 = l[:, None] ** 2 + m[None, :] ** 2
    nm1 = -r2 / (np.sqrt(1.0 - r2) + 1.0)
    cu = 1.0 / kernel_ft(ipx / float(plan.nu), W, plan.beta)
    cv = 1.0 / kernel_ft(ipy / float(plan.nv), W, plan.beta)
    corr = cu[:, None] * cv[None, :]
    if plan.do_wgridding:
        nu_ = nm1 + plan.nshift
        cw = 1.0 / _kernel_ft_many(nu_ * plan.dw, W, plan.beta)
        corr = corr * cw
    else:
        nu_ = np.zeros_like(nm1)
    if plan.divide_by_n:
        corr = corr / (nm1 + 1.0)
    sgn = 1.0 - 2.0 * ((ipx[:, None] + ipy[None, :]) & 1)  # (-1)^(i'+j'): grid origin at cell (nu/2, nv/2)
    return corr * sgn, nu_, ipx, ipy


def vis2dirty_np(plan, uvw, freq, vis, wgt=None, mask=None, chunk=20000):
    """Adjoint (gridding) direction, fp64, all planes resident."""
    b = bin_indices(plan, uvw, freq, mask)
    W, P, nu, nv = plan.W, plan.nplanes, plan.nu, plan.nv
    a = np.asarray(vis).astype(np.complex128).ravel()[b["idx"]]
    a = np.where(b["conj"], np.conj(a), a)
    if wgt is not None:
        a = a * np.asarray(wgt, dtype=np.float64).ravel()[b["idx"]]
    a = a * np.exp(2j * np.pi * _vis_phase(plan, b))
    grid = np.zeros((P, nu, nv), dtype=np.complex128)
    n = a.size
    ar = np.arange(W)
    for s0 in range(0, n, chunk):
        sl = slice(s0, s0 + chunk)
        iu0, iv0, ip0 = (b[k][sl].astype(np.int64) for k in ("iu0", "iv0", "ip0"))
        ku = _weights(b["gu"][sl], iu0, W, plan.beta)
        kv = _weights(b["gv"][sl], iv0, W, plan.beta)
        if plan.do_wgridding:
            kw = _weights(b["gw"][sl], ip0, W, plan.beta)
            npl = W
        else:
            kw = np.ones((iu0.size, 1))
            npl = 1
        iu = np.mod(iu0[:, None] + ar, nu)
        iv = np.mod(iv0[:, None] + ar, nv)
        for q in range(npl):
            val = (a[sl] * kw[:, q])[:, None, None] * ku[:, :, None] * kv[:, None, :]
            pidx, iub, ivb, neg = _mirror(plan, np.broadcast_to((ip0 + q)[:, None, None], val.shape),
                                          np.broadcast_to(iu[:, :, None], val.shape),
                                          np.broadcast_to(iv[:, None, :], val.shape))
            np.add.at(grid, (pidx, iub, ivb), np.where(neg, np.conj(val), val))
    corr, nu_, ipx, ipy = _image_factors(plan)
    ix = np.mod(ipx, nu)
    iy = np.mod(ipy, nv)
    img = np.zeros((plan.nx, plan.ny))
    for p in range(P):
        f = np.fft.ifft2(grid[p]) * (nu * nv)  # unnormalised, sign +
        f = f[np.ix_(ix, iy)]
        if plan.do_wgridding:
            wp = plan.w0 + p * plan.dw
            f = f * np.exp(-2j * np.pi * wp * nu_)
        img += f.real
    return img * corr


def dirty2vis_np(plan, uvw, freq, dirty, mask=None, chunk=20000):
    """Forward (degridding) direction, fp64."""
    b = bin_indices(plan, uvw, freq, mask)
    W, P, nu, nv = plan.W, plan.nplanes, plan.nu, plan.nv
    corr, nu_, ipx, ipy = _image_factors(plan)
    ix = np.mod(ipx, nu)
    iy = np.mod(ipy, nv)
    x = np.asarray(dirty, dtype=np.float64) * corr
    grid = np.empty((P, nu, nv), dtype=np.complex128)
    for p in range(P):
        pl = np.zeros((nu, nv), dtype=np.complex128)
        if plan.do_wgridding:
            wp = plan.w0 + p * plan.dw
            pl[np.ix_(ix, iy)] = x * np.exp(2j * np.pi * wp * nu_)
        else:
            pl[np.ix_(ix, iy)] = x
        grid[p] = np.fft.fft2(pl)
    n = b["idx"].size
    out = np.zeros(n, dtype=np.complex128)
    ar = np.arange(W)
    for s0 in range(0, n, chunk):
        sl = slice(s0, s0 + chunk)
        iu0, iv0, ip0 = (b[k][sl].astype(np.int64) for k in ("iu0", "iv0", "ip0"))
        ku = _weights(b["gu"][sl], iu0, W, plan.beta)
        kv = _weights(b["gv"][sl], iv0, W, plan.beta)
        if plan.do_wgridding:
            kw = _weights(b["gw"][sl], ip0, W, plan.beta)
            npl = W
        else:
            kw = np.ones((iu0.size, 1))
            npl = 1
        iu = np.mod(iu0[:, None] + ar, nu)
        iv = np.mod(iv0[:, None] + ar, nv)
        acc = np.zeros(iu0.size, dtype=np.complex128)
        for q in range(npl):
            shp = (iu0.size, W, W)
            pidx, iub, ivb, neg = _mirror(plan, np.broadcast_to((ip0 + q)[:, None, None], shp),
                                          np.broadcast_to(iu[:, :, None], shp), np.broadcast_to(iv[:, None, :], shp))
            g = grid[pidx, iub, ivb]
            g = np.where(neg, np.conj(g), g)
            acc += kw[:, q] * np.einsum("nij,ni,nj->n", g, ku, kv)
        out[sl] = acc
    out *= np.exp(-2j * np.pi * _vis_phase(plan, b))
    out = np.where(b["conj"], np.conj(out), out)
    nrow, nchan = np.asarray(uvw).shape[0], np.asarray(freq).size
    vis = np.zeros(nrow * nchan, dtype=np.complex128)
    vis[b["idx"]] = out
    return vis.reshape(nrow, nchan)
