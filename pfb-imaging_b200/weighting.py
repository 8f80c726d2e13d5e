"""Imaging weights on the B200: drop-ins for the numba functions of
``/root/reference/src/pfb_imaging/utils/weighting.py`` —
``_compute_counts`` (:81-140), ``counts_to_weights`` (:143-208),
``filter_extreme_counts`` (:212-226), ``box_sum_counts`` (:229-254), and the l2 re-weighting block of
``image_data_products`` (``operators/gridder.py:509-532`` -> ``l2_reweight``) — with the
same positional signatures and in-place behaviour (``counts_to_weights`` mutates
both ``weight`` and ``counts``), plus ``counts_to_weights_batch``, the same pair for each snapshot of a
``pfb hci`` batch in one call.  The histogram / gather run in
``libpfbgrid.so`` (``csrc/weighting.cuh``); the median filter and the box sum are
small image-sized host operations and stay in numpy/scipy.
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .wgridder import current_device


def _prec(dt):
    dt = np.dtype(dt)
    if dt == np.float32:
        return _lib.PFBG_F32
    if dt == np.float64:
        return _lib.PFBG_F64
    raise TypeError(f"weights must be float32 or float64, got {dt}")


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _geom(uvw, freq, mask, nrow, nchan):
    uvw = np.ascontiguousarray(uvw, dtype=np.float64)
    freq = np.ascontiguousarray(freq, dtype=np.float64)
    if uvw.shape != (nrow, 3) or freq.shape != (nchan,):
        raise ValueError("uvw/freq shapes do not match the weights")
    if mask is not None:
        mask = np.asarray(mask)
        if mask.shape != (nrow, nchan):
            raise ValueError("mask shape does not match the weights")
        mask = np.ascontiguousarray(mask if mask.dtype == np.uint8 else mask != 0, dtype=np.uint8)
    return uvw, freq, mask


def _compute_counts(uvw, freq, mask, wgt, nx, ny, cell_size_x, cell_size_y, dtype, ngrid=1, usign=1.0, vsign=-1.0):
    """(ncorr, nx, ny) sum of weights per uv cell.  `ngrid` is accepted and ignored."""
    wgt = np.asarray(wgt)
    if wgt.ndim != 3:
        raise ValueError("wgt must have shape (ncorr, nrow, nchan)")
    ncorr, nrow, nchan = wgt.shape
    dt = np.dtype(dtype)
    w = np.ascontiguousarray(wgt, dtype=dt)
    uvw, freq, mask = _geom(uvw, freq, mask, nrow, nchan)
    counts = np.empty((ncorr, int(nx), int(ny)), dtype=dt)
    lib = _lib.load()
    _lib.check(lib.pfbg_counts(_prec(dt), current_device(), _p(uvw), _p(freq), _p(mask), _p(w), nrow, nchan, ncorr,
                               int(nx), int(ny), float(cell_size_x), float(cell_size_y), float(usign), float(vsign),
                               _p(counts), _lib.HOST_PTRS, None))
    return counts


def counts_cells(uvw, freq, mask, nx, ny, cell_size_x, cell_size_y, usign=1.0, vsign=-1.0):
    """Bit-exact check hook: (nrow, nchan, 2) int32 cell index per sample (-1 = skipped)."""
    uvw = np.ascontiguousarray(uvw, dtype=np.float64)
    freq = np.ascontiguousarray(freq, dtype=np.float64)
    nrow, nchan = uvw.shape[0], freq.size
    uvw, freq, mask = _geom(uvw, freq, mask, nrow, nchan)
    cells = np.empty((nrow, nchan, 2), dtype=np.int32)
    lib = _lib.load()
    _lib.check(lib.pfbg_counts_cells(current_device(), _p(uvw), _p(freq), _p(mask), nrow, nchan, int(nx), int(ny),
                                     float(cell_size_x), float(cell_size_y), float(usign), float(vsign), _p(cells)))
    return cells


def counts_to_weights(counts, uvw, freq, weight, mask, nx, ny, cell_size_x, cell_size_y, robust, usign=1.0, vsign=-1.0):
    """Briggs/uniform re-weighting, in place on `weight` and `counts` (weighting.py:173-174,206)."""
    if not isinstance(weight, np.ndarray) or weight.ndim != 3:
        raise ValueError("weight must be an ndarray of shape (ncorr, nrow, nchan)")
    ncorr, nrow, nchan = weight.shape
    dt = weight.dtype
    if counts.dtype != dt or counts.shape != (ncorr, int(nx), int(ny)):
        raise ValueError("counts must be (ncorr, nx, ny) of the weights' dtype")
    uvw, freq, mask = _geom(uvw, freq, mask, nrow, nchan)
    w = weight if weight.flags.c_contiguous else np.ascontiguousarray(weight)
    c = counts if counts.flags.c_contiguous else np.ascontiguousarray(counts)
    lib = _lib.load()
    _lib.check(lib.pfbg_counts_to_weights(_prec(dt), current_device(), _p(c), _p(uvw), _p(freq), _p(w), _p(mask),
                                          nrow, nchan, ncorr, int(nx), int(ny), float(cell_size_x),
                                          float(cell_size_y), float(robust), float(usign), float(vsign),
                                          _lib.HOST_PTRS, None))
    if w is not weight:
        weight[...] = w
    if c is not counts:
        counts[...] = c
    return weight


def counts_to_weights_batch(uvw, freq, weight, mask, row_offsets, nx_pad, ny_pad, cellx, celly, robust, usign=1.0,
                            vsign=-1.0, counts=None):
    """Briggs/uniform weights of a batch of snapshots sharing `freq`, in place on `weight` (nrow, nchan) and returned.

    Rows ``[row_offsets[s], row_offsets[s+1])`` of `uvw`, `weight` and `mask` are snapshot s.  Each snapshot ends
    with the weights this pair of calls gives it on its own (the per-snapshot weighting of utils/stokes2im.py:563-604):

        c = _compute_counts(uvw_s, freq, mask_s, weight_s[None], nx_pad, ny_pad, cellx, celly, weight.dtype, 1, usign, vsign)
        counts_to_weights(c, uvw_s, freq, weight_s[None], mask_s, nx_pad, ny_pad, cellx, celly, robust, usign, vsign)

    One counts grid per snapshot, all on the device in one launch sequence.  `counts`, when given, is an
    (nsnap, nx_pad, ny_pad) array of the weights' dtype that receives the grids as ``counts_to_weights`` leaves them.
    ``filter_extreme_counts`` / ``box_sum_counts`` are not applied; callers that need them keep the per-snapshot calls."""
    if not isinstance(weight, np.ndarray) or weight.ndim != 2:
        raise ValueError("weight must be an ndarray of shape (nrow, nchan)")
    nrow, nchan = weight.shape
    dt = weight.dtype
    prec = _prec(dt)
    uvw, freq, mask = _geom(uvw, freq, mask, nrow, nchan)
    ro = np.ascontiguousarray(row_offsets, dtype=np.int64)
    if ro.ndim != 1 or ro.size < 2 or ro[-1] != nrow:
        raise ValueError(f"row_offsets must be 1-D, one entry more than the snapshots, and end at nrow = {nrow}")
    nsnap = ro.size - 1
    if counts is not None and (not isinstance(counts, np.ndarray) or counts.dtype != dt
                               or counts.shape != (nsnap, int(nx_pad), int(ny_pad))):
        raise ValueError(f"counts must be an ({nsnap}, {int(nx_pad)}, {int(ny_pad)}) array of the weights' dtype")
    w = weight if weight.flags.c_contiguous else np.ascontiguousarray(weight)
    c = None if counts is None else (counts if counts.flags.c_contiguous else np.empty(counts.shape, dt))
    lib = _lib.load()
    _lib.check(lib.pfbg_counts_to_weights_batch(prec, current_device(), nsnap, _p(ro), _p(uvw), _p(freq), _p(mask),
                                                _p(w), nrow, nchan, int(nx_pad), int(ny_pad), float(cellx),
                                                float(celly), float(robust), float(usign), float(vsign), _p(c),
                                                _lib.HOST_PTRS, None))
    if w is not weight:
        weight[...] = w
    if c is not None and c is not counts:
        counts[...] = c
    return weight


def l2_reweight(residual_vis, weight, mask, l2_reweight_dof, wgtp=None):
    """Student-t re-weighting from residual visibilities: the ``if l2_reweight_dof:`` block of
    ``image_data_products`` (operators/gridder.py:509-532).  ``weight`` (ncorr,nrow,nchan) is scaled in
    place by ``(dof + 2) / (dof + |r|^2 wgtp / ovar)`` and returned; ``None`` comes back when the residual
    variance is exactly zero (:531-532), the weights are then left untouched.

    The reference's ``if ovar:`` only has a truth value for ncorr == 1; for more correlations this
    routine continues when every per-correlation variance is non-zero."""
    if not isinstance(weight, np.ndarray) or weight.ndim != 3:
        raise ValueError("weight must be an ndarray of shape (ncorr, nrow, nchan)")
    ncorr, nrow, nchan = weight.shape
    dt = weight.dtype
    prec = _prec(dt)
    cdt = np.complex64 if dt == np.float32 else np.complex128
    rv = np.asarray(residual_vis)
    if rv.shape != weight.shape or rv.dtype != cdt:
        raise ValueError(f"residual_vis must be {np.dtype(cdt)} of shape {weight.shape}")
    rv = np.ascontiguousarray(rv)
    if wgtp is not None and not np.isscalar(wgtp):
        wgtp = np.ascontiguousarray(np.broadcast_to(np.asarray(wgtp, dtype=dt), weight.shape))
    elif wgtp is not None:
        wgtp = None if float(wgtp) == 1.0 else np.full(weight.shape, wgtp, dtype=dt)
    if mask is not None:
        mask = np.asarray(mask)
        if mask.shape != (nrow, nchan):
            raise ValueError("mask shape does not match the weights")
        mask = np.ascontiguousarray(mask if mask.dtype == np.uint8 else mask != 0, dtype=np.uint8)
    w = weight if weight.flags.c_contiguous else np.ascontiguousarray(weight)
    ovar = np.zeros(ncorr, dtype=np.float64)
    applied = C.c_int32(0)
    lib = _lib.load()
    _lib.check(lib.pfbg_l2_reweight(prec, current_device(), _p(rv), _p(wgtp), _p(mask), _p(w), nrow * nchan, ncorr,
                                    float(l2_reweight_dof), _p(ovar), C.cast(C.byref(applied), C.c_void_p),
                                    _lib.HOST_PTRS, None))
    if not applied.value:
        return None
    if w is not weight:
        weight[...] = w
    return weight


def filter_extreme_counts(counts, level=10.0):
    if not level:
        return counts
    ic, ix, iy = np.where(counts > 0)
    cnts = counts[ic, ix, iy]
    counts[ic, ix, iy] = np.maximum(cnts, np.median(cnts) / level)
    return counts


def box_sum_counts(counts, npix_super):
    if npix_super is None or npix_super <= 0:
        return counts
    if not np.issubdtype(counts.dtype, np.floating):
        raise AssertionError(f"box_sum_counts requires a floating-point counts array; got dtype={counts.dtype}")
    from scipy.ndimage import uniform_filter

    size = 2 * npix_super + 1
    out = np.empty_like(counts)
    for c in range(counts.shape[0]):
        out[c] = uniform_filter(counts[c], size=size, mode="constant", cval=0.0) * (size * size)
    return out


def weight_data_corr(data, weight, jones, tbin_idx, tbin_counts, ant1, ant2):
    """Visibilities and weights of one correlation behind diagonal Jones terms: the body of
    ``pfb_imaging.utils.correlations._weight_data_impl`` (``/root/reference/src/pfb_imaging/utils/correlations.py:
    195-232``, what `pfb init` hands to the gridder for single-correlation products), same arguments and outputs:

        data (nrow, nchan, ncorr) complex, weight (nrow, nchan, ncorr) real, jones (ntime, nant, nchan, ndir, ncorr_j)
        complex [direction 0, correlation 0 are used], tbin_idx / tbin_counts (ntime) first row and length of every
        time bin (any common offset), ant1 / ant2 (nrow)  ->  vis (nrow, nchan) complex, wgt (nrow, nchan) real

        wgt = Re(w0 gp gq conj(gp) conj(gq)),   vis = w0 gq v0 conj(gp)

    Runs on the device (``pfbg_weight_data_corr``), bit-identical to the numba loop.  Unlike the reference this does
    not modify `tbin_idx` in place.  The per-Stokes ``utils.weighting.weight_data`` (:274-468) takes its expressions
    from ``radiomesh.generated._stokes_expr``, which is not available here, and is not provided."""
    data = np.asarray(data)
    if data.ndim != 3 or data.dtype not in (np.complex64, np.complex128):
        raise TypeError("data must be a complex64 / complex128 array of shape (nrow, nchan, ncorr)")
    rdt = np.float32 if data.dtype == np.complex64 else np.float64
    nrow, nchan, ncorr = data.shape
    weight = np.asarray(weight)
    if weight.shape != data.shape:
        raise ValueError("weight shape does not match data")
    jones = np.asarray(jones)
    if jones.ndim != 5:
        raise NotImplementedError("only diagonal Jones terms (ntime, nant, nchan, ndir, ncorr) are supported")
    d = np.ascontiguousarray(data)
    w = np.ascontiguousarray(weight, dtype=rdt)
    j = np.ascontiguousarray(jones, dtype=data.dtype)
    tbin_idx = np.asarray(tbin_idx, dtype=np.int64)
    tbin_counts = np.asarray(tbin_counts, dtype=np.int64)
    start = tbin_idx - (tbin_idx.min() if tbin_idx.size else 0)
    row_t = np.full(nrow, -1, dtype=np.int32)
    for t in range(start.size):  # later bins win where bins overlap, like the sequential loop of the reference
        row_t[start[t]:start[t] + tbin_counts[t]] = t
    a1 = np.ascontiguousarray(ant1, dtype=np.int32)
    a2 = np.ascontiguousarray(ant2, dtype=np.int32)
    if a1.shape != (nrow,) or a2.shape != (nrow,):
        raise ValueError("ant1 / ant2 must have one entry per row")
    nt, nant, nch_j, ndir, ncj = j.shape
    if nch_j != nchan:
        raise ValueError("jones and data disagree on the number of channels")
    if nrow and (max(a1.max(), a2.max()) >= nant or row_t.max() >= nt):
        raise ValueError("antenna or time index outside the Jones array")
    vis = np.empty((nrow, nchan), dtype=data.dtype)
    wgt = np.empty((nrow, nchan), dtype=rdt)
    lib = _lib.load()
    es = j.itemsize
    _lib.check(lib.pfbg_weight_data_corr(_prec(rdt), current_device(), _p(d), _p(w), _p(j), _p(row_t), _p(a1), _p(a2), nrow,
                                         nchan, ncorr, j.size, j.strides[0] // es, j.strides[1] // es, j.strides[2] // es,
                                         _p(vis), _p(wgt), _lib.HOST_PTRS, None))
    return vis, wgt
