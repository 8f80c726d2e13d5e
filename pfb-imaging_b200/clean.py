"""Clark CLEAN minor cycle on the device: the backward step of ``pfb kclean`` (reference ``core/kclean.py:203-218``
calls ``deconv/clark.py``).  fp64, numpy in, numpy out; kernels in ``csrc/clean.cuh``.

Semantics (Clark 1980 with an MFS search over bands), images ``(nband, nx, ny)``, raster index ``p = i*ny + j``:

* ``s(p) = |R_0(p) + ... + R_{nband-1}(p)|`` (band order) over the pixels the mask keeps;
* major loop: ``Rmax = max s``; on the first pass ``tol = max(pf Rmax, threshold)``; stop when ``Rmax <= tol`` or
  after ``maxit`` major iterations; active set ``A = {p : s(p) >= subpf Rmax}``;
* subminor loop on ``A`` while the peak ``s(a*) > max(subpf Rmax, threshold)``, at most ``submaxit`` components:
  ``a*`` the first maximum in raster order, ``d_b = gamma R_b(a*) / peak_b`` (a band whose PSF peak is <= 0 gets no
  model), ``model_b(a*) += d_b``, ``R_b(a) -= d_b PSF_b(c + a - a*)`` on ``A``;
* ``R = ID - PSF (*) model`` through ``psfhat`` (the PSF convolver of :mod:`pfb_imaging_b200.psf`).

Parity with the reference's numba ``clark`` is not pinned (no golden of it exists); see INTEGRATION.md §2b.
"""

from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _lib
from .wgridder import HandleCache, content_hash, current_device

MAX_BANDS = 1024  # PFBS_CLARK_MAX_BANDS


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


class Clark:
    """The PSF of one deconvolution, uploaded once (with one PSF convolver per band) and reused by every call.

    `psf`: ``(nband, nx_psf, ny_psf)`` with its centre at ``(nx_psf//2, ny_psf//2)``; `psfhat`: its r2c spectrum
    ``rfft2(ifftshift(psf))`` as ``image_data_products_arrays`` returns it (computed here when None)."""

    def __init__(self, psf, psfhat=None, nx=None, ny=None, device=None):
        psf = np.asarray(psf)
        if psf.dtype != np.float64:
            raise TypeError(f"psf must be float64, got {psf.dtype}")
        if psf.ndim != 3:
            raise ValueError(f"psf must be (nband, nx_psf, ny_psf), got shape {psf.shape}")
        self.nband, self.nx_psf, self.ny_psf = psf.shape
        if not 1 <= self.nband <= MAX_BANDS:
            raise ValueError(f"nband {self.nband} not in 1..{MAX_BANDS}")
        if nx is None or ny is None:
            raise ValueError("nx and ny are required")
        self.nx, self.ny = int(nx), int(ny)
        if not (0 < self.nx <= self.nx_psf and 0 < self.ny <= self.ny_psf):
            raise ValueError(f"image ({nx}, {ny}) must be non-empty and no larger than the PSF {psf.shape[1:]}")
        if self.nx * self.ny >= 2**31:
            raise ValueError("nx * ny must be below 2^31")
        if psfhat is None:
            psfhat = np.fft.rfft2(np.fft.ifftshift(psf, axes=(1, 2)), axes=(1, 2))
        psfhat = np.asarray(psfhat)
        if psfhat.dtype != np.complex128:
            raise TypeError(f"psfhat must be complex128, got {psfhat.dtype}")
        if psfhat.shape != (self.nband, self.nx_psf, self.ny_psf // 2 + 1):
            raise ValueError(f"psfhat shape {psfhat.shape} != {(self.nband, self.nx_psf, self.ny_psf // 2 + 1)}")
        self.device = current_device() if device is None else int(device)
        self._lib = _lib.load()
        self._h = C.c_void_p()
        psf_c = np.ascontiguousarray(psf)
        hat_c = np.ascontiguousarray(psfhat)
        _lib.check(self._lib.pfbs_clark_create(_lib.PFBG_F64, self.device, self.nband, self.nx, self.ny, self.nx_psf,
                                               self.ny_psf, _ptr(psf_c), _ptr(hat_c), _lib.HOST_PTRS, None,
                                               C.byref(self._h)))

    def __call__(self, dirty, mask=None, threshold=0.0, gamma=0.05, pf=0.05, maxit=50, subpf=0.5, submaxit=1000,
                 timings=False):
        """Returns ``(model, residual, info)``; `info` holds ``niter`` and, per major iteration, ``rmax``,
        ``nactive`` (|A|), ``nsub`` (components) and ``peaks`` (their raster indices in order).  With `timings`,
        ``info["times_ms"]`` is ``(niter, 3)``: search + compaction, subminor, residual step (CUDA events)."""
        dirty = np.asarray(dirty)
        if dirty.dtype != np.float64:
            raise TypeError(f"dirty must be float64, got {dirty.dtype}")
        if dirty.shape != (self.nband, self.nx, self.ny):
            raise ValueError(f"dirty shape {dirty.shape} != {(self.nband, self.nx, self.ny)}")
        if mask is not None:
            mask = np.asarray(mask)
            if mask.shape != (self.nx, self.ny):
                raise ValueError(f"mask shape {mask.shape} != {(self.nx, self.ny)}")
            if mask.dtype != np.bool_ and not np.issubdtype(mask.dtype, np.number):
                raise TypeError(f"mask must be boolean or numeric, got {mask.dtype}")
            mask = np.ascontiguousarray(mask != 0, dtype=np.uint8)
        for name, v in (("threshold", threshold), ("gamma", gamma), ("pf", pf), ("subpf", subpf)):
            if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, float, np.integer, np.floating)):
                raise TypeError(f"{name} must be a real number")
            if not math.isfinite(v):
                raise ValueError(f"{name} must be finite")
        for name, v in (("maxit", maxit), ("submaxit", submaxit)):
            if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, np.integer)):
                raise TypeError(f"{name} must be an integer")
        if threshold < 0:
            raise ValueError("threshold must be >= 0")
        if not 0 < gamma <= 1:
            raise ValueError("gamma must be in (0, 1]")
        if pf < 0:
            raise ValueError("pf must be >= 0")
        if not 0 < subpf < 1:
            raise ValueError("subpf must be in (0, 1)")
        if not 0 <= maxit < 2**31 or not 1 <= submaxit < 2**31:
            raise ValueError("need 0 <= maxit and 1 <= submaxit (32-bit)")
        if not self._h.value:
            raise RuntimeError("this Clark handle has been closed")
        dirty = np.ascontiguousarray(dirty)
        model = np.empty_like(dirty)
        residual = np.empty_like(dirty)
        m = max(int(maxit), 1)
        niter = C.c_int32(0)
        rmax = np.zeros(m)
        nactive = np.zeros(m, dtype=np.int64)
        nsub = np.zeros(m, dtype=np.int32)
        peaks = np.empty(int(maxit) * int(submaxit), dtype=np.int64)  # untouched pages are never committed
        times = np.zeros((m, 3), dtype=np.float32) if timings else None
        _lib.check(self._lib.pfbs_clark_run(
            self._h, _ptr(dirty), None if mask is None else _ptr(mask), _ptr(model), _ptr(residual), float(threshold),
            float(gamma), float(pf), int(maxit), float(subpf), int(submaxit), C.byref(niter), _ptr(rmax),
            _ptr(nactive), _ptr(nsub), _ptr(peaks), peaks.size, None if times is None else _ptr(times),
            _lib.HOST_PTRS, None))
        k = niter.value
        offs = np.concatenate([[0], np.cumsum(nsub[:k])]).astype(np.int64)
        info = dict(niter=k, rmax=rmax[:k].tolist(), nactive=nactive[:k].tolist(), nsub=nsub[:k].tolist(),
                    peaks=[peaks[offs[i]:offs[i + 1]].copy() for i in range(k)])
        if timings:
            info["times_ms"] = times[:k].copy()
        return model, residual, info

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.pfbs_clark_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_CLARK_CACHE = HandleCache(2)  # a handle holds the PSF, its spectra and the work arrays: gigabytes at scale


def _clark_for(psf, psfhat, nx, ny):
    """A cached :class:`Clark`, keyed like ``psf._convolver_for``: the PSF and spectrum buffers, their shapes, the image
    size and a hash of the full content of both (a PSF or spectrum rewritten in place rebuilds the handle)."""
    psf = np.asarray(psf)
    key = (psf.ctypes.data, psf.shape, psf.dtype.str, int(nx), int(ny),
           None if psfhat is None else (np.asarray(psfhat).ctypes.data, np.asarray(psfhat).shape))
    chk = (content_hash(psf), None if psfhat is None else content_hash(psfhat))
    return _CLARK_CACHE.get(key, chk, lambda: Clark(psf, psfhat, nx=nx, ny=ny), keep=(psf, psfhat))


def clear_clark_cache():
    _CLARK_CACHE.clear()


def clark(ID, PSF, PSFHAT=None, mask=None, threshold=0.0, gamma=0.05, pf=0.05, maxit=50, subpf=0.5, submaxit=1000):
    """Clark minor cycle of `ID` (nband, nx, ny) with `PSF` (nband, nx_psf, ny_psf) and its spectrum `PSFHAT`;
    returns ``(model, residual, info)``.  The device copy of the PSF is cached across calls (kclean runs one call
    per major cycle with the same PSF)."""
    ID = np.asarray(ID)
    if ID.ndim != 3:
        raise ValueError(f"ID must be (nband, nx, ny), got shape {ID.shape}")
    cl = _clark_for(PSF, PSFHAT, ID.shape[1], ID.shape[2])
    return cl(ID, mask=mask, threshold=threshold, gamma=gamma, pf=pf, maxit=maxit, subpf=subpf, submaxit=submaxit)
