"""PSF-convolution Hessians on the device (SURVEY §8 f1): the operator pfb-imaging iterates inside
pcg, the power method and the primal-dual loop.  Drop-ins for (/root/reference/src/pfb_imaging):

  psf_convolve_slice / _cube / _fscube   operators/psf.py:8-96
  hessian_psf_slice    operators/hessian.py:103-143
  hess_direct / hess_direct_slice        operators/hessian.py:178-248
  HessPSF.dot / idot(mode="psf" | "direct")   operators/hessian.py:251-436
  HessianTree          operators/hessian.py:439-522   (sum over a band's partitions)
  HessTreeRay          operators/hessian.py:525-615   (cube-level facade over a band pool)

numpy in, numpy out; the transforms run in ``libpfbgrid.so`` (``csrc/psfconv.cuh``: row pass, one
transform-multiply-transform column kernel that never leaves shared memory, row pass back).  The
``xpad`` / ``xhat`` scratch arguments of the reference signatures are accepted and ignored.
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .wgridder import content_hash, current_device

_RDT = {np.dtype(np.float32): (_lib.PFBG_F32, np.complex64), np.dtype(np.float64): (_lib.PFBG_F64, np.complex128)}


class PsfConvolver:
    """out = beam * crop(IFFT(FFT(pad(beam * x)) * khat)) + eta * x for one band.  After :meth:`set_gauss` the
    multiplier is the transfer function of a pixel-sampled Gaussian (or a ratio of two), evaluated on the device."""

    def __init__(self, nx, ny, nx_psf, ny_psf, dtype=np.float64, device=None):
        self.rdt = np.dtype(dtype)
        if self.rdt not in _RDT:
            raise TypeError("dtype must be float32 or float64")
        self.prec, self.cdt = _RDT[self.rdt]
        self.nx, self.ny, self.nx_psf, self.ny_psf = int(nx), int(ny), int(nx_psf), int(ny_psf)
        self.device = current_device() if device is None else int(device)
        self._lib = _lib.load()
        self._h = C.c_void_p()
        _lib.check(self._lib.pfbg_conv_create(self.prec, self.device, self.nx, self.ny, self.nx_psf, self.ny_psf,
                                              C.byref(self._h)))

    def set_kernel(self, khat):
        """khat: (nx_psf, ny_psf//2+1) r2c half spectrum (real ``abspsf`` or complex ``psfhat``) or the
        full (nx_psf, ny_psf) spectrum."""
        khat = np.asarray(khat)
        if khat.shape == (self.nx_psf, self.ny_psf // 2 + 1):
            half = 1
        elif khat.shape == (self.nx_psf, self.ny_psf):
            half = 0
        else:
            raise ValueError(f"kernel shape {khat.shape} matches neither the half nor the full spectrum")
        k = np.ascontiguousarray(khat, dtype=self.cdt)
        _lib.check(self._lib.pfbg_conv_set_kernel(self._h, C.c_void_p(k.ctypes.data), half, _lib.HOST_PTRS, None))
        return self

    def set_gauss(self, beam_to, beam_from=None, norm_kernel=False):
        """Switch to the analytic kernel of ``restore.py``: convolution with the pixel-sampled Gaussian `beam_to`, or,
        with `beam_from`, the conversion of an image at resolution `beam_from` to `beam_to`.  Beams are
        ``(emaj, emin, pa)`` in pixels (FWHMs, ``emaj >= emin >= 1``); `norm_kernel`: unit-sum instead of peak-1
        kernels.  ValueError for a sub-pixel beam or a `beam_to` that does not contain `beam_from`.  The stored
        spectrum of :meth:`set_kernel`, if any, is released."""
        def arr(b):
            b = np.asarray(b, dtype=np.float64).reshape(-1)
            if b.size != 3:
                raise ValueError("a beam is (emaj, emin, pa)")
            return (C.c_double * 3)(*b)

        rc = self._lib.pfbg_conv_set_gauss(self._h, arr(beam_to), None if beam_from is None else arr(beam_from),
                                           int(bool(norm_kernel)))
        if rc == _lib.PFBG_ERR_ARG:
            raise ValueError(self._lib.pfbg_last_error().decode())
        _lib.check(rc)
        return self

    def apply(self, x, beam=None, eta=None, out=None, add=None):
        """`add`: ``crop(IFFT(FFT(pad(x)) * K)) + add``, the sum taken on the device (no `beam`, no `eta`)."""
        x = np.ascontiguousarray(x, dtype=self.rdt)
        if x.shape != (self.nx, self.ny):
            raise ValueError(f"x shape {x.shape} != ({self.nx}, {self.ny})")
        if beam is not None:
            beam = np.ascontiguousarray(beam, dtype=self.rdt)
            if beam.shape != x.shape:
                raise ValueError("beam shape does not match the image")
        if add is not None:
            if beam is not None or eta:
                raise ValueError("add= takes neither beam nor eta")
            add = np.ascontiguousarray(add, dtype=self.rdt)
            if add.shape != x.shape:
                raise ValueError("add shape does not match the image")
        res = np.empty_like(x) if out is None else out
        tmp = res if (res.flags.c_contiguous and res.dtype == self.rdt) else np.empty_like(x)
        if add is not None:
            _lib.check(self._lib.pfbg_conv_apply_add(self._h, C.c_void_p(x.ctypes.data), C.c_void_p(add.ctypes.data),
                                                     C.c_void_p(tmp.ctypes.data), _lib.HOST_PTRS, None))
        else:
            _lib.check(self._lib.pfbg_conv_apply(self._h, C.c_void_p(x.ctypes.data),
                                                 None if beam is None else C.c_void_p(beam.ctypes.data),
                                                 float(eta) if eta else 0.0, C.c_void_p(tmp.ctypes.data),
                                                 _lib.HOST_PTRS, None))
        if tmp is not res:
            res[...] = tmp
        return res

    def apply_dev(self, x_ptr, out_ptr, beam_ptr=None, eta=None, stream=None, add_ptr=None):
        """Same operator on device pointers (asynchronous on `stream`): what the device-resident deconvolution loops call.
        `add_ptr`: ``out = crop(IFFT(FFT(pad(x)) * K)) + add`` (no beam, no eta)."""
        if add_ptr is not None:
            if beam_ptr is not None or eta:
                raise ValueError("add_ptr takes neither beam_ptr nor eta")
            _lib.check(self._lib.pfbg_conv_apply_add(self._h, C.c_void_p(int(x_ptr)), C.c_void_p(int(add_ptr)),
                                                     C.c_void_p(int(out_ptr)), _lib.DEVICE_PTRS, stream))
            return
        _lib.check(self._lib.pfbg_conv_apply(self._h, C.c_void_p(int(x_ptr)), None if beam_ptr is None else C.c_void_p(int(beam_ptr)),
                                             float(eta) if eta else 0.0, C.c_void_p(int(out_ptr)), _lib.DEVICE_PTRS, stream))

    def apply_shifted(self, x, taper=None, c=0.0, inverse=True):
        """``taper * crop(IFFT(FFT(pad(taper * x)) * (Re khat + c)^(+-1)))`` (fp64, stored spectrum): the direct
        inverse of :func:`hess_direct_slice` from this convolver's own spectrum (`inverse`: the reciprocal)."""
        x = np.ascontiguousarray(x, dtype=self.rdt)
        if x.shape != (self.nx, self.ny):
            raise ValueError(f"x shape {x.shape} != ({self.nx}, {self.ny})")
        if taper is not None:
            taper = np.ascontiguousarray(taper, dtype=self.rdt)
            if taper.shape != x.shape:
                raise ValueError("taper shape does not match the image")
        res = np.empty_like(x)
        _lib.check(self._lib.pfbg_conv_apply_shifted(self._h, C.c_void_p(x.ctypes.data),
                                                     None if taper is None else C.c_void_p(taper.ctypes.data), float(c),
                                                     int(bool(inverse)), C.c_void_p(res.ctypes.data), _lib.HOST_PTRS, None))
        return res

    def apply_shifted_dev(self, x_ptr, out_ptr, taper_ptr=None, c=0.0, inverse=True, stream=None):
        """:meth:`apply_shifted` on device pointers (asynchronous on `stream`)."""
        _lib.check(self._lib.pfbg_conv_apply_shifted(self._h, C.c_void_p(int(x_ptr)),
                                                     None if taper_ptr is None else C.c_void_p(int(taper_ptr)), float(c),
                                                     int(bool(inverse)), C.c_void_p(int(out_ptr)), _lib.DEVICE_PTRS, stream))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.pfbg_conv_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_CONV_CACHE: dict = {}


def _convolver_for(khat, nx, ny, lastsize, rdt):
    khat = np.asarray(khat)
    nx_psf = khat.shape[0]
    ny_psf = int(lastsize) if lastsize is not None else 2 * (khat.shape[1] - 1)
    key = (khat.ctypes.data, khat.shape, khat.dtype.str, nx, ny, ny_psf, np.dtype(rdt).str)
    chk = content_hash(khat)  # the whole spectrum: an in-place edit of any element rebuilds the convolver
    hit = _CONV_CACHE.get(key)
    if hit is not None and hit[1] == chk:
        return hit[0]
    if hit is not None:
        hit[0].close()
    while len(_CONV_CACHE) >= 16:
        _CONV_CACHE.pop(next(iter(_CONV_CACHE)))[0].close()
    cv = PsfConvolver(nx, ny, nx_psf, ny_psf, dtype=rdt).set_kernel(khat)
    _CONV_CACHE[key] = (cv, chk, khat)
    return cv


def clear_convolver_cache():
    while _CONV_CACHE:
        _CONV_CACHE.popitem()[1][0].close()


def psf_convolve_slice(xpad, xhat, xout, psfhat, lastsize, x, nthreads=1):
    """operators/psf.py:8-31."""
    x = np.asarray(x)
    cv = _convolver_for(psfhat, x.shape[0], x.shape[1], lastsize, x.dtype)
    xout[...] = cv.apply(x)
    return xout


def hessian_psf_slice(x, xpad=None, xhat=None, xout=None, abspsf=None, beam=None, lastsize=None, nthreads=1, eta=None):
    """Tikhonov regularised PSF-convolution Hessian (operators/hessian.py:103-143)."""
    x = np.asarray(x)
    cv = _convolver_for(abspsf, x.shape[0], x.shape[1], lastsize, x.dtype)
    res = cv.apply(x, beam=beam, eta=eta)
    if xout is None:
        return res
    np.copyto(xout, res)
    return xout


def psf_convolve_cube(xpad, xhat, xout, psfhat, lastsize, x, nthreads=1):
    """operators/psf.py:36-67: band-wise convolution of an (nband, nx, ny) cube with (nband, nx_psf, nyo2) kernels."""
    x = np.asarray(x)
    for b in range(x.shape[0]):
        cv = _convolver_for(psfhat[b], x.shape[1], x.shape[2], lastsize, x.dtype)
        xout[b] = cv.apply(x[b])
    return xout


def psf_convolve_fscube(xpad, xhat, xout, psfhat, lastsize, x, nthreads=1):
    """operators/psf.py:70-96: the same over (nband, ncorr, nx, ny)."""
    x = np.asarray(x)
    for b in range(x.shape[0]):
        for c in range(x.shape[1]):
            cv = _convolver_for(psfhat[b, c], x.shape[2], x.shape[3], lastsize, x.dtype)
            xout[b, c] = cv.apply(x[b, c])
    return xout


def taperf(shape, taper_width):
    """Cosine edge taper (utils/misc.py:968-975)."""
    tapers1d = ()
    for npix in shape:
        taper = np.ones(npix)
        taper[:taper_width] = 0.5 * (1 + np.cos(np.linspace(1.1 * np.pi, 2 * np.pi, taper_width)))
        taper[-taper_width:] = 0.5 * (1 + np.cos(np.linspace(0, 0.9 * np.pi, taper_width)))
        tapers1d += (taper,)
    return np.outer(*tapers1d)


_DIRECT_CACHE: dict = {}


def hess_direct_slice(x, xpad=None, xhat=None, xout=None, abspsf=None, taperxy=None, lastsize=None, nthreads=1, eta=1,
                      mode="forward"):
    """``taper * IFFT((abspsf + eta)^{+-1} FFT(pad(taper * x)))`` (hessian.py:213-248): the same device convolver with
    the kernel ``abspsf + eta`` (forward) or its reciprocal (backward); the taper rides in the beam slot."""
    x = np.asarray(x)
    abspsf = np.asarray(abspsf)
    key = (abspsf.ctypes.data, abspsf.shape, float(eta), mode, x.shape, np.dtype(x.dtype).str, int(lastsize))
    chk = content_hash(abspsf)
    hit = _DIRECT_CACHE.get(key)
    if hit is None or hit[1] != chk:
        if hit is not None:
            hit[0].close()
        while len(_DIRECT_CACHE) >= 8:
            _DIRECT_CACHE.pop(next(iter(_DIRECT_CACHE)))[0].close()
        k = abspsf.astype(np.float64) + float(eta)
        if mode != "forward":
            k = 1.0 / k
        cv = PsfConvolver(x.shape[0], x.shape[1], abspsf.shape[0], int(lastsize), dtype=x.dtype).set_kernel(k)
        hit = _DIRECT_CACHE[key] = (cv, chk, abspsf)
    res = hit[0].apply(x, beam=None if taperxy is None else np.ascontiguousarray(taperxy, dtype=x.dtype))
    if xout is None:
        return res
    np.copyto(xout, res)
    return xout


def hess_direct(x, xpad=None, xhat=None, xout=None, abspsf=None, taperxy=None, lastsize=None, nthreads=1, eta=1,
                mode="forward"):
    """Cube form (hessian.py:178-210): one `eta`, one taper, per-band kernels."""
    x = np.asarray(x)
    out = np.empty_like(x) if xout is None else xout
    for b in range(x.shape[0]):
        out[b] = hess_direct_slice(x[b], abspsf=abspsf[b], taperxy=taperxy, lastsize=lastsize, eta=eta, mode=mode)
    return out


class HessianTree:
    """Sum-over-partitions PSF-convolution Hessian of one band (operators/hessian.py:439-522):

        H x = (1 / sum_p wsum_p) sum_p B_p (PSF_p conv (B_p x)) + eta x

    `partitions`: dicts with ``psfhat`` (corr, nx_psf, nyo2), ``beam`` (corr, nx, ny), ``wsum`` (corr,).  Partitions
    that share a beam (bit for bit) are merged by linearity — their kernels are summed once at construction — so
    the common case of one beam per band costs one device convolution per correlation whatever the number of
    partitions; distinct beams keep one convolver each.

    numpy in, numpy out as in the reference.  A float64 CUDA tensor on the tree's :attr:`device`, ``(ncorr, nx, ny)``
    or ``(nx, ny)`` when ``ncorr == 1``, stays there: ``dot`` returns a new ``(ncorr, nx, ny)`` tensor computed on
    torch's current stream (``pfbg_conv_apply_scaled`` per group, the groups of a correlation summed through a second
    buffer).  The beams are uploaded on the first device call."""

    def __init__(self, partitions, nx, ny, nx_psf, ny_psf, eta=0.0, nthreads=1, wsum=None, device=None):
        if not partitions:
            raise ValueError("HessianTree requires at least one partition")
        self.parts = partitions
        self.nx, self.ny, self.nx_psf, self.ny_psf = nx, ny, nx_psf, ny_psf
        self.eta, self.nthreads = eta, nthreads
        self.ncorr = np.asarray(partitions[0]["wsum"]).size
        if wsum is None:
            self.wsum = np.zeros(self.ncorr)
            for p in partitions:
                self.wsum += p["wsum"]
        else:
            self.wsum = np.broadcast_to(np.asarray(wsum, dtype=float), (self.ncorr,)).copy()
        groups: dict = {}
        for p in partitions:
            beam = np.asarray(p["beam"], dtype=np.float64)
            psfhat = np.asarray(p["psfhat"])
            for c in range(self.ncorr):
                key = (c, content_hash(beam[c]))
                g = groups.get(key)
                if g is None:
                    groups[key] = [c, None if (beam[c] == 1).all() else np.ascontiguousarray(beam[c]),
                                   np.array(psfhat[c], dtype=np.complex128)]
                else:
                    g[2] += psfhat[c]
        self._groups = []
        for c, beam, khat in groups.values():
            cv = PsfConvolver(nx, ny, nx_psf, ny_psf, dtype=np.float64, device=device).set_kernel(khat)
            self._groups.append((c, beam, cv))
        self.device = self._groups[0][2].device
        self._dev_beams = None  # device copies of the group beams, uploaded on the first device call

    def _beams_dev(self):
        import torch

        if self._dev_beams is None:
            dev = torch.device("cuda", self.device)
            self._dev_beams = [None if bm is None else torch.from_numpy(bm).to(dev) for _, bm, _ in self._groups]
        return self._dev_beams

    def corr_groups(self, c):
        """(convolver, device beam or None) of every group of correlation c."""
        return [(cv, bm) for (gc, _, cv), bm in zip(self._groups, self._beams_dev()) if gc == c]

    def _dot_dev(self, x, out=None):
        import torch

        if x.dtype != torch.float64:
            raise TypeError(f"device input must be float64, got {x.dtype}")
        if x.device.index != self.device:
            raise ValueError(f"input is on {x.device}, the operator on cuda:{self.device}")
        xt = x if x.dim() == 3 else x[None]
        ncorr, nx, ny = xt.shape
        assert ncorr == self.ncorr, f"expected {self.ncorr} correlations on axis 0, got {ncorr}"
        assert nx == self.nx and ny == self.ny
        xt = xt.contiguous()
        out = torch.empty_like(xt) if out is None else out
        s = torch.cuda.current_stream(xt.device).cuda_stream
        pong = None
        for c in range(ncorr):
            gs = self.corr_groups(c)
            if len(gs) > 1 and pong is None:
                pong = torch.empty_like(xt[0])
            prev = None
            for i, (cv, bm) in enumerate(gs):
                # the last group writes out[c]; the ridge term comes in with the first, the running sum with the others
                dst = out[c] if (len(gs) - 1 - i) % 2 == 0 else pong
                xin, eta = (xt[c], float(self.eta)) if i == 0 else (prev, 1.0)
                _lib.check(cv._lib.pfbg_conv_apply_scaled(
                    cv._h, C.c_void_p(xt[c].data_ptr()), None if bm is None else C.c_void_p(bm.data_ptr()),
                    C.c_void_p(xin.data_ptr()), eta, 1.0 / float(self.wsum[c]), C.c_void_p(dst.data_ptr()),
                    _lib.DEVICE_PTRS, s))
                prev = dst
        return out

    def dot(self, x):
        if getattr(x, "is_cuda", False):
            return self._dot_dev(x)
        x = np.asarray(x)
        xtmp = x if x.ndim == 3 else x[None, :, :]
        ncorr, nx, ny = xtmp.shape
        assert ncorr == self.ncorr, f"expected {self.ncorr} correlations on axis 0, got {ncorr}"
        assert nx == self.nx and ny == self.ny
        out = np.zeros_like(xtmp, dtype=np.float64)
        for c, beam, cv in self._groups:
            out[c] += cv.apply(np.ascontiguousarray(xtmp[c], dtype=np.float64), beam=beam)
        out /= self.wsum[:, None, None]
        out += self.eta * xtmp
        return out

    hdot = dot  # Hermitian

    def close(self):
        for _, _, cv in self._groups:
            cv.close()
        self._groups = []
        self._dev_beams = None


CG_STOP = {1: "converged", 2: "maxit", 3: "stalled", 4: "initial residual zero", 5: "exact"}  # pfbsara.h PFBS_CG_*


def tree_cg(trees, rhs_t, x0_t, tol, maxit, minit, stream=None):
    """Batched CG over the corr-0 systems of `trees` (HessianTrees on one device, sharing (nx, ny)): solves
    ``trees[s].dot(v)[0] = rhs_t[s]`` for every s with one ``pfbs_tree_cg``, the stopping rules of ``solvers.pcg``.

    `rhs_t`: ``(len(trees), nx, ny)`` float64 CUDA tensor on the trees' device; `x0_t`: None (start from zero) or a
    tensor like it, read and not modified.  Runs on `stream` (a ``torch.cuda.Stream``; default: torch's current stream
    of the device).  Returns the solution and a dict of per-system ``iters``, ``eps`` and ``stop`` (``CG_STOP``
    strings).  A tree with more than one correlation fails the assertion the host solve fails."""
    import torch

    n = len(trees)
    if n == 0:
        raise ValueError("tree_cg needs at least one tree")
    t0 = trees[0]
    for t in trees:
        assert t.ncorr == 1, f"expected {t.ncorr} correlations on axis 0, got 1"
        if t.device != t0.device or (t.nx, t.ny) != (t0.nx, t0.ny):
            raise ValueError("the trees of one batched solve must share the device and (nx, ny)")
    shape = (n, t0.nx, t0.ny)
    for name, v in (("rhs", rhs_t), ("x0", x0_t)):
        if v is None:
            continue
        if v.dtype != torch.float64:
            raise TypeError(f"{name} must be float64, got {v.dtype}")
        if tuple(v.shape) != shape:
            raise ValueError(f"{name} shape {tuple(v.shape)} does not match {shape}")
        if not v.is_cuda or v.device.index != t0.device:
            raise ValueError(f"{name} is on {v.device}, the trees on cuda:{t0.device}")
    dev = torch.device("cuda", t0.device)
    stream = torch.cuda.current_stream(dev) if stream is None else stream
    with torch.cuda.stream(stream):
        rhs = rhs_t.contiguous()
        sol = torch.zeros(shape, dtype=torch.float64, device=dev) if x0_t is None else x0_t.clone(
            memory_format=torch.contiguous_format)
        group_start, convs, beams = [0], [], []
        for t in trees:
            gs = t.corr_groups(0)
            convs += [cv._h.value for cv, _ in gs]
            beams += [None if bm is None else bm.data_ptr() for _, bm in gs]
            group_start.append(len(convs))
        lib, ng, npix = _lib.load(), len(convs), t0.nx * t0.ny
        gs_arr = (C.c_int32 * (n + 1))(*group_start)
        nbytes = int(lib.pfbs_tree_cg_work_bytes(n, gs_arr, npix))
        work = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        iters, eps, stop = (C.c_int32 * n)(), (C.c_double * n)(), (C.c_int32 * n)()
        _lib.check(lib.pfbs_tree_cg(t0.device, n, gs_arr, (C.c_void_p * ng)(*convs), (C.c_void_p * ng)(*beams),
                                    (C.c_double * n)(*[1.0 / float(t.wsum[0]) for t in trees]),
                                    (C.c_double * n)(*[float(t.eta) for t in trees]), C.c_void_p(rhs.data_ptr()),
                                    C.c_void_p(sol.data_ptr()), npix, float(tol), int(maxit), int(minit),
                                    C.c_void_p(work.data_ptr()), nbytes, iters, eps, stop, stream.cuda_stream))
    info = dict(iters=np.array(iters[:], dtype=np.int64), eps=np.array(eps[:]), stop=[CG_STOP.get(v, str(v)) for v in stop])
    return sol, info


class HessTreeRay:
    """Cube-level Hessian over per-band :class:`HessianTree` operators held by a band pool
    (operators/hessian.py:525-615); `workers` is a :class:`pfb_imaging_b200.operators.BandWorkerPool`.  ``dot`` and
    ``cg`` take numpy cubes or ``(nband, nx, ny)`` float64 CUDA tensors, which stay on the device."""

    def __init__(self, partitions_per_band, nx, ny, nx_psf, ny_psf, etas=0.0, nthreads=1, wsums=None, cg_tol=1e-3,
                 cg_maxit=150, cg_minit=1, cg_verbose=0, workers=None):
        from .operators import BandWorkerPool

        if partitions_per_band is None:
            if workers is None:
                raise ValueError("partitions_per_band=None requires a workers pool with loaded bands")
            self.nband = workers.nband
        else:
            self.nband = len(partitions_per_band)
        self.nx, self.ny = nx, ny
        self.cg_tol, self.cg_maxit, self.cg_minit, self.cg_verbose = cg_tol, cg_maxit, cg_minit, cg_verbose
        etas = np.broadcast_to(np.asarray(etas, dtype=float), (self.nband,))
        wsums = [None] * self.nband if wsums is None else np.broadcast_to(np.asarray(wsums, dtype=float), (self.nband,))
        if workers is None:
            workers = BandWorkerPool(self.nband, nthreads)
        elif workers.nband != self.nband:
            raise ValueError(f"workers pool has {workers.nband} bands, expected {self.nband}")
        self._pool = workers
        self._pool.init_hess(partitions_per_band, nx, ny, nx_psf, ny_psf, etas, wsums)

    def dot(self, x):
        return self._pool.hess_dot(x)

    hdot = dot

    def cg(self, rhs, x0=None, tol=None, maxit=None, minit=None):
        """Per-band CG solve of ``hess @ update = rhs`` inside the pool."""
        tol = self.cg_tol if tol is None else tol
        maxit = self.cg_maxit if maxit is None else maxit
        minit = self.cg_minit if minit is None else minit
        return self._pool.hess_cg(rhs, x0, tol, maxit, minit, self.cg_verbose)

    def get_mem(self):
        return self._pool.get_mem()

    @property
    def last_cg_info(self):
        """Per-band ``iters`` / ``eps`` / ``stop`` of the last device :meth:`cg` (``BandWorkerPool.last_cg_info``)."""
        return self._pool.last_cg_info


class HessPSF:
    """Cube-level PSF-convolution Hessian with the reference's constructor and ``dot`` / ``idot(mode="psf")``
    (operators/hessian.py:251-436); one device convolver per band.

    numpy in, numpy out as in the reference.  A float64 CUDA tensor on the convolvers' device, ``(nband, nx, ny)`` or
    ``(nx, ny)`` when ``nband == 1``, stays on the device: ``dot`` and ``idot`` then return a new ``(nband, nx, ny)``
    tensor computed on torch's current stream, ``idot(mode="psf")`` solves every band in one batched CG
    (``pfbs_psf_cg``) and leaves the per-band ``iters`` / ``eps`` / ``stop`` in :attr:`last_idot_info`."""

    def __init__(self, nx, ny, abspsf, beam=None, eta=1.0, nthreads=1, cgtol=1e-3, cgmaxit=300, cgverbose=2, cgrf=25,
                 taper_width=32, min_beam=5e-3):
        self.nx, self.ny = nx, ny
        self.abspsf = abspsf
        self.nband, self.nx_psf, self.nyo2 = abspsf.shape
        self.ny_psf = 2 * (self.nyo2 - 1)
        if beam is not None and not (np.asarray(beam) == 1).all():
            if beam.shape != (self.nband, nx, ny):
                raise AssertionError("beam must have shape (nband, nx, ny)")
            self.beam = beam
        else:
            self.beam = (None,) * self.nband
        self.eta = np.tile(eta, self.nband) if isinstance(eta, float) else np.array(eta)
        if self.eta.size != self.nband:
            raise AssertionError("eta must be a float or have one entry per band")
        self.cgtol, self.cgmaxit, self.cgverbose, self.cgrf = cgtol, cgmaxit, cgverbose, cgrf
        self.taperxy = taperf((nx, ny), taper_width)  # direct mode (hessian.py:304)
        self.min_beam = min_beam
        self.conv = [PsfConvolver(nx, ny, self.nx_psf, self.ny_psf, dtype=np.float64).set_kernel(abspsf[b])
                     for b in range(self.nband)]
        self._dev_consts = None  # device copies of the beams and the taper, uploaded on the first device call
        self.last_idot_info = None

    def set_beam(self, beam):
        assert beam.shape == (self.nband, self.nx, self.ny)
        self.beam = beam
        self._dev_consts = None

    def _cube(self, x):
        if x.ndim == 3:
            return x
        if x.ndim == 2:
            return x[None]
        raise ValueError("Unsupported number of input dimensions")

    def _dev_input(self, x):
        """The (nband, nx, ny) contiguous view of a device input; raises before anything is launched."""
        import torch

        if x.dtype != torch.float64:
            raise TypeError(f"device input must be float64, got {x.dtype}")
        if x.dim() == 2 and self.nband == 1:
            x = x[None]
        if tuple(x.shape) != (self.nband, self.nx, self.ny):
            raise ValueError(f"input shape {tuple(x.shape)} does not match ({self.nband}, {self.nx}, {self.ny})")
        if x.device.index != self.conv[0].device:
            raise ValueError(f"input is on {x.device}, the operator on cuda:{self.conv[0].device}")
        return x.contiguous()

    def _consts(self, device):
        import torch

        if self._dev_consts is None:
            up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(device)  # noqa: E731
            self._dev_consts = dict(beam=[None if b is None else up(b) for b in self.beam], taper=up(self.taperxy))
        return self._dev_consts

    def _direct_dev(self, xt, out, consts, stream):
        """Device :meth:`_direct` of every band: the same shifted spectrum from each band's own convolver."""
        c0 = np.sqrt(self.nx * self.ny)
        for b in range(self.nband):
            self.conv[b].apply_shifted_dev(xt[b].data_ptr(), out[b].data_ptr(), consts["taper"].data_ptr(),
                                           c=float(self.eta[b]) * c0, inverse=True, stream=stream)

    def _dot_dev(self, x, out=None):
        import torch

        xt = self._dev_input(x)
        consts = self._consts(xt.device)
        s = torch.cuda.current_stream(xt.device).cuda_stream
        out = torch.empty_like(xt)
        for b in range(self.nband):
            bm = consts["beam"][b]
            self.conv[b].apply_dev(xt[b].data_ptr(), out[b].data_ptr(), None if bm is None else bm.data_ptr(),
                                   float(self.eta[b]), s)
        return out

    def _idot_dev(self, x, mode, x0, init_x0):
        import torch

        xt = self._dev_input(x)
        if mode not in ("direct", "psf"):
            raise ValueError(f"Unknown mode {mode}")
        consts = self._consts(xt.device)
        s = torch.cuda.current_stream(xt.device).cuda_stream
        if mode == "direct":
            out = torch.empty_like(xt)
            self._direct_dev(xt, out, consts, s)
            for b, bm in enumerate(consts["beam"]):
                if bm is not None:
                    mask = (out[b] > 0) & (bm > self.min_beam)
                    out[b] = torch.where(mask, out[b] / (bm * bm), out[b])
            return out
        # the starting point of the host path: the direct estimate, or zero (a passed x0 is not used, as there)
        if x0 is None and init_x0:
            sol = torch.empty_like(xt)
            self._direct_dev(xt, sol, consts, s)
        else:
            sol = torch.zeros_like(xt)
        lib, nb, npix = self.conv[0]._lib, self.nband, self.nx * self.ny
        nbytes = int(lib.pfbs_psf_cg_work_bytes(nb, npix))
        work = torch.empty(nbytes, dtype=torch.uint8, device=xt.device)
        iters, eps, stop = (C.c_int32 * nb)(), (C.c_double * nb)(), (C.c_int32 * nb)()
        _lib.check(lib.pfbs_psf_cg(self.conv[0].device, nb, (C.c_void_p * nb)(*[c._h.value for c in self.conv]),
                                   (C.c_void_p * nb)(*[None if bm is None else bm.data_ptr() for bm in consts["beam"]]),
                                   (C.c_double * nb)(*[float(e) for e in self.eta]), C.c_void_p(xt.data_ptr()),
                                   C.c_void_p(sol.data_ptr()), npix, float(self.cgtol), int(self.cgmaxit), 3,
                                   C.c_void_p(work.data_ptr()), nbytes, iters, eps, stop, s))
        self.last_idot_info = dict(iters=np.array(iters[:], dtype=np.int64), eps=np.array(eps[:]),
                                   stop=[CG_STOP.get(v, str(v)) for v in stop])
        return sol

    def dot(self, x):
        if getattr(x, "is_cuda", False):
            return self._dot_dev(x)
        xt = self._cube(x)
        if xt.shape != (self.nband, self.nx, self.ny):
            raise AssertionError("input shape does not match the operator")
        out = np.empty((self.nband, self.nx, self.ny))
        for b in range(self.nband):
            self.conv[b].apply(xt[b], beam=self.beam[b], eta=float(self.eta[b]), out=out[b])
        return out

    hdot = dot

    def _direct(self, b, x, mode="backward"):
        """hess_direct_slice of band b (hessian.py:213-248) with eta scaled as idot does (:381)."""
        nx, ny = self.nx, self.ny
        return hess_direct_slice(x, abspsf=self.abspsf[b], taperxy=self.taperxy, lastsize=self.ny_psf,
                                 eta=float(self.eta[b]) * np.sqrt(nx * ny), mode=mode)

    def idot(self, x, mode="psf", x0=None, init_x0=True):
        """Inverse of `dot` per band (hessian.py:357-436): ``mode="direct"`` divides by ``abspsf + eta sqrt(nx ny)``
        between the tapers, ``mode="psf"`` runs CG on the PSF-convolution Hessian.  As in the reference, the CG
        starts from the direct estimate when ``x0 is None and init_x0`` and from zero otherwise (a passed `x0` is
        not used there either, hessian.py:372-390)."""
        from .solvers import pcg

        if getattr(x, "is_cuda", False):
            return self._idot_dev(x, mode, x0, init_x0)
        xt = self._cube(x)
        if xt.shape != (self.nband, self.nx, self.ny):
            raise AssertionError("input shape does not match the operator")
        if x0 is None and init_x0:
            x0 = np.zeros_like(xt, dtype=np.float64)
            for b in range(self.nband):
                x0[b] = self._direct(b, xt[b])
        else:
            x0 = np.zeros_like(xt, dtype=np.float64)
        out = np.empty((self.nband, self.nx, self.ny))
        if mode == "direct":
            for b in range(self.nband):
                out[b] = self._direct(b, xt[b])
                if self.beam[b] is not None:
                    mask = (out[b] > 0) & (self.beam[b] > self.min_beam)
                    out[b, mask] /= self.beam[b][mask] ** 2
        elif mode == "psf":
            for b in range(self.nband):
                hess = lambda v, b=b: self.conv[b].apply(v, beam=self.beam[b], eta=float(self.eta[b]))
                out[b] = pcg(hess, np.ascontiguousarray(xt[b], dtype=np.float64), x0=np.array(x0[b], dtype=np.float64),
                             tol=self.cgtol, maxit=self.cgmaxit, minit=3,
                             verbosity=min(self.cgverbose, 1) if self.cgverbose < 2 else 0,
                             report_freq=self.cgrf, backtrack=False, return_resid=False)
        else:
            raise ValueError(f"Unknown mode {mode}")
        return out

    def close(self):
        for c in self.conv:
            c.close()
        self._dev_consts = None


class PsfGradient:
    """Gradient of the smooth term of the deconvolution sub-problem, ``grad(x) = hess(x) - dirty`` with the
    PSF-convolution Hessian (the `grad` callables built in ``core/sara.py:300-340`` / ``deconv`` presets), usable both as
    the reference's numpy callable and, through ``device_apply``, inside the device-resident loops of
    ``pfb_imaging_b200.sara`` (no host round trip per iteration).  `hess` is a :class:`HessPSF` or, for ``pfb deconv``,
    a :class:`HessTreeRay` (its bands may sit on other devices: the pool copies them there and back)."""

    def __init__(self, hess, dirty):
        self.hess = hess
        self.dirty = np.ascontiguousarray(dirty, dtype=np.float64)
        if self.dirty.shape != (hess.nband, hess.nx, hess.ny):
            raise ValueError("dirty must have shape (nband, nx, ny)")
        self._dev = None

    def __call__(self, x):
        return self.hess.dot(x) - self.dirty

    def device_apply(self, x_t, out_t):
        import torch

        tree = not isinstance(self.hess, HessPSF)
        if self._dev is None:
            dev = x_t.device
            self._dev = dict(dirty=torch.from_numpy(self.dirty).to(dev),
                             beam=[] if tree else [None if b is None else
                                                   torch.from_numpy(np.ascontiguousarray(b, dtype=np.float64)).to(dev)
                                                   for b in self.hess.beam])
        if tree:
            torch.sub(self.hess.dot(x_t), self._dev["dirty"], out=out_t)
            return
        s = torch.cuda.current_stream(x_t.device).cuda_stream
        for b in range(self.hess.nband):
            bm = self._dev["beam"][b]
            self.hess.conv[b].apply_dev(x_t[b].data_ptr(), out_t[b].data_ptr(), None if bm is None else bm.data_ptr(),
                                        float(self.hess.eta[b]), s)
        out_t -= self._dev["dirty"]
