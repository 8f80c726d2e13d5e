"""Clean-beam fitting and restoration (``pfb restore``: the reference's ``core/restore.py``,
``utils/restoration.py`` and ``fitcleanbeam`` of ``utils/misc.py``).

Conventions (the contract is ``oracle/restore_np.py``; INTEGRATION.md "pfb restore"):

* A beam is ``(emaj, emin, pa)``.  `emaj` and `emin` are FWHMs in units of `pixsize`, ``emaj >= emin``; `pa` is in
  radians in ``(-pi/2, pi/2]``, the angle of the major axis in the (axis 0, axis 1) pixel plane, so the major axis
  points along ``(cos pa, sin pa)``; ``pa = 0`` when ``emaj == emin`` to 1e-12 relative.
* The kernel is the pixel-sampled Gaussian ``g(x, y) = exp(-4 ln 2 (x'^2 / emaj^2 + y'^2 / emin^2))``, ``(x, y)`` the
  pixel offsets from the kernel centre and ``(x', y')`` those offsets rotated by `pa`.  ``norm_kernel=False``: peak 1;
  ``norm_kernel=True``: unit sum.  The kernel is the sampled Gaussian, not a band-limited one: a point source at a
  pixel centre restores to exactly the samples of ``g``.
* Convolutions are circular on a padded grid of ``plan.good_size(int((1 + pfrac) * n))`` per axis, the image at the
  start of each padded axis, the output cropped back to ``(nx, ny)``.

The convolutions run on the device in the PSF convolver (``csrc/psfconv.cuh``), whose column pass evaluates the
transfer function of the Gaussian, or the ratio of two for a change of resolution, where it is used: no spectrum is
built or stored.  :func:`fitcleanbeam` stays on the host: the main lobe is at most a few thousand pixels and the PSF
arrives as numpy.
"""

from __future__ import annotations

import numpy as np

from . import plan as _plan
from .psf import PsfConvolver
from .wgridder import current_device

_FOURLN2 = 4.0 * np.log(2.0)


# --- the clean beam ----------------------------------------------------------------------------------------------------
def _main_lobe(p, level):
    """Pixels of the 4-connected island of ``p > level`` that contains the centre ``(nx//2, ny//2)``, found in a
    window around the centre that doubles until the island no longer touches its edge.  Returns the offsets from the
    centre and the values."""
    nx, ny = p.shape
    cx, cy = nx // 2, ny // 2
    if not p[cx, cy] > level:
        raise ValueError(f"the PSF centre ({cx}, {cy}) is not above level {level}")
    h = 8
    while True:
        x0, x1, y0, y1 = max(cx - h, 0), min(cx + h + 1, nx), max(cy - h, 0), min(cy + h + 1, ny)
        m = p[x0:x1, y0:y1] > level
        isl = np.zeros_like(m)
        isl[cx - x0, cy - y0] = True
        while True:  # grow the seed by 4-neighbour steps inside the mask
            g = isl.copy()
            g[1:] |= isl[:-1]
            g[:-1] |= isl[1:]
            g[:, 1:] |= isl[:, :-1]
            g[:, :-1] |= isl[:, 1:]
            g &= m
            if (g == isl).all():
                break
            isl = g
        touches = ((x0 > 0 and isl[0].any()) or (x1 < nx and isl[-1].any())
                   or (y0 > 0 and isl[:, 0].any()) or (y1 < ny and isl[:, -1].any()))
        if not touches:
            break
        h *= 2
    ix, iy = np.nonzero(isl)
    return (ix + x0 - cx).astype(np.float64), (iy + y0 - cy).astype(np.float64), p[ix + x0, iy + y0]


def _form_to_beam(a, b, c):
    """``exp(-(a x^2 + 2 b x y + c y^2))`` -> (emaj, emin, pa) in pixels."""
    m, d = 0.5 * (a + c), np.hypot(0.5 * (a - c), b)
    lo, hi = m - d, m + d  # 4 ln 2 / emaj^2, 4 ln 2 / emin^2
    if not (np.isfinite(lo) and lo > 0):
        raise ValueError(f"the fitted quadratic form ({a}, {b}, {c}) is not positive definite")
    emaj, emin = np.sqrt(_FOURLN2 / lo), np.sqrt(_FOURLN2 / hi)
    if emaj - emin <= 1e-12 * emaj:
        return emaj, emin, 0.0
    pa = 0.5 * np.arctan2(2.0 * b, a - c) + 0.5 * np.pi  # the larger eigenvalue's axis, turned to the major axis
    if pa > 0.5 * np.pi:
        pa -= np.pi
    return emaj, emin, pa


def _fit_form(x, y, v):
    """Unweighted least squares of ``exp(-(a x^2 + 2 b x y + c y^2))`` to the island values by Levenberg-Marquardt on
    (a, b, c), from the second moments of the island."""
    w = v / v.sum()
    sxx, sxy, syy = (w * x * x).sum(), (w * x * y).sum(), (w * y * y).sum()
    det = sxx * syy - sxy * sxy
    if x.size < 3 or not det > 0:
        raise ValueError(f"the main lobe ({x.size} pixels) does not determine a 2-D Gaussian; lower `level`")
    th = np.array([0.5 * syy / det, -0.5 * sxy / det, 0.5 * sxx / det])  # Q = Sigma^-1 / 2
    basis = np.stack([x * x, 2.0 * x * y, y * y], axis=1)

    def resid(t):
        return np.exp(-(basis @ t)) - v

    r = resid(th)
    cost, lam = r @ r, 1e-3
    for _ in range(200):
        mod = r + v
        J = -basis * mod[:, None]
        A, g = J.T @ J, J.T @ r
        while True:
            step = np.linalg.solve(A + lam * np.diag(np.diag(A)), -g)
            tn = th + step
            rn = resid(tn)
            cn = rn @ rn
            if cn <= cost:
                th, r, lam = tn, rn, lam * 0.1
                break
            lam *= 10.0
            if lam > 1e12:
                return th
        conv = np.abs(step).max() <= 1e-15 * np.abs(th).max() or cost - cn <= 1e-30 * max(cost, 1e-300)
        cost = cn
        if conv:
            break
    return th


def fitcleanbeam(psf, level=0.5, pixsize=1.0):
    """Gaussian fitted to the main lobe of each band of `psf` (``(nband, nx, ny)`` or ``(nx, ny)``): the band is
    divided by its maximum, the 4-connected island above `level` that holds the centre ``(nx//2, ny//2)`` is fitted
    by unweighted least squares with a centred, peak-1 Gaussian.  Returns ``(nband, 3)`` beams ``(emaj, emin, pa)``
    with the FWHMs in units of `pixsize`.  ValueError when a band's maximum is not positive, its centre is not above
    `level`, or the fit is not a positive definite form.  Signature of the ``fit_psf`` hook of
    ``operators.image_data_products`` and ``operators.grid_partition``."""
    psf = np.asarray(psf, dtype=np.float64)
    if psf.ndim == 2:
        psf = psf[None]
    out = np.empty((psf.shape[0], 3))
    for b in range(psf.shape[0]):
        pmax = psf[b].max()
        if not pmax > 0:
            raise ValueError(f"band {b}: PSF maximum {pmax} is not positive")
        x, y, v = _main_lobe(psf[b] / pmax, level)
        emaj, emin, pa = _form_to_beam(*_fit_form(x, y, v))
        out[b] = emaj * pixsize, emin * pixsize, pa
    return out


# --- convolution with Gaussians on the device --------------------------------------------------------------------------
def _beams(beam, nband, pixsize, name):
    b = np.asarray(beam, dtype=np.float64)
    b = np.broadcast_to(b, (nband, 3)) if b.ndim == 1 else b
    if b.shape != (nband, 3):
        raise ValueError(f"{name} must be one (emaj, emin, pa) or one per band, got shape {np.shape(beam)}")
    b = b.copy()
    b[:, :2] /= pixsize
    return b


class _Cube:
    """numpy (fp32 / fp64) or CUDA-tensor cube, with one convolver for all its bands."""

    def __init__(self, image, pfrac, name="image"):
        self.torch = type(image).__module__.startswith("torch")
        if self.torch:
            import torch

            if not image.is_cuda or image.dtype not in (torch.float32, torch.float64):
                raise TypeError(f"{name}: a torch tensor must be a float32 / float64 CUDA tensor")
            self.dtype = np.float32 if image.dtype == torch.float32 else np.float64
            device = image.device.index
        else:
            image = np.asarray(image)
            self.dtype = np.float32 if image.dtype == np.float32 else np.float64
            device = current_device()
        if image.ndim != 3:
            raise ValueError(f"{name} must be (nband, nx, ny), got shape {tuple(image.shape)}")
        self.nband, self.nx, self.ny = (int(n) for n in image.shape)
        nxp = _plan.good_size(int((1 + pfrac) * self.nx))
        nyp = _plan.good_size(int((1 + pfrac) * self.ny))
        self.device = device
        self.cv = PsfConvolver(self.nx, self.ny, max(nxp, self.nx), max(nyp, self.ny), dtype=self.dtype, device=device)

    def prep(self, a, name):
        if self.torch:
            import torch

            if not isinstance(a, torch.Tensor) or not a.is_cuda or a.device.index != self.device:
                raise TypeError(f"{name} must be a CUDA tensor on the image's device")
            if tuple(a.shape) != (self.nband, self.nx, self.ny):
                raise ValueError(f"{name} shape {tuple(a.shape)} does not match ({self.nband}, {self.nx}, {self.ny})")
            return a.to(torch.float32 if self.dtype == np.float32 else torch.float64).contiguous()
        a = np.ascontiguousarray(a, dtype=self.dtype)
        if a.shape != (self.nband, self.nx, self.ny):
            raise ValueError(f"{name} shape {a.shape} does not match ({self.nband}, {self.nx}, {self.ny})")
        return a

    def empty(self, like):
        if self.torch:
            import torch

            return torch.empty_like(like)
        return np.empty_like(like)

    def apply(self, x, out, b, add=None):
        """out[b] = conv(x[b]) (+ add[b]) with the convolver's current kernel."""
        if self.torch:
            import torch

            s = torch.cuda.current_stream(x.device).cuda_stream
            self.cv.apply_dev(x[b].data_ptr(), out[b].data_ptr(), stream=s,
                              add_ptr=None if add is None else add[b].data_ptr())
        else:
            self.cv.apply(x[b], out=out[b], add=None if add is None else add[b])

    def close(self):
        self.cv.close()


def convolve_to_beam(image, beam_to, beam_from=None, pixsize=1.0, pfrac=0.5, norm_kernel=False):
    """Each band of `image` (``(nband, nx, ny)``, numpy or CUDA tensor) convolved with the Gaussian `beam_to`
    (`beam_from` None: a model), or taken from resolution ``beam_from[b]`` to `beam_to` (`beam_from`: one beam per
    band, or one for all).  Beams in units of `pixsize`; `beam_to` may also be one per band.  ValueError when a beam
    is below one pixel or `beam_to` does not contain ``beam_from[b]``."""
    cube = _Cube(image, pfrac)
    try:
        x = cube.prep(image, "image")
        to = _beams(beam_to, cube.nband, pixsize, "beam_to")
        fr = None if beam_from is None else _beams(beam_from, cube.nband, pixsize, "beam_from")
        out = cube.empty(x)
        for b in range(cube.nband):
            cube.cv.set_gauss(to[b], None if fr is None else fr[b], norm_kernel=norm_kernel)
            cube.apply(x, out, b)
        return out
    finally:
        if cube.torch:
            import torch

            torch.cuda.current_stream(cube.device).synchronize()
        cube.close()


def restore(model, residual, beam, psf_beams=None, pixsize=1.0, pfrac=0.5):
    """Restored cube ``model[b] (*) G_beam + residual[b]``, or with `psf_beams` (one per band) the residual brought to
    the common resolution first: ``model[b] (*) G_beam + residual[b] (*) (G_beam / G_psf_b)``.  Peak-1 kernels, so a
    model in flux per pixel restores to flux per `beam`.  numpy (fp32 / fp64) or CUDA tensors in, the same out."""
    cube = _Cube(model, pfrac, "model")
    try:
        m = cube.prep(model, "model")
        r = cube.prep(residual, "residual")
        bt = _beams(beam, cube.nband, pixsize, "beam")
        bf = None if psf_beams is None else _beams(psf_beams, cube.nband, pixsize, "psf_beams")
        out = cube.empty(m)
        rc = None if bf is None else cube.empty(m[:1])  # one band of the converted residual (add must not alias out)
        for b in range(cube.nband):
            if bf is not None:  # residual pass, then the model pass adds it in its epilogue
                cube.cv.set_gauss(bt[b], bf[b])
                cube.apply(r[b:b + 1], rc, 0)
                cube.cv.set_gauss(bt[b])
                cube.apply(m[b:b + 1], out[b:b + 1], 0, add=rc)
            else:
                cube.cv.set_gauss(bt[b])
                cube.apply(m, out, b, add=r)
        return out
    finally:
        if cube.torch:
            import torch

            torch.cuda.current_stream(cube.device).synchronize()
        cube.close()
