"""numpy / scipy contract of ``pfb_imaging_b200.restore`` (tests only).

The Gaussian kernel is built in the image domain: the pixel-sampled Gaussian at the signed offsets of the padded grid,
summed over enough neighbouring periodic images, then ``rfft2``, multiply, ``irfft2`` and crop, in fp64.  This
shares nothing with the alias sum of the device's transfer function, so the two check each other.  The kernel and its
spectrum are computed in long double: the spectrum of a wide Gaussian falls far below the rounding of an fp64 FFT of
it, and the ratio of two spectra (a change of resolution) divides by exactly those small values.  The fitter is
restated with ``scipy.ndimage.label`` (4-connectivity) and ``scipy.optimize.curve_fit`` on ``(emaj, emin, pa)``.
"""
import numpy as np
import scipy.fft as sfft
import scipy.ndimage as ndi
from scipy.optimize import curve_fit

def good_size(n):
    """plan.good_size: smallest 2^a 3^b 5^c 7^d >= n."""
    n = max(int(n), 1)
    while True:
        m = n
        for p in (2, 3, 5, 7):
            while m % p == 0:
                m //= p
        if m == 1:
            return n
        n += 1


def gauss(x, y, emaj, emin, pa):
    """exp(-4 ln 2 (x'^2 / emaj^2 + y'^2 / emin^2)), (x', y') = (x, y) rotated so that x' runs along (cos pa, sin pa)."""
    c, s = np.cos(pa), np.sin(pa)
    xp, yp = x * c + y * s, -x * s + y * c
    return np.exp(-4 * np.log(np.asarray(2, dtype=np.result_type(x, y, pa))) * (xp * xp / emaj**2 + yp * yp / emin**2))


def periodic_kernel(nxp, nyp, beam):
    """The sampled Gaussian on the (nxp, nyp) grid, centred at index 0, with its periodic images summed."""
    emaj = beam[0]
    ox = np.arange(nxp) - nxp * (np.arange(nxp) > nxp // 2)  # signed offsets
    oy = np.arange(nyp) - nyp * (np.arange(nyp) > nyp // 2)
    # images out to 10 FWHM, where g < exp(-277); an image whose nearest pixel is farther along either axis is skipped
    reach = 10.0 * emaj
    P = int(np.ceil(reach / min(nxp, nyp))) + 1
    k = np.zeros((nxp, nyp), dtype=np.longdouble)
    ox, oy = ox.astype(np.longdouble), oy.astype(np.longdouble)
    beam = tuple(np.longdouble(v) for v in beam)
    for p in range(-P, P + 1):
        if np.abs(ox + p * nxp).min() > reach:
            continue
        for q in range(-P, P + 1):
            if np.abs(oy + q * nyp).min() > reach:
                continue
            k += gauss((ox + p * nxp)[:, None], (oy + q * nyp)[None, :], *beam)
    return k


def kernel_spectrum(nxp, nyp, beam, beam_from=None, norm_kernel=False):
    """rfft2 of the periodic kernel (or the ratio of two), peak-1 or unit-sum kernels; long double, returned as
    complex128."""
    def one(b):
        k = periodic_kernel(nxp, nyp, b)
        if norm_kernel:
            k /= k.sum()
        return sfft.rfft2(k)

    kh = one(beam)
    if beam_from is not None:
        kh = kh / one(beam_from)
    return kh.astype(np.complex128)


def alias_ratio_spectrum(nxp, nyp, beam_to, beam_from, rings=12):
    """K_to / K_from of peak-1 kernels by Poisson summation over |m_i| <= `rings`, in long double, each sum scaled by
    its largest term.  The image-domain route above cannot resolve K_from of a wide beam near Nyquist (e^-87 of the
    peak at 7 px), so conversions between wide beams are checked against this instead; with 12 rings the dropped terms
    are below e^-(2 pi^2 * 0.18 * 11.5^2) of the largest for any beam of FWHM >= 1 px."""
    LD = np.longdouble

    def cov(b):
        emaj, emin, pa = (LD(v) for v in b)
        k = 1 / (8 * np.log(LD(2)))
        va, vb, c, s = emaj * emaj * k, emin * emin * k, np.cos(pa), np.sin(pa)
        return va * c * c + vb * s * s, (va - vb) * c * s, va * s * s + vb * c * c

    k, l = np.arange(nxp), np.arange(nyp // 2 + 1)
    fx = (np.where(2 * k > nxp, k - nxp, k).astype(LD) / nxp)[:, None]
    fy = (np.where(2 * l > nyp, l - nyp, l).astype(LD) / nyp)[None, :]
    c2 = -2 * np.pi ** 2 * LD(1)
    rng = range(-rings, rings + 1)

    def scaled(S):
        q = [c2 * ((fx + mx) ** 2 * S[0] + 2 * (fx + mx) * (fy + my) * S[1] + (fy + my) ** 2 * S[2])
             for mx in rng for my in rng]
        top = np.max(q, axis=0)
        return 2 * np.pi * np.sqrt(S[0] * S[2] - S[1] ** 2), top, sum(np.exp(t - top) for t in q)

    at, tt, st = scaled(cov(beam_to))
    af, tf, sf = scaled(cov(beam_from))
    return (at / af * np.exp(tt - tf) * st / sf).astype(np.float64)


def convolve_pad(x, khat, nxp, nyp):
    nx, ny = x.shape
    xp = np.zeros((nxp, nyp))
    xp[:nx, :ny] = x
    return np.fft.irfft2(np.fft.rfft2(xp) * khat, s=(nxp, nyp))[:nx, :ny]


def convolve_to_beam(image, beam_to, beam_from=None, pfrac=0.5, norm_kernel=False, pads=None):
    """(nband, nx, ny) -> same; beams in pixels, `beam_from` one per band or None."""
    image = np.asarray(image, dtype=np.float64)
    nb, nx, ny = image.shape
    nxp, nyp = pads if pads else (good_size(int((1 + pfrac) * nx)), good_size(int((1 + pfrac) * ny)))
    out = np.empty_like(image)
    for b in range(nb):
        kh = kernel_spectrum(nxp, nyp, beam_to, None if beam_from is None else beam_from[b], norm_kernel)
        out[b] = convolve_pad(image[b], kh, nxp, nyp)
    return out


def restore(model, residual, beam, psf_beams=None, pfrac=0.5):
    out = convolve_to_beam(model, beam, pfrac=pfrac)
    if psf_beams is None:
        return out + np.asarray(residual, dtype=np.float64)
    return out + convolve_to_beam(residual, beam, psf_beams, pfrac=pfrac)


def canonical(emaj, emin, pa):
    """(emaj, emin, pa) with emaj >= emin and pa in (-pi/2, pi/2], 0 for a circular beam."""
    emaj, emin = abs(emaj), abs(emin)
    if emin > emaj:
        emaj, emin, pa = emin, emaj, pa + np.pi / 2
    pa = (pa + np.pi / 2) % np.pi - np.pi / 2
    if pa <= -np.pi / 2:
        pa += np.pi
    if emaj - emin <= 1e-12 * emaj:
        pa = 0.0
    return emaj, emin, pa


def fitcleanbeam(psf, level=0.5, pixsize=1.0, p0=None):
    psf = np.asarray(psf, dtype=np.float64)
    if psf.ndim == 2:
        psf = psf[None]
    out = []
    for b in range(psf.shape[0]):
        p = psf[b] / psf[b].max()
        nx, ny = p.shape
        lab, _ = ndi.label(p > level)  # default structure: 4-connectivity
        isl = lab == lab[nx // 2, ny // 2]
        ix, iy = np.nonzero(isl)
        x, y = ix - nx // 2.0, iy - ny // 2.0
        if p0 is None:
            w = p[isl] / p[isl].sum()
            cov = np.array([[(w * x * x).sum(), (w * x * y).sum()], [(w * x * y).sum(), (w * y * y).sum()]])
            ev, V = np.linalg.eigh(cov)
            start = (np.sqrt(8 * np.log(2) * ev[1]), np.sqrt(8 * np.log(2) * ev[0]), np.arctan2(V[1, 1], V[0, 1]))
        else:
            start = p0
        popt, _ = curve_fit(lambda xy, a, bb, c: gauss(xy[0], xy[1], a, bb, c), np.vstack((x, y)), p[isl], p0=start,
                            xtol=1e-15, ftol=1e-15, gtol=1e-15, maxfev=10000)
        emaj, emin, pa = canonical(*popt)
        out.append((emaj * pixsize, emin * pixsize, pa))
    return np.array(out)
