"""TEST INFRASTRUCTURE ONLY — numpy restatement of the Clark CLEAN minor cycle, the backward step of ``pfb kclean``
(``core/kclean.py:203-218`` of the reference calls ``deconv/clark.py``).

No golden of the reference's numba ``clark`` exists, so this is not pinned to it: it restates the contract the
device implementation (``pfb_imaging_b200.clean``) follows — Clark (1980) with an MFS search over bands:

  * images are (nband, nx, ny), raster index p = i*ny + j; the PSF is (nband, nx_psf, ny_psf) with its centre at
    (nx_psf//2, ny_psf//2); peak_b = PSF[b, centre]; a band with peak_b <= 0 gets no model;
  * search value s(p) = |R_0(p) + R_1(p) + ... + R_{nband-1}(p)|, summed in band order; masked-out pixels are never
    searched;
  * major loop: Rmax = max s; on the first pass tol = max(pf Rmax, threshold); stop when Rmax <= tol or after maxit
    major iterations; active set A = {masked p : s(p) >= subpf Rmax} in raster order;
  * subminor loop on A while the peak s(a*) > max(subpf Rmax, threshold) and fewer than submaxit components ran:
    a* = first maximum in raster order; d_b = (gamma R_b(a*)) / peak_b; model_b(a*) += d_b; every a in A inside the
    PSF support around a* gets R_b(a) = R_b(a) - d_b * PSF_b(c + a - a*) (multiply, then subtract);
  * R = ID - PSF (*) model through the r2c spectrum PSFHAT (padded at the corner to the PSF size, cropped to
    [0:nx, 0:ny]), then the next major iteration.

Only tests/ and tools/ may import this module.
"""

import numpy as np


def search_value(R):
    """s = |R_0 + R_1 + ...|, the sum taken in band order."""
    acc = R[0].copy()
    for b in range(1, R.shape[0]):
        acc = acc + R[b]
    return np.abs(acc)


def psfhat_of(psf):
    """PSFHAT = rfft2(ifftshift(PSF)), as ``image_data_products_arrays`` returns it."""
    return np.fft.rfft2(np.fft.ifftshift(psf, axes=(1, 2)), axes=(1, 2))


def psf_convolve(model, psfhat, nx_psf, ny_psf):
    """crop(IFFT(FFT(pad(model)) PSFHAT)) per band: the corner-padded circular convolution of the device convolver."""
    nx, ny = model.shape[1:]
    out = np.empty_like(model, dtype=np.float64)
    for b in range(model.shape[0]):
        xh = np.fft.rfft2(model[b], s=(nx_psf, ny_psf))
        out[b] = np.fft.irfft2(xh * psfhat[b], s=(nx_psf, ny_psf))[:nx, :ny]
    return out


def direct_convolve(model, psf):
    """Spatial convolution: out_b(p) = sum_q model_b(q) PSF_b(c + p - q), PSF indices outside the array being zero.
    Equals ``psf_convolve`` when nx_psf >= 2 nx and ny_psf >= 2 ny (no wrap-around)."""
    nband, nx, ny = model.shape
    _, nxp, nyp = psf.shape
    cx, cy = nxp // 2, nyp // 2
    out = np.zeros((nband, nx, ny))
    for b in range(nband):
        for i, j in zip(*np.nonzero(model[b])):
            # out[p] += m * PSF[cx + ip - i, cy + jp - j] for every p whose PSF index is inside the array
            i0, i1 = max(0, i - cx), min(nx, i - cx + nxp)
            j0, j1 = max(0, j - cy), min(ny, j - cy + nyp)
            out[b, i0:i1, j0:j1] += model[b, i, j] * psf[b, cx + i0 - i:cx + i1 - i, cy + j0 - j:cy + j1 - j]
    return out


def clark(ID, PSF, PSFHAT=None, mask=None, threshold=0.0, gamma=0.05, pf=0.05, maxit=50, subpf=0.5, submaxit=1000,
          callback=None):
    """Returns (model, residual, info) with info = dict(niter, rmax, nactive, nsub, peaks): per major iteration its
    Rmax, |A|, the number of components and the raster indices of their peaks in order.  `callback(k, model, R)` is
    called after every major iteration's residual step."""
    ID = np.asarray(ID, dtype=np.float64)
    PSF = np.asarray(PSF, dtype=np.float64)
    nband, nx, ny = ID.shape
    _, nxp, nyp = PSF.shape
    cx, cy = nxp // 2, nyp // 2
    if PSFHAT is None:
        PSFHAT = psfhat_of(PSF)
    peak = PSF[:, cx, cy]
    msk = np.ones(nx * ny, dtype=bool) if mask is None else np.asarray(mask).astype(bool).ravel()
    R = ID.copy()
    model = np.zeros_like(ID)
    info = dict(niter=0, rmax=[], nactive=[], nsub=[], peaks=[])
    tol = None
    k = 0
    while True:
        s = search_value(R).ravel()
        Rmax = float(s[msk].max()) if msk.any() else 0.0
        if tol is None:
            tol = max(pf * Rmax, threshold)
        if not (Rmax > tol) or k >= maxit:
            break
        A = np.flatnonzero(msk & (s >= subpf * Rmax))
        ia, ja = A // ny, A % ny
        RA = R.reshape(nband, -1)[:, A].copy()
        sA = s[A].copy()
        thr = max(subpf * Rmax, threshold)
        peaks = []
        while len(peaks) < submaxit:
            a = int(np.argmax(sA))
            if not (sA[a] > thr):
                break
            d = np.zeros(nband)
            for b in range(nband):
                if peak[b] > 0:
                    d[b] = (gamma * RA[b, a]) / peak[b]
            model[:, ia[a], ja[a]] += d
            x = cx + ia - ia[a]
            y = cy + ja - ja[a]
            sel = np.flatnonzero((x >= 0) & (x < nxp) & (y >= 0) & (y < nyp))
            RA[:, sel] = RA[:, sel] - d[:, None] * PSF[:, x[sel], y[sel]]
            sA[sel] = search_value(RA[:, sel])
            peaks.append(int(A[a]))
        R = ID - psf_convolve(model, PSFHAT, nxp, nyp)
        info["rmax"].append(Rmax)
        info["nactive"].append(int(A.size))
        info["nsub"].append(len(peaks))
        info["peaks"].append(np.array(peaks, dtype=np.int64))
        k += 1
        info["niter"] = k
        if callback is not None:
            callback(k, model, R)
    return model, R, info
