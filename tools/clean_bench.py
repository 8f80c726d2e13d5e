"""Cost of the device Clark minor cycle (pfb_imaging_b200.clean) at a kclean-sized problem.

Workload (defaults): 8 bands of 4096^2, PSF 5760^2 (the C2 PSF size), a Gaussian main lobe whose width grows with
band; the sky is seeded point sources (log-uniform fluxes, spectral slope) plus a smooth, positive extended
component; dirty = PSF (*) sky.  Bright sources make the first active sets hundreds of pixels, the extended
emission makes the late ones > 10^5 pixels.

Prints one JSON line: the device name and power limit read in this run, per major iteration the CUDA-event times of
search + compaction, subminor (with the model update) and the residual step, |A|, the components and the time per
component; and, with --host-iters N > 0, the time of the numpy restatement of the contract (oracle/clark_np.py, NOT
the reference's numba clark) on the host for the first N major iterations of the same call.

    python tools/clean_bench.py [--nband 8 --nx 4096 --nx-psf 5760 --maxit 8 --submaxit 2000 --host-iters 1]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gaussian_psf(nband, nxp, nyp, sigma0):
    x = (np.arange(nxp) - nxp // 2)[:, None].astype(np.float64)
    y = (np.arange(nyp) - nyp // 2)[None, :].astype(np.float64)
    psf = np.empty((nband, nxp, nyp))
    for b in range(nband):
        s = sigma0 * (1 + 0.05 * b)
        psf[b] = np.exp(-(x * x + y * y) / (2 * s * s))
    return psf


def sky_model(nband, nx, ny, nsrc, ext_amp, rng):
    sky = np.zeros((nband, nx, ny))
    i, j = rng.integers(64, nx - 64, nsrc), rng.integers(64, ny - 64, nsrc)
    flux = np.exp(rng.uniform(np.log(1.0), np.log(100.0), nsrc))
    alpha = rng.uniform(-1.0, 0.5, nsrc)
    nu = 1.0 + 0.1 * np.arange(nband)
    sky[:, i, j] += flux[None, :] * nu[:, None] ** alpha[None, :]
    # smooth positive extended emission: a few broad Gaussian blobs
    xx = np.arange(nx)[:, None] / nx
    yy = np.arange(ny)[None, :] / ny
    ext = np.zeros((nx, ny))
    for _ in range(6):
        cx, cy, w = rng.uniform(0.2, 0.8), rng.uniform(0.2, 0.8), rng.uniform(0.05, 0.15)
        ext += np.exp(-((xx - cx) ** 2 + (yy - cy) ** 2) / (2 * w * w))
    sky += ext_amp * ext[None] * nu[:, None, None] ** -0.7
    return sky


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, plim = (s.strip() for s in out.split(","))
        return name, plim
    except Exception as e:  # noqa: BLE001
        return None, f"unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nband", type=int, default=8)
    ap.add_argument("--nx", type=int, default=4096)
    ap.add_argument("--nx-psf", type=int, default=5760)
    ap.add_argument("--sigma", type=float, default=3.0, help="PSF main-lobe sigma in pixels (band 0)")
    ap.add_argument("--nsrc", type=int, default=300)
    ap.add_argument("--ext-amp", type=float, default=0.03, help="extended emission per pixel, before the PSF")
    ap.add_argument("--gamma", type=float, default=0.1)
    ap.add_argument("--pf", type=float, default=0.0)
    ap.add_argument("--subpf", type=float, default=0.5)
    ap.add_argument("--maxit", type=int, default=8)
    ap.add_argument("--submaxit", type=int, default=2000)
    ap.add_argument("--host-iters", type=int, default=1, help="major iterations of the numpy restatement to time")
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()

    from pfb_imaging_b200 import psf as P
    from pfb_imaging_b200.clean import Clark

    rng = np.random.default_rng(a.seed)
    nb, nx, nxp = a.nband, a.nx, a.nx_psf
    psf = gaussian_psf(nb, nxp, nxp, a.sigma)
    psfhat = np.fft.rfft2(np.fft.ifftshift(psf, axes=(1, 2)), axes=(1, 2))
    sky = sky_model(nb, nx, nx, a.nsrc, a.ext_amp, rng)
    dirty = np.empty_like(sky)
    for b in range(nb):  # the library's own PSF convolver: dirty = PSF (*) sky
        cv = P.PsfConvolver(nx, nx, nxp, nxp).set_kernel(psfhat[b])
        dirty[b] = cv.apply(sky[b])
        cv.close()
    del sky

    name, plim = card()
    t0 = time.perf_counter()
    cl = Clark(psf, psfhat, nx=nx, ny=nx)
    t_create = time.perf_counter() - t0
    kw = dict(gamma=a.gamma, pf=a.pf, subpf=a.subpf, submaxit=a.submaxit)
    cl(dirty, maxit=1, **dict(kw, submaxit=min(a.submaxit, 50)))  # warm-up: modules, CUB, convolvers
    t0 = time.perf_counter()
    model, resid, info = cl(dirty, maxit=a.maxit, timings=True, **kw)
    t_call = time.perf_counter() - t0
    tm = np.asarray(info["times_ms"], dtype=np.float64)
    nsub = np.asarray(info["nsub"])
    per_comp = (tm[:, 1] * 1e3 / np.maximum(nsub, 1)).round(3).tolist()
    res = dict(
        tool="clean_bench", device=name, power_limit=plim, nband=nb, nx=nx, ny=nx, nx_psf=nxp, ny_psf=nxp,
        gamma=a.gamma, pf=a.pf, subpf=a.subpf, maxit=a.maxit, submaxit=a.submaxit, niter=info["niter"],
        create_s=round(t_create, 3), call_wall_s=round(t_call, 3),
        ms_search_compact=tm[:, 0].round(3).tolist(), ms_subminor=tm[:, 1].round(3).tolist(),
        ms_residual_step=tm[:, 2].round(3).tolist(), ms_per_major=tm.sum(axis=1).round(3).tolist(),
        nactive=info["nactive"], nsub=info["nsub"], us_per_component=per_comp,
        rmax=[float(f"{r:.6g}") for r in info["rmax"]],
    )
    if a.host_iters > 0:
        from oracle import clark_np as cn

        k = min(a.host_iters, info["niter"])
        t0 = time.perf_counter()
        mo, ro, io = cn.clark(dirty, psf, psfhat, maxit=k, **kw)
        th = time.perf_counter() - t0
        same = io["nsub"] == info["nsub"][:k] and all(np.array_equal(x, y) for x, y in zip(io["peaks"], info["peaks"]))
        res.update(host_numpy_restatement_iters=k, host_numpy_restatement_s=round(th, 3),
                   host_numpy_restatement_ms_per_major=round(th * 1e3 / max(k, 1), 1),
                   device_ms_first_iters=round(float(tm[:k].sum()), 3), host_same_peaks=bool(same))
    cl.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
