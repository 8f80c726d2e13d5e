"""Cost of inverting the PSF-convolution Hessian, ``HessPSF.idot``, on the host loop (numpy in: ``solvers.pcg`` per band
around host-pointer convolutions) and on the device (CUDA tensors in: one batched ``pfbs_psf_cg``).

Workload (defaults): the C3 shape, 8 bands of 4096^2 with a 5760^2 PSF grid, fp64; the PSF is a Gaussian main lobe
whose width grows with band (its transfer function, as in tools/clean_bench.py), a beam in [0.5, 1], eta = 1e-3.  The
right-hand side is the Hessian applied to a seeded sky (point sources on smooth extended emission) plus noise.

Measured, in one run, with the card's name and power limit read in the same run:
  * ms per CG iteration per band, host and device: cgtol = 0 with cgmaxit = K1 and K2, the difference of the two
    solves over (K2 - K1) * nband, so that the start-up (initial apply, direct estimate) cancels;
  * one realistic device solve (cgtol = 1e-3, cgmaxit = 300): wall time and iterations / stop reason per band;
  * the direct estimate (mode="direct"): host first call (builds the second spectrum per band), host cached call,
    and device;
  * the rel-L2 per band between the host and device solutions after K2 iterations.
Device times are CUDA events around the call after a warm-up call; host times end in a synchronise.

    python tools/psf_idot_bench.py [--nband 8 --nx 4096 --nx-psf 5760 --k1 2 --k2 6 --out FILE]
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


def gaussian_abspsf(nband, nxp, nyp, sigma):
    fx = np.fft.fftfreq(nxp)[:, None]
    fy = np.fft.rfftfreq(nyp)[None, :]
    out = np.empty((nband, nxp, nyp // 2 + 1))
    for b in range(nband):
        s2 = (sigma * (1 + 0.05 * b)) ** 2
        out[b] = 2 * np.pi * s2 * np.exp(-2 * np.pi ** 2 * s2 * fx * fx) * np.exp(-2 * np.pi ** 2 * s2 * fy * fy)
    return out


def sky_model(nband, nx, ny, nsrc, rng):
    sky = np.zeros((nband, nx, ny))
    i, j = rng.integers(64, nx - 64, nsrc), rng.integers(64, ny - 64, nsrc)
    flux = np.exp(rng.uniform(np.log(1.0), np.log(100.0), nsrc))
    sky[:, i, j] += flux[None, :]
    xx = np.arange(nx)[:, None] / nx
    yy = np.arange(ny)[None, :] / ny
    for _ in range(6):
        cx, cy, w = rng.uniform(0.2, 0.8), rng.uniform(0.2, 0.8), rng.uniform(0.05, 0.15)
        sky += 0.03 * np.exp(-((xx - cx) ** 2 + (yy - cy) ** 2) / (2 * w * w))[None]
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
    ap.add_argument("--eta", type=float, default=1e-3)
    ap.add_argument("--k1", type=int, default=2)
    ap.add_argument("--k2", type=int, default=6)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()

    import torch

    from pfb_imaging_b200 import psf as P

    rng = np.random.default_rng(a.seed)
    nb, nx, nxp = a.nband, a.nx, a.nx_psf
    abspsf = gaussian_abspsf(nb, nxp, nxp, a.sigma)
    beam = rng.uniform(0.5, 1.0, (nb, nx, nx))
    H = P.HessPSF(nx, nx, abspsf, beam=beam, eta=a.eta, cgverbose=0)
    dev = torch.device("cuda", H.conv[0].device)
    sky = torch.from_numpy(sky_model(nb, nx, nx, 300, rng)).to(dev)
    bt = H.dot(sky)
    gen = torch.Generator(device=dev).manual_seed(a.seed)
    bt += 1e-3 * torch.randn(bt.shape, dtype=torch.float64, device=dev, generator=gen)
    del sky
    b = bt.cpu().numpy()
    name, plim = card()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def dev_ms(fn):
        fn()  # warm-up
        torch.cuda.synchronize(dev)
        ev0.record()
        out = fn()
        ev1.record()
        ev1.synchronize()
        return ev0.elapsed_time(ev1), out

    def host_s(fn):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize(dev)
        return time.perf_counter() - t0, out

    # ms per CG iteration per band (cgtol = 0: exactly cgmaxit iterations on both paths)
    H.cgtol = 0.0
    t_host, t_dev, sol_host, sol_dev = {}, {}, None, None
    for k in (a.k1, a.k2):
        H.cgmaxit = k
        t_host[k], sol_host = host_s(lambda: H.idot(b, mode="psf", init_x0=False))
        t_dev[k], sol_dev = dev_ms(lambda: H.idot(bt, mode="psf", init_x0=False))
    dk = (a.k2 - a.k1) * nb
    host_ms_it = (t_host[a.k2] - t_host[a.k1]) * 1e3 / dk
    dev_ms_it = (t_dev[a.k2] - t_dev[a.k1]) / dk
    sd = sol_dev.cpu().numpy()
    rel = [float(np.linalg.norm(sd[i] - sol_host[i]) / np.linalg.norm(sol_host[i])) for i in range(nb)]
    del sol_host, sd, sol_dev

    # one realistic device solve
    H.cgtol, H.cgmaxit = 1e-3, 300
    t_solve, _ = dev_ms(lambda: H.idot(bt, mode="psf"))
    info = H.last_idot_info

    # the direct estimate
    P._DIRECT_CACHE.clear()
    t_dir_first, _ = host_s(lambda: H.idot(b, mode="direct"))
    t_dir_cached, _ = host_s(lambda: H.idot(b, mode="direct"))
    t_dir_dev, _ = dev_ms(lambda: H.idot(bt, mode="direct"))

    res = dict(
        tool="psf_idot_bench", device=name, power_limit=plim, nband=nb, nx=nx, ny=nx, nx_psf=nxp, ny_psf=nxp,
        dtype="float64", eta=a.eta, sigma=a.sigma, k1=a.k1, k2=a.k2,
        host_ms_per_iter_per_band=round(host_ms_it, 3), device_ms_per_iter_per_band=round(dev_ms_it, 3),
        speedup_per_iter=round(host_ms_it / dev_ms_it, 1),
        host_s_k=[round(t_host[k], 3) for k in (a.k1, a.k2)], device_ms_k=[round(t_dev[k], 3) for k in (a.k1, a.k2)],
        rel_l2_device_vs_host_k2=[float(f"{r:.3g}") for r in rel],
        solve_cgtol=1e-3, solve_cgmaxit=300, solve_device_ms=round(t_solve, 3),
        solve_iters=info["iters"].tolist(), solve_stop=info["stop"], solve_eps=[float(f"{e:.3g}") for e in info["eps"]],
        direct_host_first_s=round(t_dir_first, 3), direct_host_cached_s=round(t_dir_cached, 3),
        direct_device_ms=round(t_dir_dev, 3),
    )
    H.close()
    P.clear_convolver_cache()
    P._DIRECT_CACHE.clear()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
