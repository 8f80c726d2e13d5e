"""Cost of restoration on the device (pfb_imaging_b200.restore) at the C2 shape, and of the analytic Gaussian column
pass against the stored-spectrum one.

Workload (defaults): 8 bands of 4096^2 in fp64, pfrac = 0.5 (padded 6144^2); a sparse model (2000 components per band)
and a noise residual as CUDA tensors; restoring beam (6.0, 4.5, 0.3) px, per-band PSF beams growing with band.

Prints one JSON line: the device name and power limit read in this run; CUDA-event ms per band and per cube of the
plain restore (one apply_add per band) and of the common-resolution restore (a residual pass and a model pass per
band), after a warm-up call; ms per apply of the Gaussian-mode and khat-mode convolver on the same image, alternated,
at 6144^2 and at the 5760^2 PSF size; and the host time of the same plain restore of the cube with scipy.fft on all
cores (a host restatement of the operation, not the reference's code).

    python tools/restore_bench.py [--nband 8 --nx 4096 --reps 5]
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


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    name, plim = (s.strip() for s in out.split(","))
    return name, plim


def timed(torch, fn, reps):
    fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nband", type=int, default=8)
    ap.add_argument("--nx", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import scipy.fft as sfft
    import torch

    from oracle import restore_np as O
    from pfb_imaging_b200 import plan, restore as R
    from pfb_imaging_b200.psf import PsfConvolver

    if not torch.cuda.is_available():
        raise SystemExit("restore_bench needs a GPU")
    name, plim = card()
    nb, nx = a.nband, a.nx
    rng = np.random.default_rng(0)
    model = np.zeros((nb, nx, nx))
    for b in range(nb):
        model[b, rng.integers(0, nx, 2000), rng.integers(0, nx, 2000)] = rng.exponential(1.0, 2000)
    resid = 0.01 * rng.standard_normal((nb, nx, nx))
    beam = (6.0, 4.5, 0.3)
    psf_beams = [(4.0 + 0.2 * b, 3.0 + 0.1 * b, 0.2) for b in range(nb)]
    mt, rt = torch.from_numpy(model).cuda(), torch.from_numpy(resid).cuda()
    nxp = plan.good_size(int(1.5 * nx))

    plain = timed(torch, lambda: R.restore(mt, rt, beam), a.reps)
    common = timed(torch, lambda: R.restore(mt, rt, beam, psf_beams=psf_beams), a.reps)
    res = {"device": name, "power_limit": plim, "nband": nb, "nx": nx, "nx_pad": nxp, "dtype": "float64",
           "restore_ms_cube": round(plain, 2), "restore_ms_band": round(plain / nb, 3),
           "restore_common_ms_cube": round(common, 2), "restore_common_ms_band": round(common / nb, 3),
           "note_restore": "each call creates its convolver (tables, 400 MB of scratch) and releases it"}

    # one apply, Gaussian column pass against the stored spectrum, alternated, at two padded sizes
    x = mt[0].contiguous()
    y = torch.empty_like(x)
    s = torch.cuda.current_stream().cuda_stream
    for npad in (nxp, 5760):
        cg = PsfConvolver(nx, nx, npad, npad).set_gauss(beam)
        ck = PsfConvolver(nx, nx, npad, npad).set_kernel(O.kernel_spectrum(npad, npad, beam))
        cr = PsfConvolver(nx, nx, npad, npad).set_gauss(beam, psf_beams[0])
        tg, tk, tr = [], [], []
        for _ in range(a.reps):
            tk.append(timed(torch, lambda: ck.apply_dev(x.data_ptr(), y.data_ptr(), stream=s), 10))
            tg.append(timed(torch, lambda: cg.apply_dev(x.data_ptr(), y.data_ptr(), stream=s), 10))
            tr.append(timed(torch, lambda: cr.apply_dev(x.data_ptr(), y.data_ptr(), stream=s), 10))
        res[f"apply_ms_{npad}"] = {"khat": round(float(np.median(tk)), 3), "gauss": round(float(np.median(tg)), 3),
                                   "gauss_ratio": round(float(np.median(tr)), 3)}
        for c in (cg, ck, cr):
            c.close()

    # host restatement: scipy.fft on all cores, the same plain restore of the cube (kernel spectrum built once)
    t = time.perf_counter()
    kh = O.kernel_spectrum(nxp, nxp, beam)
    t_k = time.perf_counter() - t
    t = time.perf_counter()
    host = np.empty_like(model)
    for b in range(nb):
        xp = np.zeros((nxp, nxp))
        xp[:nx, :nx] = model[b]
        host[b] = sfft.irfft2(sfft.rfft2(xp, workers=-1) * kh, s=(nxp, nxp), workers=-1)[:nx, :nx] + resid[b]
    t_h = time.perf_counter() - t
    dev = R.restore(model, resid, beam)
    res.update({"host_scipy_restatement_s_cube": round(t_h, 2), "host_kernel_spectrum_s": round(t_k, 2),
                "host_threads": os.cpu_count(),
                "device_vs_host_rel_l2": float(np.linalg.norm(dev - host) / np.linalg.norm(host))})
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
