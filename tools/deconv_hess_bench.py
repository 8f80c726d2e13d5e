"""Cost of ``pfb deconv``'s Hessian, the per-band ``HessianTree`` behind ``BandWorkerPool`` / ``HessTreeRay``, on the host
loop (numpy in: ``solvers.pcg`` per band around host-pointer convolutions) and on the device (CUDA tensors in: one
batched ``pfbs_tree_cg`` per device).

Workload (defaults): the C3 shape, 8 bands of 4096^2 with a 5760^2 PSF grid, fp64, 2 partitions per band.  Each
partition's PSF is a Gaussian main lobe whose width grows with band and partition (its transfer function, as in
tools/psf_idot_bench.py), beams in [0.5, 1], eta = 1e-3 of the largest eigenvalue bound.  Two runs: the partitions of a
band share one beam (merged into one group: one convolution per CG iteration) or have distinct beams (two groups).
The right-hand side is the Hessian applied to a seeded sky plus noise.

Measured per run, in one process on one GPU, with the card's name and power limit read in the same run:
  * ms per CG iteration per band, host and device: cgtol = 0 with cgmaxit = K1 and K2, the difference of the two
    solves over (K2 - K1) * bands, so that the start-up cancels (host: on --host-bands bands);
  * a device solve at cgtol 1e-3 (cgmaxit 300): wall time, iterations and stop reason per band;
  * hess_dot of the cube, host and device;
  * one primal-dual iteration (3 bases, 2 levels) with PsfGradient(HessTreeRay): the difference of maxit = 1 and 3 over 2;
  * shared-beam run only: the same one-group systems solved by HessPSF.idot (pfbs_psf_cg) next to pfbs_tree_cg.
With two or more visible GPUs, a second process times the distinct-beam solve with the bands spread over every GPU
against all bands on one.  Times are host clocks around work that ends in a device synchronise, after a warm-up call.

    python tools/deconv_hess_bench.py [--nband 8 --nx 4096 --nx-psf 5760 --k1 2 --k2 6 --out FILE]
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
sys.path.insert(0, os.path.join(ROOT, "tools"))


def gpu_count():
    try:
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=60).stdout
        return sum(1 for line in out.splitlines() if line.startswith("GPU "))
    except Exception:  # noqa: BLE001
        return 0


def problem(a, distinct, rng):
    from psf_idot_bench import gaussian_abspsf

    nb, nx, nxp = a.nband, a.nx, a.nx_psf
    parts = []
    for b in range(nb):
        pb = []
        shared = rng.uniform(0.5, 1.0, (1, nx, nx))
        for p in range(a.npart):
            beam = rng.uniform(0.5, 1.0, (1, nx, nx)) if distinct else shared
            khat = gaussian_abspsf(1, nxp, nxp, a.sigma * (1 + 0.02 * b) * (1 + 0.1 * p))[0]
            pb.append(dict(psfhat=khat[None], beam=beam, wsum=np.array([1.0e4 * (1 + p)])))
        parts.append(pb)
    lam = max(sum(p["psfhat"][0].max() for p in pb) / sum(p["wsum"][0] for p in pb) for pb in parts)
    return parts, lam * a.eta


def timed(fn, sync):
    sync()
    t0 = time.perf_counter()
    out = fn()
    sync()
    return time.perf_counter() - t0, out


def run_single(a, distinct):
    import torch

    from pfb_imaging_b200 import operators as ops, psf as P, solvers
    from pfb_imaging_b200.sara import L21, PrimalDual, PsiNocopyt
    from psf_idot_bench import sky_model

    rng = np.random.default_rng(a.seed)
    nb, nx, nxp = a.nband, a.nx, a.nx_psf
    parts, eta = problem(a, distinct, rng)
    dev = torch.device("cuda", 0)
    sync = lambda: torch.cuda.synchronize(dev)  # noqa: E731
    pool = ops.BandWorkerPool(nb)
    hess = P.HessTreeRay(parts, nx, nx, nxp, nxp, etas=eta, workers=pool, cg_tol=1e-3, cg_maxit=300)
    trees = [pool._workers[b].hess for b in range(nb)]
    sky = torch.from_numpy(sky_model(nb, nx, nx, 300, rng)).to(dev)
    bt = hess.dot(sky)
    bt += 1e-3 * bt.abs().max() * torch.randn(bt.shape, dtype=torch.float64, device=dev,
                                             generator=torch.Generator(device=dev).manual_seed(a.seed))
    del sky
    b = bt.cpu().numpy()
    res = dict(beams="distinct" if distinct else "shared", groups_per_band=len(trees[0]._groups), eta=eta)

    # ms per CG iteration per band
    t_dev, t_host = {}, {}
    for k in (a.k1, a.k2):
        P.tree_cg(trees, bt, None, 0.0, k, k)  # warm-up
        t_dev[k], _ = timed(lambda: P.tree_cg(trees, bt, None, 0.0, k, k), sync)
        t_host[k], _ = timed(lambda: [solvers.pcg(lambda z, t=trees[i]: t.dot(z)[0], b[i], tol=0.0, maxit=k, minit=k,
                                                  verbosity=0) for i in range(a.host_bands)], sync)
    dk = a.k2 - a.k1
    res["device_ms_per_iter_per_band"] = round((t_dev[a.k2] - t_dev[a.k1]) * 1e3 / (dk * nb), 3)
    res["host_ms_per_iter_per_band"] = round((t_host[a.k2] - t_host[a.k1]) * 1e3 / (dk * a.host_bands), 3)
    res["host_bands_timed"] = a.host_bands

    # a realistic solve on the device, through the facade
    hess.cg(bt)
    t_solve, _ = timed(lambda: hess.cg(bt), sync)
    info = hess.last_cg_info
    res.update(solve_cgtol=1e-3, solve_cgmaxit=300, solve_device_ms=round(t_solve * 1e3, 3),
               solve_iters=info["iters"].tolist(), solve_stop=info["stop"], solve_host="not measured")

    # hess_dot of the cube
    hess.dot(bt)
    t_dot_dev, _ = timed(lambda: hess.dot(bt), sync)
    t_dot_host, _ = timed(lambda: hess.dot(b), sync)
    res.update(hess_dot_device_ms=round(t_dot_dev * 1e3, 3), hess_dot_host_ms=round(t_dot_host * 1e3, 3))

    # one primal-dual iteration with the tree gradient
    bases = ["self", "db1", "db2"]
    psi = PsiNocopyt(nb, nx, nx, bases, 2, 1)
    reg = L21(psi, bases, nu=len(bases))
    pd = PrimalDual(tol=0.0, maxit=1, verbosity=0, positivity=1)
    pd.setup(reg, float(eta / a.eta) * 1.01)
    pd.set_grad(P.PsfGradient(hess, b))
    x0 = np.zeros_like(b)
    t_pd = {}
    for m in (1, 3):
        pd.maxit = m
        pd.reset()
        pd.solve(x0.copy(), 1e-4)
        pd.reset()
        t_pd[m], _ = timed(lambda: pd.solve(x0.copy(), 1e-4), sync)
    res["pd_iter_ms"] = round((t_pd[3] - t_pd[1]) * 1e3 / 2, 3)
    del pd, reg
    psi.close()

    # the one-group systems through HessPSF.idot (pfbs_psf_cg): same kernels, same loop
    if not distinct:
        abspsf = np.stack([sum(p["psfhat"][0] for p in pb) / sum(p["wsum"][0] for p in pb) for pb in parts])
        beam = np.stack([pb[0]["beam"][0] for pb in parts])
        H = P.HessPSF(nx, nx, abspsf, beam=beam, eta=float(eta), cgtol=0.0, cgverbose=0)
        t_psf = {}
        for k in (a.k1, a.k2):
            H.cgmaxit = k
            H.idot(bt, mode="psf", init_x0=False)
            t_psf[k], _ = timed(lambda: H.idot(bt, mode="psf", init_x0=False), sync)
        res["psf_cg_ms_per_iter_per_band"] = round((t_psf[a.k2] - t_psf[a.k1]) * 1e3 / (dk * nb), 3)
        res["tree_over_psf_cg"] = round(res["device_ms_per_iter_per_band"] / res["psf_cg_ms_per_iter_per_band"], 4)
        H.close()
    pool.close()
    P.clear_convolver_cache()
    return res


def run_multi(a):
    """Distinct-beam solve at cgtol 1e-3: bands spread over every visible GPU (the pool's placement) against all
    bands on GPU 0."""
    import torch

    from pfb_imaging_b200 import operators as ops, psf as P

    rng = np.random.default_rng(a.seed)
    nb, nx, nxp = a.nband, a.nx, a.nx_psf
    parts, eta = problem(a, True, rng)
    ndev = torch.cuda.device_count()

    def sync():
        for d in range(ndev):
            torch.cuda.synchronize(d)

    pool = ops.BandWorkerPool(nb)
    hess = P.HessTreeRay(parts, nx, nx, nxp, nxp, etas=eta, workers=pool, cg_tol=1e-3, cg_maxit=300)
    one = [P.HessianTree(pb, nx, nx, nxp, nxp, eta=eta, device=0) for pb in parts]
    bt = torch.from_numpy(np.random.default_rng(a.seed + 1).standard_normal((nb, nx, nx))).cuda(0)
    hess.cg(bt)
    t_n, sol_n = timed(lambda: hess.cg(bt), sync)
    P.tree_cg(one, bt, None, 1e-3, 300, 1)
    t_1, (sol_1, info_1) = timed(lambda: P.tree_cg(one, bt, None, 1e-3, 300, 1), sync)
    rel = float(torch.linalg.vector_norm(sol_n - sol_1) / torch.linalg.vector_norm(sol_1))
    res = dict(gpus=ndev, spread_solve_ms=round(t_n * 1e3, 3), one_gpu_solve_ms=round(t_1 * 1e3, 3),
               spread_speedup=round(t_1 / t_n, 2), spread_iters=hess.last_cg_info["iters"].tolist(),
               one_gpu_iters=info_1["iters"].tolist(), spread_vs_one_rel_l2=float(f"{rel:.3g}"))
    for t in one:
        t.close()
    pool.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nband", type=int, default=8)
    ap.add_argument("--npart", type=int, default=2)
    ap.add_argument("--nx", type=int, default=4096)
    ap.add_argument("--nx-psf", type=int, default=5760)
    ap.add_argument("--sigma", type=float, default=3.0, help="PSF main-lobe sigma in pixels (band 0, partition 0)")
    ap.add_argument("--eta", type=float, default=1e-3, help="ridge term as a fraction of the largest eigenvalue bound")
    ap.add_argument("--k1", type=int, default=2)
    ap.add_argument("--k2", type=int, default=6)
    ap.add_argument("--host-bands", type=int, default=2, help="bands the host loop is timed on")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--multi", action="store_true", help="(internal) the multi-GPU solve comparison only")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if a.multi:
        print(json.dumps(run_multi(a)))
        return
    from psf_idot_bench import card

    name, plim = card()
    multi = None
    if gpu_count() > 1:
        argv = [sys.executable, os.path.abspath(__file__), "--multi"] + [f"--{k.replace('_', '-')}={v}" for k, v in
                                                                          vars(a).items() if k not in ("multi", "out")]
        out = subprocess.run(argv, capture_output=True, text=True)
        multi = json.loads(out.stdout.strip().splitlines()[-1]) if out.returncode == 0 else dict(error=out.stderr[-2000:])
    os.environ["CUDA_VISIBLE_DEVICES"] = os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]
    runs = [run_single(a, distinct) for distinct in (False, True)]
    res = dict(tool="deconv_hess_bench", device=name, power_limit=plim, nband=a.nband, npart=a.npart, nx=a.nx,
               ny=a.nx, nx_psf=a.nx_psf, ny_psf=a.nx_psf, dtype="float64", k1=a.k1, k2=a.k2, runs=runs,
               multi_gpu=multi if multi is not None else "not measured (one visible GPU)")
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
