#!/usr/bin/env python
"""bench.py — Mvis/s per Hessian apply (degrid + grid) on synthetic MeerKAT-like bands.

Contract (see README / DESIGN.md §measurement):
  python bench.py --gpus N --steps K --warmup W            our arm (B200 kernels)
  python bench.py --impl reference --gpus N ...           CPU arm (oracle port; ducc0 unavailable)
  python bench.py ... --dump-outputs DIR                    also write what the last timed step computed (DIR/*.npy)
One JSON line on stdout from rank 0.  N>1 is launched with torch.distributed.run, one rank per GPU.
Multi-band workloads (c2) are ONE job whose bands are partitioned over the N GPUs (strong scaling:
longest-processing-time-first assignment, then the plane transforms of the heaviest bands are offloaded
to the least loaded GPUs over NVLink peer memory, pfb_imaging_b200/split.py); --replicas runs the
round-1 mode instead (every GPU owns a complete job, weak scaling).
"""
import argparse
import json
import os

# The helper side of a plane offload spins on flags in device memory while the same GPU runs its own band on other
# streams: every stream needs its own hardware queue, or the band's kernels line up behind a waiting helper kernel
# (the default of 8 connections aliases streams).  Must be set before the CUDA context exists.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]/[2] geometry, one band per GPU (BASELINE.md C2/C3)
    "c2": dict(nx=4096, ntime=775, nchan=16, precision="single", epsilon=1e-5, nbands=8,
               name="pfb grid/sara C2: 8 bands x 4096^2, 25.0M vis/band (200M vis), MeerKAT-like, fp32, eps=1e-5"),
    # configs[0]: the reference's own CPU-runnable case
    "c1": dict(nx=2048, ntime=62, nchan=8, precision="double", epsilon=1e-5,
               name="C1: 2048^2, 1.0M vis, fp64, eps=1e-5, single band"),
    # pfb's production default: double precision, epsilon=1e-7 (core/grid.py:50), C2 geometry
    "c2d": dict(nx=4096, ntime=775, nchan=16, precision="double", epsilon=1e-7,
                name="C2 geometry in fp64 at pfb's default eps=1e-7: 4096^2, 25.0M vis/band"),
    # configs[3]: wide field, 16 bands x 10240^2, 62.5 M vis per band (1 G vis); the field is twice as wide as
    # config 2's (finer cells AND more of them), which is what multiplies the w-planes.  The bands of a GPU take
    # turns on shared plane stacks (wgridder.StackArena): 62 GB of planes per band would not fit 16 times
    "c4": dict(nx=10240, ntime=1938, nchan=16, precision="single", epsilon=1e-5, nbands=16, nband_total=16,
               cell_div=1.25, share_stack=True,
               name="wide field C4: 16 bands x 10240^2, 62.5M vis/band (1.0G vis), MeerKAT-like, fp32, eps=1e-5, "
                    "plane stacks shared by the bands of a GPU"),
    # configs[2]: pfb sara, the backward step of the deconvolution: primal-dual iterations (Psi^T, l21 dual update with
    # the cross-band all-reduce, Psi, PSF-convolution Hessian gradient, positivity) on the device, bands over the GPUs
    "c3": dict(nx=4096, nbands=8, nlevel=3, bases=("self", "db1", "db2", "db3"), precision="double",
               name="pfb sara C3: 8 bands x 4096^2, primal-dual iterations with bases self,db1,db2,db3 x 3 levels, "
                    "PSF-convolution Hessian at 5760^2, fp64, NCCL all-reduce of the l21 band sum"),
    # configs[4]: pfb hci, 1024 high-cadence snapshots of 512^2 (utils/stokes2im.py:635-683: sigma_min = 2,
    # divide_by_n = True; tests/test_hci.py:33-34: single precision, epsilon 1e-4), batched
    "c5": dict(nx=512, nsnap=1024, nchan=16, precision="single", epsilon=1e-4, chunk=256, band=4,
               name="pfb hci C5: 1024 snapshots x 512^2, 2016 baselines x 16 channels each (33.0M vis), fp32, eps=1e-4, "
                    "sigma_min=2, divide_by_n, batched 256 snapshots per launch sequence"),
}


def algorithmic_bytes(info, nvis, nchan, p):
    """SURVEY.md §8(d): B = nvis(5p+2+48/nchan) + 2 P (6 nu nv 2p + 3 nx ny p)."""
    P, nu, nv, nx, ny = info["nplanes"], info["nu"], info["nv"], info["nx"], info["ny"]
    return nvis * (5 * p + 2 + 48.0 / nchan) + 2.0 * P * (6.0 * nu * nv * 2 * p + 3.0 * nx * ny * p)


def spread_kernel_bytes(info, nvis, nchan, p):
    """Algorithmic bytes of one launch of the gridding (spreading) kernel: compulsory visibility
    traffic (uvw 24/nchan + sorted index 4 + wgt p + vis 2p per sample) plus the plane stack
    written once (SURVEY §8d: "grid written once by the spreader": P nu nv 2p)."""
    P, nu, nv = info["nplanes"], info["nu"], info["nv"]
    return nvis * (3 * p + 4 + 24.0 / nchan) + 1.0 * P * nu * nv * 2 * p


class ClockSampler(threading.Thread):
    def __init__(self, dev):
        super().__init__(daemon=True)
        self.dev, self.samples, self.reasons, self.stop_flag = dev, [], set(), False
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.dev}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def make_inputs(cfg, band, with_vis=False):
    from pfb_imaging_b200 import synth

    d = synth.make_band(cfg["ntime"], cfg["nchan"], band=band, nband=cfg.get("nband_total", 8), precision=cfg["precision"],
                        with_vis=with_vis)
    cell = synth.default_cell(d["uvw"], 1712e6) / cfg.get("cell_div", 1.0)  # one cell size for all bands (top of L-band)
    rdt = np.float32 if cfg["precision"] == "single" else np.float64
    x = synth.point_source_image(cfg["nx"], cfg["nx"], dtype=rdt)
    return d, cell, x


DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays, nout):
    """--dump-outputs: write each array (torch tensor or numpy, float32 / float64) as out_dir/<name>.npy.  `nout` arrays
    share DUMP_BYTES; an array larger than its share is written as a fixed seeded sample of its flattened elements (the
    same positions in every run), so that two builds can be compared output for output."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    positions = {}  # (numel, k) -> sorted sample positions, drawn once for all arrays of that size
    for name, a in arrays.items():
        t = torch.as_tensor(a)
        assert t.dtype in (torch.float32, torch.float64), (name, t.dtype)
        k = (DUMP_BYTES // nout - 4096) // t.element_size()  # (4096: room for the .npy header)
        if t.numel() > k:
            if (t.numel(), k) not in positions:  # (at most k distinct positions, without a permutation of all numel)
                idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), k))
                positions[t.numel(), k] = torch.from_numpy(idx)
            t = t.reshape(-1)[positions[t.numel(), k].to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def cpu_hessian_sample(cfg, band, row_step, nthreads_note=True):
    """Time the CPU restatement (oracle/cwgridder) on a bounded sample: the plane work (FFTs, screens)
    in full, the per-visibility loops on every `row_step`-th row; extrapolate the latter."""
    from oracle import cwgridder as cw
    from pfb_imaging_b200.plan import make_plan, w_range

    cw.set_threads()  # every host core, whatever OMP_NUM_THREADS torchrun exported
    d, cell, x = make_inputs(cfg, band)
    uvw, freq = d["uvw"], d["freq"]
    wmin, wmax = w_range(uvw, freq)
    nvis_full = uvw.shape[0] * freq.size
    plan = make_plan(nx=cfg["nx"], ny=cfg["nx"], pixsize_x=cell, pixsize_y=cell, epsilon=cfg["epsilon"], flip_v=True,
                     divide_by_n=False, sigma_min=1.1, sigma_max=3.0, precision=cfg["precision"], wmin=wmin, wmax=wmax,
                     nvis=nvis_full)
    sub = uvw[::row_step]
    wgt = d["wgt"][::row_step].astype(np.float64)
    mask = d["mask"][::row_step]
    nvis_s = sub.shape[0] * freq.size
    from oracle import wgridder_np as wg

    wg._image_factors(plan)  # plan-level constants: set-up, not part of an apply (same on the GPU side)
    t0 = time.perf_counter()
    b = cw._bin(plan, sub, freq, mask)
    t_bin = time.perf_counter() - t0
    td, tg = {}, {}
    mv = cw.dirty2vis_c(plan, sub, freq, x.astype(np.float64), mask, b=b, timings=td)
    img = cw.vis2dirty_c(plan, sub, freq, mv, wgt, mask, b=b, timings=tg)
    scale = nvis_full / nvis_s
    t_planes = td["planes"] + tg["planes"]
    t_vis = (td["vis"] + tg["vis"] + td["prep"] + tg["prep"]) * scale
    t_full = t_planes + t_vis
    return dict(value=nvis_full / t_full / 1e6, t_full=t_full, t_planes=t_planes, t_vis_sample=t_vis / scale,
                t_bin_sample=t_bin, nvis_sample=nvis_s, nvis_full=nvis_full, cores=cw.nthreads(),
                plan=dict(W=plan.W, sigma=plan.sigma, nu=plan.nu, nplanes=plan.nplanes), image=img)


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps  # each step = one Hessian apply of band 0 on the host (seconds of CPU work)
    vals, last = [], None
    for it in range(min(args.warmup, 1) + steps):
        last = cpu_hessian_sample(cfg, 0, args.cpu_row_step)
        if it >= min(args.warmup, 1):
            vals.append(last["value"])
    if args.dump_outputs:  # (fp64; with --cpu-row-step n > 1 the image of every n-th row only)
        name = "hessian_band0" if args.cpu_row_step == 1 else f"hessian_band0_rows_every{args.cpu_row_step}"
        dump_outputs(args.dump_outputs, {name: last["image"]}, 1)
    v = float(np.mean(vals))
    how = ("all rows" if args.cpu_row_step == 1 else
           f"every {args.cpu_row_step}th row for the per-visibility loops ({last['nvis_sample']} vis, extrapolated)")
    sample = (f"band 0 of the workload ({last['nvis_full']} vis), {how}; plane FFTs/screens at full size; fp64 C/OpenMP "
              f"restatement + scipy.fft on {last['cores']} threads (the port computes in fp64 whatever the workload's "
              f"dtype; ducc0 itself is not installable here, parity with it is unpinned)")
    line = {
        "impl": "reference", "metric": "Mvis/s per Hessian apply (degrid+grid)", "value": v, "unit": "Mvis/s",
        "n_gpus": args.gpus, "steps": len(vals), "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * last["t_full"],
        "higher_is_better": True, "scaling": "strong" if cfg.get("nbands", 1) > 1 and not args.replicas else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["name"], "plan": last["plan"]},
        "cpu_baseline": {"value": v, "unit": "Mvis/s", "cores": last["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "Mvis/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)



def run_c3(args, cfg):
    """BASELINE configs[2]: `steps` primal-dual iterations of the SARA backward step, everything resident on the
    device, the bands of ONE job dealt to the ranks (strong scaling); the l21 band sum is the NCCL all-reduce
    north_star names.  A step is one iteration; the end-to-end number is a whole `solve()` call from host arrays."""
    import torch

    from pfb_imaging_b200 import _lib, dist
    from pfb_imaging_b200.plan import good_size
    from pfb_imaging_b200.psf import HessPSF, PsfGradient
    from pfb_imaging_b200.sara import L21, PrimalDual, PsiNocopyt

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init()
    rank = dist.rank()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    nx = ny = cfg["nx"]
    nxp = nyp = good_size(int(1.4 * nx))
    bands = dist.local_bands(cfg["nbands"])
    nb = len(bands)
    bases = list(cfg["bases"])
    rng = np.random.default_rng(100 + rank)
    xx = np.fft.fftfreq(nxp)[:, None] * nxp
    yy = np.fft.rfftfreq(nyp)[None, :] * nyp
    abspsf = np.stack([np.exp(-2.0 * (np.pi * (1.5 + 0.2 * b)) ** 2 * ((xx / nxp) ** 2 + (yy / nyp) ** 2)) for b in bands])
    truth = np.zeros((nb, nx, ny))
    truth[:, rng.integers(0, nx, 200), rng.integers(0, ny, 200)] = np.exp(rng.standard_normal(200))
    hess = HessPSF(nx, ny, abspsf, beam=None, eta=1e-3)
    dirty = hess.dot(truth) + 1e-3 * rng.standard_normal(truth.shape)
    psi = PsiNocopyt(nb, nx, ny, bases, cfg["nlevel"], 1, device=local)
    reg = L21(psi, bases, nu=len(bases))
    hooks = dict(reduce_tensor=dist.allreduce_sum, reduce_scalars=dist.allreduce_sum) if world > 1 else {}
    pd = PrimalDual(tol=0.0, maxit=max(args.warmup, 3), verbosity=0, positivity=1, **hooks)
    pd.setup(reg, 1.0 + 1e-3)
    pd.set_grad(PsfGradient(hess, dirty))
    x0 = np.zeros_like(dirty)
    pd.solve(x0, 1e-4)  # warm-up iterations (allocations, first launches)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    launches0 = _lib.load().pfbg_launch_count()
    # a solve() call = upload of weights / start model, K iterations, download of the model: two calls of different
    # length separate the per-iteration cost (device-resident `value`) from the per-call copies (`e2e`)
    times = {}
    nshort = 5
    for n in (nshort, nshort + args.steps):
        pd.maxit = n
        pd.reset()
        barrier()
        t0 = time.perf_counter()
        x = pd.solve(x0, 1e-4)
        torch.cuda.synchronize()
        times[n] = time.perf_counter() - t0
    launches = _lib.load().pfbg_launch_count() - launches0
    sampler.stop_flag = True
    sampler.join()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {f"model_band{b}": x[i] for i, b in enumerate(bands)}, cfg["nbands"])
    ms_it = (times[nshort + args.steps] - times[nshort]) / args.steps * 1e3
    t = torch.tensor([ms_it, times[nshort + args.steps] * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.allreduce_max(t)
    ms_it, ms_call = float(t[0].item()), float(t[1].item())
    split = {}
    if rank == 0:
        x_t = torch.from_numpy(np.ascontiguousarray(x)).to(dev)
        v_t = torch.empty(psi.coeff_shape, dtype=torch.float64, device=dev)
        o_t = torch.empty_like(x_t)
        grad = PsfGradient(hess, dirty)

        def timed(fn, n=5):
            fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n

        split = {"psi_dot_ms": timed(lambda: psi.dot_dev(x_t, v_t)), "psi_hdot_ms": timed(lambda: psi.hdot_dev(v_t, o_t)),
                 "psf_hessian_grad_ms": timed(lambda: grad.device_apply(x_t, o_t))}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        ncoef = int(np.prod(psi.coeff_shape))
        # compulsory traffic of Psi^T + Psi on rank 0: the coefficient cube written once and read once (fp64), the image
        # cube read and written once each way
        psi_bytes = 2.0 * ncoef * 8 + 4.0 * nb * nx * ny * 8
        psi_ms = split["psi_dot_ms"] + split["psi_hdot_ms"]
        line = {
            "metric": "primal-dual iterations/s (SARA backward step, config 3)", "value": 1e3 / ms_it, "unit": "iterations/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3) + nshort, "ms_per_step": ms_it,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["name"], "bands_total": cfg["nbands"], "bands_on_rank0": list(bands),
                       "nx_psf": nxp, "coefficients_rank0": ncoef,
                       "l2": "inputs larger than L2 (coefficient cube %.1f GB on rank 0)" % (ncoef * 8 / 1e9),
                       "collective": ("NCCL all-reduce (SUM) of the (nbasis, nymax, nxmax) l21 band sum + 2 doubles per iteration"
                                      if world > 1 else "none (all bands on one GPU)"),
                       "parallelism": f"{cfg['nbands']} bands of ONE job over {world} GPU(s)"},
            "e2e": {"value": (nshort + args.steps) / (ms_call * 1e-3), "unit": "iterations/s",
                    "h2d_bytes_per_step": int(2 * x0.nbytes / (nshort + args.steps)),
                    "d2h_bytes_per_step": int(x0.nbytes / (nshort + args.steps)),
                    "call": f"PrimalDual.solve(x0 host cube, ...) -> host model, {nshort + args.steps} iterations per call (opt/primal_dual.py:284-448)"},
            "gpu_launches": int(launches), "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "kernel": "Psi + Psi^T (db1-db3 x 3 levels wavelet analysis / synthesis, pfbs_psi_dot / pfbs_psi_hdot)",
                         "achieved": psi_bytes / (psi_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": psi_bytes / (psi_ms * 1e-3) / 1e9 / peak, "traffic": None,
                         "rank0_split_ms": split,
                         "note": "achieved = compulsory bytes of one Psi^T + Psi pair on rank 0 over their time"},
            "cpu_baseline": None,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def run_c5(args, cfg):
    """Batched small-image workload (BASELINE configs[4]): the snapshots of one job are dealt round-robin to the
    ranks; every rank images its share in batches of cfg["chunk"] snapshots (one bin / sort and one launch of every
    kernel per batch)."""
    import torch
    import torch.distributed as dist

    from pfb_imaging_b200 import _lib, synth, wgridder as W

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    nx, nsnap, nchan, chunk = cfg["nx"], cfg["nsnap"], cfg["nchan"], cfg["chunk"]
    rng = np.random.default_rng(1234)
    enu = synth.meerkat_like_antennas(rng)
    uvw_all = synth.uvw_tracks(enu, nsnap)  # time-major: rows [t * nbl, (t+1) * nbl) are snapshot t
    nbl = uvw_all.shape[0] // nsnap
    freq = synth.band_freqs(cfg["band"], 8, nchan)
    cell = synth.default_cell(uvw_all, 1712e6)
    mine = list(range(rank, nsnap, world))
    brng = np.random.default_rng([5, rank])
    geom = dict(npix_x=nx, npix_y=nx, pixsize_x=cell, pixsize_y=cell, epsilon=cfg["epsilon"], flip_v=True,
                divide_by_n=True, sigma_min=2.0, sigma_max=2.6, precision=cfg["precision"])
    batches = []
    for c0 in range(0, len(mine), chunk):
        ids = mine[c0:c0 + chunk]
        uvw = [uvw_all[t * nbl:(t + 1) * nbl] for t in ids]
        wgt = brng.uniform(0.5, 1.5, (len(ids) * nbl, nchan)).astype(np.float32)
        gp = W.batch_plan_for(uvw, freq, device=local, **geom)
        gp.bind_weights(wgt)
        x = np.zeros((len(ids), nx, nx), np.float32)
        for k in range(len(ids)):
            x[k] = synth.point_source_image(nx, nx, nsrc=20, seed=ids[k], dtype=np.float32)
        x_d = torch.from_numpy(x).to(dev)
        batches.append(dict(ids=ids, uvw=uvw, wgt=wgt, gp=gp, x=x, x_d=x_d, out_d=torch.empty_like(x_d),
                            wsum=float(wgt.sum(dtype=np.float64)), nvis=len(ids) * nbl * nchan, info=gp.info()))
    nvis_local = sum(b["nvis"] for b in batches)
    stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_dev():
        for b in batches:
            b["gp"].hessian_dev(b["x_d"].data_ptr(), None, b["wsum"], 0.0, b["out_d"].data_ptr(), stream)

    for _ in range(max(args.warmup, 3)):
        step_dev()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = _lib.load().pfbg_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step_dev()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = _lib.load().pfbg_launch_count() - launches0
    sampler.stop_flag = True
    sampler.join()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {f"hessian_rank{rank}_batch{i}": b["out_d"] for i, b in enumerate(batches)},
                     world * len(batches))
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    nv = torch.tensor([float(nvis_local)], dtype=torch.float64, device=dev)
    la = torch.tensor([float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(nv, op=dist.ReduceOp.SUM)
        dist.all_reduce(la, op=dist.ReduceOp.SUM)
    ms_step = float(t.item()) / args.steps
    value = float(nv.item()) / (ms_step * 1e-3) / 1e6
    # phases of the first batch
    names = ["stage_in", "pad_screen_fft", "degrid", "zero_grid", "spread", "fft_crop_screen", "stage_out"]
    b0 = batches[0]
    b0["gp"].set_profiling(True)
    rec = []
    for _ in range(3):
        b0["gp"].hessian_dev(b0["x_d"].data_ptr(), None, b0["wsum"], 0.0, b0["out_d"].data_ptr(), stream)
        torch.cuda.synchronize()
        rec.append(b0["gp"].timings())
    b0["gp"].set_profiling(False)
    phases = dict(zip(names, np.median(np.array(rec), axis=0).tolist()))
    # ---- end to end: host cubes in and out through the bound batch plans (the apply a solver makes) -----------
    outs = [np.empty_like(b["x"]) for b in batches]
    for _ in range(2):
        for b, o in zip(batches, outs):
            b["gp"].hessian(b["x"], wsum=b["wsum"], out=o)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for b, o in zip(batches, outs):
            b["gp"].hessian(b["x"], wsum=b["wsum"], out=o)
    torch.cuda.synchronize()
    te = torch.tensor([(time.perf_counter() - t0) / args.steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = float(nv.item()) / float(te.item()) / 1e6
    img_bytes = int(sum(b["x"].nbytes for b in batches)) * world
    # ---- the hci pattern itself: one-shot imaging of snapshots from host arrays (bind + residual + PSF), batched
    # against one pooled vis2dirty call pair per snapshot (what round 1 offered) --------------------------------
    one_shot = None
    if rank == 0:
        b = batches[0]
        ns = min(64, len(b["ids"]))
        cdt = np.complex64
        vis = [(brng.standard_normal((nbl, nchan)) + 1j * brng.standard_normal((nbl, nchan))).astype(cdt) for _ in range(ns)]
        ones = [np.ones((nbl, nchan), cdt) for _ in range(ns)]
        wl = [b["wgt"][k * nbl:(k + 1) * nbl] for k in range(ns)]
        com = dict(freq=freq, npix_x=nx, npix_y=nx, pixsize_x=cell, pixsize_y=cell, epsilon=cfg["epsilon"], flip_v=True,
                   divide_by_n=True, sigma_min=2.0, sigma_max=2.6)
        for _ in range(2):
            cube, psf = W.vis2dirty_batch(uvw=b["uvw"][:ns], vis=vis, wgt=wl, extra_vis=(ones,), **com)
        t0 = time.perf_counter()
        cube, psf = W.vis2dirty_batch(uvw=b["uvw"][:ns], vis=vis, wgt=wl, extra_vis=(ones,), **com)
        t_batch = (time.perf_counter() - t0) / ns
        for k in range(2):
            W.vis2dirty(uvw=b["uvw"][k], vis=vis[k], wgt=wl[k], **com)
        t0 = time.perf_counter()
        for k in range(ns):
            d1 = W.vis2dirty(uvw=b["uvw"][k], vis=vis[k], wgt=wl[k], **com)
            W.vis2dirty(uvw=b["uvw"][k], vis=ones[k], wgt=wl[k], **com)
        t_single = (time.perf_counter() - t0) / ns
        err = float(np.linalg.norm(cube[ns - 1] - d1) / np.linalg.norm(d1))
        one_shot = {"snapshots": ns, "ms_per_snapshot_batched": 1e3 * t_batch, "ms_per_snapshot_pooled_one_shot_calls": 1e3 * t_single,
                    "speedup": t_single / t_batch, "batched_vs_one_shot_rel_l2": err,
                    "what": "residual + PSF image of a snapshot from host arrays (bind, grid twice, images back), as utils/stokes2im.py:635-683"}
        W.clear_plan_pool()
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        info = b0["info"]
        B = sum(algorithmic_bytes(dict(bb["info"], nx=nx, ny=nx), bb["nvis"], nchan, 4) for bb in batches)
        my_ms = ms_total / args.steps
        kb = spread_kernel_bytes(info, b0["nvis"], nchan, 4)
        line = {
            "metric": "Mvis/s per Hessian apply (degrid+grid)", "value": value, "unit": "Mvis/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["name"], "snapshots_total": nsnap, "snapshots_rank0": len(mine),
                       "batches_rank0": len(batches), "nvis_total": int(nv.item()),
                       "us_per_snapshot_apply": 1e3 * ms_step / (nsnap / world) ,
                       "l2": "inputs larger than L2 (plane stack %.1f GB per batch)" % (info["grid_bytes"] / 1e9),
                       "plan": {k: info[k] for k in ("W", "sigma", "nu", "nv", "nplanes", "beta")},
                       "parallelism": f"snapshots dealt round-robin to {world} GPU(s), no data-path collective",
                       "one_shot_snapshot_imaging": one_shot},
            "e2e": {"value": e2e_value, "unit": "Mvis/s", "h2d_bytes_per_step": img_bytes, "d2h_bytes_per_step": img_bytes,
                    "call": "GridderPlan.hessian(x (nsnap, nx, ny) host numpy, out=) on the bound batch plans, batch after batch"},
            "gpu_launches": int(la.item()), "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "kernel": "k_grid_runs (spreading kernel, one launch per batch of snapshots)",
                         "achieved": kb / (phases["spread"] * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": kb / (phases["spread"] * 1e-3) / 1e9 / peak, "traffic": None,
                         "kernel_ms": phases["spread"], "algorithmic_bytes_per_launch": kb,
                         "step_algorithmic_bytes_rank0": B, "step_frac": B / (my_ms * 1e-3) / 1e9 / peak,
                         "phases_ms_first_batch": phases,
                         "note": "small-image workload: 1024-point transforms, W = 6 (general flush path of the run kernels)"},
            "cpu_baseline": None,
        }
        print(json.dumps(line), flush=True)
    for b in batches:
        b["gp"].close()
    if world > 1:
        dist.destroy_process_group()


def run_ours(args, cfg):
    import torch
    import torch.distributed as dist

    from pfb_imaging_b200 import _lib, operators as ops, split as bsplit, synth, wgridder as W
    from pfb_imaging_b200.plan import make_plan, w_range

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner (NCCL_DEBUG=VERSION / WARN) to stdout; rank 0 must print ONE JSON line there
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    p = 4 if cfg["precision"] == "single" else 8
    job_bands = list(range(cfg.get("nbands", 1)))
    if args.bands:
        job_bands = [int(b) for b in args.bands.split(",")]
    nbands = len(job_bands)
    # Default for a multi-band workload on N > 1 GPUs: ONE job, its bands partitioned over the ranks (strong scaling,
    # what north_star specifies).  --replicas: every GPU owns a complete job (weak scaling, the round-1 mode).
    strong = nbands > 1 and world > 1 and not args.replicas

    def gather_obj(obj):
        if world == 1:
            return [obj]
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    owner = None
    if strong:
        probe, cell0, _ = make_inputs(cfg, job_bands[0])
        est = []
        for b in job_bands:
            fr = synth.band_freqs(b, cfg.get("nband_total", 8), cfg["nchan"])
            wmin, wmax = w_range(probe["uvw"], fr)
            pl = make_plan(nx=cfg["nx"], ny=cfg["nx"], pixsize_x=cell0, pixsize_y=cell0, epsilon=cfg["epsilon"],
                           flip_v=True, divide_by_n=False, sigma_min=1.1, sigma_max=3.0, precision=cfg["precision"],
                           wmin=wmin, wmax=wmax, nvis=probe["uvw"].shape[0] * cfg["nchan"])
            est.append(pl.est_cost)
        owner = bsplit.lpt_assign(est, world)  # index into job_bands -> rank
        my_bands = [b for i, b in enumerate(job_bands) if owner[i] == rank]
    else:
        my_bands = list(job_bands) if nbands > 1 else [rank % 8]

    def bind_band(b, **extra):
        d, cell, x = make_inputs(cfg, b)
        gp = W.plan_for(d["uvw"], d["freq"], npix_x=cfg["nx"], npix_y=cfg["nx"], pixsize_x=cell, pixsize_y=cell,
                        epsilon=cfg["epsilon"], flip_v=True, divide_by_n=False, precision=cfg["precision"],
                        mask=d["mask"], sigma_min=1.1, sigma_max=3.0, device=local,
                        external_stack=bool(cfg.get("share_stack")), **extra)
        gp.bind_weights(d["wgt"])
        x_d = torch.from_numpy(x).to(dev)
        return dict(b=b, d=d, cell=cell, x=x, gp=gp, x_d=x_d, out_d=torch.empty_like(x_d), info=gp.info(),
                    wsum=float(d["wgt"].sum(dtype=np.float64)), nvis=d["uvw"].shape[0] * d["freq"].size)

    bands = [bind_band(b) for b in my_bands]
    if cfg.get("share_stack") and bands:
        # the bands of this GPU take turns on one shared plane stack: a band whose cheapest plan needs a larger stack
        # than what is left next to the bound data of all of them is planned again under that limit
        # (make_plan(max_stack_bytes=))
        torch.cuda.synchronize()
        free_b, _tot = torch.cuda.mem_get_info(dev)
        # (what the first Hessian apply still allocates per band: the bucket-ordered model visibilities)
        limit = int(free_b) - sum(bd["nvis"] for bd in bands) * 2 * p - (6 << 30)
        for i, bd in enumerate(bands):
            if int(bd["info"]["grid_bytes"]) > limit:
                bd["gp"].close()
                del bd["x_d"], bd["out_d"]
                bands[i] = bind_band(bd["b"], max_stack_bytes=limit)
    nvis_local = sum(bd["nvis"] for bd in bands)
    stream = torch.cuda.current_stream().cuda_stream
    arena = None
    if cfg.get("share_stack") and bands:
        # two stacks (one per compute stream) when they fit next to everything else that is resident, else one
        need = max(int(bd["info"]["grid_bytes"]) for bd in bands)
        free_b, _tot = torch.cuda.mem_get_info(dev)
        arena = W.StackArena([bd["gp"] for bd in bands], nslots=2 if free_b > 2 * need + (24 << 30) else 1, device=local)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- per-phase timing of every band on its own (events inside the library, same stream): the input of the
    # offload schedule and of the roofline section ------------------------------------------------------------
    names = ["stage_in", "pad_screen_fft", "degrid", "zero_grid", "spread", "fft_crop_screen", "stage_out"]
    phases = dict.fromkeys(names, 0.0)
    per_band, band_stats = {}, {}
    for bd in bands:
        gp = bd["gp"]
        for _ in range(2):
            gp.hessian_dev(bd["x_d"].data_ptr(), None, bd["wsum"], 0.0, bd["out_d"].data_ptr(), stream)
        gp.set_profiling(True)
        rec = []
        for _ in range(3):
            gp.hessian_dev(bd["x_d"].data_ptr(), None, bd["wsum"], 0.0, bd["out_d"].data_ptr(), stream)
            torch.cuda.synchronize()
            rec.append(gp.timings())
        gp.set_profiling(False)
        ph = np.median(np.array(rec), axis=0).tolist()
        bd["phases"] = dict(zip(names, ph))
        per_band[bd["b"]] = round(float(sum(ph)), 3)
        band_stats[bd["b"]] = dict(ms=float(sum(ph)), P=int(bd["info"]["nplanes"]),
                                   t_plane=float(bd["phases"]["pad_screen_fft"] + bd["phases"]["fft_crop_screen"]) /
                                   int(bd["info"]["nplanes"]))
        for k, v in zip(names, ph):
            phases[k] += v
    all_stats = {}
    for dct in gather_obj(band_stats):
        all_stats.update(dct)

    # ---- strong scaling: offload planes of the heaviest bands to the least loaded GPUs -----------------------
    offloads, model_loads, split = {}, None, None
    if strong:
        costs = [all_stats[b]["ms"] for b in job_bands]
        tpl = [all_stats[b]["t_plane"] for b in job_bands]
        npl = [all_stats[b]["P"] for b in job_bands]
        off_idx, model_loads = (({}, None) if args.no_offload or cfg.get("share_stack") else
                                bsplit.plan_offloads(costs, tpl, npl, owner, world))  # (lent stacks are not exported to helpers)
        offloads = {job_bands[i]: o for i, o in off_idx.items()}
        if offloads:
            split = bsplit.BandSplit({bd["b"]: bd["gp"] for bd in bands}, offloads, rank, local, gather_obj)
    # helper work runs on its own high-priority stream(s): its CTAs go first whenever an SM frees up, so the owner
    # of the heavy band never waits for a helper that is busy with its own band
    hstreams = {b: torch.cuda.Stream(dev, priority=-1) for b in (split.helpers if split else {})}
    # the bands of a GPU are independent: they alternate between two compute streams, so the tail of one band's
    # kernels overlaps the head of the next band's (measured: 100.4 -> 89.5 ms for the 8 bands of C2; more than
    # two streams bring nothing).  Every step forks from / joins the current stream, where the events are recorded.
    cstreams = [torch.cuda.Stream(dev) for _ in range(2)] if len(bands) > 1 and (arena is None or arena.nslots > 1) else []

    def step_dev():
        cur = torch.cuda.current_stream()
        for hs in hstreams.values():
            hs.wait_stream(cur)
        if split:
            split.serve({b: hs.cuda_stream for b, hs in hstreams.items()})
        if not cstreams:
            for bd in bands:
                bd["gp"].hessian_dev(bd["x_d"].data_ptr(), None, bd["wsum"], 0.0, bd["out_d"].data_ptr(), stream)
        else:
            for cs in cstreams:
                cs.wait_stream(cur)
            for i, bd in enumerate(bands):
                bd["gp"].hessian_dev(bd["x_d"].data_ptr(), None, bd["wsum"], 0.0, bd["out_d"].data_ptr(),
                                     cstreams[i % 2].cuda_stream)
            for cs in cstreams:
                cur.wait_stream(cs)
        for hs in hstreams.values():
            cur.wait_stream(hs)

    # ---- device-resident timing -------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        step_dev()
    barrier()
    if split:
        split.check()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = _lib.load().pfbg_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step_dev()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = _lib.load().pfbg_launch_count() - launches0
    sampler.stop_flag = True
    sampler.join()
    if split:
        split.check()
    if args.dump_outputs and (strong or rank == 0):  # (one job per GPU: rank 0's job)
        dump_outputs(args.dump_outputs, {f"hessian_band{bd['b']}": bd["out_d"] for bd in bands},
                     nbands if strong else len(bands))
    ms_ranks = [float(v) / args.steps for v in gather_obj(ms_total)]
    launches_all = int(sum(gather_obj(int(launches))))
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    nvis_all = torch.tensor([float(nvis_local)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(nvis_all, op=dist.ReduceOp.SUM)
    value = float(nvis_all.item()) / (ms_step * 1e-3) / 1e6
    helper_phases = {}
    if split:  # one more (untimed) step with library events on the helper plans: where the helper's time goes
        for h in split.helpers.values():
            h.set_profiling(True)
        step_dev()
        torch.cuda.synchronize()
        for b, h in split.helpers.items():
            tm = h.timings()
            h.set_profiling(False)
            if len(tm) >= 4:
                helper_phases[b] = dict(wait_x=round(tm[0], 3), copy_x_fwd_planes=round(tm[1], 3),
                                        wait_grid=round(tm[2], 3), inv_planes_partial=round(tm[3], 3))
        barrier()
        split.check()
        barrier()
        split.close()
        split = None
        barrier()
    helper_all = {}
    for dct in gather_obj(helper_phases):
        helper_all.update(dct)

    # ---- end to end through the operator call a pfb solver makes (host numpy in/out) ------
    ops._CACHE_SIZE = max(ops._CACHE_SIZE, len(bands))
    ops.clear_plan_cache()

    def step_e2e():
        for bd in bands:
            d = bd["d"]
            ops.hessian_slice(bd["x"], xout=bd["xo"], uvw=d["uvw"], weight=d["wgt"], vis_mask=d["mask"], freq=d["freq"],
                              cell=bd["cell"], epsilon=cfg["epsilon"], wsum=bd["wsum"], flip_v=True)

    shared = bool(cfg.get("share_stack"))
    nslots = arena.nslots if arena is not None else 0
    for bd in bands:
        bd["gp"].close()  # free the device-resident plans before the operator-level cache binds its own
        bd["xo"] = np.empty_like(bd["x"])
        bd["x_d"] = bd["out_d"] = None
    arena = None
    torch.cuda.empty_cache()
    e2e_value = None
    if not shared:  # (the operator-level plan cache gives every band its own stack: not for config 4)
        for _ in range(2):
            step_e2e()  # first call binds the band (like load_band); later calls hit the plan cache
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        torch.cuda.synchronize()
        t_e2e = (time.perf_counter() - t0) / args.steps
        te = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_value = float(nvis_all.item()) / float(te.item()) / 1e6
    info = bands[0]["info"] if bands else None
    if bands and not shared:
        gp0 = ops._cached_plan(bands[0]["d"]["uvw"], bands[0]["d"]["freq"], bands[0]["d"]["mask"], bands[0]["d"]["wgt"],
                               npix_x=cfg["nx"], npix_y=cfg["nx"], pixsize_x=float(bands[0]["cell"]),
                               pixsize_y=float(bands[0]["cell"]), center_x=0.0, center_y=0.0, epsilon=float(cfg["epsilon"]),
                               flip_u=False, flip_v=True, flip_w=False, do_wgridding=True, divide_by_n=False,
                               precision=cfg["precision"])
        info = gp0.info()
    ops.clear_plan_cache()

    # ---- the same through the pool call a multi-band solver makes (band_worker.py:276-281): one host cube in,
    # one host cube out; the bands' copies overlap the neighbouring bands' kernels -----------------------------
    pool_ops = {}
    for i, bd in enumerate(bands):
        d = bd["d"]
        pool_ops[i] = ops.BandHessian(d["uvw"], d["freq"], d["wgt"], d["mask"], cfg["nx"], cfg["nx"], float(bd["cell"]),
                                      epsilon=float(cfg["epsilon"]), precision=cfg["precision"], wsum=bd["wsum"],
                                      device=local, external_stack=shared)
    pool = ops.BandPool(pool_ops, nband=len(bands), share_stacks=nslots if shared else False)
    xcube = np.stack([bd["x"] for bd in bands]) if bands else None
    e2e_pool_value = None
    t_pool = 0.0
    if bands:
        res = None
        for _ in range(3):  # same hold-one-result pattern as the timed loop (the pinned result blocks get allocated here)
            res = pool.hess_dot(xcube)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = pool.hess_dot(xcube)
        torch.cuda.synchronize()
        t_pool = (time.perf_counter() - t0) / args.steps
        assert np.isfinite(res[0, :8, :8]).all()
        del res
    tp = torch.tensor([t_pool], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tp, op=dist.ReduceOp.MAX)
    e2e_pool_value = float(nvis_all.item()) / float(tp.item()) / 1e6
    pool.close()
    img_bytes = int(sum(gather_obj(int(sum(bd["x"].nbytes for bd in bands)))))

    # ---- the path pfb's own entry points take by default: fp64, epsilon = 1e-7 (core/grid.py:50), one band ----
    f64 = None
    if world == 1 and args.workload == "c2" and not args.no_f64:
        cfg64 = WORKLOADS["c2d"]
        d, cell, x = make_inputs(cfg64, 0)
        gp = W.plan_for(d["uvw"], d["freq"], npix_x=cfg64["nx"], npix_y=cfg64["nx"], pixsize_x=cell, pixsize_y=cell,
                        epsilon=cfg64["epsilon"], flip_v=True, divide_by_n=False, precision="double", mask=d["mask"],
                        sigma_min=1.1, sigma_max=3.0, device=local)
        gp.bind_weights(d["wgt"])
        x_d = torch.from_numpy(x).to(dev)
        o_d = torch.empty_like(x_d)
        ws = float(d["wgt"].sum(dtype=np.float64))
        for _ in range(3):
            gp.hessian_dev(x_d.data_ptr(), None, ws, 0.0, o_d.data_ptr(), stream)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(5):
            gp.hessian_dev(x_d.data_ptr(), None, ws, 0.0, o_d.data_ptr(), stream)
        a1.record()
        torch.cuda.synchronize()
        ms64 = a0.elapsed_time(a1) / 5
        i64 = gp.info()
        gp.set_profiling(True)
        rec64 = []
        for _ in range(3):
            gp.hessian_dev(x_d.data_ptr(), None, ws, 0.0, o_d.data_ptr(), stream)
            torch.cuda.synchronize()
            rec64.append(gp.timings())
        gp.set_profiling(False)
        nv64 = d["uvw"].shape[0] * d["freq"].size
        ph64 = dict(zip(["stage_in", "pad_screen_fft", "degrid", "zero_grid", "spread", "fft_crop_screen", "stage_out"],
                        np.median(np.array(rec64), axis=0).tolist()))
        # the run kernels of this path are DMMA m8n8k4 contractions (csrc/runs_mma.cuh): 13.5 DMMA of 256 FMAs per
        # sample and direction; their roof is the fp64 rate of the tensor pipe (measured 37 TFLOP/s on B200)
        dmma_floor_ms = nv64 * 13.5 * 512 / 37.0e12 * 1e3
        f64 = {"workload": cfg64["name"] + " (band 0)", "value": nv64 / (ms64 * 1e-3) / 1e6,
               "unit": "Mvis/s", "ms_per_band": ms64, "dtype": "f64",
               "plan": {k: i64[k] for k in ("W", "sigma", "nu", "nv", "nplanes", "pmirror")},
               "phases_ms": ph64,
               "run_kernels": "k_degrid_runs_mma / k_grid_runs_mma (FP64 tensor cores, DMMA m8n8k4)" if 9 <= i64["W"] <= 12
                              else "scalar fp64 run kernels",
               "dmma_floor_ms_per_direction": dmma_floor_ms,
               "frac_of_dmma_roof": {"degrid": dmma_floor_ms / ph64["degrid"], "spread": dmma_floor_ms / ph64["spread"]}}
        gp.close()
        del x_d, o_d

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        nchan = cfg["nchan"]
        # SURVEY §8(d) byte model summed over rank 0's bands (plans differ slightly per band; use band-0-of-rank plan)
        B = sum(algorithmic_bytes(bd["info"], bd["nvis"], nchan, p) for bd in bands)
        # the same model with the plane count a stack WITHOUT mirror planes needs for the same |w| range (what a
        # ducc0-style gridder transforms): the work this implementation removed still counts there
        B_std = sum(algorithmic_bytes(dict(bd["info"], nplanes=bd["info"]["nplanes_std"]), bd["nvis"], nchan, p) for bd in bands)
        kernel_phase = {"spread": "k_grid_runs (spreading kernel)", "degrid": "k_degrid_runs (gathering kernel)",
                        "pad_screen_fft": "k_rows2_fwd + k_cols2 (fused pad/screen/FFT; fp64: k_rows_fwd + k_cols_fwd)",
                        "fft_crop_screen": "k_cols2 + k_rows2_inv (fused FFT/screen/crop; fp64: k_cols_inv + k_rows_inv)"}
        dom = max(kernel_phase, key=lambda k: phases.get(k, 0.0))
        # roofline of the gridding (spreading) kernel, the hand-written kernel SURVEY §8(d) models per sample
        kb = sum(spread_kernel_bytes(bd["info"], bd["nvis"], nchan, p) for bd in bands) / len(bands)
        k_ms = phases.get("spread", float("nan")) / len(bands)
        traffic, prof = None, {}
        try:  # measured counters per launch from the committed ncu --set full captures (tools/ncu_traffic.py)
            prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(args.workload, {})
            traffic = prof.get("k_grid_runs")
        except Exception:
            pass
        my_ms = ms_total / args.steps
        props = torch.cuda.get_device_properties(dev)
        nsm = int(props.multi_processor_count)
        clk = sampler.summary()
        clk_hz = 1e6 * float(clk["sm_mhz"] or clk["sm_max_mhz"] or 1965.0)
        # ---- the roofs that actually bind (ncu: every kernel sits at 6-10 % of DRAM throughput) -------------
        # run kernels: fp32/fp64 FMA pipe.  Floor = nactive * W^3 complex multiply-adds = 2 W^3 real FMAs per sample,
        # at 128 (fp32) / 64 (fp64) FMA lanes per clock and SM, against the SM count and the clock sampled above.
        binding = {}
        lanes = 128.0 if p == 4 else 64.0
        for key, ph_name, kname in (("k_grid_runs", "spread", "k_grid_runs"), ("k_degrid_runs", "degrid", "k_degrid_runs")):
            ents = []
            for bd in bands:
                Wk = bd["info"]["W"]
                fmas = 2.0 * bd["info"]["nactive"] * Wk ** (3 if bd["info"]["nplanes"] > 1 else 2)
                floor_ms = fmas / (nsm * lanes * clk_hz) * 1e3
                ents.append((floor_ms, bd["phases"][ph_name]))
            fl, km = sum(e[0] for e in ents), sum(e[1] for e in ents)
            pb = prof.get("band0", {}).get(kname, {})
            binding[key] = {"roof": f"FMA pipe: {int(lanes)} FMA lanes/clk/SM x {nsm} SMs x {clk_hz / 1e6:.0f} MHz (sampled)",
                            "floor_ms": round(fl, 3), "kernel_ms": round(km, 3), "frac_of_roof": round(fl / km, 4),
                            "floor": "2 W^3 real FMAs per active sample (the W x W x W footprint update itself)",
                            "ncu_fma_pipe_pct_band0": pb.get("fma_pipe_pct"), "ncu_issue_active_pct_band0": pb.get("issue_active_pct"),
                            "ncu_dram_pct_band0": pb.get("dram_pct")}
        # transform kernels: shared-memory data pipe, one wavefront per clock and SM; wavefronts measured by ncu
        # (bank conflicts included) on the profiled bands
        for tag, ph_name, ks in (("rows_fwd+cols_fwd", "pad_screen_fft", ("k_rows_fwd", "k_cols_fwd")),
                                 ("cols_inv+rows_inv", "fft_crop_screen", ("k_cols_inv", "k_rows_inv"))):
            for bd in bands:
                pb = prof.get("band%d" % bd["b"])
                if not pb or not all(k in pb and "smem_wavefronts" in pb[k] for k in ks):
                    continue
                wf = sum(pb[k]["smem_wavefronts"] for k in ks)
                floor_ms = wf / (nsm * clk_hz) * 1e3
                binding[f"{tag} (band {bd['b']})"] = {
                    "roof": f"shared-memory wavefronts: 1 per clk and SM x {nsm} SMs x {clk_hz / 1e6:.0f} MHz",
                    "floor_ms": round(floor_ms, 3), "kernel_ms": round(bd["phases"][ph_name], 3),
                    "frac_of_roof": round(floor_ms / bd["phases"][ph_name], 4), "ncu_smem_wavefronts": wf,
                    "ncu_bank_conflict_wavefronts": sum(pb[k].get("smem_bank_conflicts", 0) for k in ks),
                    "ncu_warps_active_pct": [pb[k].get("warps_active_pct") for k in ks]}
                break
        # measured DRAM traffic of a whole step: ncu captures of bands 0 and 7, the bands in between interpolated on
        # their plane counts
        dram_step = None
        b_lo, b_hi = prof.get("band0"), prof.get("band7")
        if b_lo and b_hi:
            t_lo = sum(v.get("dram_bytes", 0) for v in b_lo.values())
            t_hi = sum(v.get("dram_bytes", 0) for v in b_hi.values())
            P_lo, P_hi = all_stats.get(0, {}).get("P"), all_stats.get(7, {}).get("P")
            if P_lo and P_hi and P_hi != P_lo:
                tot = 0.0
                for bd in bands:
                    tot += t_lo + (t_hi - t_lo) * (bd["info"]["nplanes"] - P_lo) / (P_hi - P_lo)
                dram_step = {"bytes_rank0": tot, "achieved_GBs": tot / (my_ms * 1e-3) / 1e9,
                             "frac_of_peak": tot / (my_ms * 1e-3) / 1e9 / peak,
                             "how": "ncu dram__bytes_read+write of the six kernels, bands 0 and 7 captured (profiles/traffic.json), bands 1-6 interpolated on their plane counts"}
        roof = {
            "bound": "hbm", "kernel": "k_grid_runs (spreading kernel, one launch per band and Hessian apply)",
            "achieved": kb / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
            "frac": kb / (k_ms * 1e-3) / 1e9 / peak, "traffic": traffic, "peak_source": peak_src,
            "kernel_ms": k_ms, "algorithmic_bytes_per_launch": kb,
            "note": ("frac is SURVEY 8(d)'s algorithmic bytes of the kernel over its time against the measured HBM peak; HBM is NOT the "
                     "roof that binds this kernel (measured DRAM traffic is `traffic`, 6-10 % of peak for every kernel): see "
                     "binding_roofs for the FMA-pipe floor of the run kernels and the shared-memory floor of the transforms. "
                     "kernel_ms is the spreading phase of one band run alone (library events)"),
            "binding_roofs": binding, "measured_dram_step": dram_step,
            "step_algorithmic_bytes_rank0": B, "step_achieved_rank0": B / (my_ms * 1e-3) / 1e9,
            "step_frac": B / (my_ms * 1e-3) / 1e9 / peak, "step_frac_of_nominal_8TBs": B / (my_ms * 1e-3) / 1e9 / 8000.0,
            "step_frac_unmirrored_planes": B_std / (my_ms * 1e-3) / 1e9 / peak,
            "step_frac_note": "SURVEY 8(d) byte model (6 passes over the plane stack per direction); the fused, pruned transforms move ~6x less than that model, so step_frac measures speed against the survey's model, not HBM utilisation",
            "planes_per_band": {str(bd["b"]): [bd["info"]["nplanes"], bd["info"]["nplanes_std"]] for bd in bands},
            "dominant_phase": dom, "dominant_phase_kernels": kernel_phase[dom], "phases_ms_rank0": phases,
            "ms_per_band_rank0": per_band,
        }
        cpu = None
        if world == 1 and not args.no_cpu_baseline and not cfg.get("share_stack"):  # (c4: the fp64 host planes alone are 124 GB)
            c = cpu_hessian_sample(cfg, bands[0]["b"], args.cpu_row_step)
            how = "all rows" if args.cpu_row_step == 1 else f"every {args.cpu_row_step}th row for the per-visibility loops (extrapolated)"
            cpu = {"value": c["value"], "unit": "Mvis/s", "cores": c["cores"], "kind": "port",
                   "sample": (f"one Hessian apply of band {bands[0]['b']} ({c['nvis_full']} vis), {how}, plane FFTs at full size; fp64 "
                              f"C/OpenMP restatement + scipy.fft (ducc0 not installable: parity with it unpinned); planes "
                              f"{c['t_planes']:.1f}s, vis {c['t_vis_sample']:.1f}s")}
        line = {
            "metric": "Mvis/s per Hessian apply (degrid+grid)", "value": value, "unit": "Mvis/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            # ONE job whose bands are partitioned over the GPUs: the total work is fixed as N grows, also at N = 1
            "scaling": "strong" if (nbands > 1 and not args.replicas) else "weak", "vs_baseline": None,
            "dtype": "f32" if p == 4 else "f64",
            "data": "synthetic",
            "config": {"workload": cfg["name"], "bands_total": nbands if strong else nbands * world,
                       "bands_on_rank0": [bd["b"] for bd in bands],
                       "ms_per_band": {str(b): round(all_stats[b]["ms"], 3) for b in sorted(all_stats)},
                       "ms_per_rank": [round(v, 3) for v in ms_ranks],
                       "band_owner": ({str(b): owner[i] for i, b in enumerate(job_bands)} if strong else None),
                       "plane_offloads": {str(b): o for b, o in sorted(offloads.items())},
                       "modelled_ms_per_rank": [round(v, 3) for v in model_loads] if model_loads else None,
                       "helper_phases_ms": {str(b): v for b, v in sorted(helper_all.items())},
                       "sum_over_max_of_bands": round(sum(v["ms"] for v in all_stats.values()) /
                                                      max(v["ms"] for v in all_stats.values()), 2),
                       "nvis_total": int(nvis_all.item()),
                       "l2": "inputs larger than L2 (plane stack %.1f GB per band)" % (info["grid_bytes"] / 1e9),
                       "plan_first_band": {k: info[k] for k in ("W", "sigma", "nu", "nv", "nplanes", "nplanes_std", "pmirror", "beta")},
                       "streams": "the bands of a GPU alternate between 2 compute streams" if cstreams else "one stream",
                       "plane_stacks_rank0": (f"{nslots} shared by {len(bands)} bands" if shared else f"{len(bands)} (one per band)"),
                       "parallelism": (f"{nbands} bands of ONE job partitioned over {world} GPUs (longest-processing-time first); "
                                       f"plane transforms of {len(offloads)} band(s) offloaded to the least loaded GPUs over NVLink "
                                       "peer memory (fused into the transform kernels, flags in device memory, no collective)"
                                       if strong else
                                       f"{world} job(s) of {nbands} band(s), one job per GPU, no data-path collective")},
            "e2e": {"value": e2e_pool_value, "unit": "Mvis/s", "h2d_bytes_per_step": img_bytes, "d2h_bytes_per_step": img_bytes,
                    "call": "operators.BandPool.hess_dot(x (nband, nx, ny) host numpy) -> new host numpy cube (the reference's BandWorkerPool.hess_dot); bands pinned on the device at construction (like load_band), copies of neighbouring bands overlap the kernels",
                    "hessian_slice_value": e2e_value,
                    "hessian_slice_call": "operators.hessian_slice(x, xout=, uvw=, weight=, vis_mask=, freq=, ...) band after band, host numpy in/out, nothing overlapped"},
            "gpu_launches": launches_all, "clocks": sampler.summary(), "roofline": roof, "cpu_baseline": cpu,
            "f64_default_path": f64,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-row-step", type=int, default=1, help="CPU arm: per-visibility loops on every n-th row (1 = all)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-f64", action="store_true", help="skip the fp64 / eps=1e-7 single-band measurement")
    ap.add_argument("--replicas", action="store_true", help="every GPU owns a complete job (weak scaling, the round-1 mode)")
    ap.add_argument("--strong", action="store_true", help="(default for multi-band workloads) kept for compatibility")
    ap.add_argument("--no-offload", action="store_true", help="band partition only, no plane offload")
    ap.add_argument("--bands", default="", help="restrict the job to these bands, e.g. 7,0 (development)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (at most 64 MB, "
                         "a fixed seeded sample of larger outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, cfg)
    elif args.workload == "c5":
        run_c5(args, cfg)
    elif args.workload == "c3":
        run_c3(args, cfg)
    else:
        run_ours(args, cfg)


if __name__ == "__main__":
    main()
