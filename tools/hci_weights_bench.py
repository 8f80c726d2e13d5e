"""Cost of robust (Briggs) weighting in `pfb hci` at the C5 shape: per-snapshot calls against the batched device path.

Workload (defaults, BASELINE config 5): 1024 snapshots of 2016 MeerKAT-like baselines x 16 channels, 512^2 images,
fp32, epsilon 1e-4, sigma_min 2, divide_by_n, imaged in batches of 256; Briggs robust 0 on a 1024^2 counts pad
(good_size(2 nx), utils/stokes2im.py:563-604).  Each snapshot gets its residual and its PSF image.

  loop:    per snapshot  weighting._compute_counts + weighting.counts_to_weights  (two host-pointer calls), then
           wgridder.vis2dirty_batch(wgt=those weights) per batch
  device:  wgridder.vis2dirty_batch(robustness=0) per batch: the weights are computed from the natural weights on the
           device, in the plan, and never come back to the host

Both are timed after one warm-up batch each, `--reps` times, alternating, with host wall time around work that ends
in a device synchronise and with CUDA events on the default stream; `weights_ms_per_snapshot` is the weighting's share
(the loop's calls within the same pass; the plan's bind_robust_weights on an already bound batch).  Prints one JSON
line with the card name and power limit read in the same run, and the rel-L2 between the two paths' cubes.

    python tools/hci_weights_bench.py [--nsnap 1024 --chunk 256 --nx 512 --pad 1024 --robust 0]
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
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, plim = (s.strip() for s in out.split(","))
        return name, plim
    except Exception as e:  # noqa: BLE001
        return None, f"unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nsnap", type=int, default=1024)
    ap.add_argument("--chunk", type=int, default=256)
    ap.add_argument("--nx", type=int, default=512)
    ap.add_argument("--pad", type=int, default=1024)
    ap.add_argument("--nchan", type=int, default=16)
    ap.add_argument("--robust", type=float, default=0.0)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()

    import torch

    from pfb_imaging_b200 import synth, weighting as gw, wgridder as W

    rng = np.random.default_rng(1234)
    enu = synth.meerkat_like_antennas(rng)
    uvw_all = synth.uvw_tracks(enu, a.nsnap)  # time-major: rows [t nbl, (t+1) nbl) are snapshot t
    nbl = uvw_all.shape[0] // a.nsnap
    freq = synth.band_freqs(4, 8, a.nchan)
    cell = synth.default_cell(uvw_all, 1712e6)
    wgt = rng.uniform(0.5, 1.5, (a.nsnap * nbl, a.nchan)).astype(np.float32)
    vis = (rng.standard_normal(wgt.shape) + 1j * rng.standard_normal(wgt.shape)).astype(np.complex64)
    ones = np.ones((nbl, a.nchan), np.complex64)
    geom = dict(freq=freq, npix_x=a.nx, npix_y=a.nx, pixsize_x=cell, pixsize_y=cell, epsilon=1e-4, flip_v=True,
                divide_by_n=True, sigma_min=2.0, sigma_max=2.6)
    us, vs = -1.0, 1.0  # the counts signs of flip_u=False, flip_v=True (operators.image_data_products_arrays)
    batches = [list(range(c0, min(c0 + a.chunk, a.nsnap))) for c0 in range(0, a.nsnap, a.chunk)]
    rows = lambda s: slice(s * nbl, (s + 1) * nbl)  # noqa: E731

    def loop_weights(ids):
        out = []
        for s in ids:
            u, w = uvw_all[rows(s)], wgt[None, rows(s)].copy()
            c = gw._compute_counts(u, freq, None, w, a.pad, a.pad, cell, cell, np.float32, 1, us, vs)
            gw.counts_to_weights(c, u, freq, w, None, a.pad, a.pad, cell, cell, a.robust, us, vs)
            out.append(w[0])
        return out

    loop_w_s = []

    def loop(ids):
        t0 = time.perf_counter()
        wl = loop_weights(ids)
        loop_w_s.append(time.perf_counter() - t0)
        return W.vis2dirty_batch(uvw=[uvw_all[rows(s)] for s in ids], vis=[vis[rows(s)] for s in ids], wgt=wl,
                                 extra_vis=([ones] * len(ids),), **geom)

    def device(ids):
        return W.vis2dirty_batch(uvw=[uvw_all[rows(s)] for s in ids], vis=[vis[rows(s)] for s in ids],
                                 wgt=[wgt[rows(s)] for s in ids], extra_vis=([ones] * len(ids),),
                                 robustness=a.robust, nx_pad=a.pad, ny_pad=a.pad, **geom)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record()
        res = [fn(ids) for ids in batches]
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        return res, 1e3 * wall / a.nsnap, e0.elapsed_time(e1) / a.nsnap

    name, plim = card()
    torch.cuda.init()
    loop(batches[0])  # warm-up: modules, pooled plan, CUB
    device(batches[0])
    runs, err = [], 0.0
    for _ in range(a.reps):  # the two paths alternate: other work shares the host
        loop_w_s.clear()
        res_loop, loop_wall, loop_ev = timed(loop)
        loop_w = 1e3 * sum(loop_w_s) / a.nsnap
        res_dev, dev_wall, dev_ev = timed(device)
        runs.append((loop_wall, loop_ev, loop_w, dev_wall, dev_ev))
        err = max([err] + [float(np.linalg.norm(d - r) / np.linalg.norm(r))
                           for rd, rl in zip(res_dev, res_loop) for d, r in zip(rd, rl)])
        del res_loop, res_dev

    # the device path's weighting alone: bind_robust_weights on a bound batch plan
    W.clear_plan_pool()
    dev_w, info = 0.0, None
    for ids in batches:  # one bound plan at a time: a 256-snapshot plane stack is many GB
        gp = W.batch_plan_for([uvw_all[rows(s)] for s in ids], freq, precision="single",
                              **{k: v for k, v in geom.items() if k != "freq"})
        w = wgt[rows(ids[0]).start:rows(ids[-1]).stop]
        gp.bind_robust_weights(w, a.pad, a.pad, cell, cell, a.robust, us, vs)  # warm-up: the counts scratch
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gp.bind_robust_weights(w, a.pad, a.pad, cell, cell, a.robust, us, vs)
        torch.cuda.synchronize()
        dev_w += 1e3 * (time.perf_counter() - t0) / a.nsnap
        info = info or gp.info()
        gp.close()

    print(json.dumps(dict(
        tool="hci_weights_bench", device=name, power_limit=plim, nsnap=a.nsnap, chunk=a.chunk, nx=a.nx, pad=a.pad,
        baselines=nbl, nchan=a.nchan, robust=a.robust, precision="single", epsilon=1e-4, W=int(info["W"]),
        nu=int(info["nu"]), planes_first_batch=int(info["nplanes"]),
        loop=dict(ms_per_snapshot_wall=[round(r[0], 4) for r in runs], ms_per_snapshot_events=[round(r[1], 4) for r in runs],
                  weights_ms_per_snapshot=[round(r[2], 4) for r in runs]),
        device_path=dict(ms_per_snapshot_wall=[round(r[3], 4) for r in runs],
                         ms_per_snapshot_events=[round(r[4], 4) for r in runs],
                         weights_ms_per_snapshot=round(dev_w, 4)),
        speedup_total_median=round(float(np.median([r[0] / r[3] for r in runs])), 2),
        speedup_weights_median=round(float(np.median([r[2] for r in runs])) / dev_w, 2),
        max_rel_l2_device_vs_loop=err,
        what="residual + PSF of every snapshot with Briggs weights (utils/stokes2im.py:563-604, 635-683)")))


if __name__ == "__main__":
    main()
