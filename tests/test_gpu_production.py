"""GPU: the batched-snapshot workload (BASELINE config 5, `pfb hci`) at its real shape, built as bench.py's c5 arm
builds one batch: 256 snapshots of 512^2 from `synth.uvw_tracks` (2016 baselines x 16 channels), fp32, eps 1e-4,
sigma_min 2, divide_by_n.  Such plans take W < 8, so the run kernels' general flush / fetch is the path under test.
Sampled snapshots against the explicit DFT at the plan's error bound (tests/test_gpu_widths.py), and the batched
Hessian against grid(degrid)."""
import numpy as np
import pytest

from oracle import dft
from pfb_imaging_b200 import synth, wgridder as W
from pfb_imaging_b200.plan import make_batch_plan
from pfbg_testutil import rel_l2

pytestmark = pytest.mark.gpu

BOUND_C, FLOOR = 2.0, 3e-6  # as tests/test_gpu_widths.py


def test_c5_batch_at_its_real_shape(gpu):
    nx, nsnap_job, nbatch, nchan = 512, 1024, 256, 16
    rng = np.random.default_rng(1234)
    enu = synth.meerkat_like_antennas(rng)
    uvw_all = synth.uvw_tracks(enu, nsnap_job)  # time-major: rows [t * nbl, (t+1) * nbl) are snapshot t
    nbl = uvw_all.shape[0] // nsnap_job
    assert nbl == 2016
    freq = synth.band_freqs(4, 8, nchan)
    cell = synth.default_cell(uvw_all, 1712e6)
    uvw = [uvw_all[t * nbl:(t + 1) * nbl] for t in range(nbatch)]
    geom = dict(npix_x=nx, npix_y=nx, pixsize_x=cell, pixsize_y=cell, epsilon=1e-4, flip_v=True, divide_by_n=True,
                sigma_min=2.0, sigma_max=2.6, precision="single")
    kw = dict(center_x=0.0, center_y=0.0, flip_u=False, flip_v=True, flip_w=False, do_wgridding=True, divide_by_n=True)
    gp = W.batch_plan_for(uvw, freq, **geom)
    plan = gp.plan
    assert plan.W < 8, f"fixture no longer exercises the general flush / fetch path: {plan.info()}"
    wr = np.array([W.w_range(u, freq) for u in uvw])
    _, _, npl = make_batch_plan(wr, nvis_per_snapshot=nbl * nchan, nx=nx, ny=nx, pixsize_x=cell, pixsize_y=cell,
                                epsilon=1e-4, flip_v=True, divide_by_n=True, sigma_min=2.0, sigma_max=2.6,
                                precision="single")
    assert gp.info()["nplanes"] == int(npl.sum())
    brng = np.random.default_rng(5)
    wgt = brng.uniform(0.5, 1.5, (nbatch * nbl, nchan)).astype(np.float32)
    vis = (brng.standard_normal((nbatch * nbl, nchan)) + 1j * brng.standard_normal((nbatch * nbl, nchan))).astype(np.complex64)
    gp.bind_weights(wgt)
    x = np.stack([synth.point_source_image(nx, nx, nsrc=20, seed=k, dtype=np.float32) for k in range(nbatch)])
    v = gp.degrid(x)
    d = gp.grid(vis, wgt)
    # first and last snapshot, the ones with the narrowest and the widest w-range (the fewest and the most planes; at
    # this field of view every snapshot of the batch has the same count), and random ones
    span = wr[:, 1] - wr[:, 0]
    pick = list(dict.fromkeys([0, nbatch - 1, int(np.argmin(span)), int(np.argmax(span))]))
    for s in np.random.default_rng(7).permutation(nbatch):
        if len(pick) == 16:
            break
        if int(s) not in pick:
            pick.append(int(s))
    tol = BOUND_C * plan.kernel_err + FLOOR
    prng = np.random.default_rng(11)
    for s in pick:
        rows = slice(s * nbl, (s + 1) * nbl)
        ref = dft.dft_dirty2vis(uvw[s], freq, x[s].astype(np.float64), cell, cell, **kw)
        ev = rel_l2(v[rows], ref)
        px = (prng.integers(0, nx, 64), prng.integers(0, nx, 64))
        dref = dft.dft_vis2dirty(uvw[s], freq, vis[rows], wgt[rows], None, nx, nx, cell, cell, pixels=px, **kw)
        # 64 sampled pixels against the image-wide scale (the bound is the L2 norm over the image)
        ed = np.linalg.norm(d[s][px] - dref) / (np.sqrt(64.0) * np.sqrt(np.mean(d[s].astype(np.float64) ** 2)))
        print(f"c5 snapshot {s} ({npl[s]} planes): degrid {ev:.1e} grid {ed:.1e} "
              f"(kernel_err {plan.kernel_err:.1e}, tol {tol:.1e})")
        assert ev <= tol, (s, ev, tol)
        assert ed <= tol, (s, ed, tol)
    h = gp.hessian(x, wsum=1.0, eta=0.0)
    h2 = gp.grid(v, wgt)
    assert rel_l2(h, h2) <= 2e-6
    gp.close()
