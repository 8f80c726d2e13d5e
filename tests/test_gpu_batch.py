"""GPU: batched snapshots (BASELINE config 5, `pfb hci`): many small images of one geometry through ONE bin / sort
and one launch of every kernel (pfbg_plan_set_batch / pfbg_bind_vis_batch).  Every snapshot is checked against the
explicit DFT with the settings of the reference's snapshot imager (utils/stokes2im.py:635-683: divide_by_n=True,
sigma_min = min_padding = 2) and against the one-shot call on that snapshot alone.  These are toy sizes (5 snapshots
of 64 x 48); tests/test_gpu_batch_production.py runs the benchmark's production shape (256 snapshots of 512^2)."""
import numpy as np
import pytest

from oracle import dft
from pfb_imaging_b200 import wgridder as W
from pfb_imaging_b200.plan import make_batch_plan
from pfbg_testutil import rel_l2, small_problem

pytestmark = pytest.mark.gpu


def _snapshots(nsnap, nx, ny, seed=0):
    out = []
    for s in range(nsnap):
        p = small_problem(nrow=150 + 37 * s, nchan=3, nx=nx, ny=ny, seed=seed + s, wscale=0.3 + 1.5 * s)
        out.append(p)
    for p in out:  # one geometry: the cell of the first snapshot, and one frequency axis
        p["cell"], p["freq"] = out[0]["cell"], out[0]["freq"]
    return out


@pytest.mark.parametrize("prec,eps", [("single", 1e-4), ("double", 1e-7)])
def test_batched_snapshots_match_dft_and_one_shot_calls(gpu, prec, eps):
    nx, ny = 64, 48
    snaps = _snapshots(5, nx, ny)
    rdt, cdt = (np.float32, np.complex64) if prec == "single" else (np.float64, np.complex128)
    cell, freq = snaps[0]["cell"], snaps[0]["freq"]
    kw = dict(center_x=0.01, center_y=-0.015, flip_u=False, flip_v=True, flip_w=False, do_wgridding=True, divide_by_n=True)
    com = dict(freq=freq, pixsize_x=cell, pixsize_y=cell, epsilon=eps, sigma_min=2.0, sigma_max=2.6, **kw)
    uvw = [p["uvw"] for p in snaps]
    vis = [p["vis"].astype(cdt) for p in snaps]
    wgt = [p["wgt"].astype(rdt) for p in snaps]
    mask = [p["mask"] for p in snaps]
    ones = [np.ones(p["vis"].shape, cdt) for p in snaps]
    cube, psf = W.vis2dirty_batch(uvw=uvw, vis=vis, wgt=wgt, mask=mask, npix_x=nx, npix_y=ny, extra_vis=(ones,), **com)
    assert cube.shape == (5, nx, ny) and cube.dtype == rdt and psf.shape == cube.shape
    for s, p in enumerate(snaps):
        ref = dft.dft_vis2dirty(p["uvw"], freq, vis[s], wgt[s], mask[s], nx, ny, cell, cell, **kw)
        assert rel_l2(cube[s], ref) <= eps, s
        pref = dft.dft_vis2dirty(p["uvw"], freq, ones[s], wgt[s], mask[s], nx, ny, cell, cell, **kw)
        assert rel_l2(psf[s], pref) <= eps, s
        one = W.vis2dirty(uvw=p["uvw"], vis=vis[s], wgt=wgt[s], mask=mask[s], npix_x=nx, npix_y=ny, **com)
        assert rel_l2(cube[s], one) <= (2 * eps if prec == "single" else 1e-8)  # plans may differ in their plane grids
    imgs = np.stack([np.roll(p["img"].astype(rdt), s, axis=1) for s, p in enumerate(snaps)])
    vs = W.dirty2vis_batch(uvw=uvw, dirty=imgs, mask=mask, **com)
    for s, p in enumerate(snaps):
        ref = dft.dft_dirty2vis(p["uvw"], freq, imgs[s].astype(np.float64), cell, cell, **kw)
        act = mask[s] != 0
        assert vs[s].shape == p["vis"].shape and rel_l2(vs[s][act], ref[act]) <= eps, s
        assert np.all(vs[s][~act] == 0)
    W.clear_plan_pool()


def test_batch_plan_layout_and_hessian(gpu):
    """Plane blocks per snapshot, adjointness of the batched pair, and the fused batched Hessian."""
    nx = 48
    snaps = _snapshots(4, nx, nx, seed=20)
    cell, freq = snaps[0]["cell"], snaps[0]["freq"]
    uvw = [p["uvw"] for p in snaps]
    gp = W.batch_plan_for(uvw, freq, npix_x=nx, npix_y=nx, pixsize_x=cell, pixsize_y=cell, epsilon=1e-8, flip_v=True,
                          divide_by_n=False, sigma_min=2.0, mask_list=[p["mask"] for p in snaps])
    info = gp.info()
    wr = [W.w_range(u, freq) for u in uvw]
    plan, w0, npl = make_batch_plan(wr, nx=nx, ny=nx, pixsize_x=cell, pixsize_y=cell, epsilon=1e-8, flip_v=True,
                                    divide_by_n=False, sigma_min=2.0)
    assert info["nplanes"] == int(npl.sum()) and gp.image_shape == (4, nx, nx)
    assert all(npl >= plan.W) and len(set(npl.tolist())) > 1  # different w-ranges -> different plane counts
    for (lo, hi), a, n in zip(wr, w0, npl):  # every snapshot's samples are covered by its own block
        assert a <= lo and a + (n - 1) * plan.dw >= hi
    rng = np.random.default_rng(1)
    x = rng.standard_normal((4, nx, nx))
    v = gp.degrid(x)
    vis = np.concatenate([p["vis"] for p in snaps])
    wgt = np.concatenate([p["wgt"] for p in snaps])
    act = np.concatenate([p["mask"] for p in snaps]) != 0
    d = gp.grid(vis, wgt)
    lhs = np.vdot(v, vis * wgt * act).real
    rhs = float((d * x).sum())
    assert abs(lhs - rhs) <= 1e-11 * abs(rhs)
    gp.bind_weights(wgt)
    h = gp.hessian(x, wsum=3.0, eta=0.1)
    ref = gp.grid(v, wgt) / 3.0 + 0.1 * x
    assert rel_l2(h, ref) <= 1e-11
    with pytest.raises(ValueError):
        gp.grid(vis, wgt, dirty=np.empty((nx, nx)))  # a batched plan returns the cube
    gp.close()
