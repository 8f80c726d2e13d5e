"""GPU: per-snapshot Briggs weights of a batch of `pfb hci` snapshots (weighting.counts_to_weights_batch,
GridderPlan.bind_robust_weights, vis2dirty_batch(robustness=)) against one _compute_counts / counts_to_weights pair
per snapshot, which tests/test_gpu_weighting.py pins to the reference's numba (tests/golden/weighting.npz)."""
import os

import numpy as np
import pytest

from pfb_imaging_b200 import _lib, synth, weighting as gw, wgridder as W
from pfb_imaging_b200.plan import LIGHTSPEED
from pfbg_testutil import GOLDEN, rel_l2, small_problem

pytestmark = pytest.mark.gpu

TOL = {np.float64: 1e-12, np.float32: 2e-6}  # test_counts_and_weights_match_reference


def _loop(uvw, freq, wgt, mask, ro, nxp, nyp, cellx, celly, robust, us, vs):
    """One _compute_counts + counts_to_weights pair per snapshot: (raw counts, re-weighted counts, weights)."""
    raw, cnt, out = [], [], wgt.copy()
    for s in range(len(ro) - 1):
        sl = slice(ro[s], ro[s + 1])
        m = None if mask is None else mask[sl]
        c = gw._compute_counts(uvw[sl], freq, m, wgt[None, sl], nxp, nyp, cellx, celly, wgt.dtype, 1, us, vs)
        raw.append(c[0].copy())
        w = wgt[None, sl].copy()
        gw.counts_to_weights(c, uvw[sl], freq, w, m, nxp, nyp, cellx, celly, robust, us, vs)
        out[sl] = w[0]
        cnt.append(c[0])
    return np.stack(raw), np.stack(cnt), out


def _snapshots(rows, nchan=4, seed=0, reach=1.3, flagged=()):
    """Random snapshots whose |u|, |v| reach `reach` times the edge of the pad grid, so some samples fall off it."""
    rng = np.random.default_rng(seed)
    nrow = int(sum(rows))
    freq = np.linspace(1.0e9, 1.4e9, nchan)
    cell = 2e-4
    edge = 0.5 / cell * LIGHTSPEED / freq.max()
    uvw = rng.uniform(-reach, reach, (nrow, 3)) * edge
    wgt = rng.uniform(0.5, 1.5, (nrow, nchan))
    mask = (rng.uniform(size=(nrow, nchan)) > 0.1).astype(np.uint8)
    ro = np.concatenate([[0], np.cumsum(rows)]).astype(np.int64)
    for s in flagged:
        mask[ro[s]:ro[s + 1]] = 0
    return uvw, freq, wgt, mask, ro, cell


def _check(uvw, freq, wgt, mask, ro, nxp, nyp, cell, robust, us, vs, dt):
    w0 = wgt.astype(dt)
    raw, ref_c, ref_w = _loop(uvw, freq, w0, mask, ro, nxp, nyp, cell, cell, robust, us, vs)
    w = w0.copy()
    c = np.empty((len(ro) - 1, nxp, nyp), dt)
    assert gw.counts_to_weights_batch(uvw, freq, w, mask, ro, nxp, nyp, cell, cell, robust, us, vs, counts=c) is w
    tol = TOL[dt]
    empty = raw == 0
    assert np.array_equal(c[empty], ref_c[empty])  # cells without samples: exactly 0 (or 1 after the Briggs scale)
    np.testing.assert_allclose(c, ref_c, rtol=10 * tol, atol=0)
    np.testing.assert_allclose(w, ref_w, rtol=10 * tol, atol=0)
    return raw, w, w0


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("robust", [-3.0, -2.0, 0.0, 2.0])
@pytest.mark.parametrize("signs", [(-1.0, 1.0), (1.0, -1.0)])
def test_batch_matches_per_snapshot_calls(gpu, dt, robust, signs):
    rows = [37, 0, 120, 55, 81, 3]  # unequal, one empty, snapshot 3 fully flagged
    uvw, freq, wgt, mask, ro, cell = _snapshots(rows, flagged=(3,))
    raw, w, w0 = _check(uvw, freq, wgt, mask, ro, 24, 20, cell, robust, *signs, dt)
    off = gw.counts_cells(uvw, freq, mask, 24, 20, cell, cell, *signs)[..., 0] < 0
    assert (off & (mask != 0)).sum() > 50  # unflagged samples off the pad grid
    assert not raw[3].any() and np.array_equal(w[ro[3]:ro[4]], w0[ro[3]:ro[4]])
    assert all(raw[s].any() for s in (0, 2, 4, 5))


@pytest.mark.parametrize("nsnap", [1, 2 * 64 + 3])  # 64 grids per launch along blockIdx.y (weighting.cuh)
def test_one_snapshot_and_more_than_one_launch_tile(gpu, nsnap):
    rows = np.random.default_rng(nsnap).integers(0, 40, nsnap)
    uvw, freq, wgt, mask, ro, cell = _snapshots(rows, seed=nsnap)
    _check(uvw, freq, wgt, mask, ro, 16, 18, cell, 0.5, -1.0, 1.0, np.float64)
    _check(uvw, freq, wgt, mask, ro, 16, 18, cell, 0.5, 1.0, -1.0, np.float32)


@pytest.mark.parametrize("tag,dt", [("f8", np.float64), ("f4", np.float32)])
@pytest.mark.parametrize("signs", [(-1.0, 1.0), (1.0, -1.0)])
def test_golden_rows_split_into_snapshots(gpu, tag, dt, signs):
    """The golden has two correlations and the batch takes one: every correlation on its own.  Split into snapshots,
    the batch reproduces the per-snapshot calls; as one snapshot, the reference's numba output itself."""
    g = np.load(os.path.join(GOLDEN, "weighting.npz"))
    nx, ny, cell = int(g["nx"]), int(g["ny"]), float(g["cell"])
    us, vs = signs
    st = f"{tag}_{int(us)}_{int(vs)}"
    tol = TOL[dt]
    split = np.array([0, 150, 150, 400, 610, 700], np.int64)
    for corr in range(g[f"wgt_{tag}"].shape[0]):
        wgt = g[f"wgt_{tag}"][corr]
        for r in (-2.0, 0.0, 1.5):
            _check(g["uvw"], g["freq"], wgt, g["mask"], split, nx, ny, cell, r, us, vs, dt)
            w = wgt.copy()
            c = np.empty((1, nx, ny), dt)
            gw.counts_to_weights_batch(g["uvw"], g["freq"], w, g["mask"], [0, 700], nx, ny, cell, cell, r, us, vs,
                                       counts=c)
            np.testing.assert_allclose(w, g[f"w_{st}_r{r}"][corr], rtol=10 * tol, atol=0)
            np.testing.assert_allclose(c[0], g[f"c_{st}_r{r}"][corr], rtol=10 * tol, atol=0)


@pytest.mark.parametrize("prec,flips,robust", [("double", (True, False), 0.0), ("double", (False, True), -1.0),
                                                ("single", (False, True), 0.0), ("single", (True, False), 1.0)])
def test_vis2dirty_batch_robustness_matches_per_snapshot_loop(gpu, prec, flips, robust):
    nx, ny = 64, 48
    snaps = [small_problem(nrow=150 + 37 * s, nchan=3, nx=nx, ny=ny, seed=s, wscale=0.3 + 1.5 * s) for s in range(5)]
    cell, freq = snaps[0]["cell"], snaps[0]["freq"]
    rdt, cdt = (np.float32, np.complex64) if prec == "single" else (np.float64, np.complex128)
    flip_u, flip_v = flips
    com = dict(freq=freq, npix_x=nx, npix_y=ny, pixsize_x=cell, pixsize_y=cell, epsilon=1e-4 if prec == "single" else 1e-7,
               flip_u=flip_u, flip_v=flip_v, divide_by_n=True, sigma_min=2.0, sigma_max=2.6)
    uvw = [p["uvw"] for p in snaps]
    vis = [p["vis"].astype(cdt) for p in snaps]
    ones = [np.ones(p["vis"].shape, cdt) for p in snaps]
    wgt = [p["wgt"].astype(rdt) for p in snaps]
    mask = [p["mask"] for p in snaps]
    ro = np.concatenate([[0], np.cumsum([u.shape[0] for u in uvw])])
    _, _, wl = _loop(np.concatenate(uvw), freq, np.concatenate(wgt), np.concatenate(mask), ro, 128, 96, cell, cell,
                     robust, 1.0 if flip_u else -1.0, 1.0 if flip_v else -1.0)
    ref = W.vis2dirty_batch(uvw=uvw, vis=vis, wgt=[wl[ro[s]:ro[s + 1]] for s in range(5)], mask=mask,
                            extra_vis=(ones,), **com)
    got = W.vis2dirty_batch(uvw=uvw, vis=vis, wgt=wgt, mask=mask, extra_vis=(ones,), robustness=robust, **com)
    lim = 1e-6 if prec == "single" else 1e-12
    for a, b in zip(got, ref):  # residual, PSF
        assert rel_l2(a, b) <= lim
    assert rel_l2(ref[0], W.vis2dirty_batch(uvw=uvw, vis=vis, wgt=wgt, mask=mask, **com)) > 1e-3  # weights matter
    W.clear_plan_pool()


def test_c5_batch_of_256_snapshots(gpu):
    """One C5 batch: 256 snapshots of 2016 baselines x 16 channels at 512^2, 1024^2 pad, fp32, W as the plan picks
    it; 16 sampled snapshots against the per-snapshot loop."""
    nsnap, nx = 256, 512
    rng = np.random.default_rng(1234)
    enu = synth.meerkat_like_antennas(rng)
    uvw_all = synth.uvw_tracks(enu, 1024)
    nbl = uvw_all.shape[0] // 1024
    uvw_all = uvw_all[:nsnap * nbl]
    freq = synth.band_freqs(4, 8, 16)
    cell = synth.default_cell(uvw_all, 1712e6)
    wgt = rng.uniform(0.5, 1.5, (nsnap * nbl, 16)).astype(np.float32)
    ro = np.arange(nsnap + 1, dtype=np.int64) * nbl
    us, vs = -1.0, 1.0  # flip_v=True
    _, _, wl = _loop(uvw_all, freq, wgt, None, ro, 1024, 1024, cell, cell, 0.0, us, vs)
    wb = gw.counts_to_weights_batch(uvw_all, freq, wgt.copy(), None, ro, 1024, 1024, cell, cell, 0.0, us, vs)
    pick = np.sort(rng.choice(nsnap, 16, replace=False))
    for s in pick:
        np.testing.assert_allclose(wb[ro[s]:ro[s + 1]], wl[ro[s]:ro[s + 1]], rtol=10 * TOL[np.float32], atol=0)
    uvw = [uvw_all[ro[s]:ro[s + 1]] for s in range(nsnap)]
    vis = [(rng.standard_normal((nbl, 16)) + 1j * rng.standard_normal((nbl, 16))).astype(np.complex64)
           for _ in range(nsnap)]
    ones = [np.ones((nbl, 16), np.complex64)] * nsnap
    com = dict(freq=freq, npix_x=nx, npix_y=nx, pixsize_x=cell, pixsize_y=cell, epsilon=1e-4, flip_v=True,
               divide_by_n=True, sigma_min=2.0, sigma_max=2.6, extra_vis=(ones,))
    got = W.vis2dirty_batch(uvw=uvw, vis=vis, wgt=[wgt[ro[s]:ro[s + 1]] for s in range(nsnap)], robustness=0.0,
                            nx_pad=1024, ny_pad=1024, **com)
    ref = W.vis2dirty_batch(uvw=uvw, vis=vis, wgt=[wl[ro[s]:ro[s + 1]] for s in range(nsnap)], **com)
    for a, b in zip(got, ref):
        for s in pick:
            assert rel_l2(a[s], b[s]) <= 1e-6, s
    W.clear_plan_pool()


def test_rejections_come_before_any_launch(gpu):
    lib = _lib.load()
    uvw, freq, wgt, mask, ro, cell = _snapshots([20, 30, 10])
    base = dict(uvw=uvw, freq=freq, mask=mask, row_offsets=ro, nx_pad=16, ny_pad=16, cellx=cell, celly=cell, robust=0.0)

    def rejected(exc, **kw):
        a = {**base, "weight": wgt.copy(), **kw}
        w0 = a["weight"].copy()
        n0 = lib.pfbg_launch_count()
        with pytest.raises(exc):
            gw.counts_to_weights_batch(**a)
        assert lib.pfbg_launch_count() == n0
        assert np.array_equal(a["weight"], w0)

    rejected(RuntimeError, row_offsets=[0, 30, 20, 60])  # decreasing
    rejected(RuntimeError, row_offsets=[5, 20, 50, 60])  # not from 0
    rejected(ValueError, row_offsets=[0, 20, 50, 59])  # not ending at nrow
    rejected(ValueError, row_offsets=[60])  # no snapshot
    rejected(RuntimeError, nx_pad=0)
    rejected(RuntimeError, ny_pad=-8)
    rejected(RuntimeError, cellx=np.nan)
    rejected(RuntimeError, celly=np.inf)
    rejected(ValueError, counts=np.empty((3, 16, 15)))  # not the pad
    rejected(ValueError, counts=np.empty((2, 16, 16)))  # not one grid per snapshot
    rejected(ValueError, weight=wgt[:, :3].copy())  # not the uvw / freq / mask shape
    rejected(ValueError, weight=wgt[None].copy())

    ul = [uvw[ro[s]:ro[s + 1]] for s in range(3)]
    plain = W.plan_for(uvw, freq, npix_x=32, npix_y=32, pixsize_x=cell, pixsize_y=cell, epsilon=1e-7, mask=mask)
    batch = W.batch_plan_for(ul, freq, npix_x=32, npix_y=32, pixsize_x=cell, pixsize_y=cell, epsilon=1e-7,
                             mask_list=[mask[ro[s]:ro[s + 1]] for s in range(3)])
    for gp, w, kw, exc in [(plain, wgt, {}, RuntimeError),  # not a batch
                           (batch, wgt[:-1], {}, ValueError),  # not the bound rows
                           (batch, wgt, dict(nx_pad=0), RuntimeError),
                           (batch, wgt, dict(cellx=np.inf), RuntimeError)]:
        a = dict(nx_pad=16, ny_pad=16, cellx=cell, celly=cell, robust=0.0)
        a.update(kw)
        n0 = lib.pfbg_launch_count()
        with pytest.raises(exc):
            gp.bind_robust_weights(w, **a)
        assert lib.pfbg_launch_count() == n0
    batch.bind_robust_weights(wgt, 16, 16, cell, cell, 0.0)  # the same plan takes valid arguments afterwards
    plain.close()
    batch.close()
