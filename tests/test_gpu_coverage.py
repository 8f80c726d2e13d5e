"""GPU parity tests of the code paths BASELINE's larger configs take by default and the small tests did not
reach: narrow (half / quarter sector) column blocks of the fused transforms, the 5760^2 PSF grid of config 2,
the 10240^2 / nu = 15360 geometry of config 4, gridding of a full C2 band over ALL rows, and the reference-level
``vis2im`` / ``im2vis`` wrappers.  Truth is the explicit DFT (oracle/dft.py), tolerances are BASELINE.json's:
rel-L2 <= epsilon against the DFT (hence <= 2 epsilon against ducc0, which is not installable here: parity with
ducc0's own binary output is unpinned)."""
import numpy as np
import pytest

from oracle import dft
from pfb_imaging_b200 import operators as ops, synth, wgridder as W
from pfbg_testutil import rel_l2, small_problem

pytestmark = pytest.mark.gpu

PFB = dict(flip_u=False, flip_v=True, flip_w=False, do_wgridding=True, divide_by_n=False)


@pytest.mark.parametrize("colc", ["1", "2"])
@pytest.mark.parametrize("prec,eps", [("single", 1e-5), ("double", 1e-8)])
def test_narrow_column_blocks_against_dft(gpu, monkeypatch, colc, prec, eps):
    """k_cols_fwd / k_cols_inv<T, 2> and <T, 1> are what every fp32 grid with nu > ~6.8 k and every fp64 grid with
    nu > ~3.4 k runs (the 8640^2 PSF grid of config 2, all of config 4).  PFBG_COLC forces them at a small size."""
    monkeypatch.setenv("PFBG_COLC", colc)
    W.clear_plan_pool()
    p = small_problem(nrow=700, nchan=3, nx=96, ny=80, seed=31, wscale=2.0)
    rdt, cdt = (np.float32, np.complex64) if prec == "single" else (np.float64, np.complex128)
    kw = dict(center_x=0.01, center_y=-0.02, **PFB)
    with W.plan_for(p["uvw"], p["freq"], npix_x=96, npix_y=80, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=eps,
                    precision=prec, mask=p["mask"], **kw) as gp:
        act = p["mask"] != 0
        v = gp.degrid(p["img"].astype(rdt))
        ref = dft.dft_dirty2vis(p["uvw"], p["freq"], p["img"], p["cell"], p["cell"], **kw)
        assert rel_l2(v[act], ref[act]) <= eps
        vis, wgt = p["vis"].astype(cdt), p["wgt"].astype(rdt)
        d = gp.grid(vis, wgt)
        dref = dft.dft_vis2dirty(p["uvw"], p["freq"], vis, wgt, p["mask"], 96, 80, p["cell"], p["cell"], **kw)
        assert rel_l2(d, dref) <= eps
        gp.bind_weights(wgt)
        h = gp.hessian(p["img"].astype(rdt), wsum=2.0, eta=0.25)
        href = dft.dft_vis2dirty(p["uvw"], p["freq"], ref, wgt, p["mask"], 96, 80, p["cell"], p["cell"], **kw) / 2.0 \
            + 0.25 * p["img"]
        assert rel_l2(h, href) <= 2 * eps
    # same numbers as the full-sector kernels
    monkeypatch.delenv("PFBG_COLC")
    with W.plan_for(p["uvw"], p["freq"], npix_x=96, npix_y=80, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=eps,
                    precision=prec, mask=p["mask"], **kw) as gp:
        assert rel_l2(gp.degrid(p["img"].astype(rdt))[act], v[act]) <= (3e-6 if prec == "single" else 1e-12)
        assert rel_l2(gp.grid(vis, wgt), d) <= (3e-6 if prec == "single" else 1e-11)
    W.clear_plan_pool()


def _c2_band(band, prec, flag_frac=0.03):
    d = synth.make_band(775, 16, band=band, nband=8, precision=prec, with_vis=True, flag_frac=flag_frac)
    return d, synth.default_cell(d["uvw"], 1712e6)


def test_c2_band_gridding_all_rows_rel_l2(gpu):
    """vis2dirty of a complete config-2 band (25.0 M samples, fp32, eps 1e-5) against the explicit DFT over ALL
    samples on 48 random pixels, relative L2 over those pixels."""
    d, cell = _c2_band(6, "single")
    nx, eps = 4096, 1e-5
    with W.plan_for(d["uvw"], d["freq"], npix_x=nx, npix_y=nx, pixsize_x=cell, pixsize_y=cell, epsilon=eps,
                    mask=d["mask"], sigma_min=1.1, sigma_max=3.0, precision="single", **PFB) as gp:
        dimg = gp.grid(d["vis"], d["wgt"])
    rng = np.random.default_rng(17)
    px = (rng.integers(0, nx, 48), rng.integers(0, nx, 48))
    dref = dft.dft_vis2dirty_fast(d["uvw"], d["freq"], d["vis"], d["wgt"], d["mask"], nx, nx, cell, cell,
                                  pixels=px, **PFB)
    err = rel_l2(dimg[px], dref)
    print(f"C2 band 6, all {d['vis'].size} samples, 48 pixels: rel-L2 vs DFT {err:.2e}")
    assert err <= eps


@pytest.mark.parametrize("prec,eps", [("single", 1e-5), ("double", 1e-7)])
def test_c2_psf_grid_5760(gpu, prec, eps):
    """The PSF of config 2 is gridded at nx_psf = good_size(1.4 * 4096) = 5760 (grid 8640^2: half-sector column
    blocks in fp32, quarter-sector in fp64): unit visibilities -> PSF against the DFT (all samples, 32 pixels incl.
    the peak), and dirty2vis of a point-source image at that size on sampled rows."""
    d, cell = _c2_band(2, prec)
    nxp = 5760
    rdt = np.float32 if prec == "single" else np.float64
    cdt = np.complex64 if prec == "single" else np.complex128
    with W.plan_for(d["uvw"], d["freq"], npix_x=nxp, npix_y=nxp, pixsize_x=cell, pixsize_y=cell, epsilon=eps,
                    mask=d["mask"], sigma_min=1.1, sigma_max=3.0, precision=prec, **PFB) as gp:
        info = gp.info()
        assert info["nu"] > (6900 if prec == "single" else 3500), info  # narrower-than-sector column blocks
        ones = np.broadcast_to(np.ones((1,), dtype=cdt), d["vis"].shape)
        psf = gp.grid(ones, d["wgt"])
        x = synth.point_source_image(nxp, nxp, dtype=rdt)
        v = gp.degrid(x)
    rng = np.random.default_rng(3)
    px = (np.concatenate([[nxp // 2], rng.integers(0, nxp, 31)]), np.concatenate([[nxp // 2], rng.integers(0, nxp, 31)]))
    pref = dft.dft_vis2dirty_fast(d["uvw"], d["freq"], np.ones(d["vis"].shape, np.complex128), d["wgt"], d["mask"],
                                  nxp, nxp, cell, cell, pixels=px, **PFB)
    # the PSF is dominated by its peak: compare off-peak pixels against the image-wide L2 scale (the contract is
    # the L2 norm over the image) and the peak relatively
    assert abs(psf[nxp // 2, nxp // 2] - pref[0]) <= eps * abs(pref[0])
    scale = np.sqrt(np.mean(psf.astype(np.float64) ** 2))
    assert np.sqrt(np.mean((psf[px][1:] - pref[1:]) ** 2)) <= eps * scale
    rows = rng.integers(0, d["uvw"].shape[0], 200)
    ref = dft.dft_dirty2vis(d["uvw"], d["freq"], x.astype(np.float64), cell, cell, rows=rows, **PFB)
    act = d["mask"][rows] != 0
    err = rel_l2(v[rows][act], ref[act])
    print(f"PSF grid {nxp}^2 ({prec}): nu={info['nu']} P={info['nplanes']} degrid rel-L2 {err:.2e}")
    assert err <= eps


def test_c4_geometry_quarter_sector_blocks(gpu):
    """Config-4 geometry: 10240^2 image, fp32, grid nu = nv = 15360 (quarter-sector column blocks, C = 1); both
    directions and the fused Hessian against the sampled DFT."""
    d = synth.make_band(24, 16, band=5, nband=8, precision="single", with_vis=True, flag_frac=0.02)
    nx, eps = 10240, 1e-5
    cell = synth.default_cell(d["uvw"], 1712e6) / 2.5  # same field of view as config 2, finer pixels
    with W.plan_for(d["uvw"], d["freq"], npix_x=nx, npix_y=nx, pixsize_x=cell, pixsize_y=cell, epsilon=eps,
                    mask=d["mask"], sigma_min=1.1, sigma_max=3.0, precision="single", **PFB) as gp:
        info = gp.info()
        assert info["nu"] >= 13600, info
        x = synth.point_source_image(nx, nx, dtype=np.float32)
        v = gp.degrid(x)
        dimg = gp.grid(d["vis"], d["wgt"])
        gp.bind_weights(d["wgt"])
        h = gp.hessian(x)
        h2 = gp.grid(v, d["wgt"])
    rng = np.random.default_rng(5)
    rows = rng.integers(0, d["uvw"].shape[0], 200)
    ref = dft.dft_dirty2vis(d["uvw"], d["freq"], x.astype(np.float64), cell, cell, rows=rows, **PFB)
    act = d["mask"][rows] != 0
    e1 = rel_l2(v[rows][act], ref[act])
    px = (rng.integers(0, nx, 48), rng.integers(0, nx, 48))
    dref = dft.dft_vis2dirty_fast(d["uvw"], d["freq"], d["vis"], d["wgt"], d["mask"], nx, nx, cell, cell, pixels=px, **PFB)
    e2 = rel_l2(dimg[px], dref)
    print(f"C4 geometry: nu={info['nu']} P={info['nplanes']} W={info['W']}: degrid {e1:.2e}, grid {e2:.2e}")
    assert e1 <= eps and e2 <= eps
    assert rel_l2(h, h2) <= 3e-6


@pytest.mark.parametrize("precision", ["single", "double"])
def test_vis2im_and_im2vis_wrappers(gpu, precision):
    """operators/gridder.py:37-144: `vis2im` casts by `precision` and grids with pfb's conventions;
    `im2vis` loops over the imaging bands of a cube and fills the channel ranges of one visibility array."""
    p = small_problem(nrow=500, nchan=6, nx=64, ny=72, seed=41)
    l0, m0 = 0.012, -0.02
    eps = 1e-5 if precision == "single" else 1e-8
    fu, fv, fw, x0, y0 = ops.wgridder_conventions(l0, m0)
    kw = dict(center_x=x0, center_y=y0, flip_u=fu, flip_v=fv, flip_w=fw, do_wgridding=True, divide_by_n=False)
    img = ops.vis2im(p["uvw"], p["freq"], p["vis"], p["wgt"], p["mask"], 64, 72, p["cell"], p["cell"], l0, m0, eps,
                     precision, True, False, 1, 1.1, 3.0, True)
    assert img.dtype == (np.float32 if precision == "single" else np.float64) and img.shape == (64, 72)
    cdt = np.complex64 if precision == "single" else np.complex128
    rdt = np.float32 if precision == "single" else np.float64
    dref = dft.dft_vis2dirty(p["uvw"], p["freq"], p["vis"].astype(cdt), p["wgt"].astype(rdt), p["mask"], 64, 72,
                             p["cell"], p["cell"], **kw)
    assert rel_l2(img, dref) <= eps
    with pytest.raises(ValueError):
        ops.vis2im(p["uvw"], p["freq"], p["vis"], p["wgt"], p["mask"], 64, 72, p["cell"], p["cell"], l0, m0, eps,
                   "half", True, False, 1, 1.1, 3.0, True)
    if precision == "single":
        return
    # two imaging bands of 2 and 4 channels
    cube = np.stack([p["img"], np.roll(p["img"], 5, axis=0)])
    fbi, fbc = np.array([3, 5]), np.array([2, 4])  # offsets are relative to the first band (gridder.py:114)
    vis = ops.im2vis(p["uvw"], p["freq"], cube, p["cell"], p["cell"], fbi, fbc, l0=l0, m0=m0, epsilon=1e-8,
                     do_wgridding=True, divide_by_n=False, nthreads=1)
    assert vis.shape == (500, 6) and vis.dtype == np.complex128
    ref = np.empty_like(vis)
    ref[:, :2] = dft.dft_dirty2vis(p["uvw"], p["freq"][:2], cube[0], p["cell"], p["cell"], **kw)
    ref[:, 2:] = dft.dft_dirty2vis(p["uvw"], p["freq"][2:], cube[1], p["cell"], p["cell"], **kw)
    assert rel_l2(vis, ref) <= 1e-8
