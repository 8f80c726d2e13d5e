"""GPU: the device Clark minor cycle (pfb_imaging_b200.clean) against the numpy restatement of its contract
(oracle/clark_np.py): identical peak sequences and active-set sizes, model and residual within 1e-12 relative (the
residual step runs through a different FFT), plus the reference's own kclean acceptance on this library's products."""
import numpy as np
import pytest

from oracle import clark_np as cn

pytestmark = pytest.mark.gpu


def _psf(nband, nxp, nyp, rng, width=2.5):
    x = np.arange(nxp)[:, None] - nxp // 2
    y = np.arange(nyp)[None, :] - nyp // 2
    psf = np.empty((nband, nxp, nyp))
    for b in range(nband):
        w = width * (1 + 0.1 * b)
        psf[b] = np.exp(-(x**2 + y**2) / (2 * w**2)) + 0.05 * rng.standard_normal((nxp, nyp)) / (1 + np.hypot(x, y))
        psf[b, nxp // 2, nyp // 2] = 1.0 + 0.01 * b
    return psf


def _dirty(psf, nx, ny, rng, nsrc=8, edges=False, noise=0.01):
    nband = psf.shape[0]
    sky = np.zeros((nband, nx, ny))
    i, j = rng.integers(0, nx, nsrc), rng.integers(0, ny, nsrc)
    if edges:
        i[:4], j[:4] = [0, nx - 1, 0, nx - 1], [0, ny - 1, ny - 1, 0]
    sky[:, i, j] = rng.uniform(1, 10, (nband, nsrc))
    return cn.psf_convolve(sky, cn.psfhat_of(psf), *psf.shape[1:]) + noise * rng.standard_normal((nband, nx, ny))


def _run_both(psf, dirty, mask=None, **kw):
    from pfb_imaging_b200.clean import Clark

    cl = Clark(psf, nx=dirty.shape[1], ny=dirty.shape[2])
    model, resid, info = cl(dirty, mask=mask, **kw)
    mo, ro, io = cn.clark(dirty, psf, mask=mask, **kw)
    assert info["niter"] == io["niter"]
    assert info["nactive"] == io["nactive"]
    assert info["nsub"] == io["nsub"]
    for a, b in zip(info["peaks"], io["peaks"]):
        assert np.array_equal(a, b)
    np.testing.assert_allclose(info["rmax"], io["rmax"], rtol=1e-12, atol=0)
    scale = np.abs(dirty).max()
    assert np.abs(model - mo).max() <= 1e-12 * max(np.abs(mo).max(), scale)
    assert np.abs(resid - ro).max() <= 1e-12 * scale
    cl.close()
    return model, resid, info


@pytest.mark.parametrize("nband,nx,ny,nxp,nyp", [
    (1, 32, 32, 48, 48),     # nx_psf < 2 nx
    (3, 40, 28, 80, 56),     # nx_psf = 2 nx, non-square
    (8, 24, 36, 40, 50),     # 8 bands, non-square, nx_psf < 2 nx
    (3, 36, 36, 72, 72),
])
def test_matches_oracle(gpu, nband, nx, ny, nxp, nyp):
    rng = np.random.default_rng(nband * 1000 + nx)
    psf = _psf(nband, nxp, nyp, rng)
    dirty = _dirty(psf, nx, ny, rng)
    model, _, info = _run_both(psf, dirty, gamma=0.1, pf=0.01, maxit=8, subpf=0.4, submaxit=150)
    assert info["niter"] >= 3 and sum(info["nsub"]) > 50
    assert np.abs(model).sum() > 0


def test_active_set_of_one(gpu):
    rng = np.random.default_rng(5)
    psf = _psf(2, 48, 48, rng)
    dirty = _dirty(psf, 32, 32, rng, nsrc=3)
    _, _, info = _run_both(psf, dirty, gamma=0.2, pf=0.0, maxit=1, subpf=0.9999, submaxit=10)
    assert info["nactive"] == [1] and info["nsub"][0] >= 1


def test_active_set_smaller_than_one_cta(gpu):
    rng = np.random.default_rng(6)
    psf = _psf(3, 24, 20, rng)
    dirty = _dirty(psf, 12, 12, rng, nsrc=4)
    _, _, info = _run_both(psf, dirty, gamma=0.1, pf=0.0, maxit=3, subpf=0.01, submaxit=200)
    assert 1 < info["nactive"][0] < 256 and info["nsub"][0] > 20


def test_active_set_larger_than_resident_grid(gpu):
    # 640^2 = 409600 active entries: more than 148 SMs x 8 CTAs x 256 threads, so every thread owns several
    rng = np.random.default_rng(7)
    nx = ny = 640
    psf = _psf(2, nx, ny, rng, width=6.0)
    dirty = _dirty(psf, nx, ny, rng, nsrc=30, noise=0.0) + 0.05 + 0.01 * rng.uniform(size=(2, nx, ny))
    _, _, info = _run_both(psf, dirty, gamma=0.1, pf=0.0, maxit=2, subpf=0.001, submaxit=25)
    assert min(info["nactive"]) > 148 * 8 * 256 and info["nsub"] == [25, 25]


def test_peaks_at_image_edges(gpu):
    rng = np.random.default_rng(8)
    psf = _psf(2, 40, 44, rng)
    nx, ny = 30, 34
    sky = np.zeros((2, nx, ny))
    sky[:, [0, nx - 1, 0, nx - 1], [0, ny - 1, ny - 1, 0]] = rng.uniform(5, 10, (2, 4))
    dirty = cn.psf_convolve(sky, cn.psfhat_of(psf), 40, 44) + 0.01 * rng.standard_normal((2, nx, ny))
    model, _, info = _run_both(psf, dirty, gamma=0.1, pf=0.01, maxit=6, subpf=0.5, submaxit=200)
    corners = {0, ny - 1, (nx - 1) * ny, nx * ny - 1}
    assert corners <= set(np.concatenate(info["peaks"]).tolist())


def test_brightest_pixel_masked(gpu):
    rng = np.random.default_rng(9)
    psf = _psf(3, 48, 48, rng)
    dirty = _dirty(psf, 32, 32, rng)
    mask = rng.uniform(size=(32, 32)) > 0.2
    mask.flat[np.argmax(cn.search_value(dirty))] = False
    model, _, info = _run_both(psf, dirty, mask=mask, gamma=0.1, pf=0.01, maxit=6, subpf=0.4, submaxit=200)
    assert sum(info["nsub"]) > 0 and not model[:, ~mask].any()


def test_band_with_zero_peak_gets_no_model(gpu):
    rng = np.random.default_rng(10)
    psf = _psf(3, 48, 48, rng)
    psf[1, 24, 24] = 0.0
    dirty = _dirty(psf, 32, 32, rng)
    model, _, info = _run_both(psf, dirty, gamma=0.1, pf=0.01, maxit=5, subpf=0.4, submaxit=100)
    assert sum(info["nsub"]) > 0 and not model[1].any() and model[0].any() and model[2].any()


def test_repeat_runs_are_bitwise_identical(gpu):
    from pfb_imaging_b200.clean import Clark

    rng = np.random.default_rng(11)
    psf = _psf(3, 96, 96, rng)
    dirty = _dirty(psf, 64, 64, rng, nsrc=20)
    cl = Clark(psf, nx=64, ny=64)
    a = cl(dirty, gamma=0.1, pf=0.01, maxit=6, subpf=0.3, submaxit=300)
    b = cl(dirty, gamma=0.1, pf=0.01, maxit=6, subpf=0.3, submaxit=300)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert a[2]["nsub"] == b[2]["nsub"] and all(np.array_equal(x, y) for x, y in zip(a[2]["peaks"], b[2]["peaks"]))
    cl.close()


def test_kclean_acceptance_on_library_products(gpu):
    """Point sources -> visibilities (DFT) -> dirty, PSF, PSFHAT (image_data_products_arrays) -> clark -> exact
    residual (hessian_slice): positions exact, fluxes within 5 x threshold."""
    from pfbg_testutil import small_problem

    from oracle import dft
    from pfb_imaging_b200 import operators as ops
    from pfb_imaging_b200.clean import clark, clear_clark_cache

    nx = ny = 64
    p = small_problem(nrow=600, nchan=2, nx=nx, ny=ny, seed=3, fov=0.05, wscale=0.0)  # w = 0: a shift-invariant PSF
    cell = p["cell"]
    src = [(20, 17, 1.0), (41, 45, 0.6), (12, 50, 0.35)]
    x = np.zeros((nx, ny))
    for i, j, f in src:
        x[i, j] = f
    vis = dft.dft_dirty2vis(p["uvw"], p["freq"], x, cell, cell, 0, 0, False, True, False, True, False)
    out = ops.image_data_products_arrays(p["uvw"], p["freq"], vis[None], p["wgt"][None], p["mask"], nx, ny, 2 * nx,
                                         2 * ny, cell, cell, epsilon=1e-10)
    wsum = out["wsum"][0]
    ID, PSF, PSFHAT = out["dirty"] / wsum, out["psf"] / wsum, out["psfhat"] / wsum
    thr = 1e-3
    model, resid, info = clark(ID, PSF, PSFHAT, threshold=thr, gamma=0.1, pf=0.0, maxit=50, subpf=0.5, submaxit=1000)
    assert info["niter"] < 50
    got = {tuple(ij) for ij in np.argwhere(model[0] != 0)}
    assert got == {(i, j) for i, j, _ in src}
    for i, j, f in src:
        assert abs(model[0, i, j] - f) <= 5 * thr
    exact = ID[0] - ops.hessian_slice(model[0], uvw=p["uvw"], weight=p["wgt"], vis_mask=p["mask"], freq=p["freq"],
                                      cell=cell, epsilon=1e-10, wsum=wsum)
    assert np.abs(exact).max() <= 5 * thr
    assert np.abs(exact - resid[0]).max() <= 1e-6
    clear_clark_cache()


def test_bad_arguments_raise_before_launch(gpu):
    from pfb_imaging_b200.clean import Clark, clark

    rng = np.random.default_rng(12)
    psf = _psf(2, 48, 48, rng)
    dirty = _dirty(psf, 32, 32, rng)
    with pytest.raises(TypeError):
        Clark(psf.astype(np.float32), nx=32, ny=32)
    with pytest.raises(ValueError):
        Clark(psf[0], nx=32, ny=32)
    with pytest.raises(ValueError):
        Clark(psf, nx=64, ny=32)  # image larger than the PSF
    with pytest.raises(ValueError):
        Clark(psf, psfhat=np.zeros((2, 48, 24), dtype=np.complex128), nx=32, ny=32)
    with pytest.raises(TypeError):
        Clark(psf, psfhat=np.zeros((2, 48, 25), dtype=np.complex64), nx=32, ny=32)
    cl = Clark(psf, nx=32, ny=32)
    for kw in (dict(gamma=0.0), dict(gamma=1.5), dict(pf=-0.1), dict(subpf=1.0), dict(subpf=0.0), dict(maxit=-1),
               dict(submaxit=0), dict(threshold=-1.0), dict(threshold=float("nan"))):
        with pytest.raises(ValueError):
            cl(dirty, **kw)
    with pytest.raises(TypeError):
        cl(dirty, maxit=2.5)
    with pytest.raises(TypeError):
        cl(dirty.astype(np.float32))
    with pytest.raises(ValueError):
        cl(dirty[:, :16])
    with pytest.raises(ValueError):
        cl(dirty, mask=np.ones((16, 32), dtype=bool))
    with pytest.raises(ValueError):
        clark(dirty[0], psf)
    cl.close()
    with pytest.raises(RuntimeError):
        cl(dirty)
