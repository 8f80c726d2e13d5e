"""CPU: the numpy restatement of the Clark minor cycle (oracle/clark_np.py) against properties it must have on its
own — the residual it carries equals the dirty image minus the PSF applied to its model, a delta PSF converges
geometrically, every stopping rule is honoured exactly, and masked pixels never receive model."""
import numpy as np
import pytest

from oracle import clark_np as cn


def _psf(nband, nxp, nyp, rng, width=2.0):
    """A centred Gaussian main lobe with random sidelobes, peak 1 at (nxp//2, nyp//2)."""
    x = np.arange(nxp)[:, None] - nxp // 2
    y = np.arange(nyp)[None, :] - nyp // 2
    psf = np.empty((nband, nxp, nyp))
    for b in range(nband):
        w = width * (1 + 0.2 * b)
        psf[b] = np.exp(-(x**2 + y**2) / (2 * w**2)) + 0.05 * rng.standard_normal((nxp, nyp)) / (1 + np.hypot(x, y))
        psf[b, nxp // 2, nyp // 2] = 1.0
    return psf


def _sky(nband, nx, ny, rng, nsrc=6):
    m = np.zeros((nband, nx, ny))
    i, j = rng.integers(0, nx, nsrc), rng.integers(0, ny, nsrc)
    m[:, i, j] = rng.uniform(1, 10, (nband, nsrc))
    return m


def test_residual_is_dirty_minus_psf_of_model():
    rng = np.random.default_rng(0)
    nband, nx, ny = 3, 24, 20
    psf = _psf(nband, 2 * nx, 2 * ny, rng)
    dirty = cn.direct_convolve(_sky(nband, nx, ny, rng), psf) + 0.01 * rng.standard_normal((nband, nx, ny))
    seen = []

    def check(k, model, R):
        ref = dirty - cn.direct_convolve(model, psf)
        assert np.abs(R - ref).max() <= 1e-12 * np.abs(dirty).max(), k
        seen.append(k)

    model, R, info = cn.clark(dirty, psf, gamma=0.1, pf=0.01, maxit=6, subpf=0.5, submaxit=200, callback=check)
    assert seen == list(range(1, info["niter"] + 1)) and info["niter"] >= 3
    assert np.abs(model).sum() > 0
    assert sum(info["nsub"]) == sum(p.size for p in info["peaks"])


@pytest.mark.parametrize("k", [1, 7, 40])
def test_delta_psf_converges_geometrically(k):
    nx, ny, gamma, flux = 16, 12, 0.3, 2.5
    psf = np.zeros((1, 2 * nx, 2 * ny))
    psf[0, nx, ny] = 1.0
    dirty = np.zeros((1, nx, ny))
    dirty[0, 5, 7] = flux
    model, R, info = cn.clark(dirty, psf, gamma=gamma, pf=0.0, maxit=1, subpf=1e-9, submaxit=k)
    expect = flux * (1 - (1 - gamma) ** k)
    assert info["nsub"] == [k] and (info["peaks"][0] == 5 * ny + 7).all()
    assert abs(model[0, 5, 7] - expect) <= 1e-12 * flux
    assert np.count_nonzero(model) == 1
    assert abs(R[0, 5, 7] - flux * (1 - gamma) ** k) <= 1e-12 * flux


def _delta(flux=1.0, nx=8, ny=8):
    psf = np.zeros((1, 2 * nx, 2 * ny))
    psf[0, nx, ny] = 1.0
    dirty = np.zeros((1, nx, ny))
    dirty[0, 3, 4] = flux
    return dirty, psf


def test_maxit_and_submaxit_stops():
    rng = np.random.default_rng(1)
    nband, nx, ny = 2, 20, 20
    psf = _psf(nband, 2 * nx, 2 * ny, rng)
    dirty = cn.direct_convolve(_sky(nband, nx, ny, rng), psf)
    for maxit in (0, 1, 3):
        model, R, info = cn.clark(dirty, psf, gamma=0.1, pf=0.0, maxit=maxit, subpf=0.5, submaxit=5)
        assert info["niter"] == maxit and info["nsub"] == [5] * maxit
    model, R, info = cn.clark(dirty, psf, maxit=0)
    assert not model.any() and np.array_equal(R, dirty)


def test_threshold_stop():
    dirty, psf = _delta()
    # residual after k components: 0.5^k; components run while it exceeds 0.1 (k = 0..3), then the major loop stops
    model, R, info = cn.clark(dirty, psf, threshold=0.1, gamma=0.5, pf=0.0, maxit=10, subpf=0.01, submaxit=100)
    assert info["niter"] == 1 and info["nsub"] == [4]
    assert R[0, 3, 4] == 0.0625 and model[0, 3, 4] == 0.9375


def test_pf_stop():
    dirty, psf = _delta()
    # tol = 0.2 * Rmax(first) = 0.2; each major iteration (subpf 0.9) runs one component of gain 0.5: 1 -> .5 -> .25 -> .125
    model, R, info = cn.clark(dirty, psf, threshold=0.0, gamma=0.5, pf=0.2, maxit=10, subpf=0.9, submaxit=100)
    assert info["niter"] == 3 and info["nsub"] == [1, 1, 1] and info["rmax"] == [1.0, 0.5, 0.25]
    assert R[0, 3, 4] == 0.125


def test_masked_pixels_receive_no_model():
    rng = np.random.default_rng(2)
    nband, nx, ny = 2, 24, 24
    psf = _psf(nband, 2 * nx, 2 * ny, rng)
    dirty = cn.direct_convolve(_sky(nband, nx, ny, rng, nsrc=10), psf)
    mask = rng.uniform(size=(nx, ny)) > 0.3
    s = cn.search_value(dirty)
    mask.flat[np.argmax(s)] = False  # the brightest pixel is masked out
    model, R, info = cn.clark(dirty, psf, mask=mask, gamma=0.1, pf=0.01, maxit=5, subpf=0.3, submaxit=300)
    assert sum(info["nsub"]) > 0
    assert not model[:, ~mask].any()
    assert all(mask.flat[p].all() for p in info["peaks"])
