"""CPU: ``restore.fitcleanbeam`` (host numpy, no scipy) against the scipy restatement in ``oracle/restore_np.py``:
exact sampled Gaussians are recovered to 1e-9 relative, PSFs from ``synth`` uv coverage agree with ``curve_fit`` to
1e-6, the main lobe is the 4-connected island above ``level`` that holds the centre, and bad PSFs raise."""
import numpy as np
import pytest

from oracle import restore_np as O
from pfb_imaging_b200 import restore as R
from pfb_imaging_b200 import synth

LIGHTSPEED = 299792458.0


def sampled(n, beam, amp=1.0, m=None):
    x = np.arange(n) - n // 2
    y = np.arange(m or n) - (m or n) // 2
    return amp * O.gauss(x[:, None], y[None, :], *beam)


def beam_err(got, want):
    """relative errors of emaj, emin and of pa (modulo pi, relative to pi/2)"""
    d = abs(got[2] - want[2]) % np.pi
    return max(abs(got[0] - want[0]) / want[0], abs(got[1] - want[1]) / want[1], min(d, np.pi - d) / (np.pi / 2))


CASES = [(emaj, emin, pa) for emaj, emin in ((1.2, 1.2), (1.6, 1.2), (2.5, 1.5), (4.0, 4.0), (7.3, 3.1), (20.0, 6.0),
                                             (20.0, 19.0))
         for pa in (0.0, 0.4, -1.0, np.pi / 2, -np.pi / 2 + 1e-3, np.pi / 2 - 1e-3)]


@pytest.mark.parametrize("beam", CASES)
def test_exact_gaussian_is_recovered(beam):
    want = O.canonical(*beam)
    # narrow beams need a lower level: at 0.5 the island of a 1.2 px beam is its centre pixel alone
    level = 0.5 if beam[1] >= 2.5 else 0.01
    for n, m in ((128, 128), (97, 130)):
        got = R.fitcleanbeam(sampled(n, beam, amp=2.5, m=m)[None], level=level, pixsize=1.0)[0]
        assert beam_err(got, want) <= 1e-9, (got, want)
        if want[0] == want[1]:
            assert got[2] == 0.0
        assert got[0] >= got[1] and -np.pi / 2 < got[2] <= np.pi / 2


def test_pixsize_scales_the_widths_only():
    p = sampled(64, (6.0, 3.0, 0.3))
    a = R.fitcleanbeam(p, pixsize=1.0)[0]
    b = R.fitcleanbeam(p, pixsize=2.5e-5)[0]
    np.testing.assert_allclose(b, [a[0] * 2.5e-5, a[1] * 2.5e-5, a[2]], rtol=1e-14)


def dft_psf(nx, cell, seed, ntime=6, nchan=2, band=3):
    d = synth.make_band(ntime, nchan, band=band, seed=seed, precision="double", with_vis=False)
    uv = (d["uvw"][:, None, :2] * d["freq"][None, :, None] / LIGHTSPEED).reshape(-1, 2)
    w = d["wgt"].reshape(-1)
    lm = (np.arange(nx) - nx // 2) * cell
    # PSF(l, m) = sum_k w_k cos(2 pi (u_k l + v_k m)), separable in cos / sin
    cu, su = np.cos(2 * np.pi * np.outer(uv[:, 0], lm)), np.sin(2 * np.pi * np.outer(uv[:, 0], lm))
    cv, sv = np.cos(2 * np.pi * np.outer(uv[:, 1], lm)), np.sin(2 * np.pi * np.outer(uv[:, 1], lm))
    return (cu * w[:, None]).T @ cv - (su * w[:, None]).T @ sv, d


@pytest.mark.parametrize("seed,srf,level", [(1, 2.0, 0.5), (2, 3.0, 0.5), (3, 4.0, 0.3), (4, 2.5, 0.6)])
def test_synth_psf_matches_curve_fit(seed, srf, level):
    d = synth.make_band(6, 2, band=3, seed=seed, precision="double", with_vis=False)
    cell = synth.default_cell(d["uvw"], d["freq"].max(), srf=srf)
    psf, _ = dft_psf(64, cell, seed)
    psf = np.stack([psf, 0.5 * psf.T])  # a second band: the transposed lobe at another scale
    got = R.fitcleanbeam(psf, level=level, pixsize=cell)
    want = O.fitcleanbeam(psf, level=level, pixsize=cell)
    for g, w in zip(got, want):
        assert beam_err(g, w) <= 1e-6, (g, w)


def test_island_is_four_connected_and_honours_level():
    beam = (5.0, 3.0, 0.6)
    p = sampled(64, beam)
    want = R.fitcleanbeam(p, level=0.5)[0]
    q = p.copy()
    q[5:12, 5:12] = 0.9  # a bright island elsewhere
    assert beam_err(R.fitcleanbeam(q, level=0.5)[0], want) <= 1e-12
    # a pixel above level that touches the main lobe only at a corner is not part of it
    isl = p > 0.5
    ix, iy = np.nonzero(isl)
    k = np.argmax(ix + iy)
    cx, cy = ix[k] + 1, iy[k] + 1
    assert not isl[cx, cy] and not isl[cx - 1, cy] and not isl[cx, cy - 1]
    q = p.copy()
    q[cx, cy] = 0.8
    assert beam_err(R.fitcleanbeam(q, level=0.5)[0], want) <= 1e-12
    # the oracle's label() agrees that the corner pixel is its own island
    assert beam_err(O.fitcleanbeam(q, level=0.5)[0], want) <= 1e-9
    # level is honoured: on an exact Gaussian every island gives the same beam
    for level in (0.2, 0.75):
        assert beam_err(R.fitcleanbeam(p, level=level)[0], O.canonical(*beam)) <= 1e-9
    # ... and on a non-Gaussian lobe the level changes the fit
    r = p ** 0.8 * (1 - 0.2 * p)
    a, b = R.fitcleanbeam(r, level=0.3)[0], R.fitcleanbeam(r, level=0.7)[0]
    assert beam_err(a, b) > 1e-3
    assert beam_err(a, O.fitcleanbeam(r, level=0.3)[0]) <= 1e-6
    assert beam_err(b, O.fitcleanbeam(r, level=0.7)[0]) <= 1e-6


def test_island_search_window_grows():
    # a lobe much wider than the first 17 x 17 window
    beam = (60.0, 45.0, 0.2)
    got = R.fitcleanbeam(sampled(256, beam), level=0.5)[0]
    assert beam_err(got, O.canonical(*beam)) <= 1e-9


def test_errors():
    p = sampled(32, (4.0, 3.0, 0.0))
    with pytest.raises(ValueError, match="not positive"):
        R.fitcleanbeam(np.zeros((1, 32, 32)))
    with pytest.raises(ValueError, match="not positive"):
        R.fitcleanbeam(-p[None])
    q = p.copy()
    q[16, 16] = 0.3
    q[3, 3] = 1.0  # the maximum is elsewhere; the centre falls below level
    with pytest.raises(ValueError, match="centre"):
        R.fitcleanbeam(q, level=0.5)
    # a fitted form that is not positive definite (a saddle, or flat along one axis) is not a beam
    for form in ((0.05, 0.1, 0.05), (0.05, 0.0, 0.0), (0.05, 0.0, -1e-3)):
        with pytest.raises(ValueError, match="positive definite"):
            R._form_to_beam(*form)
    # a main lobe of fewer pixels than the form has parameters is rejected, not fitted
    with pytest.raises(ValueError, match="lower `level`"):
        R.fitcleanbeam(sampled(32, (1.2, 1.2, 0.0)), level=0.5)
