"""CPU: the numpy SARA restatement (oracle/sara_np.py) against vectors produced by the reference's own numba code."""
import os

import numpy as np
import pytest

from oracle import sara_np as so
from pfb_imaging_b200 import wavelet_filters as wf

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "sara.npz"))


def _s(a):
    """The elements of `a` the golden file keeps of each output: every G["stride"]-th of the flattened array."""
    return np.asarray(a).reshape(-1)[::int(G["stride"])]


def _setup(tag):
    nx, ny, nband, nlevel, nxmax, nymax = (int(v) for v in G[f"{tag}_meta"])
    bases = [str(b) for b in G[f"{tag}_bases"]]
    bk = wf.bookkeeping(nx, ny, bases, nlevel)
    fbs = [None if b == "self" else wf.filter_bank(b) for b in bases]
    return bk, fbs, nband, nxmax, nymax


def test_filter_banks_are_orthonormal():
    for n in range(1, 6):
        dlo, dhi, rlo, rhi = wf.filter_bank(f"db{n}")
        K = dlo.size
        assert abs(rlo.sum() - np.sqrt(2)) < 1e-15 and abs(rhi.sum()) < 1e-15
        for s in range(0, K, 2):  # double-shift orthogonality
            want = 1.0 if s == 0 else 0.0
            assert abs(np.dot(rlo[s:], rlo[:K - s]) - want) < 1e-15
            assert abs(np.dot(rlo[s:], rhi[:K - s])) < 1e-15
        for p in range(1, n):  # vanishing moments of the high-pass filter
            assert abs(np.dot(np.arange(K) ** p, rhi)) < 1e-10
    with pytest.raises(ValueError):
        wf.filter_bank("sym4")


@pytest.mark.parametrize("tag", ["a", "b", "d"])
def test_bookkeeping_matches_reference(tag):
    bk, fbs, nband, nxmax, nymax = _setup(tag)
    assert (bk.nxmax, bk.nymax) == (nxmax, nymax)


@pytest.mark.parametrize("tag", ["a", "b", "d"])
def test_psi_dot_hdot_match_reference(tag):
    bk, fbs, nband, _, _ = _setup(tag)
    x = G[f"{tag}_x"]
    alpha = np.stack([so.psi_dot(x[b], bk, fbs) for b in range(nband)])
    np.testing.assert_allclose(_s(alpha), G[f"{tag}_x_alpha"], rtol=0, atol=1e-12)
    xrec = np.stack([so.psi_hdot(alpha[b], bk, fbs) for b in range(nband)])
    np.testing.assert_allclose(_s(xrec), G[f"{tag}_x_xrec"], rtol=0, atol=1e-11)
    # the reference's input was 0.5 * (its alpha, reversed) + 0.25; its alpha equals this one to ~2e-15
    a2 = 0.5 * alpha[..., ::-1, ::-1] + 0.25
    xr2 = np.stack([so.psi_hdot(a2[b], bk, fbs) for b in range(nband)])
    np.testing.assert_allclose(_s(xr2), G[f"{tag}_x_xr2"], rtol=0, atol=1e-11)
    # decomposition + reconstruction = nbasis * identity (tests/test_psi_operator.py:24-53)
    np.testing.assert_allclose(G[f"{tag}_x_xrec"], _s(bk.nbasis * x), atol=1e-11)
    np.testing.assert_allclose(xrec, bk.nbasis * x, atol=1e-11)


def test_transposed_layout_is_the_transpose():
    bk, fbs, nband, _, _ = _setup("a")
    x = G["a_x"][0]
    alpha_t = so.psi_dot(x, bk, fbs, transposed=True)
    np.testing.assert_allclose(_s(alpha_t), G["a_t_alpha"], atol=1e-12)
    np.testing.assert_allclose(alpha_t, so.psi_dot(x, bk, fbs).transpose(0, 2, 1), rtol=0, atol=1e-13)
    a2 = 0.5 * alpha_t[..., ::-1, ::-1] + 0.25
    np.testing.assert_allclose(_s(so.psi_hdot(a2, bk, fbs, transposed=True)), G["a_t_xr2"], atol=1e-11)


@pytest.mark.parametrize("nm", ["p", "z"])
def test_dual_update_and_prox_match_reference(nm):
    lam, sigma = G[f"du_{nm}_par"]
    vp, v, w = G["du_vp"], G["du_v"], G["du_w"]
    np.testing.assert_allclose(_s(so.dual_update_fast(vp, v, lam, sigma, w)), G[f"du_{nm}_out"], rtol=1e-13, atol=1e-14)
    np.testing.assert_allclose(_s(so.prox_21m(v, lam, sigma, w)), G[f"du_{nm}_prox"], rtol=1e-13, atol=1e-14)


def test_adjointness_of_the_dictionary():
    bk, fbs, _, _, _ = _setup("d")
    rng = np.random.default_rng(1)
    x = rng.standard_normal((bk.nx, bk.ny))
    a = so.psi_dot(x, bk, fbs)
    y = np.zeros_like(a)
    # hdot is the adjoint of dot on the coefficients dot can produce (packing leaves unused cells at zero)
    y[a != 0] = rng.standard_normal(int((a != 0).sum()))
    lhs = float((a * y).sum())
    rhs = float((x * so.psi_hdot(y, bk, fbs)).sum())
    assert abs(lhs - rhs) <= 1e-10 * max(abs(lhs), 1.0)
