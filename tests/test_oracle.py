"""CPU: the oracle against the reference's own known-answer vectors and identities."""
import dataclasses
import os

import numpy as np
import pytest

from oracle import dft, weighting as ow, wgridder_np as wg
from pfb_imaging_b200.plan import make_plan, w_range
from pfbg_testutil import GOLDEN, rel_l2, small_problem


@pytest.fixture(scope="module")
def kat():
    return np.load(os.path.join(GOLDEN, "kat_conventions.npz"))


def _kat_dirty(npix):
    d = np.zeros((npix, npix))
    d[npix // 2, npix // 2] = 1.0
    d[npix // 4, npix // 4] = 1.0
    return d


@pytest.mark.parametrize("k", range(5))
def test_dft_matches_reference_explicit_degridder(kat, k):
    """tests/test_hessian_approx.py:70-125: flips off, centre (-l0,-m0), divide_by_n."""
    npix, pix = int(kat["npix"]), float(kat["pixsize"])
    l0, m0 = kat["offsets"][k]
    v = dft.dft_dirty2vis(kat["uvw"], kat["freqs"], _kat_dirty(npix), pix, pix, -l0, -m0,
                          False, False, False, True, True)
    for neg in (0, 1):
        np.testing.assert_allclose(v, kat[f"conv_{k}_{neg}"], atol=2e-9, rtol=0)


@pytest.mark.parametrize("k", range(5))
def test_dft_matches_reference_explicit_wdegridder(kat, k):
    """tests/test_hessian_approx.py:128-185: pfb conventions (flip_v, x0=-l0, y0=-m0)."""
    npix, pix = int(kat["npix"]), float(kat["pixsize"])
    fu, fv, fw = (bool(f) for f in kat["flips"])
    assert (fu, fv, fw) == (False, True, False)
    x0, y0 = kat[f"wconv_center_{k}"]
    v = dft.dft_dirty2vis(kat["uvw"], kat["freqs"], _kat_dirty(npix), pix, pix, x0, y0, fu, fv, fw, True, True)
    np.testing.assert_allclose(v, kat[f"wconv_{k}"], atol=2e-9, rtol=0)


def _plan(p, eps, **kw):
    wmin, wmax = w_range(p["uvw"], p["freq"])
    args = dict(nx=p["nx"], ny=p["ny"], pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=eps, wmin=wmin, wmax=wmax,
                nvis=p["vis"].size, divide_by_n=True)
    args.update(kw)
    return make_plan(**args)


@pytest.mark.parametrize("eps", [1e-4, 1e-7])
@pytest.mark.parametrize("geom", [dict(), dict(center_x=0.05, center_y=-0.08, flip_v=True),
                                  dict(do_wgridding=False), dict(flip_u=True, flip_w=True, divide_by_n=False)])
def test_numpy_wgridder_restatement_matches_dft(eps, geom):
    p = small_problem()
    plan = _plan(p, eps, **geom)
    kw = dict(center_x=geom.get("center_x", 0.0), center_y=geom.get("center_y", 0.0),
              flip_u=geom.get("flip_u", False), flip_v=geom.get("flip_v", False), flip_w=geom.get("flip_w", False),
              do_wgridding=geom.get("do_wgridding", True), divide_by_n=geom.get("divide_by_n", True))
    ref = dft.dft_dirty2vis(p["uvw"], p["freq"], p["img"], p["cell"], p["cell"], **kw)
    v = wg.dirty2vis_np(plan, p["uvw"], p["freq"], p["img"], mask=p["mask"])
    act = p["mask"] != 0
    assert rel_l2(v[act], ref[act]) <= eps
    assert np.all(v[~act] == 0)
    dref = dft.dft_vis2dirty(p["uvw"], p["freq"], p["vis"], p["wgt"], p["mask"], p["nx"], p["ny"], p["cell"], p["cell"], **kw)
    d = wg.vis2dirty_np(plan, p["uvw"], p["freq"], p["vis"], p["wgt"], p["mask"])
    assert rel_l2(d, dref) <= eps
    # exact adjointness of the restatement
    lhs = np.vdot(v, p["vis"] * p["wgt"] * act).real
    rhs = float((d * p["img"]).sum())
    assert abs(lhs - rhs) <= 1e-11 * abs(rhs)


def test_bin_indices_invariants():
    p = small_problem(nrow=300)
    plan = _plan(p, 1e-5)
    b = wg.bin_indices(plan, p["uvw"], p["freq"], p["mask"])
    assert b["idx"].size == int((p["mask"] != 0).sum())
    x = b["iu0"] + np.arange(plan.W)[:, None] - b["gu"]
    assert (np.abs(x) <= plan.W / 2 + 1e-9).all()
    # mirror planes: supports may reach below plane 0 (served by the Hermitian mirror), never clamped
    assert b["ip0"].min() >= -plan.pmirror and b["ip0"].max() <= plan.nplanes - plan.W
    xw = b["ip0"] + np.arange(plan.W)[:, None] - b["gw"]
    assert (np.abs(xw) <= plan.W / 2 + 1e-9).all()
    std = wg.bin_indices(_plan(p, 1e-5, mirror=False), p["uvw"], p["freq"], p["mask"])
    assert std["ip0"].min() >= 0
    assert (np.diff(b["key"][b["order"]].astype(np.int64)) >= 0).all()


def test_bin_indices_of_a_batch():
    """Batched snapshots: each sample's plane comes from its own snapshot's w0 and plane block.  A batch of one
    snapshot whose block is the plan's own stack bins like the plan; in a batch of three, snapshot s's samples bin
    like the one-snapshot plan of its block, shifted by the planes before it."""
    from pfb_imaging_b200.plan import make_batch_plan

    ps = [small_problem(nrow=120 + 30 * s, seed=s, wscale=1.0 + 8.0 * s * s) for s in range(3)]
    freq, cell = ps[0]["freq"], ps[0]["cell"]
    wr = [w_range(p["uvw"], freq) for p in ps]
    plan, w0, npl = make_batch_plan(wr, nx=64, ny=48, pixsize_x=cell, pixsize_y=cell, epsilon=1e-5, flip_v=True)
    assert len(set(npl.tolist())) > 1
    plan.nplanes = int(npl.sum())
    uvw = np.concatenate([p["uvw"] for p in ps])
    mask = np.concatenate([p["mask"] for p in ps])
    ro = np.concatenate([[0], np.cumsum([p["uvw"].shape[0] for p in ps])])
    b = wg.bin_indices(plan, uvw, freq, mask, row_offsets=ro, snap_w0=w0, snap_np=npl)
    pbase = np.concatenate([[0], np.cumsum(npl)[:-1]])
    for s, p in enumerate(ps):
        one = dataclasses.replace(plan, w0=float(w0[s]), nplanes=int(npl[s]))
        ref = wg.bin_indices(one, p["uvw"], freq, p["mask"])
        sel = b["snap"] == s
        assert np.array_equal(b["ip0"][sel], ref["ip0"] + pbase[s])
        assert np.array_equal(b["iu0"][sel], ref["iu0"]) and np.array_equal(b["iv0"][sel], ref["iv0"])
        assert b["ip0"][sel].min() >= pbase[s] and b["ip0"][sel].max() + plan.W <= pbase[s] + npl[s]
    solo = wg.bin_indices(plan, uvw, freq, mask, row_offsets=[0, uvw.shape[0]], snap_w0=[plan.w0],
                          snap_np=[plan.nplanes])
    whole = wg.bin_indices(plan, uvw, freq, mask)
    for k in ("iu0", "iv0", "ip0", "key", "order"):
        assert np.array_equal(solo[k], whole[k]), k


# --- weighting -------------------------------------------------------------
@pytest.fixture(scope="module")
def wgold():
    return np.load(os.path.join(GOLDEN, "weighting.npz"))


@pytest.mark.parametrize("tag,dt", [("f8", np.float64), ("f4", np.float32)])
@pytest.mark.parametrize("signs", [(-1.0, 1.0), (1.0, -1.0)])
def test_weighting_oracle_matches_reference(wgold, tag, dt, signs):
    g = wgold
    nx, ny, cell = int(g["nx"]), int(g["ny"]), float(g["cell"])
    us, vs = signs
    st = f"{tag}_{int(us)}_{int(vs)}"
    tol = 1e-12 if dt == np.float64 else 2e-6
    wgt = g[f"wgt_{tag}"]
    c = ow.compute_counts(g["uvw"], g["freq"], g["mask"], wgt, nx, ny, cell, cell, dt, 1, us, vs)
    gc = g[f"counts_{st}"]
    assert np.array_equal(c > 0, gc > 0)  # same cells hit: the integer index is bit-exact
    np.testing.assert_allclose(c, gc, rtol=tol, atol=tol)
    for r in (-2.0, 0.0, 1.5):
        c2, w2 = gc.copy(), wgt.copy()
        ow.counts_to_weights(c2, g["uvw"], g["freq"], w2, g["mask"], nx, ny, cell, cell, r, us, vs)
        np.testing.assert_allclose(w2, g[f"w_{st}_r{r}"], rtol=10 * tol, atol=0)
        np.testing.assert_allclose(c2, g[f"c_{st}_r{r}"], rtol=10 * tol, atol=0)


def test_weighting_filters_match_reference(wgold):
    g = wgold
    for tag in ("f8", "f4"):
        c = g[f"counts_{tag}_-1_1"]
        assert np.array_equal(ow.filter_extreme_counts(c.copy(), 10.0), g[f"filtered_{tag}"])
        assert np.array_equal(ow.box_sum_counts(c.copy(), 2), g[f"boxsum_{tag}"])


def test_uv2xy_identity():
    """tests/test_weighting.py:113-137 (test_uv2xy): u = (-(nx//2) + i)/(nx cell) lands in cell i."""
    for nx in (128, 1034, 44, 10000):
        cell = 1.3e-5
        i = np.arange(nx)
        u = (-(nx // 2) + i + 0.5) / (nx * cell)
        freq = np.array([299792458.0])
        uvw = np.stack([u, np.full(nx, 1.0), np.zeros(nx)], axis=1)
        ui, vi = ow.uv_cells(uvw, freq, None, nx, 8, cell, 0.01, usign=1.0, vsign=1.0)
        assert np.array_equal(ui[:, 0], i)


def test_l2_reweight_restatement_matches_reference_block():
    """oracle.weighting.l2_reweight against the outputs of the reference's own `if l2_reweight_dof:` block
    (operators/gridder.py:509-532, executed by tests/golden/make_golden_l2.py): bit-exact."""
    import os

    from oracle import weighting as ow
    from pfbg_testutil import GOLDEN

    g = np.load(os.path.join(GOLDEN, "l2_reweight.npz"))
    assert int(g["ncase"]) == 8 and bool(g["zero_is_none"])
    for k in range(int(g["ncase"])):
        wp = g[f"wgtp_{k}"]
        got = ow.l2_reweight(g[f"rv_{k}"], g[f"wgt_{k}"], g[f"mask_{k}"], float(g[f"dof_{k}"]), None if wp.size == 0 else wp)
        assert got.dtype == g[f"out_{k}"].dtype and np.array_equal(got, g[f"out_{k}"])
    assert ow.l2_reweight(np.zeros((1, 4, 2), complex), np.ones((1, 4, 2)), np.ones((4, 2), np.uint8), 2.0) is None
