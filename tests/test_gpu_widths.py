"""GPU: every kernel support width and every run-kernel arm against the explicit DFT at the error bound the plan is
designed for, `C * plan.kernel_err + floor` (tests/test_oracle_bounds.py pins that bound on the numpy restatement).

Plans are forced to each (precision, W, sigma): fp64 W = 4..16 and fp32 W = 4..8 at sigma 1.5 and 2.0, in three
geometries (w-gridding with mirror planes; w-gridding without mirror planes on a stack of more than W planes; no
w-gridding).  That reaches, by construction rather than by whatever W an epsilon selects:

    W < 8, or W = 8 without w-gridding     k_grid_runs / k_degrid_runs, general flush / fetch
    W = 8 with w-gridding                  the same kernels' W = 8 fast path (fp32: fast and accurate w-screen)
    fp64 9 <= W <= 12                      the DMMA run kernels (runs_mma.cuh)
    fp64 13 <= W <= 16                     the scalar team kernels k_grid_runs_wide / k_degrid_runs_wide
    any W with PFBG_FORCE_DIRECT=1         k_grid_direct / k_degrid_direct (read when uvw is bound)

`FLOOR` is the round-off floor of each precision: fp64 the 5e-13 of the restatement (the kernels measure <= 4e-14 at
W = 15, 16, sigma 2); fp32 3e-6, three times the measured floor of the fp32 path (8e-7 .. 9.5e-7 at W = 8, sigma 2, where
kernel_err is 2.9e-7).  The fused Hessian is checked
against the DFT composition at twice the bound (one kernel error per direction).

The plane-count tests drive the fp32 row passes (pair engine for all planes of an even count, the one-plane kernel for
the last plane of an odd one) with controlled parity, and the band split's owner / helper plane subsets with all four
parity combinations, against the DFT and against the kernels they replace."""
import numpy as np
import pytest

from oracle import dft, wgridder_np as wg
from pfb_imaging_b200 import split as bs, wgridder as W
from pfb_imaging_b200.plan import make_plan, w_range
from pfbg_testutil import rel_l2, small_problem

pytestmark = pytest.mark.gpu

BOUND_C = 2.0
FLOOR = {"double": 5e-13, "single": 3e-6}
# Same plan through the numpy restatement (as test_gpu_wgridder.py), plus a share of kernel_err in fp64: the plan's
# grid-correction tables (plan.py, kernel_table.kernel_ft) and the restatement's own (200-node Gauss-Legendre) evaluate
# psihat with different quadratures, which differ by ~3e-7 of kernel_err at W = 4..6 (7.7e-10 relative at W = 4,
# sigma 1.5; 7e-14 at W = 8, sigma 2); the kernels reproduce the tables they are given.
ROUNDOFF = {"double": 1e-11, "single": 2e-5}
ROUNDOFF_KERR = {"double": 1e-6, "single": 0.0}
ADJ = {"double": 2e-11, "single": 2e-5}  # adjointness (as test_gpu_wgridder.py)
DT = {"double": (np.float64, np.complex128), "single": (np.float32, np.complex64)}
EPS = {"double": 1e-6, "single": 1e-5}  # only picks fp32's fast w-screen (epsilon >= 3e-6); (sigma, W) are forced
WSUM, ETA = 2.0, 0.25

GEOMS = {
    "mirror": dict(wscale=1.0, mirror=True, kw=dict()),
    "stack": dict(wscale=6.0, mirror=False, kw=dict(flip_v=True, divide_by_n=False)),
    "nowgrid": dict(wscale=1.0, mirror=True, kw=dict(do_wgridding=False, center_x=0.02, center_y=-0.01)),
}
CASES = [(prec, w, s) for prec, ws in (("double", range(4, 17)), ("single", range(4, 9))) for w in ws for s in (1.5, 2.0)]


def _kw(geom):
    kw = dict(center_x=0.0, center_y=0.0, flip_u=False, flip_v=False, flip_w=False, do_wgridding=True, divide_by_n=True)
    kw.update(geom)
    return kw


def _references(p, kw, prec):
    """DFT degrid / grid / Hessian of the problem's image, visibilities and weights as the kernels see them."""
    rdt, cdt = DT[prec]
    img, vis, wgt = p["img"].astype(rdt), p["vis"].astype(cdt), p["wgt"].astype(rdt)
    x = img.astype(np.float64)
    v = dft.dft_dirty2vis(p["uvw"], p["freq"], x, p["cell"], p["cell"], **kw)
    d = dft.dft_vis2dirty(p["uvw"], p["freq"], vis, wgt, p["mask"], p["nx"], p["ny"], p["cell"], p["cell"], **kw)
    h = dft.dft_vis2dirty(p["uvw"], p["freq"], v, wgt, p["mask"], p["nx"], p["ny"], p["cell"], p["cell"], **kw) / WSUM
    return dict(img=img, vis=vis, wgt=wgt, v=v, d=d, h=h + ETA * x)


@pytest.fixture(scope="module")
def problems():
    """Per geometry: the problem and its DFT references in both precisions (computed once for the module)."""
    out = {}
    for name, g in GEOMS.items():
        p = small_problem(nrow=400, nchan=3, nx=64, ny=48, seed=3, wscale=g["wscale"])
        kw = _kw(g["kw"])
        out[name] = dict(p=p, kw=kw, mirror=g["mirror"], ref={prec: _references(p, kw, prec) for prec in DT})
    return out


def _plan(prob, prec, w, sigma, eps=None):
    p = prob["p"]
    gp = W.plan_for(p["uvw"], p["freq"], npix_x=p["nx"], npix_y=p["ny"], pixsize_x=p["cell"], pixsize_y=p["cell"],
                    epsilon=EPS[prec] if eps is None else eps, precision=prec, mask=p["mask"], force_sigma=sigma,
                    force_W=w, mirror=prob["mirror"], **prob["kw"])
    gp.bind_weights(prob["ref"][prec]["wgt"])
    return gp


def _apply(gp, r):
    return gp.degrid(r["img"]), gp.grid(r["vis"], r["wgt"]), gp.hessian(r["img"], wsum=WSUM, eta=ETA)


def _dft_errors(prob, prec, out):
    act = prob["p"]["mask"] != 0
    r = prob["ref"][prec]
    v, d, h = out
    assert np.all(v[~act] == 0)
    return rel_l2(v[act], r["v"][act]), rel_l2(d, r["d"]), rel_l2(h, r["h"])


def _check_bound(gp, errs, what):
    kerr = gp.plan.kernel_err
    tol = BOUND_C * kerr + FLOOR[gp.plan.precision]
    ev, ed, eh = errs
    print(f"{what}: {gp.plan.precision} W={gp.plan.W} sigma={gp.plan.sigma} nplanes={gp.plan.nplanes} "
          f"kernel_err={kerr:.1e} rel_l2/kernel_err degrid {ev / kerr:.2f} grid {ed / kerr:.2f} hessian {eh / kerr:.2f} "
          f"(degrid {ev:.1e} grid {ed:.1e} hessian {eh:.1e}, tol {tol:.1e})")
    assert ev <= tol, (what, "degrid", ev, tol)
    assert ed <= tol, (what, "grid", ed, tol)
    assert eh <= 2 * tol, (what, "hessian", eh, 2 * tol)


def _check_geometry(gp, geom, w, sigma):
    pl = gp.plan
    assert pl.W == w and pl.sigma == sigma, f"fixture no longer exercises W = {w} at sigma {sigma}: {pl.info()}"
    assert gp.info()["W"] == w
    if geom == "mirror":
        assert pl.pmirror > 0, f"fixture no longer exercises mirror planes: {pl.info()}"
    elif geom == "stack":
        assert pl.pmirror == 0 and pl.nplanes > w, f"fixture no longer exercises a stack of more than W planes: {pl.info()}"
    else:
        assert pl.nplanes == 1 and not pl.do_wgridding, f"fixture no longer exercises 2-D gridding: {pl.info()}"


@pytest.mark.parametrize("geom", list(GEOMS))
@pytest.mark.parametrize("prec,w,sigma", CASES)
def test_run_kernels_at_the_kernel_error_bound(gpu, problems, geom, prec, w, sigma):
    """The default arm of each (precision, W): DFT at the bound, the restatement at round-off, adjointness."""
    prob = problems[geom]
    p, r = prob["p"], prob["ref"][prec]
    with _plan(prob, prec, w, sigma) as gp:
        _check_geometry(gp, geom, w, sigma)
        out = _apply(gp, r)
        _check_bound(gp, _dft_errors(prob, prec, out), f"runs/{geom}")
        v, d, _ = out
        v_np = wg.dirty2vis_np(gp.plan, p["uvw"], p["freq"], r["img"], mask=p["mask"])
        d_np = wg.vis2dirty_np(gp.plan, p["uvw"], p["freq"], r["vis"], r["wgt"], p["mask"])
        tol_np = ROUNDOFF[prec] + ROUNDOFF_KERR[prec] * gp.plan.kernel_err
        assert rel_l2(v, v_np) <= tol_np, ("degrid vs restatement", rel_l2(v, v_np), tol_np)
        assert rel_l2(d, d_np) <= tol_np, ("grid vs restatement", rel_l2(d, d_np), tol_np)
        act = p["mask"] != 0
        lhs = np.vdot(v.astype(np.complex128), (r["vis"] * r["wgt"] * act).astype(np.complex128)).real
        rhs = float((d.astype(np.float64) * r["img"]).sum())
        assert abs(lhs - rhs) <= ADJ[prec] * abs(rhs)


@pytest.mark.parametrize("geom", list(GEOMS))
@pytest.mark.parametrize("prec,w,sigma", CASES)
def test_direct_kernels_at_the_kernel_error_bound(gpu, problems, monkeypatch, geom, prec, w, sigma):
    """k_grid_direct / k_degrid_direct: PFBG_FORCE_DIRECT=1 is read when uvw is bound, so it is set before the plan."""
    prob = problems[geom]
    monkeypatch.setenv("PFBG_FORCE_DIRECT", "1")
    with _plan(prob, prec, w, sigma) as gp:
        _check_geometry(gp, geom, w, sigma)
        _check_bound(gp, _dft_errors(prob, prec, _apply(gp, prob["ref"][prec])), f"direct/{geom}")


@pytest.mark.parametrize("geom", ["mirror", "stack"])
@pytest.mark.parametrize("sigma", [1.5, 2.0])
@pytest.mark.parametrize("fast", [1, 0])
def test_fp32_w8_fast_path_with_both_w_screens(gpu, problems, monkeypatch, geom, sigma, fast):
    """fp32 W = 8 with w-gridding (the run kernels' W = 8 fast path) with the SFU w-screen (epsilon >= 3e-6) and the
    accurate one (PFBG_FAST_SCREEN=0, read when the plan is made)."""
    prob = problems[geom]
    if not fast:
        monkeypatch.setenv("PFBG_FAST_SCREEN", "0")
    with _plan(prob, "single", 8, sigma, eps=1e-5) as gp:
        _check_geometry(gp, geom, 8, sigma)
        assert gp.plan.fast_screen == fast, f"fixture no longer exercises fast_screen = {fast}: {gp.plan.info()}"
        _check_bound(gp, _dft_errors(prob, "single", _apply(gp, prob["ref"]["single"])), f"screen{fast}/{geom}")


# --------------------------------------------------------------------------------------------------------------------
# plane-count parity: fp32 row passes and the band split's plane subsets
# --------------------------------------------------------------------------------------------------------------------
def _parity_problem(nplanes_parity, w, sigma):
    """A problem (nv % 32 == 0: the pair-engine row kernels) whose stack without mirror planes has >= 3 planes of the
    wanted parity, found by widening the w-range."""
    for k in range(40):
        p = small_problem(nrow=500, nchan=3, nx=64, ny=64, seed=21, wscale=2.0 + 0.5 * k)
        wmin, wmax = w_range(p["uvw"], p["freq"])
        pl = make_plan(nx=64, ny=64, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-5, precision="single",
                       wmin=wmin, wmax=wmax, force_sigma=sigma, force_W=w, mirror=False, flip_v=True, divide_by_n=False)
        if pl.nplanes % 2 == nplanes_parity and pl.nplanes >= 3:
            return p
    raise AssertionError("no w-range gives the wanted plane parity")


PARITY = dict(flip_v=True, divide_by_n=False)


def _parity_plan(p, w, sigma, wgrid):
    gp = W.plan_for(p["uvw"], p["freq"], npix_x=p["nx"], npix_y=p["ny"], pixsize_x=p["cell"], pixsize_y=p["cell"],
                    epsilon=1e-5, precision="single", mask=p["mask"], force_sigma=sigma, force_W=w, mirror=False,
                    do_wgridding=wgrid, **PARITY)
    gp.bind_weights(p["wgt"].astype(np.float32))
    return gp


@pytest.mark.parametrize("planes", ["one", "odd", "even"])
@pytest.mark.parametrize("fast", [1, 0])
def test_row_passes_with_odd_and_even_plane_counts(gpu, monkeypatch, planes, fast):
    """nplanes = 1 (no w-gridding), odd >= 3 and even >= 4 through the fp32 row passes, fast w-screen on and off:
    against the DFT at the bound, and against the one-plane row kernels for every plane (PFBG_ROWS=old) at fp32
    round-off.  (Two planes occur only as split subsets, below.)"""
    w, sigma = 6, 2.0
    p = _parity_problem(0 if planes == "even" else 1, w, sigma)
    if not fast:
        monkeypatch.setenv("PFBG_FAST_SCREEN", "0")
    wgrid = planes != "one"
    kw = _kw(dict(PARITY, do_wgridding=wgrid))
    r = _references(p, kw, "single")
    prob = dict(p=p, ref={"single": r})
    res = {}
    with _parity_plan(p, w, sigma, wgrid) as gp:
        n = gp.plan.nplanes
        assert gp.plan.nv % 32 == 0, "fixture no longer exercises the pair-engine row kernels"
        assert (n == 1) if planes == "one" else (n >= 3 and n % 2 == (planes == "odd")), \
            f"fixture no longer exercises {planes} plane counts: {n}"
        assert gp.plan.fast_screen == (fast if wgrid else 0)
        res["split"] = _apply(gp, r)
        _check_bound(gp, _dft_errors(prob, "single", res["split"]), f"rows/{planes}")
    monkeypatch.setenv("PFBG_ROWS", "old")
    with _parity_plan(p, w, sigma, wgrid) as gp:
        res["old"] = _apply(gp, r)
    for a, b, what in zip(res["split"], res["old"], ("degrid", "grid", "hessian")):
        assert rel_l2(a, b) <= 3e-6, ("old", what, rel_l2(a, b))


@pytest.mark.parametrize("parity", [1, 0])
@pytest.mark.parametrize("nq", [1, 2])
def test_split_plane_subsets_of_both_parities(gpu, parity, nq):
    """The one-process band split (test_gpu_split.py) with the owner keeping nplanes - nq planes and the helper nq:
    odd / even nplanes and nq = 1 / 2 give all four owner / helper parity combinations.  The split Hessian against the
    unsplit one and against the DFT composition."""
    import torch

    w, sigma = 6, 2.0
    p = _parity_problem(parity, w, sigma)
    kw = _kw(PARITY)
    r = _references(p, kw, "single")
    gp = _parity_plan(p, w, sigma, True)
    n = gp.plan.nplanes
    assert n % 2 == parity and n > nq + 1, f"fixture no longer exercises {n} planes split {n - nq} + {nq}"
    dev = torch.device("cuda", 0)
    x = torch.from_numpy(r["img"]).to(dev)
    ref = torch.empty_like(x)
    gp.hessian_dev(x.data_ptr(), None, WSUM, ETA, ref.data_ptr(), None)
    torch.cuda.synchronize()
    split = bs.BandSplit({0: gp}, {0: dict(owner=0, helper=0, nq=nq)}, rank=0, device=0, gather=lambda o: [o])
    so, sh = torch.cuda.Stream(dev), torch.cuda.Stream(dev, priority=-1)
    outs = [torch.empty_like(x) for _ in range(2)]
    for o in outs:
        split.serve(sh.cuda_stream)
        gp.hessian_dev(x.data_ptr(), None, WSUM, ETA, o.data_ptr(), so.cuda_stream)
    torch.cuda.synchronize()
    split.check()
    split.close()
    gp.close()
    kerr = gp.plan.kernel_err
    tol = 2 * (BOUND_C * kerr + FLOOR["single"])
    for o in outs:
        h = o.cpu().numpy()
        assert rel_l2(h, ref.cpu().numpy()) <= 2e-6
        e = rel_l2(h, r["h"])
        print(f"split {n - nq} + {nq}: hessian rel_l2/kernel_err {e / kerr:.2f} ({e:.1e}, tol {tol:.1e})")
        assert e <= tol, (e, tol)
