"""GPU: the scalar branches of the row passes and caller device pointers below 16-byte alignment.

k_rows_fwd / k_rows2_fwd (degrid direction) and k_rows_inv / k_rows2_inv (grid direction) read and write image rows
four pixels at a time when ny % 8 == 0 and, in the forward kernels, when x, corr and beam are 16-byte aligned; every
other case takes a scalar branch.  pfb's image sizes only need to be even, so ny % 8 in {2, 4, 6} is an ordinary
input, and a caller may pass views into a larger device buffer.

Which row kernel runs: fp32 plans whose nv fits the pair engine (rows2_supported: nv % 32 == 0, which padded_size
always gives, and ~14 k cells of shared memory) run all planes of an even count and all but the last of an odd one
on k_rows2_*, the last one on k_rows_*; PFBG_ROWS=old runs every plane on k_rows_*.  fp64 plans always run
k_rows_*; beyond ROWS_BIG_SMEM (fused_common.cuh) of shared memory per row
the BIG variants (PFBG_ROWS_SMALL=1: the ordinary ones).  A plan with nv % 32 != 0 cannot be made (plan.padded_size
rounds nv up to a multiple of 32), so the one-plane kernels are reached through fp64, the odd last plane and
PFBG_ROWS=old instead.

Truth is the explicit DFT (oracle/dft.py); rel-L2 <= epsilon, 2 epsilon for the Hessian, which gets a non-unit beam
(the forward scalar branch multiplies by it on a line of its own); two arms of the same plan agree at round-off."""
import numpy as np
import pytest

from oracle import dft
from pfb_imaging_b200 import wgridder as W
from pfb_imaging_b200.plan import make_batch_plan, make_plan, w_range
from pfbg_testutil import rel_l2, small_problem

pytestmark = pytest.mark.gpu

KW = dict(center_x=0.0, center_y=0.0, flip_u=False, flip_v=True, flip_w=False, do_wgridding=True, divide_by_n=False)
EPS = {"single": 1e-5, "double": 1e-8}
ROUNDOFF = {"single": 3e-6, "double": 1e-11}
DT = {"single": (np.float32, np.complex64), "double": (np.float64, np.complex128)}
WSUM, ETA = 2.0, 0.25
ROWS_BIG_SMEM = 113 * 1024  # fused_common.cuh
COLS2_MAX_SMEM = 232448  # fft_host.h: kMaxSmem


def _fft_smem_bytes(n, prec):  # fft.cuh: one pad element per 16 (fp32) / 8 (fp64) elements
    return (n - 1 + ((n - 1) >> (4 if prec == "single" else 3)) + 1) * (8 if prec == "single" else 16)


def _rows2_on(nv, prec):  # colsfft.cu: rows2_supported
    return prec == "single" and nv % 32 == 0 and nv * 16 + ((nv + 63) // 64 + 64) * 8 <= COLS2_MAX_SMEM


def _beam(nx, ny, shift=0.0):
    """A smooth non-unit beam."""
    lx = np.linspace(-1, 1, nx)[:, None]
    ly = np.linspace(-1, 1, ny)[None, :]
    return 0.4 + 0.6 * np.exp(-((lx - shift) ** 2 + ly ** 2))


def _problem(nx, ny, prec, parity, nrow=300, seed=7):
    """A problem whose plan without mirror planes has >= 3 planes of the wanted parity (by widening the w-range)."""
    for k in range(60):
        p = small_problem(nrow=nrow, nchan=3, nx=nx, ny=ny, seed=seed, wscale=2.0 + 0.5 * k)
        wmin, wmax = w_range(p["uvw"], p["freq"])
        pl = make_plan(nx=nx, ny=ny, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=EPS[prec], precision=prec,
                       wmin=wmin, wmax=wmax, force_sigma=2.0, mirror=False, flip_v=True, divide_by_n=False)
        if pl.nplanes % 2 == parity and pl.nplanes >= 3:
            return p
    raise AssertionError("no w-range gives the wanted plane parity")


def _refs(p, prec, beam, pixels=None):
    """DFT degrid of the image, grid of the visibilities and the Hessian beam G^H W G (beam x) / wsum + eta x."""
    rdt, cdt = DT[prec]
    nx, ny, cell = p["nx"], p["ny"], p["cell"]
    img, vis, wgt, beam = p["img"].astype(rdt), p["vis"].astype(cdt), p["wgt"].astype(rdt), beam.astype(rdt)
    bx = img.astype(np.float64) * beam
    v = dft.dft_dirty2vis(p["uvw"], p["freq"], img.astype(np.float64), cell, cell, **KW)
    vb = dft.dft_dirty2vis(p["uvw"], p["freq"], bx, cell, cell, **KW)
    d = dft.dft_vis2dirty(p["uvw"], p["freq"], vis, wgt, p["mask"], nx, ny, cell, cell, pixels=pixels, **KW)
    h = dft.dft_vis2dirty(p["uvw"], p["freq"], vb, wgt, p["mask"], nx, ny, cell, cell, pixels=pixels, **KW)
    sel = (slice(None), slice(None)) if pixels is None else pixels
    h = h * beam[sel] / WSUM + ETA * img.astype(np.float64)[sel]
    return dict(img=img, vis=vis, wgt=wgt, beam=beam, v=v, d=d, h=h, px=sel)


def _plan(p, prec):
    gp = W.plan_for(p["uvw"], p["freq"], npix_x=p["nx"], npix_y=p["ny"], pixsize_x=p["cell"], pixsize_y=p["cell"],
                    epsilon=EPS[prec], precision=prec, mask=p["mask"], force_sigma=2.0, mirror=False, **KW)
    return gp


def _apply(gp, r):
    gp.bind_weights(r["wgt"])
    return gp.degrid(r["img"]), gp.grid(r["vis"], r["wgt"]), gp.hessian(r["img"], beam=r["beam"], wsum=WSUM, eta=ETA)


def _check_dft(p, r, out, eps, what):
    v, d, h = out
    act = p["mask"] != 0
    assert np.all(v[~act] == 0)
    ev, ed, eh = rel_l2(v[act], r["v"][act]), rel_l2(d[r["px"]], r["d"]), rel_l2(h[r["px"]], r["h"])
    print(f"{what}: degrid {ev:.1e} grid {ed:.1e} hessian {eh:.1e} (eps {eps:g})")
    assert ev <= eps and ed <= eps and eh <= 2 * eps, (what, ev, ed, eh)


def _check_arms(a, b, prec, what):
    for x, y, name in zip(a, b, ("degrid", "grid", "hessian")):
        assert rel_l2(x, y) <= ROUNDOFF[prec], (what, name, rel_l2(x, y))


@pytest.mark.parametrize("planes", ["odd", "even"])
@pytest.mark.parametrize("prec,fast", [("single", 1), ("single", 0), ("double", 0)])
@pytest.mark.parametrize("ny", [250, 252, 254])
def test_scalar_row_branches(gpu, monkeypatch, ny, prec, fast, planes):
    """ny % 8 in {2, 4, 6}: fp32 on the pair engine (nv = 512) with the fast w-screen on and off, fp64 on the one-plane
    kernels; odd and even plane counts.  fp32: against every plane on the one-plane kernels at round-off."""
    if not fast and prec == "single":
        monkeypatch.setenv("PFBG_FAST_SCREEN", "0")
    nx = 64
    p = _problem(nx, ny, prec, 1 if planes == "odd" else 0)
    r = _refs(p, prec, _beam(nx, ny))
    with _plan(p, prec) as gp:
        pl = gp.plan
        assert pl.ny % 8 != 0, "fixture no longer exercises ny % 8 != 0"
        assert pl.nplanes % 2 == (planes == "odd") and pl.nplanes >= 3, f"fixture no longer has {planes} planes"
        assert _fft_smem_bytes(pl.nv, prec) <= ROWS_BIG_SMEM, "fixture no longer exercises the ordinary row kernels"
        if prec == "single":
            assert _rows2_on(pl.nv, prec), f"fixture no longer exercises the pair-engine rows: nv = {pl.nv}"
            assert pl.fast_screen == fast, f"fixture no longer exercises fast_screen = {fast}"
        out = _apply(gp, r)
        _check_dft(p, r, out, EPS[prec], f"rows ny={ny} {prec} fast={fast} {planes} P={pl.nplanes}")
    if prec == "double":
        return
    monkeypatch.setenv("PFBG_ROWS", "old")  # read when the plan sets up its transforms
    with _plan(p, prec) as gp:
        _check_arms(out, _apply(gp, r), prec, "PFBG_ROWS=old")


@pytest.mark.parametrize("planes", ["odd", "even"])
def test_big_rows_fp64_scalar_branch(gpu, monkeypatch, planes):
    """fp64 rows longer than ROWS_BIG_SMEM of shared memory (k_rows_*<double, BIG>) with ny % 8 == 6: sampled DFT,
    and the ordinary row kernels (PFBG_ROWS_SMALL=1, read per call) at round-off."""
    prec, nx, ny = "double", 32, 3302
    p = _problem(nx, ny, prec, 1 if planes == "odd" else 0, nrow=200)
    rng = np.random.default_rng(3)
    px = (np.concatenate([[nx // 2, 0, nx - 1], rng.integers(0, nx, 45)]),
          np.concatenate([[ny // 2, ny - 1, 0], rng.integers(0, ny, 45)]))
    r = _refs(p, prec, _beam(nx, ny), pixels=px)
    with _plan(p, prec) as gp:
        pl = gp.plan
        assert pl.ny % 8 != 0, "fixture no longer exercises ny % 8 != 0"
        assert _fft_smem_bytes(pl.nv, prec) > ROWS_BIG_SMEM, f"fixture no longer exercises BIG rows: nv = {pl.nv}"
        assert pl.nplanes % 2 == (planes == "odd"), f"fixture no longer has {planes} planes"
        out = _apply(gp, r)
        _check_dft(p, r, out, EPS[prec], f"BIG rows nv={pl.nv} P={pl.nplanes}")
        monkeypatch.setenv("PFBG_ROWS_SMALL", "1")
        _check_arms(out, _apply(gp, r), prec, "PFBG_ROWS_SMALL=1")


@pytest.mark.parametrize("prec", ["single", "double"])
def test_batched_scalar_rows_with_per_snapshot_beams(gpu, prec):
    """Batched snapshots of 64 x 254 (ny % 8 == 6) with different plane counts, so that pair-engine CTAs straddle
    snapshots, each snapshot with its own beam: every snapshot against its DFT."""
    nx, ny, eps = 64, 254, EPS[prec]
    rdt, cdt = DT[prec]
    ps = [small_problem(nrow=150 + 40 * s, nchan=3, nx=nx, ny=ny, seed=30 + s, wscale=1.0 + 6.0 * s * s)
          for s in range(4)]
    for p in ps:
        p["cell"], p["freq"] = ps[0]["cell"], ps[0]["freq"]
    cell, freq = ps[0]["cell"], ps[0]["freq"]
    beams = np.stack([_beam(nx, ny, shift=0.3 * s) for s in range(4)]).astype(rdt)
    refs = [_refs(p, prec, beams[s]) for s, p in enumerate(ps)]
    wr = [w_range(p["uvw"], freq) for p in ps]
    _, _, npl = make_batch_plan(wr, nvis_per_snapshot=max(p["vis"].size for p in ps), nx=nx, ny=ny, pixsize_x=cell,
                                pixsize_y=cell, epsilon=eps, precision=prec, **KW)
    pbase = np.concatenate([[0], np.cumsum(npl)[:-1]])
    assert np.any(npl % 2 == 1) and np.any(pbase[1:] % 2 == 1), f"fixture no longer straddles snapshots: {npl}"
    gp = W.batch_plan_for([p["uvw"] for p in ps], freq, npix_x=nx, npix_y=ny, pixsize_x=cell, pixsize_y=cell,
                          epsilon=eps, precision=prec, mask_list=[p["mask"] for p in ps], **KW)
    try:
        assert np.array_equal(gp.info()["nplanes"], npl.sum())
        if prec == "single":
            assert _rows2_on(gp.plan.nv, prec), "fixture no longer exercises the pair-engine rows"
        x = np.stack([r["img"] for r in refs])
        wgt = np.concatenate([r["wgt"] for r in refs])
        v = gp.degrid(x)
        d = gp.grid(np.concatenate([r["vis"] for r in refs]), wgt)
        gp.bind_weights(wgt)
        h = gp.hessian(x, beam=beams, wsum=WSUM, eta=ETA)
        ro = gp.row_offsets
        for s, (p, r) in enumerate(zip(ps, refs)):
            _check_dft(p, r, (v[ro[s]:ro[s + 1]], d[s], h[s]), eps, f"batch {prec} snapshot {s} P={npl[s]}")
    finally:
        gp.close()


@pytest.mark.parametrize("planes", ["odd", "even"])
@pytest.mark.parametrize("prec", ["single", "double"])
def test_unaligned_device_pointers(gpu, prec, planes):
    """hessian_dev / degrid_dev with x and beam as views one element into a larger torch buffer (4 B / 8 B off, below
    16-byte alignment) and ny % 8 == 0, so the pointer alone selects the scalar branch: against the aligned call at
    round-off and against the DFT."""
    import torch

    nx, ny = 64, 48
    p = _problem(nx, ny, prec, 1 if planes == "odd" else 0)
    r = _refs(p, prec, _beam(nx, ny))
    tdt = torch.float32 if prec == "single" else torch.float64
    dev = torch.device("cuda", 0)

    def views(off):
        xb = torch.zeros(nx * ny + off, dtype=tdt, device=dev)
        bb = torch.zeros(nx * ny + off, dtype=tdt, device=dev)
        xv, bv = xb[off:].view(nx, ny), bb[off:].view(nx, ny)
        xv.copy_(torch.from_numpy(r["img"]))
        bv.copy_(torch.from_numpy(r["beam"]))
        return xb, bb, xv, bv

    with _plan(p, prec) as gp:
        assert gp.plan.ny % 8 == 0
        gp.bind_weights(r["wgt"])
        res = {}
        for off in (0, 1):
            xb, bb, xv, bv = views(off)
            assert (xv.data_ptr() % 16 != 0) == (off == 1) and (bv.data_ptr() % 16 != 0) == (off == 1), \
                "fixture no longer passes unaligned pointers"
            h = torch.empty((nx, ny), dtype=tdt, device=dev)
            vis = torch.empty(p["vis"].shape, dtype=torch.complex64 if prec == "single" else torch.complex128, device=dev)
            gp.hessian_dev(xv.data_ptr(), bv.data_ptr(), WSUM, ETA, h.data_ptr())
            gp.degrid_dev(xv.data_ptr(), vis.data_ptr())
            torch.cuda.synchronize(dev)
            res[off] = (vis.cpu().numpy(), h.cpu().numpy())
    for a, b, name in zip(res[0], res[1], ("degrid", "hessian")):
        assert rel_l2(b, a) <= ROUNDOFF[prec], (name, rel_l2(b, a))
    v, h = res[1]
    act = p["mask"] != 0
    ev, eh = rel_l2(v[act], r["v"][act]), rel_l2(h, r["h"])
    print(f"unaligned {prec} {planes}: degrid {ev:.1e} hessian {eh:.1e}")
    assert ev <= EPS[prec] and eh <= 2 * EPS[prec], (ev, eh)
