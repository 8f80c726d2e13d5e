"""GPU parity tests (through the C ABI): CUDA path vs the oracle / explicit DFT /
golden vectors.  Tolerances follow BASELINE.json north_star: rel-L2 <= epsilon vs the
DFT (hence <= 2 epsilon vs ducc0), bit-exact binning indices."""
import os

import numpy as np
import pytest

from oracle import dft, wgridder_np as wg
from pfb_imaging_b200 import operators as ops, synth, wgridder as W
from pfbg_testutil import GOLDEN, rel_l2, seed42_array, small_problem

pytestmark = pytest.mark.gpu


def _kat_dirty(npix, dt=np.float64):
    d = np.zeros((npix, npix), dtype=dt)
    d[npix // 2, npix // 2] = 1.0
    d[npix // 4, npix // 4] = 1.0
    return d


@pytest.mark.parametrize("k", range(5))
def test_kat_gridder_conventions(gpu, k):
    """/root/reference/tests/test_hessian_approx.py:70-125 through our dirty2vis, against the
    vectors the reference's explicit_degridder produced (tests/golden/kat_conventions.npz)."""
    g = np.load(os.path.join(GOLDEN, "kat_conventions.npz"))
    npix, pix = int(g["npix"]), float(g["pixsize"])
    l0, m0 = g["offsets"][k]
    vis = W.dirty2vis(uvw=g["uvw"], freq=g["freqs"], dirty=_kat_dirty(npix), wgt=None, pixsize_x=pix, pixsize_y=pix,
                      center_x=-l0, center_y=-m0, epsilon=1e-6, do_wgridding=True, flip_v=False, divide_by_n=True,
                      nthreads=2, verbosity=0)
    for neg in (0, 1):
        ref = g[f"conv_{k}_{neg}"]
        np.testing.assert_allclose(vis.real, ref.real, atol=1e-4)  # the reference's own tolerance
        np.testing.assert_allclose(vis.imag, ref.imag, atol=1e-4)
        assert rel_l2(vis, ref) <= 1e-6


@pytest.mark.parametrize("k", range(5))
def test_kat_wgridder_conventions(gpu, k):
    """tests/test_hessian_approx.py:128-185 (pfb conventions)."""
    g = np.load(os.path.join(GOLDEN, "kat_conventions.npz"))
    npix, pix = int(g["npix"]), float(g["pixsize"])
    l0, m0 = g["offsets"][k]
    fu, fv, fw, x0, y0 = ops.wgridder_conventions(l0, m0)
    vis = W.dirty2vis(uvw=g["uvw"], freq=g["freqs"], dirty=_kat_dirty(npix), wgt=None, pixsize_x=pix, pixsize_y=pix,
                      center_x=x0, center_y=y0, epsilon=1e-6, do_wgridding=True, flip_u=fu, flip_v=fv, flip_w=fw,
                      divide_by_n=True, nthreads=2, verbosity=0)
    ref = g[f"wconv_{k}"]
    np.testing.assert_allclose(vis.real, ref.real, atol=1e-4)
    np.testing.assert_allclose(vis.imag, ref.imag, atol=1e-4)
    assert rel_l2(vis, ref) <= 1e-6


@pytest.mark.parametrize("center", [(0.0, 0.0), (0.1, -0.17), (-0.15, -0.2)])
def test_psfvis_delta_1e10(gpu, center):
    """tests/test_hessian_approx.py:188-231: analytic off-centre point source == dirty2vis(delta), 1e-10."""
    npix, pix, uvw, freq = seed42_array(nsub=7)
    # The reference runs this on a ~km-scale MS; the seed-42 array has 10x longer baselines, whose
    # ~1e4-turn phases put the fp64 rounding floor of the *analytic* expression itself at ~1e-10.
    uvw = 0.1 * uvw
    fu, fv, fw, x0, y0 = ops.wgridder_conventions(*center)
    eps = 1e-10
    n = np.sqrt(1 - x0**2 - y0**2)
    ff = -2j * np.pi * freq[None, :] / 299792458.0
    psf_vis = np.exp(ff * (uvw[:, 0:1] * x0 + uvw[:, 1:2] * y0 - uvw[:, 2:] * (n - 1)))
    x = np.zeros((256, 256))
    x[128, 128] = 1.0
    v = W.dirty2vis(uvw=uvw, freq=freq, dirty=x, pixsize_x=pix, pixsize_y=pix, center_x=x0, center_y=y0,
                    flip_u=fu, flip_v=fv, flip_w=fw, epsilon=eps, nthreads=2, do_wgridding=True, divide_by_n=False)
    assert np.abs(psf_vis - v).max() <= eps


CASES = [
    ("double", 1e-7, dict()),
    ("double", 1e-4, dict(center_x=0.05, center_y=-0.08, flip_v=True)),
    ("double", 1e-9, dict(do_wgridding=False)),
    ("double", 1e-6, dict(flip_u=True, flip_w=True, divide_by_n=False)),
    ("single", 1e-5, dict(flip_v=True, divide_by_n=False)),
    ("single", 1e-4, dict(center_x=-0.02, center_y=0.03)),
    ("single", 1e-3, dict(do_wgridding=False)),
]


@pytest.mark.parametrize("prec,eps,geom", CASES)
def test_parity_with_dft_and_oracle(gpu, prec, eps, geom):
    p = small_problem(nrow=600, nchan=4, nx=96, ny=64)
    rdt, cdt = (np.float32, np.complex64) if prec == "single" else (np.float64, np.complex128)
    kw = dict(center_x=0.0, center_y=0.0, flip_u=False, flip_v=False, flip_w=False, do_wgridding=True, divide_by_n=True)
    kw.update(geom)
    gp = W.plan_for(p["uvw"], p["freq"], npix_x=p["nx"], npix_y=p["ny"], pixsize_x=p["cell"], pixsize_y=p["cell"],
                    epsilon=eps, precision=prec, mask=p["mask"], **kw)
    act = p["mask"] != 0
    # degrid
    ref = dft.dft_dirty2vis(p["uvw"], p["freq"], p["img"], p["cell"], p["cell"], **kw)
    v = gp.degrid(p["img"].astype(rdt))
    assert v.dtype == cdt
    assert rel_l2(v[act], ref[act]) <= eps
    assert np.all(v[~act] == 0)
    # grid
    vis, wgt = p["vis"].astype(cdt), p["wgt"].astype(rdt)
    dref = dft.dft_vis2dirty(p["uvw"], p["freq"], vis, wgt, p["mask"], p["nx"], p["ny"], p["cell"], p["cell"], **kw)
    d = gp.grid(vis, wgt)
    assert d.dtype == rdt
    assert rel_l2(d, dref) <= eps
    # adjointness <Rx,y> = <x,R^H y>
    lhs = np.vdot(v.astype(np.complex128), (vis * wgt * act).astype(np.complex128)).real
    rhs = float((d.astype(np.float64) * p["img"]).sum())
    # (fp64: the low-sigma plans the DMMA run kernels make attractive amplify the FFT round-off at the image corners
    #  by 1/psihat ~ exp(beta - sqrt(beta^2 - (pi W / 2 sigma)^2)) ~ 300 at sigma = 1.25: 7e-12 measured)
    assert abs(lhs - rhs) <= (2e-11 if prec == "double" else 2e-5) * abs(rhs)
    # same plan through the numpy restatement: CUDA kernels vs CPU restatement
    v_np = wg.dirty2vis_np(gp.plan, p["uvw"], p["freq"], p["img"], mask=p["mask"])
    d_np = wg.vis2dirty_np(gp.plan, p["uvw"], p["freq"], vis, wgt, p["mask"])
    tol = 1e-11 if prec == "double" else 2e-5
    assert rel_l2(v, v_np) <= tol and rel_l2(d, d_np) <= tol
    gp.close()


@pytest.mark.parametrize("geom", [dict(), dict(center_x=0.2, center_y=0.5, flip_v=True), dict(do_wgridding=False)])
def test_binning_bit_exact(gpu, geom):
    npix, pix, uvw, freq = seed42_array(nsub=3)
    rng = np.random.default_rng(5)
    mask = (rng.uniform(size=(uvw.shape[0], freq.size)) > 0.2).astype(np.uint8)
    gp = W.plan_for(uvw, freq, npix_x=512, npix_y=384, pixsize_x=pix * 2, pixsize_y=pix * 2, epsilon=1e-6,
                    mask=mask, **geom)
    b = wg.bin_indices(gp.plan, uvw, freq, mask)
    dmp = gp.bin_dump()
    idx = b["idx"]
    for k in ("iu0", "iv0", "ip0", "key"):
        assert np.array_equal(dmp[k][idx], b[k]), k
    assert np.array_equal(dmp["sorted_idx"].astype(np.int64), idx[b["order"]])
    assert gp.info()["nactive"] == idx.size
    gp.close()


def test_api_semantics(gpu):
    p = small_problem(nrow=200, nchan=2, nx=32, ny=32)
    com = dict(uvw=p["uvw"], freq=p["freq"], pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-6)
    # in-place fill of caller arrays, also returned (operators/gridder.py:590-613, 485-503)
    out = np.full((32, 32), np.nan)
    ret = W.vis2dirty(vis=p["vis"], wgt=p["wgt"], mask=p["mask"], npix_x=32, npix_y=32, dirty=out, **com)
    assert ret is out and np.isfinite(out).all()
    vout = np.full(p["vis"].shape, np.nan + 0j)
    ret = W.dirty2vis(dirty=p["img"][:32, :32].copy(), vis=vout, **com)
    assert ret is vout and np.isfinite(vout).all()
    # zero-stride broadcast PSF vis (operators/gridder.py:627-629) and read-only inputs
    ones = np.broadcast_to(np.ones((1,), dtype=np.complex128), p["vis"].shape)
    uvw_ro = p["uvw"].copy()
    uvw_ro.setflags(write=False)
    a = W.vis2dirty(uvw=uvw_ro, freq=p["freq"], vis=ones, wgt=p["wgt"], npix_x=32, npix_y=32,
                    pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-6)
    b = W.vis2dirty(vis=np.ones(p["vis"].shape, dtype=np.complex128), wgt=p["wgt"], npix_x=32, npix_y=32, **com)
    np.testing.assert_allclose(a, b, rtol=1e-11, atol=1e-11 * np.abs(b).max())  # atomics: order varies
    # empty input: zero rows
    z = W.vis2dirty(uvw=np.zeros((0, 3)), freq=p["freq"], vis=np.zeros((0, 2), dtype=np.complex128), npix_x=32,
                    npix_y=32, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-6)
    assert z.shape == (32, 32) and not z.any()
    # fully flagged
    z = W.vis2dirty(vis=p["vis"], mask=np.zeros(p["vis"].shape, np.uint8), npix_x=32, npix_y=32, **com)
    assert not z.any()
    # dtype coupling / shape errors raise
    with pytest.raises(TypeError):
        W.vis2dirty(vis=p["vis"], wgt=p["wgt"].astype(np.float32), npix_x=32, npix_y=32, **com)
    with pytest.raises(ValueError):
        W.vis2dirty(vis=p["vis"][:-1], npix_x=32, npix_y=32, **com)
    with pytest.raises(ValueError):
        W.vis2dirty(vis=p["vis"], npix_x=31, npix_y=32, **com)


@pytest.mark.parametrize("prec", ["double", "single"])
def test_hessian_slice_matches_composition(gpu, prec):
    """hessian_slice == beam * vis2dirty(W * dirty2vis(beam * x)) / wsum + eta x (operators/hessian.py:47-98)."""
    p = small_problem(nrow=500, nchan=3, nx=64, ny=64)
    rdt, cdt = (np.float32, np.complex64) if prec == "single" else (np.float64, np.complex128)
    eps = 1e-5 if prec == "single" else 1e-8
    rng = np.random.default_rng(3)
    x = rng.standard_normal((64, 64)).astype(rdt)
    beam = rng.uniform(0.5, 1.0, (64, 64)).astype(rdt)
    wgt = p["wgt"].astype(rdt)
    wsum = float(wgt[p["mask"] != 0].sum())
    kw = dict(uvw=p["uvw"], weight=wgt, vis_mask=p["mask"], freq=p["freq"], beam=beam, cell=p["cell"], x0=0.01,
              y0=-0.02, epsilon=eps, eta=0.3, wsum=wsum)
    ops.clear_plan_cache()
    h = ops.hessian_slice(x, **kw)
    com = dict(uvw=p["uvw"], freq=p["freq"], pixsize_x=p["cell"], pixsize_y=p["cell"], center_x=0.01, center_y=-0.02,
               flip_v=True, epsilon=eps, divide_by_n=False)
    mv = W.dirty2vis(dirty=x * beam, mask=p["mask"], **com)
    ref = W.vis2dirty(vis=mv, wgt=wgt, mask=p["mask"], npix_x=64, npix_y=64, **com)
    ref = ref / wsum * beam + 0.3 * x
    assert rel_l2(h, ref) <= (1e-10 if prec == "double" else 1e-5)
    # against the DFT composition
    mv_d = dft.dft_dirty2vis(p["uvw"], p["freq"], (x * beam).astype(np.float64), p["cell"], p["cell"], 0.01, -0.02,
                             False, True, False, True, False)
    ref_d = dft.dft_vis2dirty(p["uvw"], p["freq"], mv_d, wgt, p["mask"], 64, 64, p["cell"], p["cell"], 0.01, -0.02,
                              False, True, False, True, False) / wsum * beam + 0.3 * x
    assert rel_l2(h, ref_d) <= 2 * eps
    # zero input short-circuit, xout reuse, cache hit and invalidation on in-place edits
    assert not ops.hessian_slice(np.zeros_like(x), **kw).any()
    xo = np.empty_like(x)
    assert ops.hessian_slice(x, xout=xo, **kw) is xo
    assert rel_l2(xo, h) <= (1e-13 if prec == "double" else 1e-6)  # atomics: summation order varies
    wgt *= 2.0
    kw["wsum"] = 2 * wsum
    h2 = ops.hessian_slice(x, **kw)
    assert rel_l2(h2, h) <= (1e-10 if prec == "double" else 1e-5)  # 2W / 2wsum
    ops.clear_plan_cache()


def test_row_additivity_and_partitions(gpu):
    """tests/test_imager_pass2.py:45-63: gridding is additive over row partitions;
    residual_from_partitions with a zero model returns the dirty image."""
    p = small_problem(nrow=600, nchan=2, nx=48, ny=48)
    com = dict(freq=p["freq"], npix_x=48, npix_y=48, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-7,
               flip_v=True, divide_by_n=False)
    full = W.vis2dirty(uvw=p["uvw"], vis=p["vis"], wgt=p["wgt"], mask=p["mask"], **com)
    a = W.vis2dirty(uvw=p["uvw"][:250], vis=p["vis"][:250], wgt=p["wgt"][:250], mask=p["mask"][:250], **com)
    b = W.vis2dirty(uvw=p["uvw"][250:], vis=p["vis"][250:], wgt=p["wgt"][250:], mask=p["mask"][250:], **com)
    np.testing.assert_allclose(a + b, full, rtol=1e-5, atol=1e-5 * np.abs(full).max())

    class V:
        def __init__(self, v):
            self.values = v

    class Part:
        def __init__(self, sl):
            self.UVW, self.FREQ = V(p["uvw"][sl]), V(p["freq"])
            self.WEIGHT, self.MASK = V(p["wgt"][None, sl]), V(p["mask"][sl])
            self.BEAM = V(np.ones((1, 48, 48)))
            self.attrs = {}

    parts = [Part(slice(0, 250)), Part(slice(250, None))]
    dirty = full[None]
    r0 = ops.residual_from_partitions(dirty, parts, np.zeros((1, 48, 48)), p["cell"])
    assert np.array_equal(r0, dirty)
    model = np.zeros((1, 48, 48))
    model[0, 20, 30] = 1.0
    r = ops.residual_from_partitions(dirty, parts, model, p["cell"])
    one = ops.compute_residual_arrays(p["uvw"], p["wgt"][None], p["mask"], np.ones((1, 48, 48)), dirty, p["freq"],
                                      False, True, False, 0.0, 0.0, 48, 48, p["cell"], p["cell"], model)
    np.testing.assert_allclose(r, one, rtol=1e-6, atol=1e-6 * np.abs(one).max())
    ops.clear_plan_cache()


def test_full_size_properties_c1(gpu):
    """BASELINE config 1 (2048^2, 1M vis, eps 1e-5, fp64): sampled DFT parity, linearity, adjointness."""
    d = synth.make_band(62, 8, band=3, precision="double", flag_frac=0.05)
    uvw, freq = d["uvw"], d["freq"]
    cell = synth.default_cell(uvw, 1712e6)
    nx = 2048
    gp = W.plan_for(uvw, freq, npix_x=nx, npix_y=nx, pixsize_x=cell, pixsize_y=cell, epsilon=1e-5, flip_v=True,
                    divide_by_n=False, mask=d["mask"], sigma_min=1.1, sigma_max=3.0)
    x = synth.point_source_image(nx, nx)
    v = gp.degrid(x)
    rows = np.random.default_rng(0).integers(0, uvw.shape[0], 300)
    ref = dft.dft_dirty2vis(uvw, freq, x, cell, cell, 0, 0, False, True, False, True, False, rows=rows)
    act = d["mask"][rows] != 0
    assert rel_l2(v[rows][act], ref[act]) <= 1e-5
    dimg = gp.grid(d["vis"], d["wgt"])
    rng = np.random.default_rng(1)
    px = (rng.integers(0, nx, 40), rng.integers(0, nx, 40))
    dref = dft.dft_vis2dirty(uvw, freq, d["vis"], d["wgt"], d["mask"], nx, nx, cell, cell, 0, 0, False, True, False,
                             True, False, pixels=px)
    assert rel_l2(dimg[px], dref) <= 1e-5
    lhs = np.vdot(v, d["vis"] * d["wgt"] * (d["mask"] != 0)).real
    rhs = float((dimg * x).sum())
    assert abs(lhs - rhs) <= 1e-11 * abs(rhs)
    # linearity of the fused Hessian
    gp.bind_weights(d["wgt"])
    y = synth.point_source_image(nx, nx, seed=11)
    hx, hy, hxy = gp.hessian(x), gp.hessian(y), gp.hessian(2.0 * x - 3.0 * y)
    assert rel_l2(hxy, 2.0 * hx - 3.0 * hy) <= 1e-11
    gp.close()


def test_plan_pool_reuse_matches_fresh_plans(gpu):
    """One-shot calls re-use pooled plans across different w-ranges / row counts (pfb hci pattern,
    /root/reference/src/pfb_imaging/utils/stokes2im.py:635-683): results must equal those of fresh plans."""
    W.clear_plan_pool()
    outs = []
    probs = [small_problem(nrow=300 + 50 * k, nchan=2, nx=64, ny=64, seed=k, wscale=0.5 + k) for k in range(4)]
    for p in probs:
        outs.append(W.vis2dirty(uvw=p["uvw"], freq=p["freq"], vis=p["vis"], wgt=p["wgt"], mask=p["mask"], npix_x=64,
                                npix_y=64, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-7, flip_v=True,
                                sigma_min=2.0, sigma_max=2.0))
    assert sum(len(v) for v in W._POOL.values()) >= 1
    for p, o in zip(probs, outs):
        with W.plan_for(p["uvw"], p["freq"], npix_x=64, npix_y=64, pixsize_x=p["cell"], pixsize_y=p["cell"],
                        epsilon=1e-7, flip_v=True, sigma_min=2.0, sigma_max=2.0, mask=p["mask"]) as gp:
            ref = gp.grid(p["vis"], p["wgt"])
        assert rel_l2(o, ref) <= 1e-12
        dref = dft.dft_vis2dirty(p["uvw"], p["freq"], p["vis"], p["wgt"], p["mask"], 64, 64, p["cell"], p["cell"], 0, 0,
                                 False, True, False, True, True)
        assert rel_l2(o, dref) <= 1e-7
    W.clear_plan_pool()


@pytest.mark.parametrize("prec,eps", [("single", 1e-5), ("double", 1e-6), ("double", 1e-8)])
def test_aliased_uv_footprints_wrap_around_the_grid(gpu, prec, eps):
    """uv coverage three times wider than the grid: footprints straddle the periodic grid edge in u and v
    (general flush / fetch path of the run kernels) and runs are short.  The DFT is periodic in the same way."""
    p = small_problem(nrow=500, nchan=3, nx=80, ny=64, seed=3)
    uvw = p["uvw"] * np.array([3.0, 3.0, 1.0])
    rdt, cdt = (np.float32, np.complex64) if prec == "single" else (np.float64, np.complex128)
    kw = dict(center_x=0.0, center_y=0.0, flip_u=False, flip_v=True, flip_w=False, do_wgridding=True, divide_by_n=False)
    with W.plan_for(uvw, p["freq"], npix_x=80, npix_y=64, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=eps,
                    precision=prec, mask=p["mask"], **kw) as gp:
        b = wg.bin_indices(gp.plan, uvw, p["freq"], p["mask"])
        wraps = np.count_nonzero((np.mod(b["iu0"], gp.plan.nu) + gp.plan.W > gp.plan.nu) |
                                 (np.mod(b["iv0"], gp.plan.nv) + gp.plan.W > gp.plan.nv))
        assert wraps > 10, "fixture no longer exercises the wrap-around path"
        act = p["mask"] != 0
        v = gp.degrid(p["img"].astype(rdt))
        ref = dft.dft_dirty2vis(uvw, p["freq"], p["img"], p["cell"], p["cell"], **kw)
        assert rel_l2(v[act], ref[act]) <= eps
        vis, wgt = p["vis"].astype(cdt), p["wgt"].astype(rdt)
        d = gp.grid(vis, wgt)
        dref = dft.dft_vis2dirty(uvw, p["freq"], vis, wgt, p["mask"], 80, 64, p["cell"], p["cell"], **kw)
        assert rel_l2(d, dref) <= eps


def test_hermitian_fold_of_negative_w(gpu):
    """Samples with w < 0 are gridded at -(u,v,w) with the conjugate visibility: a data set and its mirror image
    (uvw -> -uvw, vis -> conj vis) must give the same dirty image, and degridding the mirror gives conj(vis)."""
    p = small_problem(nrow=700, nchan=2, nx=64, ny=96, seed=8, wscale=3.0)
    kw = dict(freq=p["freq"], pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-9, flip_v=True, divide_by_n=False)
    assert (p["uvw"][:, 2] < 0).any() and (p["uvw"][:, 2] > 0).any()
    d1 = W.vis2dirty(uvw=p["uvw"], vis=p["vis"], wgt=p["wgt"], mask=p["mask"], npix_x=64, npix_y=96, **kw)
    d2 = W.vis2dirty(uvw=-p["uvw"], vis=np.conj(p["vis"]), wgt=p["wgt"], mask=p["mask"], npix_x=64, npix_y=96, **kw)
    # identical sample set after the fold; only the order of the atomic adds differs (round-off, amplified by
    # the grid correction 1/psihat ~ 1e4 at this accuracy)
    assert rel_l2(d2, d1) <= 1e-10
    v1 = W.dirty2vis(uvw=p["uvw"], dirty=p["img"].T.copy(), mask=p["mask"], **kw)
    v2 = W.dirty2vis(uvw=-p["uvw"], dirty=p["img"].T.copy(), mask=p["mask"], **kw)
    assert rel_l2(v2, np.conj(v1)) <= 1e-10
    # the plane stack only covers |w|
    with W.plan_for(p["uvw"], p["freq"], npix_x=64, npix_y=96, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-9,
                    flip_v=True, divide_by_n=False) as gp:
        wabs = np.abs(p["uvw"][:, 2:3]) * p["freq"][None, :] / 299792458.0
        lo, hi = gp.plan.w0, gp.plan.w0 + (gp.plan.nplanes - 1) * gp.plan.dw
        assert hi >= wabs.max() and gp.plan.nplanes <= int(np.ceil((wabs.max() - wabs.min()) / gp.plan.dw)) + gp.plan.W
        if gp.plan.pmirror:  # planes at (p + 1/2) dw; those below zero are mirrors of planes 0..pmirror-1
            assert lo == 0.5 * gp.plan.dw
        else:
            assert lo <= wabs.min()


def test_full_size_properties_c2_band(gpu):
    """One band of BASELINE config 2 (4096^2, 25.0 M vis, fp32, eps 1e-5): sampled DFT parity in both directions,
    adjointness, and the fused Hessian against the composition of its halves."""
    _c2_band("single", 1e-5, adj=1e-7, hess=2e-6)


def test_full_size_properties_c2_band_fp64(gpu):
    """The same band in fp64 at eps 1e-7 (the c2d workload, pfb's default precision): the plan lands on the DMMA run
    kernels (9 <= W <= 12)."""
    _c2_band("double", 1e-7, adj=1e-12, hess=1e-12, wide=(9, 12))


def _c2_band(prec, eps, adj, hess, wide=None):
    rdt = np.float32 if prec == "single" else np.float64
    d = synth.make_band(775, 16, band=5, nband=8, precision=prec, with_vis=True, flag_frac=0.03)
    uvw, freq = d["uvw"], d["freq"]
    cell = synth.default_cell(uvw, 1712e6)
    nx = 4096
    gp = W.plan_for(uvw, freq, npix_x=nx, npix_y=nx, pixsize_x=cell, pixsize_y=cell, epsilon=eps, flip_v=True,
                    divide_by_n=False, mask=d["mask"], sigma_min=1.1, sigma_max=3.0, precision=prec)
    if wide:
        assert wide[0] <= gp.plan.W <= wide[1], f"fixture no longer exercises the DMMA run kernels: {gp.plan.info()}"
    x = synth.point_source_image(nx, nx, dtype=rdt)
    v = gp.degrid(x)
    rows = np.random.default_rng(0).integers(0, uvw.shape[0], 200)
    ref = dft.dft_dirty2vis(uvw, freq, x.astype(np.float64), cell, cell, 0, 0, False, True, False, True, False, rows=rows)
    act = d["mask"][rows] != 0
    assert rel_l2(v[rows][act], ref[act]) <= eps
    # gridding parity on a row subset small enough for the DFT (row additivity makes the subset a valid problem)
    sub = slice(0, uvw.shape[0], 997)
    with W.plan_for(uvw[sub], freq, npix_x=nx, npix_y=nx, pixsize_x=cell, pixsize_y=cell, epsilon=eps, flip_v=True,
                    divide_by_n=False, mask=d["mask"][sub], sigma_min=1.1, sigma_max=3.0, precision=prec) as gs:
        ds = gs.grid(d["vis"][sub], d["wgt"][sub])
    rng = np.random.default_rng(1)
    px = (rng.integers(0, nx, 48), rng.integers(0, nx, 48))
    dref = dft.dft_vis2dirty(uvw[sub], freq, d["vis"][sub], d["wgt"][sub], d["mask"][sub], nx, nx, cell, cell, 0, 0,
                             False, True, False, True, False, pixels=px)
    # the contract is the L2 norm over the image; on 48 sampled pixels compare against the image-wide scale
    assert np.linalg.norm(ds[px] - dref) / (np.sqrt(48.0) * np.sqrt(np.mean(ds.astype(np.float64) ** 2))) <= eps
    dimg = gp.grid(d["vis"], d["wgt"])
    a = (d["vis"] * d["wgt"] * (d["mask"] != 0)).astype(np.complex128)
    lhs = np.vdot(v.astype(np.complex128), a).real
    rhs = float((dimg.astype(np.float64) * x).sum())
    # random visibilities against a sparse model: both inner products cancel to ~1e-4 of ||Rx|| ||a||, so the
    # natural (Cauchy-Schwarz) scale is used, as in SURVEY §8(d) "adjointness ... / ||...||"
    scale = np.linalg.norm(v.astype(np.complex128)) * np.linalg.norm(a)
    print(f"adjointness defect {abs(lhs - rhs) / scale:.2e} of ||Rx|| ||a||, {abs(lhs - rhs) / abs(rhs):.2e} of the product")
    assert abs(lhs - rhs) <= adj * scale
    gp.bind_weights(d["wgt"])
    h = gp.hessian(x)
    h2 = gp.grid(v, d["wgt"])
    assert rel_l2(h, h2) <= hess
    gp.close()


@pytest.mark.parametrize("prec", ["double", "single"])
@pytest.mark.parametrize("sign", [1.0, -1.0])
def test_psf_phase_ramp_generated_on_device(gpu, prec, sign):
    """SURVEY §8 a13: the off-centre PSF visibilities exp(s 2 pi i f/c (u x0 + v y0 - w (n0-1))) are generated on the
    device; gridding them must equal gridding the array the reference materialises on the host
    (operators/gridder.py:616-629 with s=+1, utils/stokes2im.py:483-486 with s=-1)."""
    p = small_problem(nrow=500, nchan=3, nx=64, ny=80, seed=12)
    l0, m0 = 0.03, -0.02
    fu, fv, fw, x0, y0 = ops.wgridder_conventions(l0, m0)
    rdt, cdt = (np.float32, np.complex64) if prec == "single" else (np.float64, np.complex128)
    eps = 1e-5 if prec == "single" else 1e-9
    n0 = np.sqrt(1 - x0 ** 2 - y0 ** 2)
    ramp = np.exp(sign * 2j * np.pi * p["freq"][None, :] / 299792458.0 *
                  (p["uvw"][:, 0:1] * x0 + p["uvw"][:, 1:2] * y0 - p["uvw"][:, 2:] * (n0 - 1)))
    with W.plan_for(p["uvw"], p["freq"], npix_x=64, npix_y=80, pixsize_x=p["cell"], pixsize_y=p["cell"], center_x=x0,
                    center_y=y0, flip_u=fu, flip_v=fv, flip_w=fw, epsilon=eps, precision=prec, mask=p["mask"],
                    divide_by_n=False) as gp:
        wgt = p["wgt"].astype(rdt)
        a = gp.grid(ramp.astype(cdt), wgt)
        b = gp.grid_psf(x0, y0, wgt=wgt, sign=sign)
        assert b.dtype == rdt
        assert rel_l2(b, a) <= (1e-11 if prec == "double" else 3e-6)
    if sign < 0 or prec == "single":
        return
    # through the reference-level entry point: same PSF as gridding the host-materialised ramp with the sign written
    # at operators/gridder.py:618 (+2j; see SURVEY §8 a13 for the sign trap)
    out = ops.image_data_products_arrays(p["uvw"], p["freq"], p["vis"][None], p["wgt"][None], p["mask"], 64, 80, 96, 120,
                                         p["cell"], p["cell"], l0=l0, m0=m0, epsilon=1e-7, do_dirty=False)
    with W.plan_for(p["uvw"], p["freq"], npix_x=96, npix_y=120, pixsize_x=p["cell"], pixsize_y=p["cell"], center_x=x0,
                    center_y=y0, flip_u=fu, flip_v=fv, flip_w=fw, epsilon=1e-7, precision="double", mask=p["mask"],
                    divide_by_n=False, sigma_min=1.1, sigma_max=3.0) as gp:
        want = gp.grid(ramp, p["wgt"])
    assert rel_l2(out["psf"][0], want) <= 1e-10


def test_recurring_host_buffers_are_page_locked_and_results_unchanged(gpu):
    """Solver-style use: the same x / xout arrays come back every iteration.  From the second call on they are
    registered with CUDA (direct DMA); results must be identical and the registration must die with the array."""
    import gc

    p = small_problem(nrow=400, nchan=2, nx=512, ny=512, seed=5)  # 2 MB images: above the pinning threshold
    W.clear_pinned()
    with W.plan_for(p["uvw"], p["freq"], npix_x=512, npix_y=512, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-6,
                    flip_v=True, divide_by_n=False, mask=p["mask"]) as gp:
        gp.bind_weights(p["wgt"])
        x = np.random.default_rng(0).standard_normal((512, 512))
        out = np.empty_like(x)
        ref = gp.hessian(x).copy()
        for it in range(3):
            gp.hessian(x, out=out)
            # (the order of the fp64 atomic adds differs from call to call; 1/psihat amplifies that round-off)
            np.testing.assert_allclose(out, ref, rtol=0, atol=1e-8 * np.abs(ref).max())
        assert len(W._PIN_REG) == 2  # x and out, registered at their second sighting
        x *= 2.0  # in-place update of a registered buffer is seen by the next call
        gp.hessian(x, out=out)
        np.testing.assert_allclose(out, 2.0 * ref, rtol=0, atol=2e-8 * np.abs(ref).max())
        del x, out
        gc.collect()
        assert len(W._PIN_REG) == 0


def test_beam_is_cached_on_the_device_between_applies(gpu):
    """hessian_slice gets the band's beam on every call (operators/hessian.py:15-35); it is uploaded once and re-used
    while (address, size, strided checksum) stay the same, and re-uploaded when the beam changes."""
    p = small_problem(nrow=300, nchan=2, nx=128, ny=96, seed=9)
    rng = np.random.default_rng(2)
    x = rng.standard_normal((128, 96))
    beam = rng.uniform(0.2, 1.0, (128, 96))
    kw = dict(uvw=p["uvw"], weight=p["wgt"], vis_mask=p["mask"], freq=p["freq"], cell=p["cell"], epsilon=1e-7, wsum=2.0, eta=0.3)
    ops.clear_plan_cache()
    a = ops.hessian_slice(x, beam=beam, **kw)
    b = ops.hessian_slice(x, beam=beam, **kw)       # cached beam
    np.testing.assert_allclose(b, a, rtol=0, atol=1e-9 * np.abs(a).max())
    beam2 = beam * 0.5
    c = ops.hessian_slice(x, beam=beam2, **kw)      # new beam: uploaded again
    ref = 0.25 * (a - 0.3 * x) + 0.3 * x             # beam enters twice, the ridge term not at all
    np.testing.assert_allclose(c, ref, rtol=0, atol=1e-9 * np.abs(a).max())
    beam[...] = beam2                                # in-place change of the first array is noticed (checksum)
    d = ops.hessian_slice(x, beam=beam, **kw)
    np.testing.assert_allclose(d, ref, rtol=0, atol=1e-9 * np.abs(a).max())
    ops.clear_plan_cache()


@pytest.mark.parametrize("prec,eps", [("single", 1e-4), ("double", 1e-7)])
@pytest.mark.parametrize("nx,ny", [(50, 76), (130, 42)])
def test_image_sizes_off_the_vector_path(gpu, prec, eps, nx, ny):
    """ny not a multiple of 8: the fused transforms take their scalar fill / drain loops."""
    p = small_problem(nrow=400, nchan=2, nx=nx, ny=ny, seed=nx)
    rdt, cdt = (np.float32, np.complex64) if prec == "single" else (np.float64, np.complex128)
    kw = dict(center_x=0.0, center_y=0.0, flip_u=False, flip_v=True, flip_w=False, do_wgridding=True, divide_by_n=True)
    with W.plan_for(p["uvw"], p["freq"], npix_x=nx, npix_y=ny, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=eps,
                    precision=prec, mask=p["mask"], **kw) as gp:
        act = p["mask"] != 0
        v = gp.degrid(p["img"].astype(rdt))
        ref = dft.dft_dirty2vis(p["uvw"], p["freq"], p["img"], p["cell"], p["cell"], **kw)
        assert rel_l2(v[act], ref[act]) <= eps
        d = gp.grid(p["vis"].astype(cdt), p["wgt"].astype(rdt))
        dref = dft.dft_vis2dirty(p["uvw"], p["freq"], p["vis"].astype(cdt), p["wgt"].astype(rdt), p["mask"], nx, ny,
                                 p["cell"], p["cell"], **kw)
        assert rel_l2(d, dref) <= eps


def test_fast_screen_phasors_stay_inside_the_error_budget(gpu, monkeypatch):
    """fp32 plans with epsilon >= 3e-6 take the w-screen phasors from the SFU (plan.fast_screen); the switch must
    cost well under epsilon: both variants against the explicit DFT, and against each other, on a wide field."""
    p = small_problem(nrow=800, nchan=4, nx=128, ny=96, seed=21, wscale=3.0)
    kw = dict(flip_v=True, divide_by_n=False)
    eps = 1e-5
    ref = dft.dft_dirty2vis(p["uvw"], p["freq"], p["img"], p["cell"], p["cell"], **kw)
    vis, wgt = p["vis"].astype(np.complex64), p["wgt"].astype(np.float32)
    dref = dft.dft_vis2dirty(p["uvw"], p["freq"], vis, wgt, p["mask"], 128, 96, p["cell"], p["cell"], **kw)
    act = p["mask"] != 0
    res = {}
    for fast in ("1", "0"):
        monkeypatch.setenv("PFBG_FAST_SCREEN", fast)
        W.clear_plan_pool()
        with W.plan_for(p["uvw"], p["freq"], npix_x=128, npix_y=96, pixsize_x=p["cell"], pixsize_y=p["cell"],
                        epsilon=eps, precision="single", mask=p["mask"], **kw) as gp:
            assert gp.plan.fast_screen == int(fast) and gp.plan.nplanes > 1
            v, d = gp.degrid(p["img"].astype(np.float32)), gp.grid(vis, wgt)
        assert rel_l2(v[act], ref[act]) <= eps and rel_l2(d, dref) <= eps
        res[fast] = (v, d)
    assert rel_l2(res["1"][0][act], res["0"][0][act]) <= 0.2 * eps and rel_l2(res["1"][1], res["0"][1]) <= 0.2 * eps
    # tighter requests keep the accurate phasors
    monkeypatch.setenv("PFBG_FAST_SCREEN", "1")
    W.clear_plan_pool()
    with W.plan_for(p["uvw"], p["freq"], npix_x=128, npix_y=96, pixsize_x=p["cell"], pixsize_y=p["cell"],
                    epsilon=1e-6, precision="single", mask=p["mask"], **kw) as gp:
        assert gp.plan.fast_screen == 0
    with W.plan_for(p["uvw"], p["freq"], npix_x=128, npix_y=96, pixsize_x=p["cell"], pixsize_y=p["cell"],
                    epsilon=1e-5, precision="double", mask=p["mask"], **kw) as gp:
        assert gp.plan.fast_screen == 0


def test_sparse_in_place_edits_invalidate_the_cached_binding(gpu):
    """ADVICE r1 (medium): the operator-level plan cache must notice a SINGLE-element in-place edit of the mask, the
    weights or the beam between two hessian_slice calls (the reference keeps no state between calls)."""
    p = small_problem(nrow=3000, nchan=4, nx=64, ny=64, seed=13)
    rng = np.random.default_rng(4)
    x = rng.standard_normal((64, 64))
    beam = rng.uniform(0.5, 1.0, (64, 64))
    mask, wgt = p["mask"].copy(), p["wgt"].copy()
    mask[:] = 1
    kw = dict(uvw=p["uvw"], weight=wgt, vis_mask=mask, freq=p["freq"], cell=p["cell"], epsilon=1e-8, beam=beam)
    ops.clear_plan_cache()

    def fresh():
        ops.clear_plan_cache()
        r = ops.hessian_slice(x, **kw)
        ops.clear_plan_cache()
        return r

    h0 = ops.hessian_slice(x, **kw)
    assert rel_l2(ops.hessian_slice(x, **kw), h0) <= 1e-12  # cache hit
    mask[1717, 2] = 0  # one more flagged sample, off every stride a sampled checksum would look at
    h1 = ops.hessian_slice(x, **kw)
    assert rel_l2(h1, fresh()) <= 1e-12 and rel_l2(h1, h0) > 1e-9
    wgt[1234, 1] *= 3.0  # one re-weighted sample
    h2 = ops.hessian_slice(x, **kw)
    assert rel_l2(h2, fresh()) <= 1e-12 and rel_l2(h2, h1) > 1e-9
    beam[17, 33] = 0.1  # one patched beam pixel
    h3 = ops.hessian_slice(x, **kw)
    assert rel_l2(h3, fresh()) <= 1e-12 and rel_l2(h3, h2) > 1e-9
    ops.clear_plan_cache()


def test_no_mask_zero_leaves_flagged_samples_untouched_on_the_wide_path(gpu):
    """include/pfbgrid.h PFBG_NO_MASK_ZERO: masked output samples keep the caller's values, also for W > 8 (the
    cooperative-team kernels add into the output and used to clear all of it)."""
    import ctypes as C

    from pfb_imaging_b200 import _lib

    p = small_problem(nrow=600, nchan=3, nx=64, ny=64, seed=2)
    for eps, wide in ((1e-10, True), (1e-4, False)):
        with W.plan_for(p["uvw"], p["freq"], npix_x=64, npix_y=64, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=eps,
                        mask=p["mask"], flip_v=True, divide_by_n=False) as gp:
            assert (gp.plan.W > 8) == wide
            ref = gp.degrid(p["img"])
            out = np.full(ref.shape, 7.0 - 3.0j)
            img = np.ascontiguousarray(p["img"])
            _lib.check(gp._lib.pfbg_degrid(gp._h, C.c_void_p(img.ctypes.data), C.c_void_p(out.ctypes.data), None,
                                           _lib.HOST_PTRS | _lib.NO_MASK_ZERO, None))
            act = p["mask"] != 0
            assert np.all(out[~act] == 7.0 - 3.0j) and (~act).sum() > 0
            assert rel_l2(out[act], ref[act]) <= 1e-12
