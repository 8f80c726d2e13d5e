"""fp64 run kernels on the DMMA path (csrc/runs_mma.cuh, 9 <= W <= 12) against the explicit DFT and against the
direct kernels (k_grid_direct / k_degrid_direct, PFBG_FORCE_DIRECT=1), which evaluate every tap with the library's
exp / sqrt straight from uvw.  Tolerance: rel-L2 <= epsilon vs the DFT (north_star), and fp64 round-off between the
two kernel families (the same kernel, different tap arithmetic and summation order)."""
import numpy as np
import pytest

from oracle import dft
from pfb_imaging_b200 import wgridder as W
from pfbg_testutil import rel_l2, small_problem

pytestmark = pytest.mark.gpu


def _both(monkeypatch, make):
    """make() bound as usual (the DMMA kernels) and bound with PFBG_FORCE_DIRECT=1 (the direct kernels: the variable
    is read when uvw is bound)"""
    gp = make()
    with monkeypatch.context() as m:
        m.setenv("PFBG_FORCE_DIRECT", "1")
        gd = make()
    return gp, gd


# (epsilon, sigma range) chosen so that the plan lands on W = 9 .. 12
@pytest.mark.parametrize("eps,smin,smax,geom", [
    (1e-7, 1.4, 1.4, dict()),
    (1e-7, 2.0, 2.0, dict(flip_v=True, divide_by_n=False)),
    (1e-8, 1.9, 1.9, dict(center_x=0.03, center_y=-0.02)),
    (1e-8, 2.0, 2.0, dict(do_wgridding=False)),
    (3e-7, 1.35, 1.35, dict(flip_u=True, flip_w=True)),
    (3e-7, 1.85, 1.85, dict(flip_v=True)),
])
def test_mma_kernels_vs_dft_and_direct_kernels(gpu, monkeypatch, eps, smin, smax, geom):
    p = small_problem(nrow=900, nchan=4, nx=96, ny=64, wscale=3.0)
    kw = dict(center_x=0.0, center_y=0.0, flip_u=False, flip_v=False, flip_w=False, do_wgridding=True, divide_by_n=True)
    kw.update(geom)
    gp, gd = _both(monkeypatch, lambda: W.plan_for(
        p["uvw"], p["freq"], npix_x=p["nx"], npix_y=p["ny"], pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=eps,
        precision="double", mask=p["mask"], sigma_min=smin, sigma_max=smax, **kw))
    assert 9 <= gp.info()["W"] <= 12, gp.info()
    act = p["mask"] != 0
    v_mma, v_dir = gp.degrid(p["img"]), gd.degrid(p["img"])
    ref = dft.dft_dirty2vis(p["uvw"], p["freq"], p["img"], p["cell"], p["cell"], **kw)
    assert rel_l2(v_mma[act], ref[act]) <= eps
    assert np.all(v_mma[~act] == 0)
    d_mma, d_dir = gp.grid(p["vis"], p["wgt"]), gd.grid(p["vis"], p["wgt"])
    print(f"W={gp.info()['W']}: DMMA vs direct: degrid {rel_l2(v_mma, v_dir):.2e}, grid {rel_l2(d_mma, d_dir):.2e}")
    assert rel_l2(v_mma, v_dir) <= 1e-13
    dref = dft.dft_vis2dirty(p["uvw"], p["freq"], p["vis"], p["wgt"], p["mask"], p["nx"], p["ny"], p["cell"],
                             p["cell"], **kw)
    assert rel_l2(d_mma, dref) <= eps
    assert rel_l2(d_mma, d_dir) <= 1e-13
    # adjointness of the DMMA pair
    lhs = np.vdot(v_mma, p["vis"] * p["wgt"] * act).real
    rhs = float((d_mma * p["img"]).sum())
    assert abs(lhs - rhs) <= 1e-12 * abs(rhs)
    gp.close()
    gd.close()


def test_mma_hessian_long_runs_and_tail_batches(gpu, monkeypatch):
    """Many samples per footprint origin (runs longer than a batch), a sample count that is not a multiple of the
    batch, and the fused Hessian (bucket-order model visibilities, phases skipped)."""
    rng = np.random.default_rng(5)
    p = small_problem(nrow=37, nchan=2, nx=64, ny=64, wscale=2.0)
    uvw = np.repeat(p["uvw"], 41, axis=0) + rng.normal(scale=1e-3, size=(37 * 41, 3))  # 41 near-copies of every row
    wgt = rng.uniform(0.5, 1.5, (uvw.shape[0], 2))
    mask = (rng.uniform(size=wgt.shape) > 0.1).astype(np.uint8)
    x = p["img"]
    kw = dict(npix_x=64, npix_y=64, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-7, precision="double",
              mask=mask, sigma_min=1.4, sigma_max=1.4, flip_v=True, divide_by_n=False)
    gp, gd = _both(monkeypatch, lambda: W.plan_for(uvw, p["freq"], **kw))
    assert 9 <= gp.info()["W"] <= 12
    gp.bind_weights(wgt)
    gd.bind_weights(wgt)
    h_mma, h_dir = gp.hessian(x, wsum=1.0, eta=0.0), gd.hessian(x, wsum=1.0, eta=0.0)
    v = gp.degrid(x)
    ref = gp.grid(v, wgt)
    print(f"W={gp.info()['W']}: DMMA vs direct: hessian {rel_l2(h_mma, h_dir):.2e}")
    assert rel_l2(h_mma, h_dir) <= 1e-13
    assert rel_l2(h_mma, ref) <= 1e-12
    gp.close()
    gd.close()


@pytest.mark.parametrize("beta", [13.7, 16.4, 23.34, 31.0, 37.0])
def test_lean_fp64_tap_against_numpy(gpu, beta):
    """The taps of the DMMA kernels (a * rsqrt(a) + Cody-Waite exp, no special cases) against numpy's exp / sqrt over
    the whole support, including both ends and the values next to them."""
    import ctypes as C

    from pfb_imaging_b200 import _lib

    lib = _lib.load()
    x = np.concatenate([np.linspace(-1.0, 1.0, 200001), [np.nextafter(1.0, 0.0), np.nextafter(-1.0, 0.0), 0.0],
                        1.0 - np.logspace(-16, -1, 64)])
    out = np.empty_like(x)
    _lib.check(lib.pfbg_debug_es_fast64(0, x.size, x.ctypes.data_as(C.c_void_p), float(beta), out.ctypes.data_as(C.c_void_p)))
    ref = np.exp(beta * (np.sqrt((1.0 - x) * (1.0 + x)) - 1.0))
    rel = np.abs(out - ref) / ref
    print(f"beta {beta}: max rel err {rel.max():.2e}")
    assert rel.max() <= 2e-14  # ~ beta ulps; the requested accuracies end at 1e-10
