"""CPU: the numpy restatement of the gridder (oracle/wgridder_np.py) against the explicit DFT at the error bound the
planner designs for, `plan.kernel_err` (plan.py: the 1-D kernel error of the table at (sigma, W)), rather than at the
requested epsilon.  The planner picks W so that kernel_err <= epsilon / safety (3 in fp64, sqrt(3) in fp32), so a test
at epsilon lets a kernel 2-3x worse than its design pass; at `C * kernel_err + floor` it does not.

Measured rel-L2 / kernel_err of the restatement (64 x 48 image, 300 rows x 3 channels, w-gridding with mirror planes,
degrid / grid):

    W    sigma 1.5     sigma 2.0          W    sigma 1.5     sigma 2.0
    4    0.73 / 0.78   0.86 / 1.02        11   0.30 / 0.35   0.58 / 0.53
    5    0.65 / 0.60   0.84 / 0.81        12   0.27 / 0.32   0.49 / 0.51
    6    0.63 / 0.46   0.88 / 0.69        13   0.30 / 0.32   0.45 / 0.46
    7    0.51 / 0.42   0.77 / 0.62        14   0.35 / 0.31   0.48 / 0.44
    8    0.36 / 0.36   0.60 / 0.55        15   0.24 / 0.25   0.59 / 0.54
    9    0.26 / 0.32   0.78 / 0.63        16   0.31 / 0.29   1.72 / 1.70
    10   0.42 / 0.37   0.70 / 0.59

(W = 16 at sigma 2: kernel_err is 1.2e-14 and the fp64 round-off of the transforms, ~2e-14, dominates.)  Without
w-gridding, and with a plane stack without mirror planes, the ratios are within 0.05 of these.  The bound is therefore
sharp: `BOUND_C = 2` leaves twice the worst ratio as headroom, and `FLOOR_F64` covers the round-off.  The GPU tests
(tests/test_gpu_widths.py) hold the CUDA kernels to the same bound, so a failure there points at a kernel, not at the
table."""
import numpy as np
import pytest

from oracle import dft, wgridder_np as wg
from pfb_imaging_b200.plan import make_plan, w_range
from pfbg_testutil import rel_l2, small_problem

BOUND_C = 2.0
FLOOR_F64 = 5e-13

GEOMS = {
    "mirror": (1.0, True, dict()),
    "stack": (4.0, False, dict()),
    "nowgrid": (1.0, True, dict(do_wgridding=False)),
}


@pytest.fixture(scope="module")
def refs():
    out = {}
    for name, (wscale, _, geom) in GEOMS.items():
        p = small_problem(nrow=300, nchan=3, nx=64, ny=48, wscale=wscale)
        kw = dict(center_x=0.0, center_y=0.0, flip_u=False, flip_v=False, flip_w=False, do_wgridding=True,
                  divide_by_n=True)
        kw.update(geom)
        v = dft.dft_dirty2vis(p["uvw"], p["freq"], p["img"], p["cell"], p["cell"], **kw)
        d = dft.dft_vis2dirty(p["uvw"], p["freq"], p["vis"], p["wgt"], p["mask"], p["nx"], p["ny"], p["cell"],
                              p["cell"], **kw)
        out[name] = (p, kw, v, d)
    return out


@pytest.mark.parametrize("geom", list(GEOMS))
@pytest.mark.parametrize("sigma", [1.5, 2.0])
@pytest.mark.parametrize("W", range(4, 17))
def test_restatement_meets_the_kernel_error_bound(refs, geom, sigma, W):
    p, kw, vref, dref = refs[geom]
    mirror = GEOMS[geom][1]
    wmin, wmax = w_range(p["uvw"], p["freq"]) if kw["do_wgridding"] else (0.0, 0.0)
    plan = make_plan(nx=p["nx"], ny=p["ny"], pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-3, wmin=wmin,
                     wmax=wmax, nvis=p["vis"].size, force_sigma=sigma, force_W=W, mirror=mirror, **kw)
    assert plan.W == W and plan.sigma == sigma
    if geom == "mirror":
        assert plan.pmirror > 0, "fixture no longer exercises mirror planes"
    if geom == "stack":
        assert plan.pmirror == 0 and plan.nplanes > W, "fixture no longer exercises a stack of more than W planes"
    act = p["mask"] != 0
    tol = BOUND_C * plan.kernel_err + FLOOR_F64
    v = wg.dirty2vis_np(plan, p["uvw"], p["freq"], p["img"], mask=p["mask"])
    d = wg.vis2dirty_np(plan, p["uvw"], p["freq"], p["vis"], p["wgt"], p["mask"])
    e_v, e_d = rel_l2(v[act], vref[act]), rel_l2(d, dref)
    assert e_v <= tol, (e_v / plan.kernel_err, plan.kernel_err)
    assert e_d <= tol, (e_d / plan.kernel_err, plan.kernel_err)
    # the bound is sharp: a restatement far better than the table would mean the table (or the DFT) is off
    assert max(e_v, e_d) >= 0.1 * plan.kernel_err, (e_v, e_d, plan.kernel_err)
