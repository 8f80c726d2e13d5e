"""GPU parity of the device SARA backward step (SURVEY §8 f2) against vectors produced by the reference's own
numba code (tests/golden/sara.npz) and against the numpy restatement (oracle/sara_np.py).  fp64 tolerance 1e-11
absolute on O(1) data (the reference compiles with fastmath, so summation order differs); fp32 1e-5 relative."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "sara.npz"))


def _s(a):
    """The elements of `a` the golden file keeps of each output: every G["stride"]-th of the flattened array."""
    return np.asarray(a).reshape(-1)[::int(G["stride"])]


def _case(tag):
    nx, ny, nband, nlevel, nxmax, nymax = (int(v) for v in G[f"{tag}_meta"])
    return nx, ny, nband, nlevel, [str(b) for b in G[f"{tag}_bases"]]


@pytest.mark.parametrize("tag", ["a", "b", "d"])
def test_psi_nocopyt_matches_reference(tag):
    from oracle import sara_np as so
    from pfb_imaging_b200 import wavelet_filters as wf
    from pfb_imaging_b200.sara import PsiNocopyt

    nx, ny, nband, nlevel, bases = _case(tag)
    psi = PsiNocopyt(nband, nx, ny, bases, nlevel, 1)
    x = G[f"{tag}_x"]
    alpha = np.random.default_rng(0).standard_normal(psi.coeff_shape)  # must be overwritten
    psi.dot(x, alpha)
    np.testing.assert_allclose(_s(alpha), G[f"{tag}_x_alpha"], rtol=0, atol=1e-11)
    # every coefficient: against the numpy restatement, which the golden samples pin to the reference
    bk = wf.bookkeeping(nx, ny, bases, nlevel)
    fbs = [None if b == "self" else wf.filter_bank(b) for b in bases]
    np.testing.assert_allclose(alpha, np.stack([so.psi_dot(x[b], bk, fbs) for b in range(nband)]), rtol=0, atol=1e-11)
    xr = np.random.default_rng(1).standard_normal(x.shape)
    psi.hdot(alpha, xr)
    np.testing.assert_allclose(_s(xr), G[f"{tag}_x_xrec"], rtol=0, atol=1e-11)
    np.testing.assert_allclose(xr, len(bases) * x, rtol=0, atol=1e-11)  # tests/test_psi_operator.py:24-53
    # the reference's input was 0.5 * (its alpha, reversed) + 0.25; its alpha equals this one to ~2e-15
    a2 = np.ascontiguousarray(0.5 * alpha[..., ::-1, ::-1] + 0.25)
    psi.hdot(a2, xr)
    np.testing.assert_allclose(_s(xr), G[f"{tag}_x_xr2"], rtol=0, atol=1e-11)
    np.testing.assert_allclose(xr, np.stack([so.psi_hdot(a2[b], bk, fbs) for b in range(nband)]), rtol=0, atol=1e-11)
    psi.close()


def test_psi_transposed_layout_matches_reference():
    from pfb_imaging_b200.sara import Psi

    nx, ny, nband, nlevel, bases = _case("a")
    nxmax, nymax = (int(v) for v in G["a_meta"][4:])
    psi = Psi(nband, nx, ny, bases, nlevel, 1)
    assert psi.coeff_shape == (nband, len(bases), nymax, nxmax)
    alpha = np.empty(psi.coeff_shape)
    psi.dot(G["a_x"], alpha)
    np.testing.assert_allclose(_s(alpha), G["a_t_alpha"], rtol=0, atol=1e-11)
    xr = np.empty_like(G["a_x"])
    psi.hdot(np.ascontiguousarray(0.5 * alpha[..., ::-1, ::-1] + 0.25), xr)
    np.testing.assert_allclose(_s(xr), G["a_t_xr2"], rtol=0, atol=1e-11)
    with pytest.raises(ValueError):
        psi.dot(G["a_x"], np.empty(psi.coeff_shape[:2] + (3, 3)))


@pytest.mark.parametrize("nx,ny,nband,nlevel", [(128, 64, 3, 1), (250, 78, 2, 2), (240, 150, 6, 2), (64, 64, 1, 3)])
def test_psi_against_oracle_and_identity(nx, ny, nband, nlevel):
    from oracle import sara_np as so
    from pfb_imaging_b200 import wavelet_filters as wf
    from pfb_imaging_b200.sara import PsiNocopyt

    bases = ["self", "db1", "db2", "db3", "db4"] if nlevel < 3 else ["db1", "db2", "self"]
    rng = np.random.default_rng(420)
    x = rng.standard_normal((nband, nx, ny))
    psi = PsiNocopyt(nband, nx, ny, bases, nlevel, 1)
    alpha = np.empty(psi.coeff_shape)
    psi.dot(x, alpha)
    bk = wf.bookkeeping(nx, ny, bases, nlevel)
    fbs = [None if b == "self" else wf.filter_bank(b) for b in bases]
    for b in range(nband):
        np.testing.assert_allclose(alpha[b], so.psi_dot(x[b], bk, fbs), rtol=0, atol=1e-11)
    xr = np.empty_like(x)
    psi.hdot(alpha, xr)
    np.testing.assert_allclose(xr, len(bases) * x, rtol=0, atol=1e-11)


def test_psi_single_precision():
    from pfb_imaging_b200.sara import PsiNocopyt

    rng = np.random.default_rng(3)
    x = rng.standard_normal((2, 192, 130)).astype(np.float32)
    psi = PsiNocopyt(2, 192, 130, ["self", "db2", "db5"], 2, 1, dtype=np.float32)
    alpha = np.empty(psi.coeff_shape, np.float32)
    psi.dot(x, alpha)
    xr = np.empty_like(x)
    psi.hdot(alpha, xr)
    assert np.linalg.norm(xr - 3 * x) / np.linalg.norm(3 * x) < 1e-5


@pytest.mark.parametrize("nm", ["p", "z"])
def test_l21_dual_update_and_prox_match_reference(nm):
    from oracle import sara_np as so
    from pfb_imaging_b200.sara import L21, Psi

    lam, sigma = (float(t) for t in G[f"du_{nm}_par"])
    vp, v0, w = G["du_vp"], G["du_v"], G["du_w"]

    class Shape:  # the regulariser only needs the PsiOperator attributes for these two calls
        nband, nbasis, nymax, nxmax = v0.shape
        coeff_shape = v0.shape
        rdt, prec, device = np.dtype(np.float64), 1, 0
        dot = hdot = None

    from pfb_imaging_b200 import _lib

    Shape._lib = _lib.load()
    Shape._transposed = True
    reg = L21(Shape, bases=("a", "b", "c", "d"))
    reg.l1weight = w
    v = v0.copy()
    reg.dual_update(vp, v, lam, sigma)
    np.testing.assert_allclose(_s(v), G[f"du_{nm}_out"], rtol=1e-13, atol=1e-14)
    np.testing.assert_allclose(v, so.dual_update_fast(vp, v0, lam, sigma, w), rtol=1e-13, atol=1e-14)
    res = np.empty_like(v0)
    reg.prox(v0, res, lam, sigma)
    np.testing.assert_allclose(_s(res), G[f"du_{nm}_prox"], rtol=1e-13, atol=1e-14)
    np.testing.assert_allclose(res, so.prox_21m(v0, lam, sigma, w), rtol=1e-13, atol=1e-14)


def test_dual_update_split_over_ranks_equals_fused():
    """Bands sharded over two 'ranks': local band sums, one reduction, scale == the fused single-rank update."""
    import torch

    from pfb_imaging_b200.sara import L21

    vp, v0, w = G["du_vp"], G["du_v"], G["du_w"]
    lam, sigma = 0.7, 1.3

    class Shape:
        nband, nbasis, nymax, nxmax = v0.shape
        coeff_shape = v0.shape
        rdt, prec, device = np.dtype(np.float64), 1, 0
        dot = hdot = None
        _transposed = True

    from pfb_imaging_b200 import _lib

    Shape._lib = _lib.load()
    reg = L21(Shape)
    dev = torch.device("cuda", 0)
    wt = torch.from_numpy(w).to(dev)
    parts = [(torch.from_numpy(vp[:2]).to(dev), torch.from_numpy(v0[:2].copy()).to(dev)),
             (torch.from_numpy(vp[2:]).to(dev), torch.from_numpy(v0[2:].copy()).to(dev))]
    sums = []

    def first_pass(t):  # record the local sums; nothing to add yet
        sums.append(t.clone())

    for vpt, vt in parts:
        reg.dual_update_dev(vpt, vt, wt, lam, sigma, reduce=first_pass)
    total = sums[0] + sums[1]
    outs = []
    for (vpt, _), vsrc in zip(parts, (v0[:2], v0[2:])):
        vt = torch.from_numpy(vsrc.copy()).to(dev)
        reg.dual_update_dev(vpt, vt, wt, lam, sigma, reduce=lambda t: t.copy_(total))
        outs.append(vt.cpu().numpy())
    np.testing.assert_allclose(_s(np.concatenate(outs)), G["du_p_out"], rtol=1e-13, atol=1e-14)


@pytest.mark.parametrize("positivity", [0, 1, 2])
@pytest.mark.parametrize("device_grad", [False, True])
def test_primal_dual_matches_oracle(positivity, device_grad):
    """Denoising f(x) = 1/2 ||x - y||^2 (grad = x - y, hessnorm 1): 25 iterations of the device loop against
    the numpy restatement of opt/primal_dual.py:404-448."""
    from oracle import sara_np as so
    from pfb_imaging_b200 import wavelet_filters as wf
    from pfb_imaging_b200.sara import L21, PrimalDual, Psi

    nband, nx, ny, nlevel = 3, 96, 80, 2
    bases = ["self", "db1", "db2", "db3"]
    rng = np.random.default_rng(11)
    truth = np.zeros((nband, nx, ny))
    truth[:, 20:30, 30:50] = 1.0
    truth[:, 60, 10] = 5.0
    y = truth * np.array([1.0, 0.8, 0.6])[:, None, None] + 0.1 * rng.standard_normal(truth.shape)
    psi = Psi(nband, nx, ny, bases, nlevel, 1)
    reg = L21(psi, bases, nu=len(bases))
    reg.l1weight = rng.uniform(0.5, 1.5, reg.l1weight.shape)
    lam, maxit = 0.05, 25

    class Grad:
        def __call__(self, x):
            return x - y

    grad = Grad()
    if device_grad:
        import torch

        y_t = torch.from_numpy(y).cuda()
        grad.device_apply = lambda x_t, out_t: torch.sub(x_t, y_t, out=out_t)
    pd = PrimalDual(tol=1e-14, maxit=maxit, verbosity=0, positivity=positivity)
    pd.setup(reg, 1.0)
    pd.set_grad(grad)
    x = pd.solve(np.zeros_like(y), lam)

    bk = wf.bookkeeping(nx, ny, bases, nlevel)
    fbs = [None if b == "self" else wf.filter_bank(b) for b in bases]
    dot = lambda xx: np.stack([so.psi_dot(xx[b], bk, fbs, transposed=True) for b in range(nband)])  # noqa: E731
    hdot = lambda aa: np.stack([so.psi_hdot(aa[b], bk, fbs, transposed=True) for b in range(nband)])  # noqa: E731
    v0 = np.zeros(psi.coeff_shape)
    xr, vr, k, eps = so.primal_dual(np.zeros_like(y), v0, lam, dot, hdot, lambda xx: xx - y, 1.0, len(bases),
                                    reg.l1weight, 1e-14, maxit, positivity=positivity)
    np.testing.assert_allclose(x, xr, rtol=0, atol=1e-10)
    np.testing.assert_allclose(pd.dual, vr, rtol=0, atol=1e-10)
    assert pd.niter == k and abs(pd.eps - eps) <= 1e-9 * max(eps, 1e-30) + 1e-12
    if positivity:
        assert x.min() >= 0.0


def test_psi_full_size_identity_and_rate():
    """BASELINE-size cube slice (4096^2, 'self,db1,db2,db3', 3 levels): Psi^H Psi = nbasis * I, timing printed."""
    import time

    import torch

    from pfb_imaging_b200.sara import PsiNocopyt

    nx = ny = 4096
    bases = ["self", "db1", "db2", "db3"]
    psi = PsiNocopyt(1, nx, ny, bases, 3, 1)
    dev = torch.device("cuda", 0)
    x_t = torch.randn((1, nx, ny), dtype=torch.float64, device=dev)
    a_t = torch.empty(psi.coeff_shape, dtype=torch.float64, device=dev)
    r_t = torch.empty_like(x_t)
    for _ in range(2):
        psi.dot_dev(x_t, a_t)
        psi.hdot_dev(a_t, r_t)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        psi.dot_dev(x_t, a_t)
        psi.hdot_dev(a_t, r_t)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / 5
    err = float((r_t - len(bases) * x_t).abs().max())
    gb = (x_t.numel() * 8 * 2 + a_t.numel() * 8 * 2) / 1e9
    print(f"\n4096^2 dot+hdot: {dt * 1e3:.2f} ms  ({gb / dt:.0f} GB/s of compulsory traffic), max err {err:.1e}")
    assert err < 1e-10


@pytest.mark.parametrize("acceleration,positivity", [(True, 0), (False, 1), (True, 2)])
def test_forward_backward_matches_oracle(acceleration, positivity):
    from oracle import sara_np as so
    from pfb_imaging_b200 import wavelet_filters as wf
    from pfb_imaging_b200.sara import L21, ForwardBackward, PsiNocopyt

    nband, nx, ny, nlevel = 2, 88, 72, 2
    bases = ["self", "db1", "db3"]
    rng = np.random.default_rng(5)
    y = rng.standard_normal((nband, nx, ny)) * 0.1
    y[:, 30:40, 20:30] += 2.0
    psi = PsiNocopyt(nband, nx, ny, bases, nlevel, 1)
    reg = L21(psi, bases, nu=len(bases))
    reg.l1weight = rng.uniform(0.5, 1.5, reg.l1weight.shape)
    fb = ForwardBackward(tol=1e-14, maxit=15, verbosity=0, acceleration=acceleration, positivity=positivity)
    fb.setup(reg, 1.0)
    fb.set_grad(lambda xx: xx - y)
    x = fb.solve(np.zeros_like(y), 0.05)
    bk = wf.bookkeeping(nx, ny, bases, nlevel)
    fbs = [None if b == "self" else wf.filter_bank(b) for b in bases]
    dot = lambda xx: np.stack([so.psi_dot(xx[b], bk, fbs) for b in range(nband)])  # noqa: E731
    hdot = lambda aa: np.stack([so.psi_hdot(aa[b], bk, fbs) for b in range(nband)])  # noqa: E731
    xr, k, eps = so.forward_backward(np.zeros_like(y), 0.05, dot, hdot, lambda xx: xx - y, 1.0, len(bases), reg.l1weight,
                                     1e-14, 15, positivity=positivity, acceleration=acceleration)
    np.testing.assert_allclose(x, xr, rtol=0, atol=1e-10)
    assert fb.niter == k


def test_l1_reweighting_matches_formula():
    from oracle import sara_np as so
    from pfb_imaging_b200 import wavelet_filters as wf
    from pfb_imaging_b200.sara import L21, Psi

    nband, nx, ny = 2, 64, 48
    bases = ["self", "db2"]
    rng = np.random.default_rng(9)
    upd, model = rng.standard_normal((nband, nx, ny)), rng.standard_normal((nband, nx, ny))
    psi = Psi(nband, nx, ny, bases, 2, 1)
    reg = L21(psi, bases, rmsfactor=0.7, alpha=2.0)
    reg.init_reweighting(upd)
    w = reg.update_weights(model)
    bk = wf.bookkeeping(nx, ny, bases, 2)
    fbs = [None, wf.filter_bank("db2")]
    tot_u = sum(so.psi_dot(upd[b], bk, fbs, transposed=True) for b in range(nband))
    rms = np.array([np.std(tot_u[i][tot_u[i] != 0]) for i in range(2)])
    tot_m = sum(so.psi_dot(model[b], bk, fbs, transposed=True) for b in range(nband))
    np.testing.assert_allclose(w, so.l1reweight(tot_m, 0.7, rms, 2.0), rtol=1e-9)


def test_primal_dual_with_device_psf_hessian_gradient():
    """pfb sara's inner problem: grad(x) = HessPSF(x) - dirty.  The device-resident loop (no host round trips) must
    equal the same loop driven through the numpy callable."""
    from pfb_imaging_b200.psf import HessPSF, PsfGradient
    from pfb_imaging_b200.sara import L21, PrimalDual, PsiNocopyt

    nband, nx, ny = 2, 96, 80
    nxp, nyp = 144, 120
    rng = np.random.default_rng(21)
    psf = np.zeros((nband, nxp, nyp))
    yy, xx = np.meshgrid(np.arange(nyp) - nyp // 2, np.arange(nxp) - nxp // 2)
    for b in range(nband):
        psf[b] = np.exp(-(xx ** 2 + yy ** 2) / (2.0 * (2.0 + b) ** 2))
    psf /= psf.sum(axis=(1, 2), keepdims=True)
    abspsf = np.abs(np.fft.rfft2(np.fft.ifftshift(psf, axes=(1, 2)), axes=(1, 2)))
    truth = np.zeros((nband, nx, ny))
    truth[:, 40, 30] = 3.0
    truth[:, 60:66, 50:58] = 1.0
    hess = HessPSF(nx, ny, abspsf, beam=None, eta=0.01)
    dirty = hess.dot(truth) + 1e-3 * rng.standard_normal(truth.shape)
    bases = ["self", "db1", "db2"]
    sols = []
    for use_dev in (False, True):
        psi = PsiNocopyt(nband, nx, ny, bases, 2, 1)
        reg = L21(psi, bases, nu=len(bases))
        grad = PsfGradient(hess, dirty)
        if not use_dev:
            grad = (lambda g: (lambda x: g(x)))(grad)  # plain numpy callable: no device_apply attribute
        pd = PrimalDual(tol=1e-14, maxit=20, verbosity=0, positivity=1)
        pd.setup(reg, 1.0 + 0.01)
        pd.set_grad(grad)
        sols.append(pd.solve(np.zeros_like(dirty), 1e-3))
    np.testing.assert_allclose(sols[1], sols[0], rtol=0, atol=1e-12)
    assert np.abs(sols[1]).max() > 0.1
    hess.close()
