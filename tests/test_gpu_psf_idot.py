"""GPU: the device inverse of the PSF-convolution Hessian, ``HessPSF.idot`` on CUDA tensors (``pfbg_conv_apply_shifted``
for the direct estimate, the batched conjugate gradients ``pfbs_tree_cg`` for ``mode="psf"``), against the numpy path of
the same operator, which runs ``solvers.pcg`` band by band.

* ``mode="direct"`` is bit-identical to the numpy path: the column pass forms ``Re khat + c`` and its reciprocal in
  fp64 from the stored spectrum, the doubles the host path stores as a second kernel.
* ``mode="psf"`` with ``cgtol=0`` runs exactly ``cgmaxit`` iterations on both paths.  The element-wise updates round
  as numpy does, so the iterates differ only through the order of the dot-product sums; that difference grows with the
  iteration count k.  Bound per band (rel-L2 of the device solution against the numpy one) and the worst value
  measured on a B200 (1000 W power limit) over the cases of ``test_fixed_iterations``:

      k     bound     measured
      1     1e-14     2.4e-16
      5     3e-14     5.0e-16
      10    1e-13     2.5e-15   (8 x 4096^2, PSF 5760^2: test_production_size)
      30    3e-13     9.1e-16

* Converged solves stop after the same number of iterations per band as the host ``pcg`` (its operator applies minus
  the initial one), with the stopping decisions made on the device.
"""
import ctypes as C

import numpy as np
import pytest

from pfb_imaging_b200 import _lib, solvers
from pfb_imaging_b200 import psf as P
from pfbg_testutil import rel_l2

pytestmark = pytest.mark.gpu

BOUND = {1: 1e-14, 5: 3e-14, 10: 1e-13, 30: 3e-13}


def gaussian_abspsf(nband, nxp, nyp, sigma, seed=1, sidelobes=0.02):
    """|rfft2| of a Gaussian main lobe (width growing with band) with seeded random sidelobes around it."""
    rng = np.random.default_rng(seed)
    x = (np.arange(nxp) - nxp // 2)[:, None]
    y = (np.arange(nyp) - nyp // 2)[None, :]
    out = np.empty((nband, nxp, nyp // 2 + 1))
    c0, c1, h = nxp // 2, nyp // 2, min(12, nxp // 4, nyp // 4)
    for b in range(nband):
        s = sigma * (1 + 0.1 * b)
        psf = np.exp(-(x * x + y * y) / (2 * s * s))
        psf[c0 - h:c0 + h + 1, c1 - h:c1 + h + 1] += sidelobes * rng.standard_normal((2 * h + 1, 2 * h + 1))
        out[b] = np.abs(np.fft.rfft2(np.fft.ifftshift(psf)))
    return out


def analytic_gaussian_abspsf(nband, nxp, nyp, sigma):
    """Transfer function of a Gaussian main lobe on the padded grid, without an FFT (production sizes)."""
    fx = np.fft.fftfreq(nxp)[:, None]
    fy = np.fft.rfftfreq(nyp)[None, :]
    out = np.empty((nband, nxp, nyp // 2 + 1))
    for b in range(nband):
        s2 = (sigma * (1 + 0.05 * b)) ** 2
        out[b] = 2 * np.pi * s2 * np.exp(-2 * np.pi ** 2 * s2 * fx * fx) * np.exp(-2 * np.pi ** 2 * s2 * fy * fy)
    return out


def dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def test_direct_bit_identical(gpu):
    nband, nx, ny, nxp, nyp = 3, 70, 64, 120, 128
    rng = np.random.default_rng(11)
    abspsf = gaussian_abspsf(nband, nxp, nyp, 1.5)
    x = rng.standard_normal((nband, nx, ny))
    beam = rng.uniform(0.0, 1.0, (nband, nx, ny))
    beam[:, :10, :] = 1e-3  # below min_beam: these pixels are not divided
    assert (beam < 5e-3).any()
    for taper_width in (8, 32):
        plain = None
        for bm in (None, beam):
            H = P.HessPSF(nx, ny, abspsf, beam=bm, eta=[1e-3, 0.1, 3.0], taper_width=taper_width, cgverbose=0)
            want = H.idot(x, mode="direct")
            got = H.idot(dev(x), mode="direct")
            assert got.shape == (nband, nx, ny)
            assert np.array_equal(host(got), want)
            if bm is None:
                plain = want
            else:  # the division by beam^2 ran, and only where the mask allows
                cut = (beam <= 5e-3) | (plain <= 0)
                assert np.array_equal(want[cut], plain[cut]) and not np.array_equal(want, plain)
            H.close()
    # both directions of apply_shifted against hess_direct_slice, through host and device pointers
    import torch

    taper = P.taperf((nx, ny), 16)
    cv = P.PsfConvolver(nx, ny, nxp, nyp).set_kernel(abspsf[1])
    xt, tt, ot = dev(x[1]), dev(taper), torch.empty((nx, ny), dtype=torch.float64, device="cuda")
    for c in (0.0, 0.37, 25.0):
        for inverse, mode in ((True, "backward"), (False, "forward")):
            want = P.hess_direct_slice(x[1], abspsf=abspsf[1], taperxy=taper, lastsize=nyp, eta=c, mode=mode)
            assert np.array_equal(cv.apply_shifted(x[1], taper, c, inverse), want)
            cv.apply_shifted_dev(xt.data_ptr(), ot.data_ptr(), tt.data_ptr(), c, inverse,
                                 torch.cuda.current_stream().cuda_stream)
            assert np.array_equal(host(ot), want)
    cv.close()
    P._DIRECT_CACHE.clear()


CASES = [  # nband, nx, ny, nxp, nyp, eta, beam, init_x0
    (1, 64, 64, 128, 128, 0.1, False, True),
    (3, 50, 70, 96, 120, [0.03, 0.3, 3.0], True, False),
    (8, 64, 48, 128, 96, list(np.geomspace(1e-3, 1.0, 8)), True, True),
    (3, 64, 64, 128, 128, [1.0, 0.01, 0.1], False, False),
]


@pytest.mark.parametrize("case", range(len(CASES)))
@pytest.mark.parametrize("k", [1, 5, 30])
def test_fixed_iterations(gpu, case, k):
    nband, nx, ny, nxp, nyp, eta, with_beam, init_x0 = CASES[case]
    rng = np.random.default_rng(100 + case)
    abspsf = gaussian_abspsf(nband, nxp, nyp, 1.5, seed=case)
    beam = rng.uniform(0.5, 1.0, (nband, nx, ny)) if with_beam else None
    eta = float(eta) if np.isscalar(eta) else eta
    H = P.HessPSF(nx, ny, abspsf, beam=beam, eta=eta, cgtol=0.0, cgmaxit=k, cgverbose=0)
    b = rng.standard_normal((nband, nx, ny))
    want = H.idot(b, mode="psf", init_x0=init_x0)
    bt = dev(b) if nband > 1 else dev(b[0])
    got = H.idot(bt, mode="psf", init_x0=init_x0)
    assert np.array_equal(host(bt), b if nband > 1 else b[0])  # input unchanged
    info = H.last_idot_info
    assert list(info["iters"]) == [k] * nband and info["stop"] == ["maxit"] * nband
    errs = [rel_l2(host(got)[i], want[i]) for i in range(nband)]
    print(f"MEASURED fixed k={k} case={case} worst rel-L2 {max(errs):.2e}")
    assert max(errs) <= BOUND[k], errs
    # dot on the device runs the same kernels as the numpy path
    assert np.array_equal(host(H.dot(dev(b))), H.dot(b))
    H.close()
    P._DIRECT_CACHE.clear()


def _host_counts(H, b, monkeypatch):
    """Iterations and eps history of the host pcg on each band, started as the numpy idot starts it: operator
    applies (a wrapped operator) minus the initial one."""
    counts, hist = [], []
    orig_nd = solvers.norm_diff
    for band in range(H.nband):
        n, h = [0], []

        def op(v, band=band, n=n):
            n[0] += 1
            return H.conv[band].apply(v, beam=H.beam[band], eta=float(H.eta[band]))

        def nd(x, xp, reduce=None, h=h):
            e = orig_nd(x, xp, reduce)
            h.append(e)
            return e

        monkeypatch.setattr(solvers, "norm_diff", nd)
        solvers.pcg(op, np.ascontiguousarray(b[band]), x0=H._direct(band, b[band]), tol=H.cgtol, maxit=H.cgmaxit,
                    minit=3, verbosity=0, backtrack=False)
        monkeypatch.setattr(solvers, "norm_diff", orig_nd)
        counts.append(n[0] - 1)
        hist.append(h)
    return counts, hist


def test_converged_solves(gpu, monkeypatch):
    nband, nx, ny, nxp, nyp = 4, 64, 64, 128, 128
    rng = np.random.default_rng(7)
    abspsf = gaussian_abspsf(nband, nxp, nyp, 1.5)
    beam = rng.uniform(0.6, 1.0, (nband, nx, ny))
    tol = 1e-4
    H = P.HessPSF(nx, ny, abspsf, beam=beam, eta=[30.0, 3.0, 0.3, 0.03], cgtol=tol, cgmaxit=300, cgverbose=0)
    b = rng.standard_normal((nband, nx, ny))
    counts, hist = _host_counts(H, b, monkeypatch)
    # the problem is chosen so that no band stops near tol: round-off cannot move a stopping decision
    for h in hist:
        assert h[-1] < 0.98 * tol and h[-2] > 1.02 * tol, h[-3:]
    assert len(set(counts)) == nband, counts  # the bands stop at clearly different iterations
    got = H.idot(dev(b), mode="psf")
    info = H.last_idot_info
    print(f"MEASURED converged host iters {counts} device {list(info['iters'])}")
    assert list(info["iters"]) == counts
    assert info["stop"] == ["converged"] * nband
    assert (info["eps"] < tol).all()
    res = host(H.dot(got)) - b
    for i in range(nband):
        assert np.linalg.norm(res[i]) / np.linalg.norm(b[i]) < 1e-3
    H.close()


def test_zero_band_and_flux_mop(gpu, monkeypatch):
    nband, nx, ny, nxp, nyp = 3, 64, 64, 128, 128
    rng = np.random.default_rng(8)
    abspsf = gaussian_abspsf(nband, nxp, nyp, 1.5)
    pb = rng.uniform(0.6, 1.0, (nband, nx, ny))
    mask = np.zeros((nx, ny))
    mask[10:25, 12:30] = 1.0  # two islands
    mask[40:52, 35:60] = 1.0
    beam = pb * mask[None]  # the flux mop: the mask rides in the beam
    H = P.HessPSF(nx, ny, abspsf, beam=beam, eta=[1.0, 0.1, 0.01], cgtol=1e-4, cgmaxit=300, cgverbose=0)
    b = rng.standard_normal((nband, nx, ny)) * beam
    b[1] = 0.0
    counts, _ = _host_counts(H, b, monkeypatch)
    got = H.idot(dev(b), mode="psf")
    info = H.last_idot_info
    assert info["stop"][1] == "initial residual zero" and info["iters"][1] == 0
    assert not host(got)[1].any()
    assert list(info["iters"]) == counts
    res = host(H.dot(got)) - b
    for i in (0, 2):
        assert info["stop"][i] == "converged"
        assert np.linalg.norm(res[i]) / np.linalg.norm(b[i]) < 1e-3
    H.close()


def test_repeatable_and_streams(gpu):
    import torch

    nband, nx, ny, nxp, nyp = 3, 64, 64, 128, 128
    rng = np.random.default_rng(9)
    abspsf = gaussian_abspsf(nband, nxp, nyp, 1.5)
    H = P.HessPSF(nx, ny, abspsf, beam=rng.uniform(0.5, 1.0, (nband, nx, ny)), eta=[0.01, 0.1, 1.0], cgtol=1e-6,
                  cgmaxit=200, cgverbose=0)
    bt = dev(rng.standard_normal((nband, nx, ny)))
    a = host(H.idot(bt, mode="psf"))
    b = host(H.idot(bt, mode="psf"))
    assert np.array_equal(a, b)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        c = H.idot(bt, mode="psf")
        d = H.idot(bt, mode="direct")
    side.synchronize()
    assert np.array_equal(host(c), a)
    assert np.array_equal(host(d), host(H.idot(bt, mode="direct")))
    H.close()


def test_set_beam(gpu):
    nband, nx, ny, nxp, nyp = 2, 64, 64, 128, 128
    rng = np.random.default_rng(10)
    abspsf = gaussian_abspsf(nband, nxp, nyp, 1.5)
    H = P.HessPSF(nx, ny, abspsf, beam=rng.uniform(0.5, 1.0, (nband, nx, ny)), eta=0.1, cgtol=0.0, cgmaxit=5,
                  cgverbose=0)
    x = rng.standard_normal((nband, nx, ny))
    xt = dev(x)
    first = host(H.idot(xt, mode="psf"))
    beam2 = rng.uniform(0.0, 1.0, (nband, nx, ny))
    H.set_beam(beam2)
    assert np.array_equal(host(H.dot(xt)), H.dot(x))
    assert np.array_equal(host(H.idot(xt, mode="direct")), H.idot(x, mode="direct"))
    second = host(H.idot(xt, mode="psf"))
    want = H.idot(x, mode="psf")
    assert rel_l2(first, want) > 1e-3
    assert max(rel_l2(second[i], want[i]) for i in range(nband)) <= BOUND[5]
    H.close()
    P._DIRECT_CACHE.clear()


def test_gradient_follows_set_beam(gpu):
    """PsfGradient.device_apply uses the Hessian's current beams: after set_beam it still equals the numpy gradient."""
    import torch

    nband, nx, ny, nxp, nyp = 2, 64, 64, 128, 128
    rng = np.random.default_rng(13)
    abspsf = gaussian_abspsf(nband, nxp, nyp, 1.5)
    H = P.HessPSF(nx, ny, abspsf, beam=rng.uniform(0.5, 1.0, (nband, nx, ny)), eta=0.1, cgverbose=0)
    grad = P.PsfGradient(H, rng.standard_normal((nband, nx, ny)))
    x = rng.standard_normal((nband, nx, ny))
    xt = dev(x)
    out = torch.empty_like(xt)
    grad.device_apply(xt, out)
    assert np.array_equal(host(out), grad(x))
    H.set_beam(rng.uniform(0.0, 1.0, (nband, nx, ny)))
    grad.device_apply(xt, out)
    assert np.array_equal(host(out), grad(x))
    H.close()


def test_errors_before_launch_tree_cg(gpu):
    import torch

    lib = _lib.load()
    nband, nx, ny, nxp, nyp = 2, 32, 32, 64, 64
    abspsf = gaussian_abspsf(nband, nxp, nyp, 1.5)
    H = P.HessPSF(nx, ny, abspsf, eta=0.1, cgverbose=0)
    x = torch.zeros((nband, nx, ny), dtype=torch.float64, device="cuda")
    n0 = lib.pfbg_launch_count()
    with pytest.raises(TypeError):
        H.idot(x.float())
    with pytest.raises(TypeError):
        H.dot(x.float())
    with pytest.raises(ValueError):
        H.idot(x[0])  # (nx, ny) only when nband == 1
    with pytest.raises(ValueError):
        H.idot(x[:, :, :16])
    with pytest.raises(ValueError):
        H.idot(x, mode="cheap")
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            H.idot(x.to("cuda:1"))
    assert lib.pfbg_launch_count() == n0

    # the C entry points
    other = P.PsfConvolver(nx, ny + 1, nxp, nyp).set_kernel(np.ones((nxp, nyp // 2 + 1)))
    npix = nx * ny
    gs = (C.c_int32 * (nband + 1))(*range(nband + 1))  # one group per system
    need = int(lib.pfbs_tree_cg_work_bytes(nband, gs, npix))
    work = torch.empty(need, dtype=torch.uint8, device="cuda")
    sol = torch.zeros_like(x)
    iters, eps, stop = (C.c_int32 * nband)(), (C.c_double * nband)(), (C.c_int32 * nband)()
    beams = (C.c_void_p * nband)(None, None)
    scales = (C.c_double * nband)(1.0, 1.0)
    etas = (C.c_double * nband)(0.1, 0.1)
    s = torch.cuda.current_stream().cuda_stream

    def run(convs, rhs=x.data_ptr(), n=npix, wb=need):
        return lib.pfbs_tree_cg(H.conv[0].device, nband, gs, (C.c_void_p * nband)(*[c._h.value for c in convs]), beams,
                                scales, etas, None if rhs is None else C.c_void_p(rhs), C.c_void_p(sol.data_ptr()), n,
                                1e-3, 10, 3, C.c_void_p(work.data_ptr()), wb, iters, eps, stop, s)

    n0 = lib.pfbg_launch_count()
    assert run([H.conv[0], other]) == _lib.PFBG_ERR_ARG  # mismatched image sizes
    assert run(H.conv, wb=need - 1) == _lib.PFBG_ERR_ARG
    assert run(H.conv, n=npix + 1) == _lib.PFBG_ERR_ARG
    assert run(H.conv, rhs=None) == _lib.PFBG_ERR_ARG
    assert lib.pfbs_tree_cg_work_bytes(0, gs, npix) == -1
    g = P.PsfConvolver(nx, ny, nxp, nyp).set_gauss((3.0, 2.0, 0.1))
    xh = np.zeros((nx, ny))
    rc = lib.pfbg_conv_apply_shifted(g._h, C.c_void_p(xh.ctypes.data), None, 1.0, 1, C.c_void_p(xh.ctypes.data),
                                     _lib.HOST_PTRS, None)
    assert rc == 4  # PFBG_ERR_STATE: no stored spectrum
    assert lib.pfbg_launch_count() == n0
    assert run(H.conv) == 0  # and the same call with good arguments runs
    for c in (other, g):
        c.close()
    H.close()


def test_production_size(gpu):
    """8 x 4096^2 with a 5760^2 PSF: 10 fixed iterations against the numpy path."""
    nband, nx, nxp, k = 8, 4096, 5760, 10
    rng = np.random.default_rng(12)
    abspsf = analytic_gaussian_abspsf(nband, nxp, nxp, 3.0)
    beam = rng.uniform(0.5, 1.0, (nx, nx))[None].repeat(nband, 0)
    H = P.HessPSF(nx, nx, abspsf, beam=beam, eta=1e-3, cgtol=0.0, cgmaxit=k, cgverbose=0)
    b = rng.standard_normal((nband, nx, nx))
    want = H.idot(b, mode="psf")
    got = host(H.idot(dev(b), mode="psf"))
    errs = [rel_l2(got[i], want[i]) for i in range(nband)]
    print(f"MEASURED production k={k} worst rel-L2 {max(errs):.2e}")
    assert list(H.last_idot_info["iters"]) == [k] * nband
    assert max(errs) <= BOUND[k], errs
    H.close()
    P._DIRECT_CACHE.clear()
