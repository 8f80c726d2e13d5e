"""GPU: restoration (``restore.py``) and the analytic Gaussian kernel of the PSF convolver (``pfbg_conv_set_gauss``,
``pfbg_conv_apply_add``) against the image-domain fp64 oracle of ``oracle/restore_np.py``, which builds the sampled,
periodised Gaussian on the padded grid and convolves with ``rfft2`` / ``irfft2``: it shares nothing with the device's
alias sum.  The bounds are those of the PSF-convolver tests, ``u`` the unit roundoff of the device precision and
``bound = 4 u log2(nx_psf ny_psf)``: global rel-L2 <= bound, max|err| / max|ref| <= 4 bound, worst row and worst
column rel-L2 <= 8 bound.  The oracle starts from the inputs rounded to the device precision."""
import ctypes as C

import numpy as np
import pytest

from oracle import restore_np as O
from pfb_imaging_b200 import _lib, operators as ops, plan, restore as R
from pfb_imaging_b200.psf import PsfConvolver
from pfbg_testutil import small_problem

pytestmark = pytest.mark.gpu
UNIT = {np.float32: 2.0**-24, np.float64: 2.0**-53}


def check(got, ref, dtype, nxp, nyp, extra=1.0):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    bound = extra * 4 * UNIT[dtype] * np.log2(nxp * nyp)
    err = got - ref
    rel = np.linalg.norm(err) / np.linalg.norm(ref)
    mx = np.abs(err).max() / np.abs(ref).max()
    assert rel <= bound and mx <= 4 * bound, (rel / bound, mx / bound)
    for ax in (-1, -2):
        if ref.shape[ax] >= 16:
            # each row against its own norm, floored at the mean row norm (rows far from a compact source are ~0)
            rn = np.sqrt((ref**2).sum(axis=ax))
            rows = np.sqrt((err**2).sum(axis=ax)) / np.maximum(rn, np.sqrt((rn**2).mean()))
            assert rows.max() <= 8 * bound, (ax, rows.max() / bound)


def col_block(cv):
    c = C.c_int32(0)
    _lib.check(cv._lib.pfbg_conv_info(cv._h, C.byref(c), None))
    return c.value


def smooth_image(rng, nb, nx, ny, dtype):
    """point sources on smooth emission, rounded to the device precision"""
    x = np.zeros((nb, nx, ny))
    x[:, rng.integers(0, nx, 40), rng.integers(0, ny, 40)] = rng.exponential(1.0, 40)
    x += 0.1 * rng.standard_normal((nb, nx, ny))
    return x.astype(dtype)


BEAMS = [(1.0, 1.0, 0.0), (2.0, 1.4, 0.7), (3.0, 2.0, -1.2), (30.0, 12.0, np.pi / 2), (4.5, 4.5, 0.0)]


# --- the convolver level: every column-block width, a factor 11, both normalisations ------------------------------------
# (nx, ny, nx_psf, ny_psf) -> the column-block width conv_setup_t picks, per precision
CONV_CASES = [
    ((2, 2, 2, 2), {np.float32: 2, np.float64: 2}),
    ((3, 2, 5, 3), {np.float32: 1, np.float64: 1}),
    ((51, 77, 99, 98), {np.float32: 2, np.float64: 2}),
    ((60, 45, 96, 96), {np.float32: 4, np.float64: 2}),
    ((700, 500, 1100, 770), {np.float32: 2, np.float64: 2}),  # factor 11 in both axes
    ((1201, 1001, 1575, 1540), {np.float32: 4, np.float64: 2}),
    ((4096, 1999, 8640, 3087), {np.float32: 1, np.float64: 1}),
    ((4096, 1024, 6144, 1536), {np.float32: 4, np.float64: 2}),
    ((5760, 512, 8640, 768), {np.float32: 2, np.float64: 1}),
]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_gauss_mode_every_column_block(gpu, dtype):
    rng = np.random.default_rng(1)
    seen = set()
    for (nx, ny, nxp, nyp), want_c in CONV_CASES:
        x = smooth_image(rng, 1, nx, ny, dtype)[0]
        cv = PsfConvolver(nx, ny, nxp, nyp, dtype=dtype)
        try:
            assert col_block(cv) == want_c[dtype], (nx, ny, nxp, nyp)
            seen.add(col_block(cv))
            for k, beam in enumerate(BEAMS):
                norm = bool(k % 2)
                cv.set_gauss(beam, norm_kernel=norm)
                got = cv.apply(x)
                ref = O.convolve_pad(x.astype(np.float64), O.kernel_spectrum(nxp, nyp, beam, norm_kernel=norm), nxp, nyp)
                check(got, ref, dtype, nxp, nyp)
        finally:
            cv.close()
    assert seen == ({1, 2, 4} if dtype == np.float32 else {1, 2})


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("nx,ny", [(2, 2), (33, 20), (257, 130), (4096, 4096), (5760, 5760)])
def test_convolve_to_beam_against_oracle(gpu, dtype, nx, ny):
    rng = np.random.default_rng(nx + ny)
    big = nx >= 4096
    nb = 1 if big else 2
    img = smooth_image(rng, nb, nx, ny, dtype)
    nxp, nyp = plan.good_size(int(1.5 * nx)), plan.good_size(int(1.5 * ny))
    cases = [((3.0, 2.0, 0.4), None, False), ((30.0, 12.0, -0.3), None, True)]
    cases += [((6.0, 4.0, 0.3), [(3.0, 2.0, 0.1), (2.0, 1.0, -1.4)][:nb], False)]
    if big:  # one case per size: the oracle's long-double kernel spectra dominate the time
        cases = cases[2:] if nx == 4096 else cases[:1]
    for to, fr, norm in cases:
        got = R.convolve_to_beam(img, to, beam_from=fr, pfrac=0.5, norm_kernel=norm)
        assert got.shape == img.shape and got.dtype == img.dtype
        ref = O.convolve_to_beam(img, to, fr, pfrac=0.5, norm_kernel=norm)
        for b in range(nb):
            check(got[b], ref[b], dtype, nxp, nyp)


def test_pixsize_and_per_band_target(gpu):
    rng = np.random.default_rng(3)
    img = smooth_image(rng, 2, 64, 48, np.float64)
    to = np.array([(3.0, 2.0, 0.4), (5.0, 2.5, -0.4)])
    got = R.convolve_to_beam(img, to * [2e-5, 2e-5, 1.0], pixsize=2e-5)
    for b in range(2):
        ref = O.convolve_to_beam(img[b:b + 1], to[b])[0]
        check(got[b], ref, np.float64, 96, 72)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_point_sources_restore_to_the_sampled_gaussian(gpu, dtype):
    n = 256
    beam = (3.0, 2.0, 0.5)
    model = np.zeros((1, n, n), dtype=dtype)
    model[0, 100, 131] = 2.5
    model[0, 40, 200] = -1.0
    out = R.convolve_to_beam(model, beam)
    x = np.arange(n)
    want = (2.5 * O.gauss((x - 100)[:, None], (x - 131)[None, :], *beam)
            - O.gauss((x - 40)[:, None], (x - 200)[None, :], *beam))
    assert abs(out[0, 100, 131] - 2.5) <= 4 * 4 * UNIT[dtype] * np.log2(384 * 384) * 2.5
    check(out[0], want, dtype, 384, 384)
    unit = R.convolve_to_beam(model, beam, norm_kernel=True)
    s = np.sum(unit, dtype=np.float64)
    assert abs(s - 1.5) <= 64 * UNIT[dtype] * np.abs(unit).sum(dtype=np.float64)


@pytest.mark.parametrize("to,fr", [((5.0, 4.0, 0.3), (3.0, 2.0, 0.1)), ((8.0, 8.0, 0.0), (8.0, 3.0, -1.2)),
                                   ((4.0, 2.0, 1.0), (4.0, 2.0, 1.0)), ((40.0, 30.0, 0.2), (1.0, 1.0, 0.0))])
def test_closure_from_beam_to_beam(gpu, to, fr):
    n = 256
    x = np.arange(n) - n // 2
    src = O.gauss(x[:, None], x[None, :], *fr)[None]
    got = R.convolve_to_beam(src, to, beam_from=[fr])
    want = O.gauss(x[:, None], x[None, :], *to)
    # the area ratio (up to 600 for the last pair) scales the rounding of the source image's spectrum
    check(got[0], want, np.float64, 384, 384, extra=(to[0] * to[1]) / (fr[0] * fr[1]))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("to,fr", [((7.2, 7.2, 0.0), (7.0, 7.0, 0.0)), ((7.05, 7.0, 0.1), (7.0, 7.0, 0.0)),
                                   ((8.5, 8.5, 0.0), (8.0, 8.0, 0.0)), ((30.3, 20.2, 0.3), (30.0, 20.0, 0.3)),
                                   ((12.0, 6.0, 0.7), (11.0, 5.0, 0.7))])
def test_white_noise_between_wide_beams(gpu, dtype, to, fr):
    """The residual pass of a common-resolution restore sees white noise, which has power up to Nyquist, where the
    alias sums of a wide beam need more than the m = 0 term to be accurate relative to their own largest term."""
    rng = np.random.default_rng(9)
    img = rng.standard_normal((1, 256, 256)).astype(dtype)
    got = R.convolve_to_beam(img, to, beam_from=[fr])
    ref = O.convolve_pad(img[0].astype(np.float64), O.alias_ratio_spectrum(384, 384, to, fr), 384, 384)
    check(got[0], ref, dtype, 384, 384)


def test_invalid_beams_raise(gpu):
    img = np.zeros((1, 32, 32))
    with pytest.raises(ValueError, match="does not contain"):
        R.convolve_to_beam(img, (5.0, 2.0, 0.0), beam_from=[(4.0, 3.0, 0.0)])
    with pytest.raises(ValueError, match="does not contain"):
        R.convolve_to_beam(img, (5.0, 2.0, 0.0), beam_from=[(5.0, 2.0, 0.3)])
    with pytest.raises(ValueError, match="below 1 pixel"):
        R.convolve_to_beam(img, (3.0, 0.9, 0.0))
    with pytest.raises(ValueError, match="below 1 pixel"):
        R.convolve_to_beam(img, (2e-5, 2e-5, 0.0), pixsize=4e-5)
    with pytest.raises(ValueError, match="below 1 pixel"):
        R.convolve_to_beam(img, (5.0, 4.0, 0.0), beam_from=[(0.5, 0.5, 0.0)])
    cv = PsfConvolver(32, 32, 48, 48)
    try:
        lib = cv._lib
        d3 = C.c_double * 3
        assert lib.pfbg_conv_set_gauss(cv._h, d3(5.0, 2.0, 0.0), d3(4.0, 3.0, 0.0), 0) == _lib.PFBG_ERR_ARG
        assert lib.pfbg_conv_set_gauss(cv._h, d3(0.99, 0.99, 0.0), None, 0) == _lib.PFBG_ERR_ARG
        assert lib.pfbg_conv_set_gauss(cv._h, d3(2.0, 3.0, 0.0), None, 0) == _lib.PFBG_ERR_ARG
        # a change of resolution between beams of axis ratio ~60 would need an alias scan beyond 2048 rings
        assert lib.pfbg_conv_set_gauss(cv._h, d3(61.0, 1.0, 0.5), d3(60.0, 1.0, 0.5), 0) == _lib.PFBG_ERR_ARG
        assert lib.pfbg_conv_set_gauss(cv._h, d3(61.0, 1.0, 0.5), None, 0) == 0
        assert lib.pfbg_conv_set_gauss(cv._h, d3(3.0, 2.0, 0.0), d3(3.0, 2.0, 0.0), 1) == 0
    finally:
        cv.close()
    with pytest.raises(RuntimeError):  # beyond the shared-memory FFT, as for PsfConvolver
        R.convolve_to_beam(np.zeros((1, 1, 40000)), (3.0, 2.0, 0.0))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_restore_against_oracle(gpu, dtype):
    rng = np.random.default_rng(5)
    nb, nx, ny = 3, 200, 170
    model = np.zeros((nb, nx, ny), dtype=dtype)
    model[:, rng.integers(0, nx, 50), rng.integers(0, ny, 50)] = rng.exponential(1.0, 50)
    resid = (0.05 * rng.standard_normal((nb, nx, ny))).astype(dtype)
    beam = (5.0, 4.0, 0.25)
    psf_beams = [(3.0, 2.0, 0.2), (2.5, 2.0, 0.4), (2.0, 2.0, 0.0)]
    nxp, nyp = plan.good_size(300), plan.good_size(255)
    got = R.restore(model, resid, beam)
    ref = O.restore(model, resid, beam)
    for b in range(nb):
        check(got[b], ref[b], dtype, nxp, nyp)
    got = R.restore(model, resid, beam, psf_beams=psf_beams)
    ref = O.restore(model, resid, beam, psf_beams=psf_beams)
    for b in range(nb):
        check(got[b], ref[b], dtype, nxp, nyp)


def test_add_epilogue_equals_the_separate_sum(gpu):
    """The epilogue may add `add` to the unrounded scaled transform (one fused multiply-add), the separate sum adds it
    to the rounded one: they agree to one rounding of the transform plus one of the sum."""
    rng = np.random.default_rng(6)
    x, a = rng.standard_normal((2, 300, 280))
    cv = PsfConvolver(300, 280, 450, 420).set_gauss((4.0, 3.0, 0.5))
    try:
        for _ in range(2):
            y = cv.apply(x)
            e = cv.apply(x, add=a)
            assert (np.abs(e - (y + a)) <= np.spacing(np.abs(y)) + np.spacing(np.abs(y + a))).all()
            cv.set_gauss((6.0, 3.0, 0.5), (4.0, 3.0, 0.5))
    finally:
        cv.close()


def test_switching_kernels_and_memory(gpu):
    """set_kernel after set_gauss runs the stored spectrum again; set_gauss after set_kernel releases it."""
    import torch

    rng = np.random.default_rng(7)
    nx, ny, nxp, nyp = 96, 80, 144, 120
    x = rng.standard_normal((nx, ny))
    beam = (3.0, 2.0, 0.3)
    kh = O.kernel_spectrum(nxp, nyp, beam)
    cv = PsfConvolver(nx, ny, nxp, nyp)
    try:
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        g = cv.set_gauss(beam).apply(x)
        k = cv.set_kernel(kh).apply(x)
        np.testing.assert_allclose(g, k, rtol=0, atol=1e-13 * np.abs(k).max())
        np.testing.assert_array_equal(cv.set_gauss(beam).apply(x), g)
        assert torch.cuda.mem_get_info()[0] >= free0 - (1 << 21)
    finally:
        cv.close()


def test_device_pointers_on_a_side_stream_match_the_host_path(gpu):
    import torch

    rng = np.random.default_rng(8)
    nb, nx, ny = 3, 256, 192
    model = np.zeros((nb, nx, ny))
    model[:, rng.integers(0, nx, 30), rng.integers(0, ny, 30)] = 1.0
    resid = 0.05 * rng.standard_normal((nb, nx, ny))
    beam, psf_beams = (6.0, 4.5, 0.25), [(4.0, 3.0, 0.2), (5.0, 3.5, 0.4), (3.0, 3.0, 0.0)]
    for dtype in (np.float32, np.float64):
        m, r = model.astype(dtype), resid.astype(dtype)
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            mt, rt = torch.from_numpy(m).cuda(), torch.from_numpy(r).cuda()
            plain = R.restore(mt, rt, beam)
            common = R.restore(mt, rt, beam, psf_beams=psf_beams)
            conv = R.convolve_to_beam(rt, (7.0, 5.0, 0.1), beam_from=psf_beams, norm_kernel=True)
        s.synchronize()
        assert plain.dtype == mt.dtype and plain.device == mt.device
        np.testing.assert_array_equal(plain.cpu().numpy(), R.restore(m, r, beam))
        np.testing.assert_array_equal(common.cpu().numpy(), R.restore(m, r, beam, psf_beams=psf_beams))
        np.testing.assert_array_equal(conv.cpu().numpy(),
                                      R.convolve_to_beam(r, (7.0, 5.0, 0.1), beam_from=psf_beams, norm_kernel=True))


# --- the fit_psf hook of the imaging products ---------------------------------------------------------------------------
class V:
    def __init__(self, v):
        self.values = np.asarray(v)


class Part:
    def __init__(self, **kw):
        for k, v in kw.items():
            setattr(self, k, V(v))


def test_grid_partition_and_image_data_products_fit_the_psf(gpu, tmp_path):
    from pfb_imaging_b200 import store

    p = small_problem(nrow=600, nchan=3, nx=40, ny=40, seed=11)
    cell = p["cell"] / 4  # a main lobe of several pixels
    part = Part(VIS=p["vis"][None], WEIGHT=p["wgt"][None], MASK=p["mask"], UVW=p["uvw"], FREQ=p["freq"],
                BEAM=np.ones((1, 3, 3)), l_beam=np.array([-1.0, 0.0, 1.0]), m_beam=np.array([-1.0, 0.0, 1.0]))
    out = ops.grid_partition(part, None, nx=40, ny=40, nx_psf=64, ny_psf=64, cell_rad=cell,
                             fit_psf=R.fitcleanbeam)
    assert out["PSFPARSN"].shape == (1, 3)
    np.testing.assert_array_equal(out["PSFPARSN"], R.fitcleanbeam(out["PSF"], level=0.5, pixsize=1.0))
    assert out["PSFPARSN"][0, 1] > 1.5
    d = store.Dataset()
    d["UVW"], d["FREQ"] = (("row", "three"), p["uvw"]), (("chan",), p["freq"])
    d["VIS"] = (("corr", "row", "chan"), p["vis"][None])
    d["WEIGHT"], d["MASK"] = (("corr", "row", "chan"), p["wgt"][None]), (("row", "chan"), p["mask"])
    d["BEAM"] = (("corr", "l_beam", "m_beam"), np.ones((1, 4, 4)))
    d["l_beam"], d["m_beam"] = (("l_beam",), np.linspace(-1, 1, 4)), (("m_beam",), np.linspace(-1, 1, 4))
    path = str(tmp_path / "band.dds")
    outs = ops.image_data_products([d], None, 40, 40, 64, 64, cell, cell, path, dict(timeid=0, bandid=0),
                                   epsilon=1e-8, fit_psf=R.fitcleanbeam)
    ds = store.open_zarr(path)
    np.testing.assert_array_equal(ds.PSFPARSN.values, R.fitcleanbeam(outs["psf"], level=0.5, pixsize=1.0))
    assert ds.PSFPARSN.values.shape == (1, 3)
