"""GPU: ``pfb deconv``'s Hessian on the device.  ``HessianTree.dot`` on CUDA tensors (``pfbg_conv_apply_scaled`` per
beam group), the batched conjugate gradients over grouped systems (``psf.tree_cg`` -> ``pfbs_tree_cg``), and
``BandWorkerPool`` / ``HessTreeRay`` / ``PsfGradient`` on CUDA tensors, against the numpy path of the same operators,
which runs ``solvers.pcg`` band by band around host-pointer convolutions.

* ``dot`` differs from the host only in rounding: the device multiplies by ``1 / wsum`` in the convolver's epilogue and
  adds each group's term there, the host divides the summed cube by ``wsum``.
  Measured on a B200 (1000 W power limit): at most 2.9e-16 rel-L2 against the reference golden, 1.9e-16 against the
  host ``dot``.
* CG with ``tol=0`` runs exactly ``k`` iterations on both paths.  The element-wise updates round as numpy does, so the
  iterates differ through the operator's rounding and the order of the dot-product sums.  Bound per band (rel-L2 of
  the device solution against the numpy one) and the worst value measured on a B200 (1000 W power limit) over the
  cases of ``test_fixed_iterations``:

      k     bound     measured
      1     1e-14     2.4e-16
      5     3e-14     2.2e-16
      30    3e-13     2.3e-16

* Converged solves stop after the same number of iterations per band as the host ``pcg``.
"""
import ctypes as C

import numpy as np
import pytest

from pfb_imaging_b200 import _lib, operators as ops, psf as P, solvers
from pfbg_testutil import GOLDEN, rel_l2
from test_store_cpu import make_dt_store

pytestmark = pytest.mark.gpu

BOUND = {1: 1e-14, 5: 3e-14, 30: 3e-13}


def dev(a, device=0):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(torch.device("cuda", device))


def host(t):
    return t.detach().cpu().numpy()


def golden_parts():
    G = np.load(f"{GOLDEN}/solvers.npz")
    parts = [dict(psfhat=G[f"ht_psfhat{p}"], beam=G[f"ht_beam{p}"], wsum=G[f"ht_wsum{p}"]) for p in range(3)]
    return G, parts


def store_parts(tmp_path, nband=3, npart=2, nx=48, nxp=72, ncorr=1, seed=0):
    """Per-band HessianTree partitions of a `make_dt_store` store (every partition has its own beam), and the
    largest eigenvalue bound of the convolution term of each band (max |psfhat| / wsum)."""
    path = str(tmp_path / f"img_{nband}_{npart}_{ncorr}_{seed}.dt")
    truth = make_dt_store(path, nband=nband, npart=npart, nx=nx, nx_psf=nxp, ncorr=ncorr, seed=seed)
    per_band, lam = [], []
    for b in range(nband):
        parts = [dict(psfhat=np.abs(t["PSFHAT"]), beam=t["BEAM"],
                      wsum=np.array([t["WEIGHT"][c][t["MASK"] > 0].sum() for c in range(ncorr)]))
                 for t in truth[b]["parts"]]
        per_band.append(parts)
        lam.append(sum(p["psfhat"][0].max() for p in parts) / sum(p["wsum"][0] for p in parts))
    return path, per_band, np.array(lam)


def make_trees(per_band, nx, nxp, etas, device=0):
    return [P.HessianTree(parts, nx, nx, nxp, nxp, eta=float(e), device=device) for parts, e in zip(per_band, etas)]


def close_all(trees):
    for t in trees:
        t.close()


def test_dot_against_the_reference_golden(gpu):
    """The golden tree has three partitions of which two share a beam: two groups per correlation, ncorr = 2."""
    G, parts = golden_parts()
    x = G["ht_x"]
    ncorr, nx, ny = x.shape
    assert ncorr == 2
    nxp, nyo2 = parts[0]["psfhat"].shape[1:]
    for kw, key in ((dict(eta=0.3), "ht_dot"), (dict(eta=0.1, wsum=17.0), "ht_dot_wsum")):
        ht = P.HessianTree(parts, nx, ny, nxp, 2 * (nyo2 - 1), **kw)
        assert len(ht._groups) == 2 * ncorr
        xt = dev(x)
        got = ht.dot(xt)
        assert got.is_cuda and tuple(got.shape) == x.shape and got.data_ptr() != xt.data_ptr()
        assert np.array_equal(host(xt), x)  # input unchanged
        print(f"MEASURED golden {key} rel-L2 {rel_l2(host(got), G[key]):.2e}")
        assert rel_l2(host(got), G[key]) <= 1e-12
        assert rel_l2(host(ht.hdot(xt)), G[key]) <= 1e-12
        with pytest.raises(AssertionError):
            ht.dot(xt[0])  # (nx, ny) only when ncorr == 1, as on the host
        ht.close()


@pytest.mark.parametrize("npart", [2, 3])
def test_dot_against_host(gpu, tmp_path, npart):
    import torch

    nx, nxp = 48, 72
    _, per_band, lam = store_parts(tmp_path, nband=2, npart=npart, nx=nx, nxp=nxp)
    trees = make_trees(per_band, nx, nxp, lam * np.array([0.01, 0.0]))  # eta = 0 reads no ridge term
    rng = np.random.default_rng(1)
    for t in trees:
        assert len(t._groups) == npart
        x = rng.standard_normal((nx, nx))
        xt = dev(x)
        got = t.dot(xt)
        assert tuple(got.shape) == (1, nx, nx)
        assert np.array_equal(host(xt), x)
        err = rel_l2(host(got), t.dot(x))
        print(f"MEASURED dot npart={npart} rel-L2 {err:.2e}")
        assert err <= 1e-13
        # on a side stream, and from a (1, nx, ny) input
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            again = t.dot(xt[None])
        side.synchronize()
        assert torch.equal(again, got)
        with pytest.raises(TypeError):
            t.dot(xt.float())
    close_all(trees)


def test_dot_two_correlations(gpu, tmp_path):
    nx, nxp = 40, 60
    _, per_band, lam = store_parts(tmp_path, nband=1, npart=2, nx=nx, nxp=nxp, ncorr=2)
    (t,) = make_trees(per_band, nx, nxp, lam * 0.1)
    assert t.ncorr == 2 and len(t._groups) == 4
    x = np.random.default_rng(2).standard_normal((2, nx, nx))
    got = host(t.dot(dev(x)))
    want = t.dot(x)
    err = max(rel_l2(got[c], want[c]) for c in range(2))
    print(f"MEASURED dot ncorr=2 rel-L2 {err:.2e}")
    assert err <= 1e-13
    # the CG systems are correlation 0 only, and a two-correlation tree fails as the host solve fails
    with pytest.raises(AssertionError):
        solvers.pcg(lambda z: t.dot(z)[0], x[0], tol=0.0, maxit=1, minit=1, verbosity=0)
    with pytest.raises(AssertionError):
        P.tree_cg([t], dev(x[:1]), None, 0.0, 1, 1)
    t.close()


def host_solve(tree, rhs, x0, tol, maxit, minit):
    return solvers.pcg(lambda z: tree.dot(z)[0], np.ascontiguousarray(rhs), x0=None if x0 is None else x0.copy(),
                       tol=tol, maxit=maxit, minit=minit, verbosity=0)


CASES = [  # nband, npart, nx, nxp, eta / lam
    (3, 2, 48, 72, [0.01, 0.1, 1.0]),
    (2, 3, 40, 64, [0.03, 0.3]),
    (1, 1, 48, 72, [0.05]),
]


@pytest.mark.parametrize("case", range(len(CASES)))
@pytest.mark.parametrize("k", [1, 5, 30])
def test_fixed_iterations(gpu, tmp_path, case, k):
    nband, npart, nx, nxp, eta = CASES[case]
    _, per_band, lam = store_parts(tmp_path, nband=nband, npart=npart, nx=nx, nxp=nxp, seed=case)
    trees = make_trees(per_band, nx, nxp, lam * np.array(eta))
    b = np.random.default_rng(100 + case).standard_normal((nband, nx, nx))
    want = np.stack([host_solve(trees[i], b[i], None, 0.0, k, k) for i in range(nband)])
    bt = dev(b)
    got, info = P.tree_cg(trees, bt, None, 0.0, k, k)
    assert np.array_equal(host(bt), b)
    assert list(info["iters"]) == [k] * nband and info["stop"] == ["maxit"] * nband
    errs = [rel_l2(host(got)[i], want[i]) for i in range(nband)]
    print(f"MEASURED fixed k={k} case={case} worst rel-L2 {max(errs):.2e}")
    assert max(errs) <= BOUND[k], errs
    close_all(trees)


def _host_counts(trees, b, tol, maxit, minit, monkeypatch):
    """Iterations and eps history of the host pcg per band."""
    counts, hist = [], []
    orig_nd = solvers.norm_diff
    for i, t in enumerate(trees):
        h = []

        def nd(x, xp, reduce=None, h=h):
            e = orig_nd(x, xp, reduce)
            h.append(e)
            return e

        monkeypatch.setattr(solvers, "norm_diff", nd)
        host_solve(t, b[i], None, tol, maxit, minit)
        monkeypatch.setattr(solvers, "norm_diff", orig_nd)
        counts.append(len(h))
        hist.append(h)
    return counts, hist


def test_converged_solves(gpu, tmp_path, monkeypatch):
    nband, nx, nxp = 4, 48, 72
    _, per_band, lam = store_parts(tmp_path, nband=nband, npart=2, nx=nx, nxp=nxp, seed=5)
    trees = make_trees(per_band, nx, nxp, lam * np.array([1.0, 0.3, 0.1, 0.03]))
    b = np.random.default_rng(7).standard_normal((nband, nx, nx))
    # the tolerance is picked so that no band stops near it: round-off cannot move a stopping decision
    _, hist = _host_counts(trees, b, 0.0, 200, 1, monkeypatch)
    tol = None
    for cand in (1e-4, 5e-5, 2e-5, 1e-5, 5e-6, 2e-6, 1e-6):
        ok = True
        for h in hist:
            i = next((j for j, e in enumerate(h) if e < cand), None)
            ok &= i is not None and i > 0 and h[i] < 0.98 * cand and h[i - 1] > 1.02 * cand
        if ok:
            tol = cand
            break
    assert tol is not None
    counts, _ = _host_counts(trees, b, tol, 300, 1, monkeypatch)
    got, info = P.tree_cg(trees, dev(b), None, tol, 300, 1)
    print(f"MEASURED converged tol={tol:g} host iters {counts} device {list(info['iters'])}")
    assert list(info["iters"]) == counts
    assert info["stop"] == ["converged"] * nband and (info["eps"] < tol).all()
    res = np.stack([trees[i].dot(host(got)[i])[0] for i in range(nband)]) - b
    for i in range(nband):
        assert np.linalg.norm(res[i]) / np.linalg.norm(b[i]) < 1e-2
    close_all(trees)


def test_zero_rhs_and_x0(gpu, tmp_path):
    import torch

    nband, nx, nxp, k = 3, 48, 72, 5
    _, per_band, lam = store_parts(tmp_path, nband=nband, npart=2, nx=nx, nxp=nxp, seed=3)
    trees = make_trees(per_band, nx, nxp, lam * 0.1)
    rng = np.random.default_rng(9)
    b = rng.standard_normal((nband, nx, nx))
    b[1] = 0.0
    got, info = P.tree_cg(trees, dev(b), None, 1e-6, 100, 1)
    assert info["stop"][1] == "initial residual zero" and info["iters"][1] == 0
    assert not host(got)[1].any()
    assert info["stop"][0] == info["stop"][2] == "converged"
    # x0 is the starting point and is left unchanged
    b[1] = rng.standard_normal((nx, nx))
    x0 = rng.standard_normal((nband, nx, nx))
    x0t = dev(x0)
    got, info = P.tree_cg(trees, dev(b), x0t, 0.0, k, k)
    assert np.array_equal(host(x0t), x0)
    zero, _ = P.tree_cg(trees, dev(b), torch.zeros_like(x0t), 0.0, k, k)
    assert rel_l2(host(got), host(zero)) > 1e-6
    for i in range(nband):
        assert rel_l2(host(got)[i], host_solve(trees[i], b[i], x0[i], 0.0, k, k)) <= BOUND[k]
    close_all(trees)


def test_pool_and_facade_on_cuda_tensors(gpu, tmp_path, capsys):
    import torch

    nband, nx, nxp, k = 3, 48, 72, 5
    path, _, lam = store_parts(tmp_path, nband=nband, npart=2, nx=nx, nxp=nxp, seed=4)
    pool = ops.BandWorkerPool(nband)
    pool.load_bands(path, [f"band{b:04d}" for b in range(nband)])
    etas = lam * np.array([0.3, 0.1, 0.03])
    pool.init_hess(None, nx, nx, nxp, nxp, etas, [None] * nband)
    rng = np.random.default_rng(11)
    x = rng.standard_normal((nband, nx, nx))
    xt = dev(x)
    hx = pool.hess_dot(x)
    hxt = pool.hess_dot(xt)
    assert hxt.is_cuda and hxt.device == xt.device and tuple(hxt.shape) == x.shape
    assert np.array_equal(host(xt), x)
    assert max(rel_l2(host(hxt)[i], hx[i]) for i in range(nband)) <= 1e-13
    # fixed iterations, with and without x0 (not modified)
    x0 = rng.standard_normal((nband, nx, nx))
    for start in (None, x0):
        want = pool.hess_cg(hx, None if start is None else start.copy(), 0.0, k, k, 0)
        x0t = None if start is None else dev(start)
        got = pool.hess_cg(hxt, x0t, 0.0, k, k, 0)
        assert got.device == hxt.device
        if start is not None:
            assert np.array_equal(host(x0t), start)
        assert max(rel_l2(host(got)[i], want[i]) for i in range(nband)) <= BOUND[k]
        assert list(pool.last_cg_info["iters"]) == [k] * nband
    # the facade: a converged solve recovers x, with pcg's end-of-solve message per band
    ht = P.HessTreeRay(None, nx, nx, nxp, nxp, etas=etas, workers=pool, cg_verbose=1)
    assert rel_l2(host(ht.dot(xt)), hx) <= 1e-13
    capsys.readouterr()
    sol = ht.cg(hxt, tol=1e-10, maxit=300)
    out = capsys.readouterr().out
    assert out.count("Success, converged after") == nband, out
    assert isinstance(sol, torch.Tensor) and rel_l2(host(sol), x) <= 1e-6
    assert ht.last_cg_info["stop"] == ["converged"] * nband
    with pytest.raises(TypeError):
        pool.hess_cg(hxt.float(), None, 0.0, 1, 1, 0)
    with pytest.raises(ValueError):
        pool.hess_dot(hxt[:, :, :16])
    pool.close()


def test_primal_dual_with_tree_gradient(gpu, tmp_path, monkeypatch):
    """pfb deconv's inner problem: grad(x) = HessTreeRay(x) - dirty inside the device primal-dual loop (no host
    convolution), against the same loop driven through the numpy callable."""
    from pfb_imaging_b200.sara import L21, PrimalDual, PsiNocopyt

    nband, nx, nxp = 2, 48, 72
    path, _, lam = store_parts(tmp_path, nband=nband, npart=2, nx=nx, nxp=nxp, seed=6)
    pool = ops.BandWorkerPool(nband)
    pool.load_bands(path, [f"band{b:04d}" for b in range(nband)])
    hess = P.HessTreeRay(None, nx, nx, nxp, nxp, etas=lam * 0.01, workers=pool)
    truth = np.zeros((nband, nx, nx))
    truth[:, 20, 15] = 3.0
    truth[:, 30:34, 25:31] = 1.0
    dirty = hess.dot(truth) + 1e-4 * np.random.default_rng(21).standard_normal(truth.shape)
    bases = ["self", "db1", "db2"]
    hessnorm = float(lam.max()) * 1.01
    sols = []
    for use_dev in (False, True):
        psi = PsiNocopyt(nband, nx, nx, bases, 2, 1)
        reg = L21(psi, bases, nu=len(bases))
        grad = P.PsfGradient(hess, dirty)
        if not use_dev:
            grad = (lambda g: (lambda x: g(x)))(grad)  # plain numpy callable: no device_apply attribute
        else:
            def no_host(*a, **k):
                raise AssertionError("host convolution inside the device loop")

            monkeypatch.setattr(P.PsfConvolver, "apply", no_host)
        pd = PrimalDual(tol=1e-14, maxit=20, verbosity=0, positivity=1)
        pd.setup(reg, hessnorm)
        pd.set_grad(grad)
        sols.append(pd.solve(np.zeros_like(dirty), lam.max() * 1e-3))
        psi.close()
    monkeypatch.undo()
    err = rel_l2(sols[1], sols[0])
    print(f"MEASURED primal-dual tree gradient rel-L2 {err:.2e}")
    assert err <= 1e-10 and np.abs(sols[1]).max() > 0
    pool.close()


def test_bands_over_devices(gpu, tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two or more visible GPUs")
    nband, nx, nxp, k = 4, 48, 72, 10
    path, per_band, lam = store_parts(tmp_path, nband=nband, npart=2, nx=nx, nxp=nxp, seed=8)
    etas = lam * 0.1
    pool = ops.BandWorkerPool(nband)  # band b on device b mod ndev
    pool.load_bands(path, [f"band{b:04d}" for b in range(nband)])
    pool.init_hess(None, nx, nx, nxp, nxp, etas, [None] * nband)
    assert len({pool._workers[b].hess.device for b in range(nband)}) > 1
    trees = make_trees(per_band, nx, nxp, etas, device=0)
    b = dev(np.random.default_rng(12).standard_normal((nband, nx, nx)))
    want, info = P.tree_cg(trees, b, None, 0.0, k, k)
    got = pool.hess_cg(b, None, 0.0, k, k, 0)
    assert got.device == b.device
    assert rel_l2(host(got), host(want)) <= 1e-14
    assert list(pool.last_cg_info["iters"]) == list(info["iters"])
    assert rel_l2(host(pool.hess_dot(b)), np.stack([host(t.dot(b[i]))[0] for i, t in enumerate(trees)])) <= 1e-14
    close_all(trees)
    pool.close()


def test_tree_cg_abi_errors(gpu, tmp_path):
    import torch

    lib = _lib.load()
    nx, nxp = 32, 48
    _, per_band, lam = store_parts(tmp_path, nband=2, npart=2, nx=nx, nxp=nxp, seed=2)
    trees = make_trees(per_band, nx, nxp, lam * 0.1)
    cv = trees[0]._groups[0][2]
    s = torch.cuda.current_stream().cuda_stream
    x = torch.randn((nx, nx), dtype=torch.float64, device="cuda")
    out, out2 = torch.empty_like(x), torch.empty_like(x)
    xh = np.zeros((nx, nx))
    vp = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731

    def scaled(xp, xin, outp, scale=1.0, eta=0.5, flags=_lib.DEVICE_PTRS):
        return lib.pfbg_conv_apply_scaled(cv._h, xp, None, xin, eta, scale, outp, flags, s)

    n0 = lib.pfbg_launch_count()
    hp = C.c_void_p(xh.ctypes.data)
    assert scaled(hp, hp, vp(out)) == _lib.PFBG_ERR_ARG  # host pointers
    assert scaled(vp(x), vp(x), hp) == _lib.PFBG_ERR_ARG
    assert scaled(vp(x), vp(x), vp(out), flags=_lib.HOST_PTRS) == _lib.PFBG_ERR_ARG
    assert scaled(vp(x), vp(out), vp(out)) == _lib.PFBG_ERR_ARG  # xin aliases out
    for bad in (0.0, -1.0, float("inf"), float("nan")):
        assert scaled(vp(x), vp(x), vp(out), scale=bad) == _lib.PFBG_ERR_ARG
    assert lib.pfbg_launch_count() == n0
    # scale 1 with xin = x is pfbg_conv_apply, bit for bit
    assert scaled(vp(x), vp(x), vp(out)) == 0
    _lib.check(lib.pfbg_conv_apply(cv._h, vp(x), None, 0.5, vp(out2), _lib.DEVICE_PTRS, s))
    assert torch.equal(out, out2)

    # pfbs_tree_cg
    nsys, npix = 2, nx * nx
    convs = [g[2] for t in trees for g in t._groups]
    beams = [t._beams_dev() for t in trees]
    beam_ptrs = [None if bm is None else bm.data_ptr() for bl in beams for bm in bl]
    ng = len(convs)
    assert ng == 4
    good_gs = [0, 2, 4]
    rhs = torch.randn((nsys, nx, nx), dtype=torch.float64, device="cuda")
    sol = torch.zeros_like(rhs)
    need = int(lib.pfbs_tree_cg_work_bytes(nsys, (C.c_int32 * 3)(*good_gs), npix))
    one_group = int(lib.pfbs_tree_cg_work_bytes(nsys, (C.c_int32 * 3)(0, 1, 2), npix))
    assert need == one_group + ((npix * 8 + 255) // 256) * 256  # one more image
    work = torch.empty(need, dtype=torch.uint8, device="cuda")
    iters, eps, stop = (C.c_int32 * nsys)(), (C.c_double * nsys)(), (C.c_int32 * nsys)()

    def run(gs=good_gs, cl=None, scale=(1e-2, 1e-2), device=0):
        cl = [c._h.value for c in convs] if cl is None else cl
        return lib.pfbs_tree_cg(device, nsys, (C.c_int32 * 3)(*gs), (C.c_void_p * ng)(*cl), (C.c_void_p * ng)(*beam_ptrs),
                                (C.c_double * nsys)(*scale), (C.c_double * nsys)(0.1, 0.1), vp(rhs), vp(sol), npix,
                                1e-3, 10, 1, vp(work), need, iters, eps, stop, s)

    f32 = P.PsfConvolver(nx, nx, nxp, nxp, dtype=np.float32).set_kernel(np.ones((nxp, nxp // 2 + 1)))
    n0 = lib.pfbg_launch_count()
    for gs in ([0, 0, 4], [1, 2, 4], [0, 3, 2], [0, 2, 2]):  # empty systems, a non-zero start, decreasing
        assert run(gs=gs) == _lib.PFBG_ERR_ARG, gs
    assert run(cl=[f32._h.value] + [c._h.value for c in convs[1:]]) == _lib.PFBG_ERR_ARG  # fp32 convolver
    assert run(device=torch.cuda.device_count()) == _lib.PFBG_ERR_ARG  # no such device
    if torch.cuda.device_count() > 1:
        assert run(device=1) == _lib.PFBG_ERR_ARG  # the convolvers are on device 0
    for bad in ((0.0, 1e-2), (1e-2, -1.0), (float("inf"), 1e-2), (float("nan"), 1e-2)):
        assert run(scale=bad) == _lib.PFBG_ERR_ARG, bad
    assert lib.pfbg_launch_count() == n0
    assert run() == 0  # and the same call with good arguments runs
    f32.close()
    close_all(trees)
