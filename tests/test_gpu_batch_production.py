"""GPU: batched snapshots (BASELINE config 5, `pfb hci`) at the shape the benchmark runs (bench.py `run_c5`): 256
snapshots of 512^2 per batch, 2016 baselines x 16 channels each (8.3 M samples), fp32, epsilon 1e-4, sigma_min 2,
divide_by_n: grid nu = nv = 1024 and W = 6, which takes the run kernels' general flush / fetch path, on a plane
stack of about 2000 planes (~16 GB).  fp64 at epsilon 1e-7 runs 64 snapshots of the same shape on the DMMA run
kernels (W = 10).

Every snapshot has its own point-source image and its own random visibilities, so a snapshot that reads a
neighbour's planes, rows or image slot gives a wrong answer rather than a plausible one.  The benchmark's snapshots
each span less than a tenth of the plane spacing in w, so every one of them gets W + 1 planes; the fixture stretches
the w coordinate of chosen snapshots to give them W + 2 or W + 3 planes instead (as a snapshot at low elevation
would), so that both plane-count parities occur and the pair-engine row CTAs (two neighbouring planes of the stack
each) straddle snapshot boundaries in both directions, and the plane total is odd (its last plane goes to the
one-plane row kernel).

Three snapshots are empty: a zero image at index 0, zero visibilities at the last index and every row flagged in
the middle, each next to a pair CTA that straddles into it; their outputs must be exactly zero.

Truth is the explicit DFT (oracle/dft.py) on sampled pixels and on every row of a snapshot; tolerances are the
contract: rel-L2 <= epsilon, 2 epsilon for the Hessian; two device arms agree at round-off."""
import functools

import numpy as np
import pytest

from oracle import dft, wgridder_np as wg
from pfb_imaging_b200 import synth, wgridder as W
from pfb_imaging_b200.plan import make_batch_plan, w_range
from pfbg_testutil import rel_l2

pytestmark = pytest.mark.gpu

NX, NTIME, NCHAN, BAND = 512, 1024, 16, 4
DFT_KW = dict(flip_u=False, flip_v=True, flip_w=False, do_wgridding=True, divide_by_n=True)
PLAN_KW = dict(npix_x=NX, npix_y=NX, flip_v=True, divide_by_n=True, sigma_min=2.0, sigma_max=2.6)
EPS = {"single": 1e-4, "double": 1e-7}
NSNAP = {"single": 256, "double": 64}
WANT_W = {"single": (6, 6), "double": (9, 12)}  # fp32: general flush / fetch; fp64: DMMA run kernels
ROUNDOFF = {"single": 3e-6, "double": 1e-11}
DT = {"single": (np.float32, np.complex64), "double": (np.float64, np.complex128)}


@functools.lru_cache(maxsize=1)
def _track():
    """The benchmark's observation: 1024 snapshots of a MeerKAT-like array (bench.py run_c5)."""
    rng = np.random.default_rng(1234)
    enu = synth.meerkat_like_antennas(rng)
    uvw_all = synth.uvw_tracks(enu, NTIME)  # time-major: rows [t nbl, (t+1) nbl) are snapshot t
    nbl = uvw_all.shape[0] // NTIME
    freq = synth.band_freqs(BAND, 8, NCHAN)
    cell = synth.default_cell(uvw_all, 1712e6)
    return uvw_all, nbl, freq, cell


def _pixels(rng, n=48):
    """n pixels: the centre, the four corners and random ones."""
    ix = np.concatenate([[NX // 2, 0, 0, NX - 1, NX - 1], rng.integers(0, NX, n - 5)])
    iy = np.concatenate([[NX // 2, 0, NX - 1, 0, NX - 1], rng.integers(0, NX, n - 5)])
    return ix, iy


def _design(nsnap, w, seed, leaks):
    """Planes per snapshot (W + 1, + 2, + 3) such that: snapshot 0 has an odd count; the flagged snapshot in the
    middle follows one with an odd count at an odd plane base; the last snapshot starts at an odd plane base and
    has an even count (so the total is odd)."""
    rng = np.random.default_rng([seed, 77])
    npl = w + rng.choice([1, 2, 3], size=nsnap, p=[0.5, 0.3, 0.2])

    def toggle_to(i, odd_base):  # make plane base i odd / even by changing the count of snapshot i - 2 (or i - 1)
        if (int(npl[:i].sum()) % 2 == 1) != odd_base:
            npl[i - 2] += -1 if npl[i - 2] > w + 1 else 1

    mid = nsnap // 2 if leaks else None
    last = nsnap - 1
    if npl[0] % 2 == 0:
        npl[0] += 1 if npl[0] < w + 3 else -1
    if leaks:
        if npl[mid - 1] % 2 == 0:
            npl[mid - 1] += 1 if npl[mid - 1] < w + 3 else -1
        toggle_to(mid, True)
    if npl[last] % 2:
        npl[last] += 1 if npl[last] < w + 3 else -1
    toggle_to(last, True)
    return npl.astype(np.int32), mid


def _build(prec, nsnap, first, seed, leaks):
    """Inputs of one batch of the benchmark's snapshots [first, first + nsnap) with the planned plane counts."""
    uvw_all, nbl, freq, cell = _track()
    eps = EPS[prec]
    rdt, cdt = DT[prec]
    uvw = [uvw_all[t * nbl:(t + 1) * nbl].copy() for t in range(first, first + nsnap)]
    wr = np.array([w_range(u, freq) for u in uvw])
    plan, _, npl0 = make_batch_plan(wr, nvis_per_snapshot=nbl * NCHAN, pixsize_x=cell, pixsize_y=cell, epsilon=eps,
                                    precision=prec, nx=NX, ny=NX, flip_v=True, divide_by_n=True, sigma_min=2.0,
                                    sigma_max=2.6)
    assert np.all(npl0 == plan.W + 1), "the benchmark's snapshots no longer have W + 1 planes each"
    want, mid = _design(nsnap, plan.W, seed, leaks)
    for s in range(nsnap):  # stretch w so that the span is (extra - 1/2) plane spacings
        extra = int(want[s]) - plan.W
        if extra > 1:
            uvw[s][:, 2] *= (extra - 0.5) * plan.dw / (wr[s, 1] - wr[s, 0])
    rng = np.random.default_rng([seed, 5])
    vis = [(rng.standard_normal((nbl, NCHAN)) + 1j * rng.standard_normal((nbl, NCHAN))).astype(cdt) for _ in uvw]
    wgt = [rng.uniform(0.5, 1.5, (nbl, NCHAN)).astype(rdt) for _ in uvw]
    mask = [(rng.uniform(size=(nbl, NCHAN)) > 0.02).astype(np.uint8) for _ in uvw]
    x = np.stack([synth.point_source_image(NX, NX, nsrc=20, seed=first + s, dtype=rdt) for s in range(nsnap)])
    empty = {}
    if leaks:
        empty = {0: "image", nsnap - 1: "vis", mid: "flagged"}
        x[0] = 0
        vis[nsnap - 1][:] = 0
        mask[mid][:] = 0
    geom = dict(pixsize_x=cell, pixsize_y=cell, epsilon=eps, **PLAN_KW)
    wr = [w_range(u, freq) for u in uvw]
    plan, w0, npl = make_batch_plan(wr, nvis_per_snapshot=nbl * NCHAN, pixsize_x=cell, pixsize_y=cell, epsilon=eps,
                                    precision=prec, nx=NX, ny=NX, flip_v=True, divide_by_n=True, sigma_min=2.0,
                                    sigma_max=2.6)
    assert np.array_equal(npl, want), "the stretched w-ranges no longer give the planned plane counts"
    ro = np.concatenate([[0], np.cumsum([u.shape[0] for u in uvw])]).astype(np.int64)
    return dict(prec=prec, eps=eps, uvw=uvw, freq=freq, cell=cell, vis=vis, wgt=wgt, mask=mask, x=x, geom=geom,
                w0=w0, npl=npl, pbase=np.concatenate([[0], np.cumsum(npl)[:-1]]), ro=ro, empty=empty, mid=mid,
                plan=plan)


def _check_fixture(b):
    pl, npl, pbase = b["plan"], b["npl"], b["pbase"]
    lo, hi = WANT_W[b["prec"]]
    assert lo <= pl.W <= hi, f"fixture no longer exercises W in [{lo}, {hi}]: {pl.info()}"
    assert pl.nu == pl.nv == 1024, f"fixture no longer has the benchmark's 1024^2 grid: {pl.info()}"
    if b["prec"] == "single":
        assert pl.nv % 32 == 0 and (pl.nx // 2) % 32 == 0, "fixture no longer selects pair-engine rows / TMA columns"
        assert pl.fast_screen == 1, "fixture no longer uses the fast w-screen of the benchmark"
    assert np.any(npl % 2 == 1) and np.any(npl % 2 == 0), "fixture no longer has odd and even snapshot plane counts"
    assert int(npl.sum()) % 2 == 1, "fixture no longer sends the last plane of the stack to the one-plane row kernel"
    if b["empty"]:
        mid, last = b["mid"], len(npl) - 1
        assert npl[0] % 2 == 1, "fixture no longer has a pair CTA straddling out of snapshot 0"
        assert pbase[mid] % 2 == 1 and npl[mid - 1] % 2 == 1, "fixture no longer straddles into the flagged snapshot"
        assert pbase[last] % 2 == 1, "fixture no longer straddles into the last snapshot"


def _cat(lst):
    return np.concatenate(lst, axis=0)


def _run(b):
    """One batched plan over the whole batch: degrid, grid and the Hessian (bound weights, eta = 0)."""
    gp = W.batch_plan_for(b["uvw"], b["freq"], precision=b["prec"], mask_list=b["mask"], **b["geom"])
    info = gp.info()
    assert info["nplanes"] == int(b["npl"].sum()) and info["W"] == b["plan"].W
    wgt = _cat(b["wgt"])
    out = dict(gp=gp, v=gp.degrid(b["x"]), d=gp.grid(_cat(b["vis"]), wgt))
    gp.bind_weights(wgt)
    out["h"] = gp.hessian(b["x"])
    return out




_BATCHES = {}


def _batch(prec):
    """The module's batch of `prec` (built, checked and run once; the plans are closed when the module ends)."""
    if prec not in _BATCHES:
        b = _build(prec, NSNAP[prec], 0, 0, True)
        _check_fixture(b)
        b.update(_run(b))
        _BATCHES[prec] = b
    return _BATCHES[prec]


@pytest.fixture(scope="module")
def batches(gpu):
    yield _batch
    for b in _BATCHES.values():
        b["gp"].close()
    _BATCHES.clear()
    W.clear_plan_pool()


def _rows(b, s):
    return slice(int(b["ro"][s]), int(b["ro"][s + 1]))


def _straddling(b):
    """Snapshots whose first plane shares a pair-engine row CTA with the previous snapshot's last plane."""
    return [s for s in range(1, len(b["npl"])) if b["pbase"][s] % 2 == 1]


def _dft_check(b, s, rng, what):
    """grid on 48 pixels, degrid on every row of snapshot s, and the Hessian as the DFT composition on 48 pixels."""
    eps, freq, cell = b["eps"], b["freq"], b["cell"]
    uvw, vis, wgt, mask, x = b["uvw"][s], b["vis"][s], b["wgt"][s], b["mask"][s], b["x"][s]
    px = _pixels(rng)
    kind = b["empty"].get(s)
    if kind is None or kind == "image":
        dref = dft.dft_vis2dirty(uvw, freq, vis, wgt, mask, NX, NX, cell, cell, pixels=px, **DFT_KW)
        e = rel_l2(b["d"][s][px], dref)
        assert e <= eps, (what, s, "grid", e)
    if kind is None or kind == "vis":
        vref = dft.dft_dirty2vis(uvw, freq, x.astype(np.float64), cell, cell, **DFT_KW)
        act = mask != 0
        e = rel_l2(b["v"][_rows(b, s)][act], vref[act])
        assert e <= eps, (what, s, "degrid", e)
        href = dft.dft_vis2dirty(uvw, freq, vref, wgt, mask, NX, NX, cell, cell, pixels=px, **DFT_KW)
        e = rel_l2(b["h"][s][px], href)
        assert e <= 2 * eps, (what, s, "hessian", e)


def test_binning_bit_exact_at_c5_shape(batches):
    """Kernel 1 of the batched plan against oracle.bin_indices with the batch description, over all 8.3 M samples;
    every active sample's footprint [ip0, ip0 + W) lies inside its own snapshot's plane block."""
    b = batches("single")
    gp, pl = b["gp"], b["plan"]
    uvw = _cat(b["uvw"])
    mask = _cat(b["mask"])
    ref = wg.bin_indices(gp.plan, uvw, b["freq"], mask, row_offsets=b["ro"], snap_w0=b["w0"], snap_np=b["npl"])
    dmp = gp.bin_dump()
    idx = ref["idx"]
    assert uvw.shape[0] * NCHAN == dmp["iu0"].size == 256 * 2016 * NCHAN
    for k in ("iu0", "iv0", "ip0", "key"):
        assert np.array_equal(dmp[k][idx], ref[k]), k
    assert np.array_equal(dmp["sorted_idx"].astype(np.int64), idx[ref["order"]])
    assert gp.info()["nactive"] == idx.size
    lo = b["pbase"][ref["snap"]]
    assert np.all(ref["ip0"] >= lo) and np.all(ref["ip0"] + pl.W <= lo + b["npl"][ref["snap"]])
    assert not np.any(ref["snap"] == b["mid"]), "the flagged snapshot has active samples"


@pytest.mark.parametrize("prec", ["single", "double"])
def test_snapshots_against_dft(batches, prec):
    """At least 8 snapshots: the first and the last, the one with the most planes, straddling ones, and the
    neighbours of the empty snapshots."""
    b = batches(prec)
    n = len(b["npl"])
    mid = b["mid"]
    st = [s for s in _straddling(b) if s not in b["empty"]]
    picks = sorted({0, 1, n // 4, n - 2, n - 1, int(np.argmax(b["npl"])), st[0], st[len(st) // 2], st[-1], mid - 1,
                    mid + 1})
    assert len(picks) >= 8 and b["npl"][int(np.argmax(b["npl"]))] == b["plan"].W + 3
    rng = np.random.default_rng(11)
    for s in picks:
        _dft_check(b, s, rng, prec)


@pytest.mark.parametrize("prec", ["single", "double"])
def test_every_snapshot_against_one_shot_calls(batches, prec):
    """Each snapshot alone through W.vis2dirty / W.dirty2vis (a plan of its own: no plane blocks, no row map)."""
    b = batches(prec)
    eps = b["eps"]
    tol = 2 * eps if prec == "single" else 1e-8  # plans may differ in their plane grids
    for s in range(len(b["npl"])):
        if s in b["empty"]:
            continue
        com = dict(uvw=b["uvw"][s], freq=b["freq"], mask=b["mask"][s], **{k: v for k, v in b["geom"].items()
                                                                       if not k.startswith("npix")})
        one = W.vis2dirty(vis=b["vis"][s], wgt=b["wgt"][s], npix_x=NX, npix_y=NX, **com)
        assert rel_l2(b["d"][s], one) <= tol, (s, "grid", rel_l2(b["d"][s], one))
        ov = W.dirty2vis(dirty=b["x"][s], **com)
        act = b["mask"][s] != 0
        e = rel_l2(b["v"][_rows(b, s)][act], ov[act])
        assert e <= tol, (s, "degrid", e)


@pytest.mark.parametrize("prec", ["single", "double"])
def test_empty_snapshots_are_exactly_zero(batches, prec):
    """Leak detectors: a zero image (index 0), zero visibilities (last index), every row flagged (middle), each with
    a pair CTA straddling into it.  Anything a neighbour leaks into them shows as a non-zero output."""
    b = batches(prec)
    kinds = {v: k for k, v in b["empty"].items()}
    s0, sv, sf = kinds["image"], kinds["vis"], kinds["flagged"]
    assert s0 == 0 and sv == len(b["npl"]) - 1 and sf == b["mid"]
    assert np.all(b["v"][_rows(b, s0)] == 0) and np.all(b["h"][s0] == 0)
    assert np.all(b["d"][sv] == 0)
    assert np.all(b["v"][_rows(b, sf)] == 0) and np.all(b["d"][sf] == 0) and np.all(b["h"][sf] == 0)
    for s in (s0 + 1, sv - 1, sf - 1, sf + 1):  # the neighbours are not empty
        assert np.any(b["d"][s] != 0) and np.any(b["h"][s] != 0) and np.any(b["v"][_rows(b, s)] != 0)
    # and the neighbours are right (the hessian of snapshot 1 and the grid of the last but one: the planes next
    # to the empty ones in a straddling CTA)
    rng = np.random.default_rng(13)
    for s in (s0 + 1, sv - 1, sf - 1, sf + 1):
        _dft_check(b, s, rng, "neighbour")


def test_adjointness_per_snapshot(batches):
    """<degrid(x)_s, (v w)_s> against <x_s, grid(v w)_s> for every snapshot.  With rel-L2 errors of at most
    epsilon in each direction, Cauchy-Schwarz bounds the difference by eps / (1 - eps) (|Gx| |y| + |x| |G^H y|)."""
    b = batches("single")
    eps = b["eps"]
    for s in range(len(b["npl"])):
        r = _rows(b, s)
        y = (b["vis"][s] * b["wgt"][s] * (b["mask"][s] != 0)).astype(np.complex128)
        v = b["v"][r].astype(np.complex128)
        x = b["x"][s].astype(np.float64)
        d = b["d"][s].astype(np.float64)
        lhs = np.vdot(v, y).real
        rhs = float((d * x).sum())
        bound = eps / (1 - eps) * (np.linalg.norm(v) * np.linalg.norm(y) + np.linalg.norm(x) * np.linalg.norm(d))
        assert abs(lhs - rhs) <= bound, (s, lhs, rhs, bound)


def test_hessian_dev_against_grid_of_degrid(batches):
    """hessian_dev on torch tensors (as the benchmark calls it) against grid(degrid(x)) of the same plan and against
    the host-pointer Hessian, every snapshot at fp32 round-off."""
    import torch

    b = batches("single")
    gp = b["gp"]
    dev = torch.device("cuda", gp.device)
    x_d = torch.from_numpy(b["x"]).to(dev)
    out = torch.empty_like(x_d)
    gp.hessian_dev(x_d.data_ptr(), None, 0.0, 0.0, out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    h = out.cpu().numpy()
    comp = gp.grid(b["v"], _cat(b["wgt"]))
    for s in range(len(b["npl"])):
        if s in (0, b["mid"]):  # zero image / flagged: exactly zero
            assert np.all(h[s] == 0) and np.all(comp[s] == 0), s
            continue
        assert rel_l2(h[s], comp[s]) <= ROUNDOFF["single"], (s, rel_l2(h[s], comp[s]))
        assert rel_l2(h[s], b["h"][s]) <= ROUNDOFF["single"], (s, rel_l2(h[s], b["h"][s]))


def test_pooled_plan_reused_across_chunks(batches):
    """vis2dirty_batch (a pooled plan) on three chunks in a row: 256, 256 and 100 snapshots with other plane counts.
    The second and third re-use the first chunk's plan (smaller stack, new row map, uv window and image slots); both
    against a fresh plan at round-off and sampled snapshots against the DFT."""
    W.clear_plan_pool()
    chunks = [_build("single", 256, 0, 1, False), _build("single", 256, 256, 2, False), _build("single", 100, 512, 3, False)]
    tot = [int(c["npl"].sum()) for c in chunks]
    assert not np.array_equal(chunks[0]["npl"], chunks[1]["npl"]) and tot[2] < min(tot[:2]), \
        f"fixture no longer changes the plane blocks and the stack between chunks: {tot}"
    pooled = None
    rng = np.random.default_rng(17)
    for k, c in enumerate(chunks):
        _check_fixture(c)
        cube = W.vis2dirty_batch(uvw=c["uvw"], freq=c["freq"], vis=c["vis"], wgt=c["wgt"], mask=c["mask"], **c["geom"])
        keys = [key for key in W._POOL if key[0] == "batch"]
        assert len(keys) == 1 and len(W._POOL[keys[0]]) == 1, "fixture no longer pools the batched plan"
        gp = W._POOL[keys[0]][0]
        assert pooled is None or gp is pooled, "fixture no longer re-uses the pooled plan for the next chunk"
        pooled = gp
        if k == 0:
            continue
        with W.batch_plan_for(c["uvw"], c["freq"], precision="single", mask_list=c["mask"], **c["geom"]) as fresh:
            ref = fresh.grid(_cat(c["vis"]), _cat(c["wgt"]))
        for s in range(len(c["npl"])):
            assert rel_l2(cube[s], ref[s]) <= ROUNDOFF["single"], (k, s, rel_l2(cube[s], ref[s]))
        c.update(d=cube)
        for s in (0, int(np.argmax(c["npl"])), len(c["npl"]) - 1):
            px = _pixels(rng)
            dref = dft.dft_vis2dirty(c["uvw"][s], c["freq"], c["vis"][s], c["wgt"][s], c["mask"][s], NX, NX, c["cell"],
                                     c["cell"], pixels=px, **DFT_KW)
            assert rel_l2(cube[s][px], dref) <= c["eps"], (k, s)
    W.clear_plan_pool()
