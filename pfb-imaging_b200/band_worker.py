"""Per-band workers and the cube-level pool: drop-in for
``/root/reference/src/pfb_imaging/operators/band_worker.py`` (``_BandWorkerImpl`` :23-206, ``BandWorkerPool``
:209-319) with the same constructor, role methods, argument order and cube ranks.

The reference spawns one Ray actor per band; here a band is pinned to a GPU (band b -> device b mod ndev inside one
process; with ``torch.distributed`` initialised, band b lives on rank b mod world and the cube-level results are
completed by one all-reduce, like ``BandPool``).  A worker holds the three roles of the reference actor:

  Hessian   ``init_hess`` / ``hess_dot`` / ``cg``     PSF-convolution ``HessianTree`` (operators/hessian.py:439-522)
  Psi       ``init_psi`` / ``psi_dot`` / ``psi_hdot``  SARA dictionary of one band (operators/psi.py:414-540)
  residual  ``load_band`` / ``residual``              exact ``dirty - sum_p R_p^H W_p R_p (beam_p model)``
                                                       (operators/gridder.py:926-1016), data pinned on the device

``hess_dot`` / ``hess_cg`` also take ``(nband, nx, ny)`` float64 CUDA tensors: the cube then stays on the devices
(bands pinned to another device are copied there and back), and ``hess_cg`` solves the bands of each device in one
batched ``psf.tree_cg``, the devices concurrently.

``load_band(store_url, node_name)`` reads the band node of a ``.dt`` zarr store itself (band_worker.py:61-106) through
``pfb_imaging_b200.store`` (xarray / zarr are not importable here); `store_url` may also be an already opened tree.
"""

from __future__ import annotations

import numpy as np

from . import dist as _dist


class _BandWorkerImpl:
    """One band's co-located deconvolution state; roles initialised on demand (band_worker.py:23-206)."""

    def __init__(self, nthreads=1, device=None):
        self._nthreads = nthreads
        self._device = device
        self._hess = None
        self._psib = None
        self._parts = None
        self._hess_parts = None
        self._dirty = None

    # --- band loading (worker-side reads; the driver never touches these arrays) ---
    def load_band(self, store_url, node_name):
        from .store import open_datatree

        tree = open_datatree(store_url) if isinstance(store_url, (str, bytes)) or hasattr(store_url, "__fspath__") else store_url
        band = tree[node_name]
        self._dirty = np.asarray(band.ds.DIRTY.values)  # (corr, nx, ny)
        parts, hess_parts = [], []
        for cname in sorted(band.children):
            child = band[cname].ds
            pds = child[["UVW", "WEIGHT", "MASK", "FREQ", "BEAM"]].load()
            pds.attrs.update(child.attrs)
            hess_parts.append({
                # HessianTree expects the real, non-negative magnitude of the stored complex PSFHAT (:91-97)
                "psfhat": np.abs(child.PSFHAT.values),
                "beam": pds.BEAM.values,
                "wsum": np.asarray(child.attrs["wsum"]),
            })
            parts.append(pds)
        self._parts, self._hess_parts = parts, hess_parts

    # --- Hessian role ---
    def init_hess(self, partitions, nx, ny, nx_psf, ny_psf, eta, wsum):
        from .psf import HessianTree

        if partitions is None:
            partitions = self._hess_parts
            if partitions is None:
                raise RuntimeError("no partitions passed and none loaded; call load_band first")
        if self._hess is not None:
            self._hess.close()
        self._hess = HessianTree(partitions, nx, ny, nx_psf, ny_psf, eta=eta, nthreads=self._nthreads, wsum=wsum,
                                 device=self._device)

    def hess_dot(self, x):
        return self._hess.dot(x)

    @property
    def hess(self):
        if self._hess is None:
            raise RuntimeError("no Hessian; call init_hess first")
        return self._hess

    def cg(self, rhs, x0, tol, maxit, minit, verbosity):
        from .solvers import pcg

        if x0 is not None:
            x0 = np.array(x0, copy=True)  # the solver updates x0 in place (band_worker.py:128-131)
        return pcg(lambda z: self._hess.dot(z)[0], rhs, x0=x0, tol=tol, maxit=maxit, minit=minit, verbosity=verbosity)

    # --- Psi (wavelet dictionary) role ---
    def init_psi(self, nx, ny, bases, nlevel):
        from .sara import PsiNocopyt

        self._psib = PsiNocopyt(1, nx, ny, bases, nlevel, device=self._device)
        self._alphao = np.empty((self._psib.nbasis, self._psib.nxmax, self._psib.nymax))
        self._xo = np.empty((nx, ny))
        return int(self._psib.nxmax), int(self._psib.nymax)

    def psi_dot(self, x):
        self._psib.dot(np.asarray(x)[None], self._alphao[None])
        return self._alphao

    def psi_hdot(self, alpha):
        self._psib.hdot(np.asarray(alpha)[None], self._xo[None])
        return self._xo

    # --- exact residual role ---
    def residual(self, model, cell_rad, epsilon, do_wgridding, double_accum):
        from .operators import residual_from_partitions

        return residual_from_partitions(self._dirty, self._parts, model, cell_rad, nthreads=self._nthreads,
                                        epsilon=epsilon, do_wgridding=do_wgridding, double_accum=double_accum)

    # --- telemetry ---
    def get_mem(self):
        import gc
        import os
        import resource

        gc.collect()
        out = {"pid": os.getpid(), "peak_gb": resource.getrusage(resource.RUSAGE_SELF).ru_maxrss * 1024 / 2**30}
        try:
            import psutil

            out["rss_gb"] = psutil.Process().memory_info().rss / 2**30
        except ImportError:
            pass
        return out

    def close(self):
        if self._hess is not None:
            self._hess.close()
            self._hess = None
        if self._psib is not None:
            self._psib.close()
            self._psib = None


class BandWorkerPool:
    """nband band workers plus cube-level dispatch for their role methods (band_worker.py:209-319).

    Args:
        nband: Number of imaging bands (one worker each).
        nthreads: accepted for signature compatibility (the device does the work)."""

    def __init__(self, nband, nthreads=1):
        from ._lib import device_count

        self.nband = nband
        self.nthreads_per_band = max(1, nthreads)
        world, rank = _dist.world_size(), _dist.rank()
        self._world = world
        if world > 1:
            import os

            dev = int(os.environ.get("LOCAL_RANK", "0"))
            self._mine = [b for b in range(nband) if b % world == rank]
            self._workers = {b: _BandWorkerImpl(self.nthreads_per_band, device=dev) for b in self._mine}
        else:
            ndev = max(1, device_count())
            self._mine = list(range(nband))
            self._workers = {b: _BandWorkerImpl(self.nthreads_per_band, device=b % ndev) for b in self._mine}
        self.actors = None  # the reference's attribute: no Ray actors here
        self.last_cg_info = None  # per-band iters / eps / stop of the last device hess_cg

    def _map(self, method, per_band_args):
        """Run ``method(*args)`` on the band workers of this process; band -> result."""
        return {b: getattr(self._workers[b], method)(*per_band_args[b]) for b in self._mine}

    def _complete(self, out):
        """Bands owned by other ranks are filled in by one all-reduce (they are zero here)."""
        return _dist.allreduce_sum(out) if self._world > 1 else out

    # --- band loading ---
    def load_bands(self, store_url, node_names):
        """Each worker reads its own band node from the ``.dt`` store."""
        if len(node_names) != self.nband:
            raise ValueError(f"got {len(node_names)} band nodes for {self.nband} workers")
        self._map("load_band", [(store_url, node_names[b]) for b in range(self.nband)])

    # --- Hessian role ---
    def init_hess(self, partitions_per_band, nx, ny, nx_psf, ny_psf, etas, wsums):
        """Build per-band HessianTrees; ``partitions_per_band=None`` uses load_bands data."""
        self._map("init_hess", [(None if partitions_per_band is None else partitions_per_band[b], nx, ny, nx_psf, ny_psf,
                                 etas[b], wsums[b]) for b in range(self.nband)])

    def hess_dot(self, x):
        if getattr(x, "is_cuda", False):
            return self._complete(self._hess_dot_dev(x))
        out = np.zeros_like(x)
        for b, res in self._map("hess_dot", [(x[b],) for b in range(self.nband)]).items():
            out[b] = res[0]
        return self._complete(out)

    def hess_cg(self, rhs, x0, tol, maxit, minit, verbosity):
        if getattr(rhs, "is_cuda", False):
            return self._complete(self._hess_cg_dev(rhs, x0, tol, maxit, minit, verbosity))
        out = np.zeros_like(rhs)
        args = [(rhs[b], None if x0 is None else x0[b], tol, maxit, minit, verbosity) for b in range(self.nband)]
        for b, res in self._map("cg", args).items():
            out[b] = res
        return self._complete(out)

    def _dev_cube(self, x, name):
        """The contiguous (nband, nx, ny) float64 CUDA tensor `x`; raises before anything is launched."""
        import torch

        if not getattr(x, "is_cuda", False) or x.dtype != torch.float64:
            raise TypeError(f"{name} must be a float64 CUDA tensor")
        t = self._workers[self._mine[0]].hess if self._mine else None
        if t is not None and tuple(x.shape) != (self.nband, t.nx, t.ny):
            raise ValueError(f"{name} shape {tuple(x.shape)} does not match ({self.nband}, {t.nx}, {t.ny})")
        return x.contiguous()

    def _hess_dot_dev(self, x):
        import torch

        x = self._dev_cube(x, "x")
        out = torch.zeros_like(x) if self._world > 1 else torch.empty_like(x)
        for b in self._mine:
            tree = self._workers[b].hess
            if tree.device == x.device.index:
                tree._dot_dev(x[b], out=out[b:b + 1])
            else:
                out[b].copy_(tree.dot(x[b].to(torch.device("cuda", tree.device)))[0])
        return out

    def _hess_cg_dev(self, rhs, x0, tol, maxit, minit, verbosity):
        import torch

        from .psf import tree_cg

        rhs = self._dev_cube(rhs, "rhs")
        if x0 is not None:
            x0 = self._dev_cube(x0, "x0")
            if x0.device != rhs.device:
                raise ValueError(f"x0 is on {x0.device}, rhs on {rhs.device}")
        by_dev: dict = {}
        for b in self._mine:
            by_dev.setdefault(self._workers[b].hess.device, []).append(b)
        jobs = []  # the copies run here, on torch's current streams, and each solve on its device's current stream
        for d, bands in by_dev.items():
            dev = torch.device("cuda", d)
            idx = torch.tensor(bands, device=rhs.device)
            jobs.append((bands, idx, rhs.index_select(0, idx).to(dev),
                         None if x0 is None else x0.index_select(0, idx).to(dev), torch.cuda.current_stream(dev)))

        def solve(job):
            bands, _, r, x, st = job
            return tree_cg([self._workers[b].hess for b in bands], r, x, tol, maxit, minit, stream=st)

        if len(jobs) == 1:
            results = [solve(jobs[0])]
        else:  # one host thread per device: the solves synchronise their own stream once per iteration
            from concurrent.futures import ThreadPoolExecutor

            with ThreadPoolExecutor(len(jobs)) as ex:
                results = list(ex.map(solve, jobs))
        out = torch.zeros_like(rhs)
        info = dict(iters=np.full(self.nband, -1, dtype=np.int64), eps=np.full(self.nband, np.nan),
                    stop=[None] * self.nband)  # bands of other ranks keep -1 / nan / None
        for (bands, idx, *_), (sol, inf) in zip(jobs, results):
            out.index_copy_(0, idx, sol.to(rhs.device))
            for i, b in enumerate(bands):
                info["iters"][b], info["eps"][b], info["stop"][b] = inf["iters"][i], inf["eps"][i], inf["stop"][i]
        self.last_cg_info = info
        if verbosity:
            for b in self._mine:
                print(_pcg_end_message(info["stop"][b], info["iters"][b], info["eps"][b]))
        return out

    # --- Psi role ---
    def init_psi(self, nx, ny, bases, nlevel):
        shapes = self._map("init_psi", [(nx, ny, bases, nlevel)] * self.nband)
        if not shapes:  # this rank owns no band: same bookkeeping, no device state
            from . import wavelet_filters as wf

            bk = wf.bookkeeping(nx, ny, tuple(bases), nlevel)
            return int(bk.nxmax), int(bk.nymax)
        return next(iter(shapes.values()))  # (nxmax, nymax), identical across bands

    def psi_dot(self, x, alphao):
        if self._world > 1:
            alphao[...] = 0
        for b, res in self._map("psi_dot", [(x[b],) for b in range(self.nband)]).items():
            alphao[b] = res
        self._complete(alphao)

    def psi_hdot(self, alpha, xo):
        if self._world > 1:
            xo[...] = 0
        for b, res in self._map("psi_hdot", [(alpha[b],) for b in range(self.nband)]).items():
            xo[b] = res
        self._complete(xo)

    # --- exact residual role ---
    def residual(self, model, cell_rad, epsilon=1e-7, do_wgridding=True, double_accum=True):
        """Exact per-band residual for a ``(nband, corr, nx, ny)`` model cube."""
        args = [(model[b], cell_rad, epsilon, do_wgridding, double_accum) for b in range(self.nband)]
        res = self._map("residual", args)
        if self._world == 1:
            return np.stack([res[b] for b in range(self.nband)], axis=0)
        out = np.zeros(np.shape(model), dtype=np.float64)
        for b, r in res.items():
            out[b] = r
        return self._complete(out)

    # --- telemetry ---
    def get_mem(self):
        """Per-worker memory telemetry (the reference returns [] for its in-process path)."""
        return [] if self.nband == 1 else [self._workers[b].get_mem() for b in self._mine]

    def close(self):
        for w in self._workers.values():
            w.close()


def _pcg_end_message(stop, k, eps):
    """What ``solvers.pcg`` prints at the end of a solve (verbosity >= 1), from a device stop code."""
    if stop == "initial residual zero":
        return "Initial residual is zero"
    if stop == "maxit":
        return f"Max iters reached. eps = {eps:.3e}"
    if stop == "stalled":
        return f"Stalled after {k} iterations with eps = {eps:.3e}"
    return f"Success, converged after {k} iterations"
