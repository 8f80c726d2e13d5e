"""Drop-in ``vis2dirty`` / ``dirty2vis`` with the keyword signatures pfb-imaging
uses for ``ducc0.wgridder[.experimental]`` (``/root/reference/src/pfb_imaging/
operators/gridder.py:78-100, 485-503``; ``operators/hessian.py:50-89``).

numpy in, numpy out; the work happens in ``libpfbgrid.so`` on a B200.
:class:`GridderPlan` is the stateful form (geometry bound and binned once,
reused across calls); the free functions build a plan per call like ducc0 does.
"""

from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from . import _lib
from .plan import LIGHTSPEED, Plan, good_size, make_batch_plan, make_plan, w_range

_PREC = {"single": _lib.PFBG_F32, "double": _lib.PFBG_F64}
_RDT = {"single": np.float32, "double": np.float64}
_CDT = {"single": np.complex64, "double": np.complex128}


def _ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def content_hash(a) -> int:
    """64-bit hash of the full content of a numpy array (threaded, in libpfbgrid.so; host memory only)."""
    a = np.asarray(a)
    if not a.flags.c_contiguous:
        a = np.ascontiguousarray(a)
    h = C.c_uint64(0)
    _lib.check(_lib.load().pfbg_host_hash64(C.c_void_p(a.ctypes.data), a.nbytes, C.byref(h)))
    return int(h.value)


def current_device() -> int:
    import os

    return int(os.environ.get("PFBG_DEVICE", os.environ.get("LOCAL_RANK", "0")))


def _plan_desc(plan: Plan, device: int):
    """The C struct of a host-side plan (+ the arrays it points to, which the caller keeps alive)."""
    keep = (np.ascontiguousarray(plan.corr_u, dtype=np.float64),
            np.ascontiguousarray(plan.corr_v, dtype=np.float64),
            np.ascontiguousarray(plan.gl_x, dtype=np.float64),
            np.ascontiguousarray(plan.gl_w, dtype=np.float64))
    d = _lib.PlanDesc(
        precision=_PREC[plan.precision], device=device, nx=plan.nx, ny=plan.ny, nu=plan.nu, nv=plan.nv,
        W=plan.W, nplanes=plan.nplanes, do_wgridding=int(plan.do_wgridding), divide_by_n=int(plan.divide_by_n),
        beta=plan.beta, pixsize_x=plan.pixsize_x, pixsize_y=plan.pixsize_y,
        center_x=plan.center_x, center_y=plan.center_y, usign=plan.usign, vsign=plan.vsign, wsign=plan.wsign,
        w0=plan.w0, dw=plan.dw, nshift=plan.nshift,
        corr_u=keep[0].ctypes.data, corr_v=keep[1].ctypes.data,
        gl_x=keep[2].ctypes.data, gl_w=keep[3].ctypes.data, n_gl=len(keep[2]),
        pmirror=int(getattr(plan, "pmirror", 0)),
        fast_screen=int(getattr(plan, "fast_screen", 0)),
    )
    return d, keep


class GridderPlan:
    """A plan bound to one set of (uvw, freq, mask): the analogue of the state a
    band worker pins (``operators/band_worker.py:61-106``)."""

    def __init__(self, plan: Plan, device: int | None = None, external_stack: bool = False):
        self.plan = plan
        self.device = current_device() if device is None else int(device)
        self._h = C.c_void_p()
        self._lib = _lib.load()
        d, self._keep = _plan_desc(plan, self.device)
        if external_stack:  # no plane stack of its own: one is lent with set_stack() (StackArena)
            d.flags |= _lib.PLAN_EXTERNAL_STACK
        self._stack_ref = None
        _lib.check(self._lib.pfbg_plan_create(C.byref(d), C.byref(self._h)))
        self.nrow = self.nchan = 0
        self.nbatch = 0  # > 0: batched snapshots, image arguments are (nbatch, nx, ny)
        self.rdt = _RDT[plan.precision]
        self.cdt = _CDT[plan.precision]

    # -- lifetime -----------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.pfbg_plan_destroy(self._h)
            self._h = C.c_void_p()
        self._stack_ref = None  # a lent plane stack goes back to its owner

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_stack(self, dev_ptr, nbytes, keep=None):
        """Lend the plan a plane stack (``pfbg_plan_set_stack``): device memory of this plan's device, at least
        ``info()["grid_bytes"]`` bytes.  The stack is scratch between calls, so the bands sharing a GPU can take
        turns on one stack per compute stream.  ``keep`` is held to keep the memory alive (e.g. a torch tensor)."""
        _lib.check(self._lib.pfbg_plan_set_stack(self._h, C.c_void_p(int(dev_ptr) if dev_ptr else None),
                                                 C.c_uint64(int(nbytes))))
        self._stack_ref = keep

    # -- binding ------------------------------------------------------------
    def bind(self, uvw, freq, mask=None, stream=None):
        self._beam_fp = None
        uvw = np.ascontiguousarray(uvw, dtype=np.float64)
        freq = np.ascontiguousarray(freq, dtype=np.float64)
        if uvw.ndim != 2 or uvw.shape[1] != 3:
            raise ValueError("uvw must have shape (nrow, 3)")
        if freq.ndim != 1 or freq.size == 0:
            raise ValueError("freq must be a non-empty 1-D array")
        nrow, nchan = uvw.shape[0], freq.size
        fscale = np.ascontiguousarray(freq / LIGHTSPEED)
        if mask is not None:
            mask = np.asarray(mask)
            if mask.shape != (nrow, nchan):
                raise ValueError(f"mask shape {mask.shape} != ({nrow}, {nchan})")
            mask = np.ascontiguousarray(mask != 0 if mask.dtype != np.uint8 else mask, dtype=np.uint8)
        _lib.check(self._lib.pfbg_bind_vis(self._h, _ptr(uvw), _ptr(fscale), _ptr(mask), nrow, nchan,
                                           _lib.HOST_PTRS, stream))
        self.nrow, self.nchan = nrow, nchan
        return self

    # -- batched snapshots (include/pfbgrid.h "Batched snapshots") --------------------------------------------
    def set_batch(self, snap_w0, snap_np):
        """Turn this plan into a batch of len(snap_w0) snapshots sharing its geometry (plan.make_batch_plan)."""
        w0 = np.ascontiguousarray(snap_w0, dtype=np.float64)
        npl = np.ascontiguousarray(snap_np, dtype=np.int32)
        if w0.ndim != 1 or w0.shape != npl.shape or w0.size == 0:
            raise ValueError("snap_w0 / snap_np must be 1-D arrays of one length")
        _lib.check(self._lib.pfbg_plan_set_batch(self._h, w0.size, _ptr(w0), _ptr(npl)))
        self.nbatch = int(w0.size)
        return self

    def bind_batch(self, uvw, freq, row_offsets, mask=None, stream=None):
        """Bind the rows of all snapshots, concatenated; rows [row_offsets[s], row_offsets[s+1]) are snapshot s."""
        if not self.nbatch:
            raise RuntimeError("set_batch first")
        self._beam_fp = None
        uvw = np.ascontiguousarray(uvw, dtype=np.float64)
        freq = np.ascontiguousarray(freq, dtype=np.float64)
        ro = np.ascontiguousarray(row_offsets, dtype=np.int64)
        if uvw.ndim != 2 or uvw.shape[1] != 3:
            raise ValueError("uvw must have shape (nrow, 3)")
        if ro.shape != (self.nbatch + 1,):
            raise ValueError(f"row_offsets must have {self.nbatch + 1} entries")
        nrow, nchan = uvw.shape[0], freq.size
        fscale = np.ascontiguousarray(freq / LIGHTSPEED)
        if mask is not None:
            mask = np.asarray(mask)
            if mask.shape != (nrow, nchan):
                raise ValueError(f"mask shape {mask.shape} != ({nrow}, {nchan})")
            mask = np.ascontiguousarray(mask != 0 if mask.dtype != np.uint8 else mask, dtype=np.uint8)
        _lib.check(self._lib.pfbg_bind_vis_batch(self._h, _ptr(uvw), _ptr(fscale), _ptr(mask), nrow, nchan, _ptr(ro),
                                                 _lib.HOST_PTRS, stream))
        self.nrow, self.nchan = nrow, nchan
        return self

    @property
    def image_shape(self):
        return (self.nbatch, self.plan.nx, self.plan.ny) if self.nbatch else (self.plan.nx, self.plan.ny)

    def bind_weights(self, wgt, stream=None):
        if wgt is not None:
            wgt = self._check_wgt(wgt)
        _lib.check(self._lib.pfbg_bind_weights(self._h, _ptr(wgt), _lib.HOST_PTRS, stream))
        return self

    def bind_robust_weights(self, wgt, nx_pad, ny_pad, cellx, celly, robust, usign=1.0, vsign=-1.0, stream=None):
        """Bind the Briggs/uniform weights of every snapshot of the bound batch, computed on the device from the
        natural weights `wgt` (nrow, nchan) as ``weighting.counts_to_weights_batch`` computes them, without the
        weights coming back to the host (``pfbg_bind_weights_robust``).  Later calls without `wgt` use them."""
        wgt = self._check_wgt(wgt)
        _lib.check(self._lib.pfbg_bind_weights_robust(self._h, _ptr(wgt), int(nx_pad), int(ny_pad), float(cellx),
                                                      float(celly), float(robust), float(usign), float(vsign),
                                                      _lib.HOST_PTRS, stream))
        return self

    def info(self) -> dict:
        i = _lib.PlanInfo()
        _lib.check(self._lib.pfbg_plan_get_info(self._h, C.byref(i)))
        out = {k: getattr(i, k) for k, _ in _lib.PlanInfo._fields_}
        out.update(self.plan.info())
        return out

    def bin_dump(self):
        """Kernel-1 outputs for the bit-exact check (host arrays)."""
        i = self.info()
        n, na = i["nvis"], i["nactive"]
        iu0, iv0, ip0 = (np.empty(n, np.int32) for _ in range(3))
        key = np.empty(n, np.uint64)
        sidx = np.empty(na, np.uint32)
        _lib.check(self._lib.pfbg_bin_dump(self._h, _ptr(iu0), _ptr(iv0), _ptr(ip0), _ptr(key), _ptr(sidx)))
        return dict(iu0=iu0, iv0=iv0, ip0=ip0, key=key, sorted_idx=sidx)

    # -- argument checks ----------------------------------------------------
    def _check_wgt(self, wgt):
        wgt = np.asarray(wgt)
        if wgt.shape != (self.nrow, self.nchan):
            raise ValueError(f"wgt shape {wgt.shape} != ({self.nrow}, {self.nchan})")
        if wgt.dtype != self.rdt:
            raise TypeError(f"wgt dtype {wgt.dtype} does not match precision '{self.plan.precision}' ({self.rdt.__name__})")
        return np.ascontiguousarray(wgt)

    def _check_img(self, x, name):
        x = np.asarray(x)
        if x.shape != self.image_shape:
            raise ValueError(f"{name} shape {x.shape} != {self.image_shape}")
        if x.dtype != self.rdt:
            raise TypeError(f"{name} dtype {x.dtype} does not match precision '{self.plan.precision}'")
        return np.ascontiguousarray(x)

    # -- operators (host arrays) ---------------------------------------------
    def grid(self, vis, wgt=None, dirty=None, stream=None):
        vis = np.asarray(vis)
        if vis.shape != (self.nrow, self.nchan):
            raise ValueError(f"vis shape {vis.shape} != ({self.nrow}, {self.nchan})")
        if vis.dtype != self.cdt:
            raise TypeError(f"vis dtype {vis.dtype} does not match precision '{self.plan.precision}' ({self.cdt.__name__})")
        if vis.size and all(s == 0 for s in vis.strides):
            rs = cs = 0  # np.broadcast_to(scalar): operators/gridder.py:627-629
        else:
            vis = np.ascontiguousarray(vis)
            rs, cs = self.nchan, 1
        if wgt is not None:
            wgt = self._check_wgt(wgt)
        out = self._out_img(dirty, "dirty")
        tmp = out if out.flags.c_contiguous else np.empty(out.shape, out.dtype)
        _lib.check(self._lib.pfbg_grid(self._h, _ptr(vis), rs, cs, _ptr(wgt), _ptr(tmp), _lib.HOST_PTRS, stream))
        if tmp is not out:
            out[...] = tmp
        return out

    def grid_psf(self, x0, y0, wgt=None, dirty=None, sign=1.0, stream=None):
        """PSF of a field centred at (x0, y0): grids exp(sign 2 pi i f/c (u x0 + v y0 - w (n0 - 1))) generated on the
        device from the bound uvw (operators/gridder.py:616-629; sign=-1 for utils/stokes2im.py:483-486)."""
        if wgt is not None:
            wgt = self._check_wgt(wgt)
        out = self._out_img(dirty, "dirty")
        tmp = out if out.flags.c_contiguous else np.empty(out.shape, out.dtype)
        _lib.check(self._lib.pfbg_grid_psf(self._h, float(x0), float(y0), float(sign), _ptr(wgt), _ptr(tmp),
                                           _lib.HOST_PTRS, stream))
        if tmp is not out:
            out[...] = tmp
        return out

    def _out_img(self, arr, name):
        if arr is None:
            return np.empty(self.image_shape, dtype=self.rdt)
        if not isinstance(arr, np.ndarray) or arr.shape != self.image_shape or arr.dtype != self.rdt:
            raise ValueError(f"`{name}` must be a {self.image_shape} {self.rdt.__name__} array")
        if not arr.flags.writeable:
            raise ValueError(f"`{name}` is read-only")
        return arr

    def degrid(self, dirty, wgt=None, vis=None, stream=None):
        x = self._check_img(dirty, "dirty")
        flags = _lib.HOST_PTRS
        if wgt is not None:
            wgt = self._check_wgt(wgt)
            flags |= _lib.APPLY_WGT
        if vis is None:
            out = np.empty((self.nrow, self.nchan), dtype=self.cdt)
        else:
            if not isinstance(vis, np.ndarray) or vis.shape != (self.nrow, self.nchan) or vis.dtype != self.cdt:
                raise ValueError(f"`vis` must be a ({self.nrow}, {self.nchan}) {self.cdt.__name__} array")
            if not vis.flags.writeable:
                raise ValueError("`vis` is read-only")
            out = vis
        tmp = out if out.flags.c_contiguous else np.empty(out.shape, out.dtype)
        _lib.check(self._lib.pfbg_degrid(self._h, _ptr(x), _ptr(tmp), _ptr(wgt), flags, stream))
        if tmp is not out:
            out[...] = tmp
        return out

    def hessian(self, x, beam=None, wsum=None, eta=None, out=None, stream=None):
        x = self._check_img(x, "x")
        if beam is not None:
            beam = self._check_img(beam, "beam")
        res = self._out_img(out, "out")
        tmp = res if res.flags.c_contiguous else np.empty(res.shape, res.dtype)
        flags = _lib.HOST_PTRS
        if beam is not None:
            # the beam of a band never changes between applies: upload it once (address + size + a hash of its full
            # content identify it, so an in-place patch of a few pixels is seen; PFBG_BEAM_CACHE=0 re-uploads every call)
            fp = (beam.ctypes.data, beam.nbytes, content_hash(beam))
            if _BEAM_CACHE and fp == getattr(self, "_beam_fp", None):
                flags |= _lib.BEAM_CACHED
            self._beam_fp = fp
        if _pinned(x):
            flags |= _lib.PINNED_IN
        if out is not None and _pinned(tmp):  # a fresh output array is never seen twice
            flags |= _lib.PINNED_OUT
        _lib.check(self._lib.pfbg_hessian(self._h, _ptr(x), _ptr(beam), float(wsum) if wsum else 0.0,
                                          float(eta) if eta else 0.0, _ptr(tmp), flags, stream))
        if tmp is not res:
            res[...] = tmp
        return res

    # -- operators (device pointers; asynchronous on `stream`) ----------------
    def hessian_dev(self, x_ptr, beam_ptr, wsum, eta, out_ptr, stream=None):
        _lib.check(self._lib.pfbg_hessian(self._h, x_ptr, beam_ptr, float(wsum) if wsum else 0.0,
                                          float(eta) if eta else 0.0, out_ptr, _lib.DEVICE_PTRS, stream))

    def grid_dev(self, vis_ptr, wgt_ptr, dirty_ptr, stream=None, rs=None, cs=1):
        rs = self.nchan if rs is None else rs
        _lib.check(self._lib.pfbg_grid(self._h, vis_ptr, rs, cs, wgt_ptr, dirty_ptr, _lib.DEVICE_PTRS, stream))

    def degrid_dev(self, dirty_ptr, vis_ptr, stream=None):
        _lib.check(self._lib.pfbg_degrid(self._h, dirty_ptr, vis_ptr, None, _lib.DEVICE_PTRS, stream))

    # -- band split across two GPUs (include/pfbgrid.h "Band split"; pfb_imaging_b200.split drives it) ---------
    def window(self):
        """(a_lo, a_len, b_lo, b_len): grid rows / columns any bound sample can touch."""
        w = (C.c_int32 * 4)()
        _lib.check(self._lib.pfbg_plan_get_window(self._h, w))
        return tuple(int(v) for v in w)

    def split_owner_init(self, nq: int) -> bytes:
        """Hand the transforms of the last `nq` planes to a helper: returns the four IPC blobs the helper needs
        (plane stack, shared image, partial image, mailbox)."""
        buf = C.create_string_buffer(4 * _lib.IPC_BLOB_BYTES)
        _lib.check(self._lib.pfbg_split_owner_init(self._h, int(nq), buf))
        return buf.raw

    def split_owner_connect(self, helper_mailbox: bytes):
        buf = C.create_string_buffer(bytes(helper_mailbox), _lib.IPC_BLOB_BYTES)
        _lib.check(self._lib.pfbg_split_owner_connect(self._h, buf))

    def split_timed_out(self, stream=None) -> bool:
        t = C.c_int32(0)
        _lib.check(self._lib.pfbg_split_status(self._h, stream, C.byref(t)))
        return bool(t.value)

    def split_end(self):
        _lib.check(self._lib.pfbg_split_end(self._h))

    def set_profiling(self, on=True):
        _lib.check(self._lib.pfbg_set_profiling(self._h, int(on)))

    def timings(self):
        ms = (C.c_float * 8)()
        n = C.c_int32(0)
        _lib.check(self._lib.pfbg_get_timings(self._h, ms, 8, C.byref(n)))
        return [ms[i] for i in range(n.value)]


class SplitHelper:
    """Transform helper of a band whose owner lives on another GPU / in another process: holds the band's geometry
    (no visibilities) and the last `nq` planes; ``serve`` enqueues one Hessian apply worth of helper work."""

    def __init__(self, plan: Plan, nq: int, window, owner_blobs: bytes, device: int | None = None):
        self.plan, self.nq = plan, int(nq)
        self.device = current_device() if device is None else int(device)
        self._lib = _lib.load()
        self._h = C.c_void_p()
        d, self._keep = _plan_desc(plan, self.device)
        win = (C.c_int32 * 4)(*[int(v) for v in window])
        blobs = C.create_string_buffer(bytes(owner_blobs), 4 * _lib.IPC_BLOB_BYTES)
        mb = C.create_string_buffer(_lib.IPC_BLOB_BYTES)
        _lib.check(self._lib.pfbg_split_helper_create(C.byref(d), self.nq, win, blobs, C.byref(self._h), mb))
        self.mailbox_blob = mb.raw

    def serve(self, stream=None):
        _lib.check(self._lib.pfbg_split_helper_serve(self._h, stream))

    def timed_out(self, stream=None) -> bool:
        t = C.c_int32(0)
        _lib.check(self._lib.pfbg_split_status(self._h, stream, C.byref(t)))
        return bool(t.value)

    def set_profiling(self, on=True):
        _lib.check(self._lib.pfbg_set_profiling(self._h, int(on)))

    def timings(self):
        ms = (C.c_float * 8)()
        n = C.c_int32(0)
        _lib.check(self._lib.pfbg_get_timings(self._h, ms, 8, C.byref(n)))
        return [ms[i] for i in range(n.value)]

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.pfbg_plan_destroy(self._h)
            self._h = C.c_void_p()
        self._stack_ref = None  # a lent plane stack goes back to its owner

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---------------------------------------------------------------------------
# Page-locking of caller arrays that keep coming back (solver work vectors, `xout=` buffers): the second time
# the same buffer is seen it is registered with CUDA, after which its copies are single DMAs instead of a
# staged copy through the library's pinned buffer (64 MB image: ~1.3 ms instead of ~3.5 ms per direction).
# The registration is dropped when the owning ndarray is garbage collected (weakref finaliser, which runs
# before numpy releases the data) or when the table overflows.
# ---------------------------------------------------------------------------
_BEAM_CACHE = __import__("os").environ.get("PFBG_BEAM_CACHE", "1") != "0"
_PIN_SEEN: dict = {}
_PIN_REG: dict = {}
_PIN_MAX_BYTES = int(__import__("os").environ.get("PFBG_PIN_MAX_MB", "4096")) << 20
_PIN_MIN_BYTES = 1 << 20


def _pin_owner(a):
    while isinstance(getattr(a, "base", None), np.ndarray):
        a = a.base
    return a if (isinstance(a, np.ndarray) and a.base is None and a.flags.owndata) else None


def _unpin(key):
    ent = _PIN_REG.pop(key, None)
    if ent is not None:
        try:
            _lib.load().pfbg_host_unregister(C.c_void_p(key[0]))
        except Exception:
            pass


def _pinned(a) -> bool:
    """True if `a`'s memory is (now) page-locked.  Registers on the second sighting of the same live buffer."""
    if _PIN_MAX_BYTES <= 0 or a.nbytes < _PIN_MIN_BYTES:
        return False
    owner = _pin_owner(a)
    if owner is None:
        return False
    key = (owner.ctypes.data, owner.nbytes)
    if key in _PIN_REG:  # the finaliser removes the entry before the memory can be re-used
        return True
    ref = _PIN_SEEN.get(key)
    if ref is None or ref() is not owner:  # first sighting of this array object
        if len(_PIN_SEEN) > 256:
            _PIN_SEEN.clear()
        _PIN_SEEN[key] = weakref.ref(owner)
        return False
    while _PIN_REG and sum(k[1] for k in _PIN_REG) + owner.nbytes > _PIN_MAX_BYTES:
        key0 = next(iter(_PIN_REG))
        fin = _PIN_REG.get(key0)
        _unpin(key0)
        if fin is not None:
            fin.detach()
    if _lib.load().pfbg_host_register(C.c_void_p(key[0]), owner.nbytes) != 0:
        _PIN_SEEN.pop(key, None)
        return False
    _PIN_REG[key] = weakref.finalize(owner, _unpin, key)
    _PIN_SEEN.pop(key, None)
    return True


def clear_pinned():
    for key in list(_PIN_REG):
        fin = _PIN_REG.get(key)
        _unpin(key)
        if fin is not None:
            fin.detach()


# ---------------------------------------------------------------------------
# plan pool for the one-shot entry points: a plan is re-used whenever image geometry, sigma and W
# agree (only the w-plane range and the bound samples change), which removes all per-call device /
# pinned allocations and table set-up.  This is what makes thousands of small snapshot images
# (pfb hci, utils/stokes2im.py:635-683) affordable.
# ---------------------------------------------------------------------------
_POOL: dict = {}
_POOL_MAX = int(__import__("os").environ.get("PFBG_PLAN_POOL", "8"))


def _pool_key(p: Plan, device):
    return (device, p.precision, p.nx, p.ny, p.nu, p.nv, p.W, round(p.beta, 12), p.pixsize_x, p.pixsize_y,
            p.center_x, p.center_y, p.usign, p.vsign, p.wsign, p.do_wgridding, p.divide_by_n, p.dw, p.nshift,
            getattr(p, "fast_screen", 0))


def clear_plan_pool():
    for lst in _POOL.values():
        for gp in lst:
            gp.close()
    _POOL.clear()


class _Pooled:
    """Context manager handing out a pooled GridderPlan and taking it back afterwards."""

    def __init__(self, gp, key):
        self.gp, self.key = gp, key

    def __enter__(self):
        return self.gp

    def __exit__(self, et, ev, tb):
        if et is not None or _POOL_MAX <= 0 or sum(len(v) for v in _POOL.values()) >= _POOL_MAX:
            self.gp.close()
        else:
            _POOL.setdefault(self.key, []).append(self.gp)


def _precision_of(dtype, what):
    dt = np.dtype(dtype)
    if dt in (np.dtype(np.complex64), np.dtype(np.float32)):
        return "single"
    if dt in (np.dtype(np.complex128), np.dtype(np.float64)):
        return "double"
    raise TypeError(f"unsupported {what} dtype {dt}")


def plan_for(uvw, freq, *, npix_x, npix_y, pixsize_x, pixsize_y, center_x=0.0, center_y=0.0, epsilon,
             flip_u=False, flip_v=False, flip_w=False, do_wgridding=True, divide_by_n=True,
             sigma_min=1.1, sigma_max=2.6, precision="double", mask=None, device=None, pooled=False,
             external_stack=False, **force) -> GridderPlan:
    """Build a plan for the geometry and bind (uvw, freq, mask) to it.  ``external_stack=True``: the plan owns no
    plane stack; lend it one (``GridderPlan.set_stack`` / ``StackArena``) before the first transform call."""
    uvw = np.asarray(uvw)
    freq = np.asarray(freq)
    wmin, wmax = w_range(uvw, freq, -1.0 if flip_w else 1.0) if do_wgridding else (0.0, 0.0)
    p = make_plan(nx=npix_x, ny=npix_y, pixsize_x=pixsize_x, pixsize_y=pixsize_y, center_x=center_x,
                  center_y=center_y, epsilon=epsilon, flip_u=flip_u, flip_v=flip_v, flip_w=flip_w,
                  do_wgridding=do_wgridding, divide_by_n=divide_by_n, sigma_min=sigma_min, sigma_max=sigma_max,
                  precision=precision, wmin=wmin, wmax=wmax, nvis=uvw.shape[0] * freq.size, **force)
    if pooled and _POOL_MAX > 0:
        dev = current_device() if device is None else int(device)
        key = _pool_key(p, dev)
        free = _POOL.get(key)
        if free:
            gp = free.pop()
            _lib.check(gp._lib.pfbg_plan_set_wrange(gp._h, p.w0, p.nplanes, int(p.pmirror)))
            gp.plan = p
        else:
            gp = GridderPlan(p, device=dev)
        try:
            gp.bind(uvw, freq, mask)
        except Exception:
            gp.close()
            raise
        return _Pooled(gp, key)
    gp = GridderPlan(p, device=device, external_stack=external_stack)
    try:
        gp.bind(uvw, freq, mask)
    except Exception:
        gp.close()
        raise
    return gp


class StackArena:
    """Plane stacks shared by the band plans of one GPU.

    A plan's plane stack (nplanes x nu x nv complex cells: 2.4-3.3 GB per config-2 band, 62 GB per config-4 band) is
    scratch between calls, so ``nslots`` stacks — one per compute stream — serve any number of bands: band i uses
    slot ``i % nslots`` and the caller keeps the calls of a slot on one stream.  The reference keeps one worker
    process per band (``operators/band_worker.py:217-246``), each with its own ducc0 grid."""

    def __init__(self, plans, nslots=1, device=None):
        import torch

        plans = list(plans)
        self.nslots = max(1, min(int(nslots), len(plans)))
        dev = plans[0].device if device is None else int(device)
        need = max(int(gp.info()["grid_bytes"]) for gp in plans)
        self.nbytes = (need + 255) // 256 * 256
        self.buffers = [torch.empty(self.nbytes, dtype=torch.uint8, device=torch.device("cuda", dev))
                        for _ in range(self.nslots)]
        for i, gp in enumerate(plans):
            buf = self.buffers[i % self.nslots]
            gp.set_stack(buf.data_ptr(), self.nbytes, keep=buf)

    def slot(self, i):
        return i % self.nslots


def vis2dirty(*, uvw, freq, vis, wgt=None, mask=None, npix_x, npix_y, pixsize_x, pixsize_y,
              center_x=0.0, center_y=0.0, epsilon, flip_u=False, flip_v=False, flip_w=False,
              do_wgridding=True, divide_by_n=True, nthreads=1, sigma_min=1.1, sigma_max=2.6,
              double_precision_accumulation=False, verbosity=0, dirty=None, allow_nshift=True, gpu=False):
    """``ducc0.wgridder.experimental.vis2dirty`` replacement (B200).

    ``nthreads``, ``verbosity``, ``double_precision_accumulation`` (the plane sum
    is always accumulated in fp64), ``allow_nshift`` and ``gpu`` are accepted
    for signature compatibility and otherwise ignored.
    """
    vis = np.asarray(vis)
    prec = _precision_of(vis.dtype, "vis")
    with plan_for(uvw, freq, npix_x=npix_x, npix_y=npix_y, pixsize_x=pixsize_x, pixsize_y=pixsize_y,
                  center_x=center_x, center_y=center_y, epsilon=epsilon, flip_u=flip_u, flip_v=flip_v,
                  flip_w=flip_w, do_wgridding=do_wgridding, divide_by_n=divide_by_n, sigma_min=sigma_min,
                  sigma_max=sigma_max, precision=prec, mask=mask, pooled=True) as gp:
        return gp.grid(vis, wgt=wgt, dirty=dirty)


def dirty2vis(*, uvw, freq, dirty, wgt=None, mask=None, pixsize_x, pixsize_y, center_x=0.0, center_y=0.0,
              epsilon, flip_u=False, flip_v=False, flip_w=False, do_wgridding=True, divide_by_n=True,
              nthreads=1, sigma_min=1.1, sigma_max=2.6, verbosity=0, vis=None, allow_nshift=True, gpu=False):
    """``ducc0.wgridder.experimental.dirty2vis`` replacement (B200)."""
    dirty = np.asarray(dirty)
    if dirty.ndim != 2:
        raise ValueError("dirty must be 2-D")
    prec = _precision_of(dirty.dtype, "dirty")
    with plan_for(uvw, freq, npix_x=dirty.shape[0], npix_y=dirty.shape[1], pixsize_x=pixsize_x,
                  pixsize_y=pixsize_y, center_x=center_x, center_y=center_y, epsilon=epsilon, flip_u=flip_u,
                  flip_v=flip_v, flip_w=flip_w, do_wgridding=do_wgridding, divide_by_n=divide_by_n,
                  sigma_min=sigma_min, sigma_max=sigma_max, precision=prec, mask=mask, pooled=True) as gp:
        return gp.degrid(dirty, wgt=wgt, vis=vis)


# ---------------------------------------------------------------------------
# batched snapshots: `pfb hci` images thousands of small snapshots, two vis2dirty calls each
# (utils/stokes2im.py:635-683: residual + PSF, sigma_min = min_padding = 2, divide_by_n = True).  One launch
# sequence per snapshot is launch-latency bound (1.24 ms per pooled call against ~10 us of work); a batch goes
# through ONE bin / sort and one launch of every kernel.
# ---------------------------------------------------------------------------
def batch_plan_for(uvw_list, freq, *, npix_x, npix_y, pixsize_x, pixsize_y, center_x=0.0, center_y=0.0, epsilon,
                   flip_u=False, flip_v=False, flip_w=False, do_wgridding=True, divide_by_n=True, sigma_min=1.1,
                   sigma_max=2.6, precision="double", mask_list=None, device=None, pooled=False, **force) -> GridderPlan:
    """One plan for the snapshots `uvw_list` (each (nrow_s, 3)) of a common geometry, bound and binned.
    ``pooled=True`` returns a context manager that hands the plan back to the pool of the one-shot calls: the next
    batch of the same geometry re-uses its device buffers and tables (hci images chunk after chunk)."""
    freq = np.asarray(freq, dtype=np.float64)
    wr = [w_range(u, freq) if do_wgridding else (0.0, 0.0) for u in uvw_list]
    nrow_max = max(int(np.asarray(u).shape[0]) for u in uvw_list)
    p, w0, npl = make_batch_plan(wr, nvis_per_snapshot=nrow_max * freq.size, nx=npix_x, ny=npix_y, pixsize_x=pixsize_x,
                                 pixsize_y=pixsize_y, center_x=center_x, center_y=center_y, epsilon=epsilon, flip_u=flip_u,
                                 flip_v=flip_v, flip_w=flip_w, do_wgridding=do_wgridding, divide_by_n=divide_by_n,
                                 sigma_min=sigma_min, sigma_max=sigma_max, precision=precision, **force)
    dev = current_device() if device is None else int(device)
    key = ("batch",) + _pool_key(p, dev)
    free = _POOL.get(key) if pooled and _POOL_MAX > 0 else None
    if free:  # same geometry, sigma, W: only the plane blocks and the bound samples change
        gp = free.pop()
    else:
        first = Plan(**{**p.__dict__, "nplanes": int(p.W if do_wgridding else 1)})  # the stack is sized by set_batch
        gp = GridderPlan(first, device=dev)
    try:
        gp.set_batch(w0, npl)
        p.nplanes = int(npl.sum())
        gp.plan = p
        ro = np.concatenate([[0], np.cumsum([np.asarray(u).shape[0] for u in uvw_list])]).astype(np.int64)
        uvw = np.concatenate([np.asarray(u, dtype=np.float64) for u in uvw_list], axis=0)
        mask = None if mask_list is None else np.concatenate([np.asarray(m) for m in mask_list], axis=0)
        gp.bind_batch(uvw, freq, ro, mask)
        gp.row_offsets = ro
    except Exception:
        gp.close()
        raise
    return _Pooled(gp, key) if pooled and _POOL_MAX > 0 else gp


def vis2dirty_batch(*, uvw, freq, vis, wgt=None, mask=None, npix_x, npix_y, pixsize_x, pixsize_y, center_x=0.0,
                    center_y=0.0, epsilon, flip_u=False, flip_v=False, flip_w=False, do_wgridding=True, divide_by_n=True,
                    nthreads=1, sigma_min=1.1, sigma_max=2.6, double_precision_accumulation=False, verbosity=0,
                    dirty=None, extra_vis=(), robustness=None, nx_pad=None, ny_pad=None):
    """``vis2dirty`` for a list of snapshots of one geometry: `uvw`, `vis`, `wgt`, `mask` are lists (one entry per
    snapshot, `freq` is shared); returns ``(nsnap, npix_x, npix_y)``.  `extra_vis`: further lists of visibilities
    gridded with the same binding (the PSF visibilities of stokes2im.py:660-683); then a tuple of cubes comes back.

    `robustness`: grid with each snapshot's Briggs weights (utils/stokes2im.py:563-604), computed on the device from
    `wgt` (ones when None) on an (nx_pad, ny_pad) counts grid with cells (pixsize_x, pixsize_y), as
    ``weighting.counts_to_weights_batch`` computes them.  The pad defaults to ``plan.good_size(2 * npix)``, which
    admits the factors 2, 3, 5, 7; the reference's ducc0 ``good_size`` also admits 11, so pass the pad where the two
    differ.  ``filter_extreme_counts`` / ``box_sum_counts`` are not applied."""
    nsnap = len(uvw)
    prec = _precision_of(np.asarray(vis[0]).dtype, "vis")
    gp = batch_plan_for(uvw, freq, npix_x=npix_x, npix_y=npix_y, pixsize_x=pixsize_x, pixsize_y=pixsize_y,
                        center_x=center_x, center_y=center_y, epsilon=epsilon, flip_u=flip_u, flip_v=flip_v, flip_w=flip_w,
                        do_wgridding=do_wgridding, divide_by_n=divide_by_n, sigma_min=sigma_min, sigma_max=sigma_max,
                        precision=prec, mask_list=mask, pooled=True)
    with gp as g:
        w = None if wgt is None else np.concatenate([np.asarray(a) for a in wgt], axis=0)
        if robustness is not None:
            g.bind_robust_weights(np.ones((g.nrow, g.nchan), g.rdt) if w is None else w,
                                  good_size(2 * npix_x) if nx_pad is None else nx_pad,
                                  good_size(2 * npix_y) if ny_pad is None else ny_pad, pixsize_x, pixsize_y, robustness,
                                  usign=1.0 if flip_u else -1.0, vsign=1.0 if flip_v else -1.0)
            w = None  # grid with the bound robust weights
        outs = []
        for k, vl in enumerate((vis,) + tuple(extra_vis)):
            if len(vl) != nsnap:
                raise ValueError("every visibility list needs one entry per snapshot")
            v = np.concatenate([np.asarray(a) for a in vl], axis=0)
            outs.append(g.grid(v, wgt=w, dirty=dirty if k == 0 else None))
        return outs[0] if not extra_vis else tuple(outs)


def dirty2vis_batch(*, uvw, freq, dirty, wgt=None, mask=None, pixsize_x, pixsize_y, center_x=0.0, center_y=0.0, epsilon,
                    flip_u=False, flip_v=False, flip_w=False, do_wgridding=True, divide_by_n=True, nthreads=1,
                    sigma_min=1.1, sigma_max=2.6, verbosity=0):
    """``dirty2vis`` for a cube of snapshot images ``(nsnap, nx, ny)``: returns the list of per-snapshot visibilities."""
    dirty = np.asarray(dirty)
    if dirty.ndim != 3 or dirty.shape[0] != len(uvw):
        raise ValueError("dirty must be (nsnap, nx, ny) with one image per snapshot")
    prec = _precision_of(dirty.dtype, "dirty")
    gp = batch_plan_for(uvw, freq, npix_x=dirty.shape[1], npix_y=dirty.shape[2], pixsize_x=pixsize_x, pixsize_y=pixsize_y,
                        center_x=center_x, center_y=center_y, epsilon=epsilon, flip_u=flip_u, flip_v=flip_v, flip_w=flip_w,
                        do_wgridding=do_wgridding, divide_by_n=divide_by_n, sigma_min=sigma_min, sigma_max=sigma_max,
                        precision=prec, mask_list=mask, pooled=True)
    with gp as g:
        w = None if wgt is None else np.concatenate([np.asarray(a) for a in wgt], axis=0)
        v = g.degrid(dirty, wgt=w)
        ro = g.row_offsets
        return [v[ro[s]:ro[s + 1]] for s in range(len(uvw))]
