"""Generate tests/golden/sara.npz by EXECUTING the reference's own numba code (run in the build container;
/root/reference does not exist on the GPU box).

  python tests/golden/make_golden_sara.py

Reference functions executed (nothing is copied into this repo):
  pfb_imaging.operators.psi.Psi / PsiNocopyt            (operators/psi.py:549-664)
  pfb_imaging.prox.prox_21m.dual_update_numba_fast / prox_21m_numba   (prox/prox_21m.py:30-62, 104-135)
PyWavelets is absent from this image: a stub `pywt` serving pfb_imaging_b200.wavelet_filters is injected, so
the goldens pin the transform structure / packing / boundary handling, with our db1..db5 tables as filters.
"""
import importlib.util
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from pfb_imaging_b200 import wavelet_filters as wf  # noqa: E402

R = "/root/reference/src/pfb_imaging"
STRIDE = 17
os.environ.setdefault("NUMBA_CACHE_DIR", "/tmp/numba_cache")


def _stub(name, path=None):
    m = types.ModuleType(name)
    if path:
        m.__path__ = [path]
    sys.modules[name] = m
    return m


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


class _Wavelet:
    def __init__(self, name):
        self.filter_bank = wf.filter_bank(name)


pywt = _stub("pywt")
pywt.Wavelet = _Wavelet
pywt.dwt_max_level = lambda n, w: wf.dwt_max_level(int(n), 2 * int(w[-1]) if isinstance(w, str) else int(w))

_stub("pfb_imaging", R)
_stub("pfb_imaging.operators", R + "/operators")
_stub("pfb_imaging.prox", R + "/prox")
psi_mod = _load("pfb_imaging.operators.psi", R + "/operators/psi.py")
prox_mod = _load("pfb_imaging.prox.prox_21m", R + "/prox/prox_21m.py")


def main():
    rng = np.random.default_rng(420)
    out = {}
    cases = [  # (tag, nx, ny, nband, nlevel, bases, layouts)  sizes of tests/test_psi_operator.py:19-22 and odd ones
        ("a", 128, 64, 1, 2, ["self", "db1", "db2", "db3", "db4", "db5"], "tx"),
        ("b", 250, 78, 1, 2, ["self", "db1", "db2", "db3", "db4", "db5"], "x"),
        ("d", 122, 96, 2, 3, ["db2", "self", "db4"], "x"),
    ]
    for tag, nx, ny, nband, nlevel, bases, layouts in cases:
        x = rng.standard_normal((nband, nx, ny))
        for cls, nm in ((psi_mod.Psi, "t"), (psi_mod.PsiNocopyt, "x")):
            if nm not in layouts:
                continue
            psi = cls(nband, nx, ny, bases, nlevel, 1)
            shape = (nband, len(bases), psi.nymax, psi.nxmax) if nm == "t" else (nband, len(bases), psi.nxmax, psi.nymax)
            alpha = rng.standard_normal(shape)  # dot must overwrite whatever is there
            psi.dot(x, alpha)
            xr = rng.standard_normal((nband, nx, ny))
            psi.hdot(alpha, xr)
            # adjoint of coefficients that are NOT in the range of dot: a fixed function of alpha (not stored)
            a2 = 0.5 * alpha[..., ::-1, ::-1] + 0.25
            xr2 = np.zeros((nband, nx, ny))
            psi.hdot(np.ascontiguousarray(a2), xr2)
            out[f"{tag}_{nm}_alpha"] = alpha
            if nm == "x":  # (the tests use no reconstruction of the transposed layout)
                out[f"{tag}_{nm}_xrec"] = xr
            out[f"{tag}_{nm}_xr2"] = xr2
        out[f"{tag}_x"] = x
        out[f"{tag}_meta"] = np.array([nx, ny, nband, nlevel, psi.nxmax, psi.nymax])
        out[f"{tag}_bases"] = np.array(bases)
    # dual update / prox on a small coefficient cube
    nband, nbasis, ny_, nx_ = 3, 4, 33, 41
    vp = rng.standard_normal((nband, nbasis, ny_, nx_))
    v = rng.standard_normal((nband, nbasis, ny_, nx_))
    w = rng.uniform(0.2, 2.0, (nbasis, ny_, nx_))
    w[0, :3] = 0.0
    vp[:, 1, 5, :] = 0.0
    v[:, 1, 5, :] = 0.0
    for lam, sigma, nm in ((0.7, 1.3, "p"), (0.0, 0.5, "z")):
        vv = v.copy()
        prox_mod.dual_update_numba_fast(vp, vv, lam, sigma=sigma, weight=w)
        res = np.zeros_like(v)
        prox_mod.prox_21m_numba(v, res, lam, sigma=sigma, weight=w)
        out[f"du_{nm}_out"] = vv
        out[f"du_{nm}_prox"] = res
        out[f"du_{nm}_par"] = np.array([lam, sigma])
    out["du_vp"], out["du_v"], out["du_w"] = vp, v, w
    # inputs in full; of every output every STRIDE-th element of the flattened array (keeps the file under 1 MB)
    for k in list(out):
        if k.endswith(("_alpha", "_xrec", "_xr2", "_out", "_prox")):
            out[k] = np.ascontiguousarray(out[k].reshape(-1)[::STRIDE])
    out["stride"] = np.array(STRIDE)
    np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "sara.npz"), **out)
    print({k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
