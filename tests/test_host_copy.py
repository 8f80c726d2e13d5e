"""The threaded host copy (`par_memcpy`) and content hash (`pfbg_host_hash64`) of csrc/pfbgrid.cu split a buffer of n
bytes over nt threads in chunks of a multiple of 64 bytes.  Chunks of floor(n / nt) rounded up to 64 bytes cover only
nt * 64 k bytes when floor(n / nt) = 64 k and n % nt != 0: the last n % nt bytes were then neither hashed (an edit of the
last flags of a mask, or of the last samples of an odd-length fp32 weight array, left the operator cache serving the
stale binding) nor staged (the last mask bytes reached the device from whatever the pinned buffer held before).

The thread count is read once per process (PFBG_COPY_THREADS), so every case runs in a child process of its own."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THREADS = [2, 3, 5, 6, 7, 8]


def tail_size(nt, lo, r, unit=1, stride=1):
    """Smallest n >= lo, a multiple of `unit` and n / unit a multiple of `stride` plus one, with floor(n / nt) a
    multiple of 64 and n % nt == r: the sizes the old chunking dropped r bytes of."""
    n = (lo // (nt * 64)) * nt * 64 + r
    while n < lo or n % unit or (n // unit) % stride != 1 % stride:
        n += nt * 64
    assert n % nt == r and (n // nt) % 64 == 0
    return n


def _run_child(tmp_path, name, code, nt):
    script = tmp_path / f"{name}.py"
    script.write_text(f"import sys\nsys.path.insert(0, {ROOT!r}); sys.path.insert(0, {ROOT!r} + '/tests')\n" + code)
    env = dict(os.environ, PFBG_COPY_THREADS=str(nt))
    r = subprocess.run([sys.executable, str(script)], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    return r.stdout


HASH_CHILD = """
import numpy as np
from pfb_imaging_b200.wgridder import content_hash
from test_host_copy import tail_size
nt = {nt}
cases = []
for r in sorted({{1, nt - 1}}):
    cases.append(np.ones(tail_size(nt, 4 << 20, r), np.uint8))  # a mask: 1 byte per sample
# an fp32 array of an odd element count (its byte count is a multiple of 4, never of 8)
r4 = next((r for r in range(4, nt, 4)), None)
n = tail_size(nt, 4 << 20, r4, unit=4, stride=2) if r4 else (((4 << 20) // 4) | 1) * 4
cases.append(np.linspace(0.5, 1.5, n // 4, dtype=np.float32))
for a in cases:
    b = a.view(np.uint8)
    n = b.size
    assert n >= 4 << 20
    h0 = content_hash(a)
    assert content_hash(a.copy()) == h0
    # the last byte, and both sides of every chunk boundary of the floor- and the ceil-based split
    pos = {{n - 1}}
    for per in ((n // nt + 63) & ~63, ((n + nt - 1) // nt + 63) & ~63):
        for t in range(1, nt + 1):
            pos.update(q for q in (t * per - 1, t * per) if q < n)
    for q in sorted(pos):
        c = b.copy()
        c[q] ^= 0x5A
        assert content_hash(c.view(a.dtype)) != h0, ("edit not seen", nt, n, q)
    print("ok", nt, n, len(pos))
"""


@pytest.mark.parametrize("nt", THREADS)
def test_content_hash_sees_every_byte(tmp_path, nt):
    out = _run_child(tmp_path, "hash", HASH_CHILD.format(nt=nt), nt)
    assert out.count("ok") >= 2, out


UPLOAD_CHILD = """
import numpy as np
from pfb_imaging_b200 import wgridder as W
from test_host_copy import tail_size
nt, nchan = {nt}, 29
# nvis = nrow * nchan: one staging chunk (1 MiB <= nvis < 32 MiB), nvis % nt != 0 and floor(nvis / nt) % 64 == 0;
# 29 bytes of mask per row against 24 of uvw, so the mask's last bytes sit beyond what the uvw upload staged
nvis = tail_size(nt, 1 << 20, nt - 1, unit=nchan)
nrow = nvis // nchan
assert (1 << 20) <= nvis < (32 << 20)
rng = np.random.default_rng(nt)
freq = np.linspace(1.0e9, 1.2e9, nchan)
nx = ny = 64
cell = 0.25 / nx
umax = 0.5 / cell * 299792458.0 / freq.max()
uvw = rng.uniform(-1, 1, (nrow, 3)) * umax * 0.9
uvw[:, 2] *= 0.1
img = np.zeros((nx, ny), np.float32)
img[nx // 2, ny // 2] = 1.0
img[5, 40] = 0.5
mask = np.ones((nrow, nchan), np.uint8)
gp = W.plan_for(uvw, freq, npix_x=nx, npix_y=ny, pixsize_x=cell, pixsize_y=cell, epsilon=1e-4, precision="single",
                mask=mask)
assert gp.info()["nactive"] == nvis, ("first binding", gp.info()["nactive"], nvis)
assert gp.degrid(img)[-1, -1] != 0
mask[-1, -1] = 0  # flag the last sample only and bind again
gp.bind(uvw, freq, mask)
assert gp.info()["nactive"] == int(np.count_nonzero(mask)), ("second binding", gp.info()["nactive"], nvis - 1)
v = gp.degrid(img)
assert v[-1, -1] == 0 and v[-1, -2] != 0, (v[-1, -1], v[-1, -2])
gp.close()
print("ok", nt, nvis)
"""


@pytest.mark.gpu
@pytest.mark.parametrize("nt", THREADS)
def test_mask_upload_stages_every_byte(gpu, tmp_path, nt):
    out = _run_child(tmp_path, "upload", UPLOAD_CHILD.format(nt=nt), nt)
    assert "ok" in out, out
