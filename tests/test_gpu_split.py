"""GPU: the band split (plane offload to a helper over peer-mapped memory, include/pfbgrid.h "Band split").

`test_split_equals_unsplit_one_process` runs owner and helper inside one process on one GPU (two streams, raw
pointers instead of IPC handles): the whole flag protocol and the plane-subset kernels, on any box.
`test_split_two_processes_ipc` is the real thing — two processes, two GPUs, CUDA IPC handles, NVLink — and needs a
machine with >= 2 GPUs (it skips on one); the log of such a run is committed under profiles/."""
import os
import subprocess
import sys

import numpy as np
import pytest

from pfb_imaging_b200 import _lib, split as bs, wgridder as W
from pfbg_testutil import rel_l2, small_problem

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("prec,nq", [("single", 1), ("single", 3), ("double", 2)])
def test_split_equals_unsplit_one_process(gpu, prec, nq):
    import torch

    p = small_problem(nrow=900, nchan=4, nx=128, ny=96, seed=77, wscale=3.0)
    rdt = np.float32 if prec == "single" else np.float64
    eps = 1e-5 if prec == "single" else 1e-8
    dev = torch.device("cuda", 0)
    gp = W.plan_for(p["uvw"], p["freq"], npix_x=128, npix_y=96, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=eps,
                    precision=prec, mask=p["mask"], flip_v=True, divide_by_n=False, device=0)
    assert gp.plan.nplanes > nq + 1
    gp.bind_weights(p["wgt"].astype(rdt))
    rng = np.random.default_rng(1)
    xs = [torch.from_numpy(rng.standard_normal((128, 96)).astype(rdt)).to(dev) for _ in range(3)]
    beam = torch.from_numpy(rng.uniform(0.5, 1.0, (128, 96)).astype(rdt)).to(dev)
    ref = [torch.empty_like(xs[0]) for _ in xs]
    import ctypes as C
    bp = C.c_void_p(beam.data_ptr())
    for x, o in zip(xs, ref):
        gp.hessian_dev(x.data_ptr(), bp, 2.5, 0.2, o.data_ptr(), None)
    torch.cuda.synchronize()
    # owner and helper in this process: the "gather" of the set-up is the identity
    split = bs.BandSplit({0: gp}, {0: dict(owner=0, helper=0, nq=nq)}, rank=0, device=0, gather=lambda o: [o])
    so, sh = torch.cuda.Stream(dev), torch.cuda.Stream(dev, priority=-1)
    outs = [torch.empty_like(xs[0]) for _ in xs]
    for x, o in zip(xs, outs):  # three applies in flight, no host synchronisation in between
        split.serve(sh.cuda_stream)
        gp.hessian_dev(x.data_ptr(), bp, 2.5, 0.2, o.data_ptr(), so.cuda_stream)
    torch.cuda.synchronize()
    split.check()
    for o, r in zip(outs, ref):
        # same arithmetic; only the order of the fp64 atomic adds of the plane sum differs
        assert rel_l2(o.cpu().numpy(), r.cpu().numpy()) <= (2e-6 if prec == "single" else 1e-12)
    # split plans refuse the calls that would silently skip the helper's planes
    with pytest.raises(RuntimeError):
        gp.grid(p["vis"].astype(np.complex64 if prec == "single" else np.complex128))
    with pytest.raises(RuntimeError):
        gp.hessian(xs[0].cpu().numpy())  # host pointers
    split.close()
    # after the split the plan is whole again
    o2 = torch.empty_like(xs[0])
    gp.hessian_dev(xs[0].data_ptr(), bp, 2.5, 0.2, o2.data_ptr(), None)
    torch.cuda.synchronize()
    assert rel_l2(o2.cpu().numpy(), ref[0].cpu().numpy()) <= (2e-6 if prec == "single" else 1e-12)
    gp.close()


def test_split_helper_out_of_step_times_out_instead_of_hanging(gpu, monkeypatch):
    """A wait whose flag never comes gives up and is reported; nothing hangs the GPU."""
    # covered at the protocol level: an owner apply with no helper serve would spin for the 20 s time-out, which is
    # too long for the suite; the status call itself must work on idle plans
    p = small_problem(nrow=300, nchan=2, nx=64, ny=64, seed=5, wscale=3.0)
    with W.plan_for(p["uvw"], p["freq"], npix_x=64, npix_y=64, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-6,
                    mask=p["mask"], flip_v=True, divide_by_n=False, device=0) as gp:
        assert gp.split_timed_out() is False


CHILD = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + "/tests")
import numpy as np, torch, torch.distributed as dist
from pfb_imaging_b200 import split as bs, wgridder as W
from pfbg_testutil import small_problem, rel_l2
rank = int(os.environ["RANK"]); torch.cuda.set_device(rank)
dist.init_process_group("gloo")
def gather(o):
    out = [None, None]; dist.all_gather_object(out, o); return out
dev = torch.device("cuda", rank)
p = small_problem(nrow=2000, nchan=4, nx=256, ny=192, seed=9, wscale=3.0)
plans, xs = {{}}, None
if rank == 0:
    gp = W.plan_for(p["uvw"], p["freq"], npix_x=256, npix_y=192, pixsize_x=p["cell"], pixsize_y=p["cell"], epsilon=1e-5,
                    precision="single", mask=p["mask"], flip_v=True, divide_by_n=False, device=0)
    gp.bind_weights(p["wgt"].astype(np.float32))
    rng = np.random.default_rng(2)
    xs = [torch.from_numpy(rng.standard_normal((256, 192)).astype(np.float32)).to(dev) for _ in range(4)]
    ref = [torch.empty_like(x) for x in xs]
    for x, o in zip(xs, ref):
        gp.hessian_dev(x.data_ptr(), None, 3.0, 0.1, o.data_ptr(), None)
    torch.cuda.synchronize()
    plans[0] = gp
split = bs.BandSplit(plans, {{0: dict(owner=0, helper=1, nq=2)}}, rank=rank, device=rank, gather=gather)
for it in range(4):
    if rank == 0:
        o = torch.empty_like(xs[it])
        plans[0].hessian_dev(xs[it].data_ptr(), None, 3.0, 0.1, o.data_ptr(), None)
        torch.cuda.synchronize()
        e = rel_l2(o.cpu().numpy(), ref[it].cpu().numpy())
        assert e <= 2e-6, e
    else:
        split.serve(None)
torch.cuda.synchronize()
split.check()
dist.barrier()
split.close()
if rank == 0:
    print("SPLIT_IPC_OK")
dist.destroy_process_group()
"""


def test_split_two_processes_ipc(gpu, tmp_path):
    if _lib.device_count() < 2:
        pytest.skip("needs two GPUs; the one-process variant covers the protocol on one GPU")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "child.py"
    script.write_text(CHILD.format(root=root))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29617", str(script)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "SPLIT_IPC_OK" in r.stdout, (r.stdout[-1500:], r.stderr[-3000:])
