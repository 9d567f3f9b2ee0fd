"""Multi-GPU check (run under torchrun, one rank per GPU): the NCCL all-reduce of the volumes -- issued on the library's collective
stream so that it overlaps with the next segmentize! -- gives every rank the volumes of the whole track set, call after call.
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29533 tools/check_nccl_volumes.py"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import raytracing_jl_b200 as rt  # noqa: E402
from raytracing_jl_b200.distributed import init_comm  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
model = rt.synth.jittered_triangle_mesh(120, 90, 2.0, 1.5, 0.25, 4321, x0=-0.5, y0=3.0)
mesh = rt.Mesh(model)
bcs = rt.BoundaryConditions(top=rt.Reflective, bottom=rt.Vacuum, right=rt.Periodic, left=rt.Periodic)
area = rt.synth.mesh_area(model)
# max_iter of the calls below: neighbouring calls differ, so that volumes from the buffer or the collective of the call before
# would not match the reference of their own call (None: the full walk)
MAX_ITERS = [None, 60, 25, 90, None]
# the whole track set on one GPU (no communicator): the yardsticks, one per max_iter
ref = rt.TrackGenerator(mesh, 16, 0.004, bcs=bcs, device=local)
rt.trace_(ref)
vrefs = {}
for mi in set(MAX_ITERS):
    rt.segmentize_(ref, rtol=1e-6, check=False, max_iter=mi or rt.MAX_ITER)
    vrefs[mi] = ref.volumes.copy()
    if mi is None:
        n_ref = ref.n_segments
vref = vrefs[None]
tg = rt.TrackGenerator(mesh, 16, 0.004, bcs=bcs, device=local, shard=(rank, world))
init_comm(tg)
rt.trace_(tg)
for rep, mi in enumerate(MAX_ITERS):
    if rep % 2 == 0:
        rt.segmentize_(tg, rtol=1e-6, check=False, max_iter=mi or rt.MAX_ITER)  # fetches the all-reduced volumes
    else:  # collective left in flight behind the next call
        rt.segmentize_(tg, rtol=1e-6, check=False, max_iter=mi or rt.MAX_ITER, fetch_volumes=False)
        continue
    v = tg.volumes.copy()
    if mi is None:
        assert abs(v.sum() - area) <= 1e-9 * area, (rep, v.sum(), area)
    assert np.allclose(v, vrefs[mi], rtol=1e-10, atol=0.0), (rep, mi, np.abs(v - vrefs[mi]).max())
    g = torch.tensor(v, device="cuda")
    lo, hi = g.clone(), g.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    assert torch.equal(lo, hi), "ranks hold different volumes"
n = torch.tensor([float(tg.n_segments)], device="cuda", dtype=torch.float64)
dist.all_reduce(n)
assert int(n.item()) == n_ref, (int(n.item()), n_ref)
# a rank whose rt_segmentize fails still joins the collective (zero contribution + failed-rank flag): nobody hangs, the failing
# rank raises its own error and its peers are told that the sums are incomplete (RT_ERR_PEER)
try:
    rt.segmentize_(tg, rtol=1e-6, check=False, k=(33 if rank == world - 1 else 5))  # k > RT_MAX_K: RT_ERR_ARG on the last rank only
    raised = None
except rt.RTError as e:
    raised = e.code
assert raised == (-2 if rank == world - 1 else -11), raised
rt.segmentize_(tg, rtol=1e-6, check=False)  # ... and the next call is clean again
assert np.allclose(tg.volumes, vref, rtol=1e-10, atol=0.0)
# one all-reduce per segmentize! on every rank, the failed one included
c = torch.tensor([tg.info("collectives")], device="cuda", dtype=torch.float64)
lo, hi = c.clone(), c.clone()
dist.all_reduce(lo, op=dist.ReduceOp.MIN)
dist.all_reduce(hi, op=dist.ReduceOp.MAX)
assert lo.item() == hi.item() == len(MAX_ITERS) + 2, (lo.item(), hi.item())
if rank == 0:
    print(f"nccl volumes ok: {world} ranks, {n_ref} segments, sum(vol)/area = {vref.sum() / area:.12f}", flush=True)
dist.destroy_process_group()
