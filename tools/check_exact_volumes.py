"""Multi-GPU check of RT_SEG_EXACT_VOLUMES (run under torchrun, one rank per GPU): the rank-order chain of rt_volumes gives every rank
the volumes of one GPU bit for bit, and its argument errors reach every rank without leaving one waiting.
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29534 tools/check_exact_volumes.py"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import raytracing_jl_b200 as rt  # noqa: E402
from raytracing_jl_b200 import _lib as L  # noqa: E402
from raytracing_jl_b200.distributed import init_comm  # noqa: E402
from oracle.oracle import OracleMesh, OracleTrackGenerator  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
model = rt.synth.jittered_triangle_mesh(120, 90, 2.0, 1.5, 0.25, 4321, x0=-0.5, y0=3.0)
mesh = rt.Mesh(model)
bcs = rt.BoundaryConditions(top=rt.Reflective, bottom=rt.Vacuum, right=rt.Periodic, left=rt.Periodic)
otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), 16, 0.004, bcs=(1, 0, 2, 2)).trace().segmentize(rtol=1e-6, check=False, fetch=False, nthreads=8)
oracle = otg.volumes()
one = rt.TrackGenerator(mesh, 16, 0.004, bcs=bcs, device=local)  # the whole track set on one GPU
rt.trace_(one)
rt.segmentize_(one, rtol=1e-6, check=False, exact_volumes=True)
single = one.volumes.copy()
assert single.tobytes() == oracle.tobytes(), "one GPU: exact volumes differ from the oracle's"


def sharded(shard):
    tg = rt.TrackGenerator(mesh, 16, 0.004, bcs=bcs, device=local, shard=shard)
    init_comm(tg)
    rt.trace_(tg)
    return tg


def code_of(call):
    try:
        call()
        return 0
    except rt.RTError as e:
        return e.code


def agree(x):
    t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    return lo.item() == hi.item()


# 1. shards in rank order: the chain gives the single-GPU bits on every rank, call after call, also with the chain left in flight
tg = sharded((rank, world))
for rep in range(3):
    rt.segmentize_(tg, rtol=1e-6, check=False, exact_volumes=True, fetch_volumes=rep != 1)
    if rep != 1:
        assert tg.volumes.tobytes() == single.tobytes(), (rank, rep)
# recv (ranks > 0) + send (ranks < world - 1) + broadcast, per call
calls = (rank > 0) + (rank < world - 1) + 1
assert tg.info("collectives") == 3 * calls, (rank, tg.info("collectives"))

# 2. a batched shard: RT_ERR_ARG on every rank, before the chain; every rank then joins the chain as failed and nobody hangs
L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, max(1, tg.n_segments // 3)))
assert code_of(lambda: rt.segmentize_(tg, rtol=1e-6, check=False, exact_volumes=True)) == -2
L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, 0))
rt.segmentize_(tg, rtol=1e-6, check=False, exact_volumes=True)  # ... and the next call is clean again
assert tg.volumes.tobytes() == single.tobytes()

# 3. a rank whose rt_segmentize fails: its own error there, RT_ERR_PEER on its peers (k > RT_MAX_K on the last rank only)
got = code_of(lambda: rt.segmentize_(tg, rtol=1e-6, check=False, exact_volumes=True, k=(33 if rank == world - 1 else 5)))
assert got == (-2 if rank == world - 1 else -11), (rank, got)
tg.close()

# 4. shards in reverse rank order: RT_ERR_ARG on every rank, nobody hangs
rev = sharded((world - 1 - rank, world))
got = code_of(lambda: rt.segmentize_(rev, rtol=1e-6, check=False, exact_volumes=True))
assert got == -2, (rank, got)
rev.close()
assert agree(1.0)
if rank == 0:
    print(f"exact volumes ok: {world} ranks, {otg.n_segments} segments, bit-equal to one GPU and to the oracle", flush=True)
dist.destroy_process_group()
