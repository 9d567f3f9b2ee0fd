"""GPU experiment: the single-walk pipeline (3) against the hybrid one (0); chunk size / order sweeps."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import raytracing_jl_b200 as rt  # noqa: E402

name = sys.argv[1] if len(sys.argv) > 1 else "cfg3"
model, n_azim, delta = rt.synth.workload(name)
mesh = rt.Mesh(model)
bcs = rt.BoundaryConditions(top=rt.Reflective, bottom=rt.Reflective, right=rt.Reflective, left=rt.Reflective)
tg = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs)
rt.trace_(tg)
print("tracks", tg.n_total_tracks, "cells", model.num_cells, flush=True)


def checksum():
    s = tg.segments
    w = (np.arange(s["len"].shape[0], dtype=np.int64) % 1021 + 1)
    return tuple(int((s[k].view(np.int64 if s[k].dtype.itemsize == 8 else np.int32).astype(np.int64) & 0xFFFFFFFF).dot(w)) for k in
                 ("px", "py", "qx", "qy", "len", "element"))


def run(label, flags=0, reps=4, chk=False, **opts):
    tg.set_option("chunk_segments", opts.get("chunk_segments", 128))
    tg.set_option("order_grid", opts.get("order_grid", 32))
    tg.set_option("pipeline", opts.get("pipeline", 0))
    best = None
    for _ in range(reps):
        tg.timer_start()
        rt.segmentize_(tg, flags=flags, rtol=1e-6, check=False, fetch_volumes=False)
        ms = tg.timer_stop()
        p = tg.phase_ms()
        if best is None or ms < best[0]:
            best = (ms, p)
    print(f"{label:36s} total {best[0]:7.3f} ms  count {best[1]['count']:6.3f} scan {best[1]['scan']:6.3f} fill {best[1]['fill']:6.3f}"
          f"  nseg {tg.n_segments} seg/s {tg.n_segments / best[0] * 1e3:.3e} fb {tg.info('verify_fallbacks'):.0f} bad {tg.bad_status}", flush=True)
    return checksum() if chk else None


small = name in ("cfg3", "cfg2", "pincell")
c0 = run("hybrid (0)", pipeline=0, chk=small)
c3 = run("single-walk (3)", pipeline=3, chk=small)
print("chunk stats:", tg.chunk_stats(), flush=True)
if small:
    print("checksums equal:", c0 == c3, flush=True)
for cs in (64, 96, 192, 256):
    run(f"single-walk chunk={cs}", pipeline=3, chunk_segments=cs)
for og in (0, 16, 64):
    run(f"single-walk order_grid={og}", pipeline=3, order_grid=og)
run("single-walk no volumes", pipeline=3, flags=rt.RT_SEG_NO_VOLUMES)
