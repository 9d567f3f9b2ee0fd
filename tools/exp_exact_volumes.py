"""GPU experiment: what RT_SEG_EXACT_VOLUMES costs on the cfg3 workload (synth.workload("cfg3"), rtol = 1e-6 as in bench.py).

The step is bench.py's: one segmentize_ with the volumes left on the device (fetch_volumes=False), timed by the context's CUDA-event
stopwatch (rt_timer_start / rt_timer_stop, which end in a synchronise).  Default and exact steps alternate in the same process after a
warm-up of both; "exact_vol_ms" (contributions, sort and fold, CUDA events) is read after every exact step.  The same is repeated with
the segment capacity at one quarter of the segments (batched fill).  The exact volumes are checked bit for bit against the first exact
step and the default ones against them within 1e-12.  The card's name and power limit are read in the same run.
  python tools/exp_exact_volumes.py --out profiles/exact_volumes_cfg3.txt"""
import argparse
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import raytracing_jl_b200 as rt  # noqa: E402
from raytracing_jl_b200 import _lib as L  # noqa: E402

RTOL = 1e-6


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True)
    except OSError as e:
        return f"nvidia-smi failed: {e}"
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def measure(tg, reps, lines, label):
    def step(exact):
        tg.timer_start()
        rt.segmentize_(tg, rtol=RTOL, check=False, fetch_volumes=False, exact_volumes=exact)
        return tg.timer_stop()

    for exact in (False, True, False, True):  # warm-up of both kinds (allocations, sort scratch, plan)
        step(exact)
    L.check(tg._ctx, L.lib().rt_volumes(tg._ctx, tg.volumes.ctypes.data_as(L._vp)))
    ref = tg.volumes.copy()
    t = {False: [], True: []}
    ex = []
    for _ in range(reps):
        for exact in (False, True):
            t[exact].append(step(exact))
            if exact:
                ex.append(tg.info("exact_vol_ms"))
    L.check(tg._ctx, L.lib().rt_volumes(tg._ctx, tg.volumes.ctypes.data_as(L._vp)))
    assert tg.volumes.tobytes() == ref.tobytes(), "exact volumes changed between steps"
    rt.segmentize_(tg, rtol=RTOL, check=False)
    assert np.allclose(tg.volumes, ref, rtol=1e-12, atol=0.0)
    d, e = statistics.median(t[False]), statistics.median(t[True])
    lines.append(f"{label}: {tg.n_segments} segments, {reps} alternating repetitions of each step")
    lines.append(f"  default step  median {d:.3f} ms  (min {min(t[False]):.3f}, max {max(t[False]):.3f})")
    lines.append(f"  exact step    median {e:.3f} ms  (min {min(t[True]):.3f}, max {max(t[True]):.3f})")
    lines.append(f"  added         {e - d:.3f} ms per step ({e / d:.2f}x)")
    lines.append(f"  exact_vol_ms  median {statistics.median(ex):.3f} ms  (min {min(ex):.3f}, max {max(ex):.3f})")
    lines.append(f"  default volumes within {np.max(np.abs(tg.volumes - ref) / np.where(ref > 0, ref, 1.0)):.2e} relative of the exact ones")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="text file for the results")
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    rt.build()
    model, n_azim, delta = rt.synth.workload("cfg3")
    mesh = rt.Mesh(model)
    lines = [f"card: {card()}", f"cfg3: {mesh.num_cells} cells, n_azim {n_azim}, delta {delta}, rtol {RTOL}"]
    tg = rt.TrackGenerator(mesh, n_azim, delta)
    rt.trace_(tg)
    measure(tg, args.reps, lines, "resident")
    n = tg.n_segments
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, n // 4 + 1))
    measure(tg, args.reps, lines, f"batched (segment capacity {n // 4 + 1})")
    tg.close()
    text = "\n".join(lines) + "\n"
    print(text, end="")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)


if __name__ == "__main__":
    main()
