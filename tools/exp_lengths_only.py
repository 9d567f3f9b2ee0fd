"""GPU experiment: what RT_SEG_LENGTHS_ONLY (segmentize_(..., lengths_only=True)) saves on cfg3 and cfg4 at their named sizes.

cfg3 (rtol = 1e-6 as in bench.py): the step is bench.py's -- one segmentize_ with the volumes left on the device, timed by the
context's CUDA-event stopwatch (rt_timer_start / rt_timer_stop, which end in a synchronise) -- with default and lengths-only steps
alternating on ONE context after a warm-up of both.  The fill phase is rt_phase_ms[4] (k_eval3 + k_track_status) of every step; its
share of the HBM roofline uses bench.py's algorithmic bytes (44 S + 72 T + 40 N per launch; 12 S + 72 T + 40 N for lengths-only,
which writes 12 instead of 44 bytes per segment) over bench.py's own peak.  Afterwards len and element of the two modes are compared
bit for bit on the device (torch), over every segment.

cfg4: per mode on one context, the evaluation batches (on_batch calls), rt_info "segment_capacity" and "count_batches" (walk
batches), and the call time after two warm-up calls.  The card's name and power limit are read in the same run.
  python tools/exp_lengths_only.py --out profiles/lengths_only_cfg3.txt"""
import argparse
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import raytracing_jl_b200 as rt  # noqa: E402
from raytracing_jl_b200 import _lib as L  # noqa: E402
from raytracing_jl_b200.api import DeviceColumn  # noqa: E402
from bench import RTOL, peaks  # noqa: E402
from tools.exp_exact_volumes import card  # noqa: E402


def alg_bytes(tg, lengths_only):
    """bench.py's algorithmic bytes of one evaluation launch, with the segment columns lengths-only writes"""
    return (12.0 if lengths_only else 44.0) * tg.n_segments + 72.0 * (tg.uid_end - tg.uid_begin) + 40.0 * tg.mesh.num_cells


def device_columns(tg):
    import torch

    view = L.rt_batch()
    L.check(tg._ctx, L.lib().rt_segments_device(tg._ctx, view))
    n = int(view.n_segments)
    return (torch.as_tensor(DeviceColumn(view.d_len, n, "<f8"), device="cuda").clone(),
            torch.as_tensor(DeviceColumn(view.d_element, n, "<i4"), device="cuda").clone())


def cfg3(lines, reps):
    import torch

    model, n_azim, delta = rt.synth.workload("cfg3")
    mesh = rt.Mesh(model)
    bcs = rt.BoundaryConditions(top=rt.Reflective, bottom=rt.Reflective, right=rt.Reflective, left=rt.Reflective)
    tg = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs)
    rt.trace_(tg)

    def step(lo):
        tg.timer_start()
        rt.segmentize_(tg, rtol=RTOL, check=False, fetch_volumes=False, lengths_only=lo)
        ms = tg.timer_stop()
        return ms, tg.phase_ms()["fill"]

    for lo in (False, True, False, True, False, True):  # warm-up of both kinds
        step(lo)
    t = {False: [], True: []}
    fill = {False: [], True: []}
    for _ in range(reps):
        for lo in (False, True):
            ms, f = step(lo)
            t[lo].append(ms)
            fill[lo].append(f)
    peak, peak_src = peaks()
    lines.append(f"cfg3: {mesh.num_cells} cells, n_azim {n_azim}, delta {delta}, rtol {RTOL}, {tg.n_segments} segments, "
                 f"{tg.uid_end - tg.uid_begin} tracks; {reps} alternating repetitions of each step on one context")
    lines.append(f"  HBM peak {peak:.0f} GB/s ({peak_src})")
    for lo, name in ((False, "default     "), (True, "lengths-only")):
        s, f = statistics.median(t[lo]), statistics.median(fill[lo])
        b = alg_bytes(tg, lo)
        lines.append(f"  {name} step median {s:.3f} ms (min {min(t[lo]):.3f}, max {max(t[lo]):.3f}); fill phase median {f:.3f} ms "
                     f"(min {min(fill[lo]):.3f}, max {max(fill[lo]):.3f}); {b / 1e9:.3f} GB algorithmic -> "
                     f"{b / (f * 1e-3) / 1e9:.0f} GB/s = {b / (f * 1e-3) / 1e9 / peak:.2f} of the roofline")
    d, o = statistics.median(t[False]), statistics.median(t[True])
    fd, fo = statistics.median(fill[False]), statistics.median(fill[True])
    lines.append(f"  difference: step {o - d:+.3f} ms ({o / d:.3f}x), fill phase {fo - fd:+.3f} ms ({fo / fd:.3f}x)")
    rt.segmentize_(tg, rtol=RTOL, check=False, fetch_volumes=False)
    a = device_columns(tg)
    rt.segmentize_(tg, rtol=RTOL, check=False, fetch_volumes=False, lengths_only=True)
    b = device_columns(tg)
    same = a[0].numel() == b[0].numel() == tg.n_segments and torch.equal(a[0].view(torch.int64), b[0].view(torch.int64)) and \
        torch.equal(a[1], b[1])
    lines.append(f"  len / element of the two modes bit-equal on the device over all {a[0].numel()} segments: {same}")
    assert same
    tg.close()


def cfg4(lines, reps):
    model, n_azim, delta = rt.synth.workload("cfg4")
    mesh = rt.Mesh(model)
    bcs = rt.BoundaryConditions(top=rt.Reflective, bottom=rt.Reflective, right=rt.Reflective, left=rt.Reflective)
    tg = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs)
    rt.trace_(tg)
    lines.append(f"cfg4: {mesh.num_cells} cells, n_azim {n_azim}, delta {delta}, rtol {RTOL}, {tg.uid_end - tg.uid_begin} tracks; "
                 f"per mode 2 warm-up calls, then {reps} timed calls (with an on_batch that counts the batches)")
    offsets = {}
    for lo, name in ((False, "default     "), (True, "lengths-only")):
        times, batches = [], []
        for i in range(2 + reps):
            seen = []
            tg.timer_start()
            rt.segmentize_(tg, rtol=RTOL, check=False, fetch_volumes=False, lengths_only=lo, on_batch=lambda b: seen.append(b.n_segments))
            ms = tg.timer_stop()
            if i >= 2:
                times.append(ms)
                batches.append(len(seen))
        offsets[lo] = tg.segment_offsets.copy()
        lines.append(f"  {name} {tg.n_segments} segments: evaluation batches {batches[-1]} (largest {max(seen)}), segment_capacity "
                     f"{tg.info('segment_capacity'):.4g}, walk batches (count_batches) {tg.info('count_batches'):.0f}, call median "
                     f"{statistics.median(times):.1f} ms (min {min(times):.1f}, max {max(times):.1f}), fill phase {tg.phase_ms()['fill']:.1f} ms")
    same = np.array_equal(offsets[False], offsets[True])
    lines.append(f"  offsets of the two modes equal: {same}")
    assert same
    tg.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="text file for the results")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--reps4", type=int, default=3)
    args = ap.parse_args()
    rt.build()
    lines = [f"card: {card()}"]
    try:
        cfg3(lines, args.reps)
        cfg4(lines, args.reps4)
    finally:
        text = "\n".join(lines) + "\n"
        print(text, end="")
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
