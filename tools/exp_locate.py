"""GPU experiment: throughput of rt_find_elements (find_element for batches of points, k_find_elements) on the cfg3 mesh.

Two point sets -- the pixel centres of a 4096 x 4096 raster over the bounding box and 1e7 uniform random points -- each at k = 2
and k = 5: points/s of the kernel alone (CUDA events, rt_info "locate_ms") and of the whole call (host clock around
TrackGenerator.find_elements: validation, H2D of the coordinates from pageable memory, kernel, D2H of the ids; it ends in a stream
synchronise), and the points that entered the k-nearest-node branch.  The CPU oracle (the restatement of the reference's
find_element, KD-tree, one host thread) runs on a 1e6-point subset of each set, which also checks the device ids bit for bit.  The
card's name and power limit are read in the same run.  Writes exp_locate.json and exp_locate.txt under the output directory."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import raytracing_jl_b200 as rt  # noqa: E402
from oracle.oracle import OracleMesh  # noqa: E402
from tests.locate_oracle import find_elements as oracle_find_elements  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True)
    except OSError as e:
        return f"nvidia-smi failed: {e}"
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for exp_locate.json and exp_locate.txt")
    ap.add_argument("--raster", type=int, default=4096)
    ap.add_argument("--random", type=int, default=10_000_000)
    ap.add_argument("--oracle-points", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    gpu = card()
    say(f"card (name, power limit, max SM clock): {gpu}")
    model, _, _ = rt.synth.workload("cfg3")
    mesh = rt.Mesh(model)
    say(f"cfg3 mesh: {mesh.num_nodes} nodes, {mesh.num_cells} triangles")
    tg = rt.TrackGenerator(mesh, 4, 0.5)
    lo, hi = mesh.bb_min, mesh.bb_max
    n = a.raster
    xs = lo[0] + (np.arange(n) + 0.5) * ((hi[0] - lo[0]) / n)
    ys = lo[1] + (np.arange(n) + 0.5) * ((hi[1] - lo[1]) / n)
    gx, gy = np.meshgrid(xs, ys)
    sets = {
        f"raster {n}x{n}": np.stack([gx.reshape(-1), gy.reshape(-1)], 1),
        f"random {a.random:.0e}": lo + np.random.default_rng(1).uniform(size=(a.random, 2)) * (hi - lo),
    }
    del gx, gy
    om = OracleMesh.from_mesh(mesh)
    rows = []
    for name, pts in sets.items():
        sub = pts[np.random.default_rng(2).choice(pts.shape[0], min(a.oracle_points, pts.shape[0]), replace=False)]
        for k in (2, 5):
            tg.find_elements(pts, k)  # warm-up of this shape (buffers grown, module loaded)
            kern, whole, knn = [], [], []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                ids, _ = tg.find_elements(pts, k)
                whole.append((time.perf_counter() - t0) * 1e3)
                kern.append(tg.info("locate_ms"))
                knn.append(tg.info("locate_knn"))
            sub_ids, _ = tg.find_elements(sub, k)
            t0 = time.perf_counter()
            want, o_knn = oracle_find_elements(om, mesh, sub, k)
            o_ms = (time.perf_counter() - t0) * 1e3
            same = bool(np.array_equal(sub_ids, want))
            km, wm = statistics.median(kern), statistics.median(whole)
            r = dict(points=name, n=int(pts.shape[0]), k=k, kernel_ms_median=km, kernel_ms_min=min(kern), kernel_ms_max=max(kern),
                     kernel_points_per_s=pts.shape[0] / (km * 1e-3), call_ms_median=wm, call_ms_min=min(whole), call_ms_max=max(whole),
                     call_points_per_s=pts.shape[0] / (wm * 1e-3), locate_knn=knn[-1], not_found=int((ids < 0).sum()),
                     cpu_restatement_points=int(sub.shape[0]), cpu_restatement_ms=o_ms,
                     cpu_restatement_points_per_s=sub.shape[0] / (o_ms * 1e-3), cpu_restatement_knn=o_knn, ids_equal_oracle=same)
            rows.append(r)
            say(f"{name:>18} k={k}: kernel {km:8.3f} ms ({r['kernel_points_per_s']:.3e} points/s, min {min(kern):.3f} max {max(kern):.3f}), "
                f"whole call {wm:8.2f} ms ({r['call_points_per_s']:.3e} points/s), locate_knn {knn[-1]:.0f}, not found {r['not_found']}; "
                f"CPU restatement (oracle, 1 thread) on {sub.shape[0]:.0e} points: {o_ms:.0f} ms ({r['cpu_restatement_points_per_s']:.3e} "
                f"points/s, knn {o_knn}), device ids equal: {same}")
    with open(os.path.join(a.out, "exp_locate.json"), "w") as fh:
        json.dump({"card": gpu, "mesh": {"nodes": mesh.num_nodes, "cells": mesh.num_cells}, "reps": a.reps, "runs": rows}, fh, indent=1)
    with open(os.path.join(a.out, "exp_locate.txt"), "w") as fh:
        fh.write("\n".join(lines) + "\n")
    if not all(r["ids_equal_oracle"] for r in rows):
        sys.exit("device ids differ from the oracle")


if __name__ == "__main__":
    main()
