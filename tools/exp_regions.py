"""GPU experiment: optical lengths from per-region cross sections (rt_optical_lengths_by_region) against the per-cell call with the
table expanded cell by cell (rt_optical_lengths), and the cost of the per-region volume sums (rt_region_volumes), on cfg3 at its
named size.

The map is a synthetic 3-region pin layout of the cfg3 unit square by cell centroid: fuel (r < 0.3 around the centre), cladding
(0.3 <= r < 0.35) and moderator.  For G = 1, 7 and 70 groups and both layouts, the two calls alternate, several runs each, with the
device buffer only (fetch=False, no tau download): "tau_ms" (k_tau alone, CUDA events) and the whole call (host clock around the
call, which ends in a stream synchronise: the table's host -> device copy from pageable memory, the kernel and the launch).  In the
first run of every case the two tau buffers are compared bit for bit on the device (torch).  rt_region_volumes (traced and exact
sums) is timed the same way after a segmentize_ with volumes.  The card's name and power limit are read in the same run.
  python tools/exp_regions.py --out profiles/regions_cfg3.txt"""
import argparse
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import raytracing_jl_b200 as rt  # noqa: E402
from bench import RTOL  # noqa: E402
from tools.exp_exact_volumes import card  # noqa: E402

NAMES = ("fuel", "cladding", "moderator")


def pin_regions(model):
    """1 fuel, 2 cladding, 3 moderator by the distance of each cell's centroid from the centre of the bounding box"""
    xy = model.node_coordinates
    c = xy[model.triangles0()].mean(axis=1)
    mid = 0.5 * (xy.min(axis=0) + xy.max(axis=0))
    r = np.hypot(c[:, 0] - mid[0], c[:, 1] - mid[1])
    return np.where(r < 0.3, 1, np.where(r < 0.35, 2, 3)).astype(np.int32)


def spread(v):
    return f"median {statistics.median(v):.3f} (min {min(v):.3f}, max {max(v):.3f})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="text file for the results")
    ap.add_argument("--reps", type=int, default=6, help="alternating runs of each call per case")
    args = ap.parse_args()
    import torch

    rt.build()
    lines = [f"card: {card()}"]
    model, n_azim, delta = rt.synth.workload("cfg3")
    tg = rt.TrackGenerator(rt.Mesh(model), n_azim, delta)
    rt.trace_(tg)
    rt.segmentize_(tg, rtol=RTOL, check=False)
    region = pin_regions(model)
    tg.set_regions(region)
    counts = np.bincount(region, minlength=4)[1:]
    lines.append(f"cfg3: {model.num_cells} cells, n_azim {n_azim}, delta {delta}, rtol {RTOL}, {tg.n_segments} segments; regions "
                 + ", ".join(f"{n} {k} cells" for n, k in zip(NAMES, counts)) + f"; {args.reps} alternating runs of each call per case")
    lines.append("  tau_ms: k_tau alone (CUDA events); call: host clock around the whole call, fetch=False (tau stays on the device)")
    rng = np.random.default_rng(7)
    for groups in (1, 7, 70):
        sig_r = rng.uniform(0.01, 10.0, size=(3, groups))
        sig_c = np.ascontiguousarray(sig_r[region - 1])
        for layout in (0, 1):
            t = {"cell": ([], []), "region": ([], [])}
            equal = None

            def run(kind):
                t0 = time.perf_counter()
                if kind == "cell":
                    _, dev = tg.optical_lengths(sig_c, layout=layout, fetch=False)
                else:
                    _, dev = tg.optical_lengths_by_region(sig_r, layout=layout, fetch=False)
                wall = (time.perf_counter() - t0) * 1e3
                t[kind][0].append(tg.info("tau_ms"))
                t[kind][1].append(wall)
                return dev

            run("cell"), run("region")  # warm-up of both (not recorded)
            for v in t.values():
                v[0].clear(), v[1].clear()
            for k in range(args.reps):
                dev = run("cell")
                if k == 0:
                    ref = torch.as_tensor(dev, device="cuda").clone()
                dev = run("region")
                if k == 0:
                    equal = bool(torch.equal(torch.as_tensor(dev, device="cuda"), ref))
                    del ref
                    torch.cuda.empty_cache()
            n_val = tg.n_segments * groups
            lines.append(f"  G {groups:2d} layout {layout} ({n_val:.3e} values, per-cell table {sig_c.nbytes / 1e6:.1f} MB, per-region "
                         f"{sig_r.nbytes} B): bit-equal {equal}")
            for kind, name in (("cell", "per-cell  "), ("region", "per-region")):
                lines.append(f"    {name} tau_ms {spread(t[kind][0])}; call ms {spread(t[kind][1])}")
    rv = []
    for _ in range(args.reps + 1):
        t0 = time.perf_counter()
        traced, exact = tg.region_volumes()
        rv.append((time.perf_counter() - t0) * 1e3)
    lines.append(f"  rt_region_volumes (traced and exact, after the first call that computes the areas) ms {spread(rv[1:])}; "
                 f"first call {rv[0]:.3f} ms")
    lines.append("    traced " + ", ".join(f"{v:.9f}" for v in traced) + "; exact " + ", ".join(f"{v:.9f}" for v in exact)
                 + "; traced / exact - 1: " + ", ".join(f"{a / b - 1:+.2e}" for a, b in zip(traced, exact)))
    tg.close()
    text = "\n".join(lines) + "\n"
    print(text, end="")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)


if __name__ == "__main__":
    main()
