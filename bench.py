#!/usr/bin/env python
"""bench.py -- segments/s of segmentize! (BASELINE.json:metric) on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3|cfg2|cfg4|cfg5|pincell] [--impl ours|reference]

A "step" is one pass of the hot path over the workload's tracks with mesh + tracks already resident in
HBM: walk (count + record) -> scan -> evaluation (+ fused per-element volumes) -> volumes normalise (+ NCCL
all-reduce when N > 1).  The default workload is BASELINE.json configs[2] (unit square, ~1.0 M jittered
triangles, n_phi = 64, delta = 1e-3), the largest named configuration whose 2.2 GB of segments fit one GPU
without batching.  For N > 1 the tracks are sharded by uid range (mesh replicated) and the track spacing is
delta / N, so per-GPU work stays fixed ("scaling": "weak"); the same line then carries a `strong` block: the
named configs[3] (cfg4) -- and configs[4] (cfg5) at N = 8 -- sharded at their named sizes, with the
unsharded single-GPU time measured in the same run.  `e2e` is the same metric through the host API with HOST
buffers: mesh upload (H2D) + trace! + segmentize! + download of every Segment record (D2H).  `parity`
compares the GPU's segments of sampled uid blocks with the CPU oracle, bit for bit, in the same run.
`--impl reference` times the reference's CPU algorithm (the oracle port: Julia is not installable here) on
all host cores over a bounded uid sample of the same workload.  `--dump-outputs DIR` writes what the last timed step
computed as DIR/<name>.npy (see dump_outputs), so that two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree, which may be read-only

# segmentize!(tg; rtol): with the default rtol = sqrt(eps) the reference's own length check (src/track.jl:171-175) throws on 88
# corner tracks of cfg3 (it drops a 2e-8 chord); 1e-6 -- the remedy its error message suggests -- lets every track complete.
RTOL = 1e-6
SEG_KEYS = ("px", "py", "qx", "qy", "len", "element")


def load_workload(name, n_gpus, strong=False):
    import raytracing_jl_b200 as rt

    if name == "pincell":
        d = np.load(os.path.join(ROOT, "tests", "golden", "pincell.npz"))
        model, n_azim, delta = rt.UnstructuredDiscreteModel(d["node_coordinates"], d["cell_ptrs"], d["cell_data"]), 8, 2e-2
    else:
        model, n_azim, delta = rt.synth.workload(name)
    return model, n_azim, delta if strong else delta / n_gpus


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe).  The timed region of the default run
    is only tens of milliseconds, so the clocks are polled through NVML every 10 ms from a thread of this process (nvidia-smi
    -lms cannot sample faster than ~100 ms, and polling NVML faster than this measurably delays the kernel launches of the
    timed loop); nvidia-smi is the fallback when NVML is unavailable."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index, period=0.01):
        self.index, self.sm, self.reasons, self.mx, self.period = index, [], set(), None, period
        self._stop, self._thr, self.how = threading.Event(), None, None

    def _nvml_loop(self):
        import pynvml as nv

        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self._stop.is_set():
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            for name, bit in bits.items():
                if r & bit:
                    self.reasons.add(name)
            self._stop.wait(self.period)

    def _smi_loop(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.sm.append(float(out[0]))
                self.mx = float(out[1])
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                return

    def start(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            # NVML indexes physical devices: honour CUDA_VISIBLE_DEVICES when it lists ordinals
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            ids = [int(v) for v in vis.split(",") if v.strip().isdigit()]
            if ids and self.index < len(ids):
                self.index = ids[self.index]
            self.how, target = f"nvml {int(self.period * 1e3)} ms", self._nvml_loop
        except Exception:
            self.how, target = "nvidia-smi", self._smi_loop
        self._thr = threading.Thread(target=target, daemon=True)
        self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=6)
        sm = self.sm
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.mx, "reasons": sorted(self.reasons),
                "samples": len(sm), "how": self.how}


# ---- the CPU side: reference algorithm (oracle port) on sampled uid blocks, timed and -- optionally -- compared with the GPU ------
class Compare:
    """What the GPU produced for this rank's shard, on the host: offsets / status of the shard's tracks and the Segment columns
    of the resident batch (the whole shard for the benched workloads).  `check(otg, u0, u1)` compares one oracle block."""

    def __init__(self, tg, seg):
        self.uid_begin, self.uid_end = tg.uid_begin, tg.uid_end
        self.off, self.status, self.seg = tg.segment_offsets, tg.segment_status, seg
        self.res = tg.resident_batch()
        self.tracks = self.segments = self.mismatches = 0
        self.first = None

    def check(self, otg, u0, u1):
        lo_u, hi_u = max(u0, self.uid_begin, self.res[0]), min(u1, self.uid_end, self.res[1])
        if hi_u <= lo_u:
            return
        o = otg.fetch(lo_u, hi_u)
        a, b = lo_u - self.uid_begin, hi_u - self.uid_begin
        bad = 0
        if not np.array_equal(np.diff(self.off[a:b + 1]), o["counts"]):
            bad += int(np.count_nonzero(np.diff(self.off[a:b + 1]) != o["counts"]))
        elif not np.array_equal(self.status[a:b], o["status"]):
            bad += int(np.count_nonzero(self.status[a:b] != o["status"]))
        else:
            s0, s1 = int(self.off[a] - self.res[2]), int(self.off[b] - self.res[2])
            for k in SEG_KEYS:  # bit-exact: element ids and order, p / q / len
                g = self.seg[k][s0:s1]
                if not np.array_equal(g, o[k]):
                    bad += int(np.count_nonzero(g != o[k]))
        if bad and self.first is None:
            self.first = f"uids [{lo_u}, {hi_u})"
        self.mismatches += bad
        self.tracks += hi_u - lo_u
        self.segments += int(o["counts"].sum())

    def result(self):
        return {"checked_tracks": int(self.tracks), "checked_segments": int(self.segments), "mismatches": int(self.mismatches),
                "ok": bool(self.mismatches == 0 and self.segments > 0), "first_mismatch": self.first,
                "what": "GPU vs CPU oracle on sampled uid blocks: per-track counts and status, element ids and order, p/q/len bit for bit"}


DUMP_CAP = 1 << 19  # elements per stored array: 13 arrays at most, 52 MiB in all


def dump_outputs(tg, out_dir, suffix=""):
    """What the last segmentize! handed its caller, as float64 .npy files in out_dir: the Segment columns of the resident batch
    (px, py, qx, qy, len, element), segment_offsets, segment_status and the normalised volumes.  Every group is stored at the
    positions <group>_index.npy names (segment positions count from the shard's first segment): all of them, or a sample of
    DUMP_CAP positions seeded by nothing but the group's length when it is longer.  The volumes are summed with atomics: their
    last bits differ from run to run, everything else is reproduced bit for bit."""
    from raytracing_jl_b200 import _lib

    # the step left the normalised volumes on the device (fetch_volumes=False): copy them, nothing is recomputed
    _lib.check(tg._ctx, _lib.lib().rt_volumes(tg._ctx, _lib.ptr(tg.volumes)))
    seg = tg.fetch_segments()
    groups = [("segment", {k: seg[k] for k in SEG_KEYS}, tg.resident_batch()[2]),
              ("segment_offsets", {"segment_offsets": tg.segment_offsets}, 0),
              ("segment_status", {"segment_status": tg.segment_status}, 0), ("volumes", {"volumes": tg.volumes}, 0)]
    os.makedirs(out_dir, exist_ok=True)
    for group, cols, base in groups:
        n = len(next(iter(cols.values())))
        idx = np.arange(n) if n <= DUMP_CAP else np.unique(np.random.default_rng(n).integers(0, n, DUMP_CAP))
        np.save(os.path.join(out_dir, f"{group}_index{suffix}.npy"), (idx + base).astype(np.float64))
        for k, a in cols.items():
            np.save(os.path.join(out_dir, f"{k}{suffix}.npy"), np.asarray(a)[idx].astype(np.float64))


def estimate_segments(model, mesh, n_azim, delta):
    return (mesh.width * mesh.height) * (n_azim / 2) / delta / (0.45 * (2 * mesh.width * mesh.height / model.num_cells) ** 0.5)


def cpu_sample(model, n_azim, delta, budget_segments=3.0e7, blocks=16, threads=None, compare=None, uid_range=None, otg=None):
    """Reference CPU algorithm (oracle port) over `blocks` uid ranges spread evenly over [uid_range) of the workload.
    Only orc_segmentize is timed; fetching and comparing the blocks (compare) is not."""
    import raytracing_jl_b200 as rt
    from oracle.oracle import OracleMesh, OracleTrackGenerator

    threads = threads or os.cpu_count() or 1
    mesh = rt.Mesh(model)
    if otg is None:
        otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), n_azim, delta, bcs=(1, 1, 1, 1)).trace()
    lo, hi = uid_range or (1, otg.n_total_tracks + 1)
    n = hi - lo
    frac = min(1.0, budget_segments / max(estimate_segments(model, mesh, n_azim, delta) * n / otg.n_total_tracks, 1.0))
    blocks = max(1, min(blocks, n))
    per = max(1, int(n * frac / blocks))
    segs, secs = 0, 0.0
    for b in range(blocks):
        u0 = lo + int(b * (n - per) / max(blocks - 1, 1)) if frac < 1.0 else lo + b * (n // blocks)
        u1 = u0 + per if frac < 1.0 else (hi if b == blocks - 1 else lo + (b + 1) * (n // blocks))
        t0 = time.perf_counter()
        otg.segmentize(rtol=RTOL, uid_begin=u0, uid_end=u1, nthreads=threads, fetch=False, check=False)
        secs += time.perf_counter() - t0
        segs += otg.n_segments
        if compare is not None:
            compare.check(otg, u0, u1)
        otg.free_segments()
    sample = f"{blocks} uid blocks x {per} tracks = {100 * min(1.0, blocks * per / otg.n_total_tracks):.1f}% of {otg.n_total_tracks} tracks"
    return segs, secs, threads, sample, otg


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model, n_azim, delta = load_workload(args.workload, args.gpus, args.strong)
    threads = os.cpu_count() or 1
    # every step is a bounded sample of the workload, in FEW LARGE blocks so that every host thread has many tracks to walk
    # (schedule(dynamic, 1) over >= 64 tracks per thread); 1e7 - 3e7 segments per step keep the whole run within a minute
    budget = min(3.0e7, max(1.0e7, 2.5e8 / max(1, args.steps + args.warmup)))
    tot_s, tot_t, sample, otg = 0, 0.0, "", None
    for it in range(args.warmup + args.steps):
        s, t, threads, sample, otg = cpu_sample(model, n_azim, delta, budget_segments=budget, blocks=4, threads=threads, otg=otg)
        if it >= args.warmup:
            tot_s += s
            tot_t += t
    v = tot_s / tot_t
    # the reference's own execution model is ONE thread (src/trackgenerator.jl:362): a smaller sample, reported next to it
    s1, t1, _, sample1, otg = cpu_sample(model, n_azim, delta, budget_segments=3.0e6, blocks=4, threads=1, otg=otg)
    out = {"impl": "reference", "metric": "segments/sec for segmentize!", "value": v, "unit": "segments/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True,
           "scaling": "strong" if args.strong else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": workload_config(args, model, n_azim, delta),
           "cpu_baseline": {"value": v, "unit": "segments/s", "cores": threads, "kind": "port",
                            "sample": sample + " per step; OpenMP over tracks, schedule(dynamic, 1) (the reference itself is serial)"},
           "cpu_baseline_1thread": {"value": s1 / t1, "unit": "segments/s", "cores": 1, "kind": "port", "sample": sample1,
                                    "note": "the reference's own execution model: one serial loop over tracks_by_uid"},
           "e2e": {"value": v, "unit": "segments/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def workload_config(args, model, n_azim, delta):
    names = {"cfg3": "BASELINE.json configs[2]: synthetic unit-square jittered triangular mesh, seed 1234",
             "cfg2": "BASELINE.json configs[1]: synthetic 4x4 BWR pin lattice", "pincell": "BASELINE.json configs[0]: demo/pincell",
             "cfg4": "BASELINE.json configs[3]: synthetic 17x17 pin lattice", "cfg5": "BASELINE.json configs[4]: synthetic 51x51 pin lattice"}
    return {"workload": names.get(args.workload, args.workload), "n_cells": int(model.num_cells), "n_nodes": int(model.num_nodes),
            "n_azim": n_azim, "delta": delta, "rtol": RTOL, "bcs": "reflective", "sharding": f"uid ranges over {args.gpus} GPU(s), mesh replicated",
            "l2": "inputs larger than L2: cell+edge records 160 B/cell and >2 GB of segment output stream through the 126 MB L2 every step"}


def strong_block(name, rank, world, local, dist, torch, steps=3):
    """The named workload `name` at its named size: first unsharded on every GPU (N independent replicas = the 1-GPU time, max
    over ranks), then sharded by uid range over the N GPUs with the volume all-reduce.  Device time between two events on the
    library's stream, max over ranks."""
    import raytracing_jl_b200 as rt
    from raytracing_jl_b200.distributed import init_comm

    model, n_azim, delta = rt.synth.workload(name)
    mesh = rt.Mesh(model)
    bcs = rt.BoundaryConditions(top=rt.Reflective, bottom=rt.Reflective, right=rt.Reflective, left=rt.Reflective)
    area = rt.synth.mesh_area(model)

    retimed = []

    def timed(tg, k):
        rt.segmentize_(tg, rtol=RTOL, check=False, fetch_volumes=False)  # warm-up (allocations, first-touch)
        for attempt in range(2):
            dist.barrier()
            torch.cuda.synchronize()
            tg.timer_start()
            ph, wall = [], []
            for _ in range(k):
                t0 = time.perf_counter()
                rt.segmentize_(tg, rtol=RTOL, check=False, fetch_volumes=False)
                wall.append(round((time.perf_counter() - t0) * 1e3, 2))
                ph.append(tg.phase_ms())
            ms = tg.timer_stop() / k
            print(f"[rank {rank}] {name} {'sharded' if tg.uid_end - tg.uid_begin < tg.n_total_tracks else 'unsharded'}: host wall per call (ms) {wall}",
                  file=sys.stderr)
            # k is small (the calls take 0.02 .. 1 s): one call disturbed on the host side (observed once: +60 ms in one of three
            # calls on a fresh box) would decide the figure, so a region whose slowest call is far off its fastest is measured again, once
            off = torch.tensor([1.0 if max(wall) > 1.15 * min(wall) + 1.0 else 0.0], dtype=torch.float64, device="cuda")
            dist.all_reduce(off, op=dist.ReduceOp.MAX)
            if attempt == 0 and off.item() > 0:
                retimed.append(name)
                continue
            break
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        mine = torch.tensor([float(np.mean([p[k] for p in ph])) for k in ("count", "fill", "volumes")] + [ms, tg.info("count_batches")],
                            dtype=torch.float64, device="cuda")
        ws = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(ws, mine)
        return float(t.item()), [[round(float(v), 3) for v in w.tolist()] for w in ws]

    out = {"workload": name, "n_cells": int(model.num_cells), "n_azim": n_azim, "delta": delta, "steps": steps}
    one = None
    if name != "cfg5":  # (cfg5 unsharded takes ~9 s per step on one GPU; its 1-GPU time is not part of the default run)
        tg1 = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs, device=local)
        rt.trace_(tg1)
        one, _ = timed(tg1, max(1, steps - 1))
        out["segments"] = int(tg1.n_segments)
        out["ms_per_step_1gpu"] = one
        tg1.close()
        del tg1
    tg = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs, device=local, shard=(rank, world))
    init_comm(tg)
    rt.trace_(tg)
    ms, walks = timed(tg, steps)
    rt.segmentize_(tg, rtol=RTOL, check=False)  # (fetches the all-reduced volumes)
    tg.segment_offsets  # (also fetches tg.segment_status)
    n = torch.tensor([float(tg.n_segments), float(np.count_nonzero(tg.segment_status))], dtype=torch.float64, device="cuda")
    dist.all_reduce(n)
    nseg = int(n[0].item())
    out.update({"value": nseg / (ms * 1e-3), "unit": "segments/s", "ms_per_step": ms, "segments_sharded": nseg, "bad_tracks": int(n[1].item()),
                "per_rank_ms[walk, evaluation, volumes, step, walk_batches]": walks,
                "walk_spread": (max(w[0] for w in walks) - min(w[0] for w in walks)) / max(float(np.mean([w[0] for w in walks])), 1e-9),
                "volumes_sum_over_area": float(tg.volumes.sum() / area)})
    out["retimed"] = bool(retimed)
    if one is not None:
        out["efficiency_vs_n1"] = one / (world * ms)
        out["segments_match_unsharded"] = bool(nseg == out["segments"])
    tg.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="cfg3")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-strong-block", action="store_true", help="N > 1: skip the cfg4 (and, at N = 8, cfg5) strong-scaling block")
    ap.add_argument("--clock-period-ms", type=float, default=20.0)
    ap.add_argument("--strong", action="store_true", help="N > 1: shard the named workload itself (fixed total work) instead of delta / N")
    ap.add_argument("--pipeline", type=int, default=None, help="rt_set_option('pipeline'): 0 hybrid, 1 sequential, 3 single-walk")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float64; one set per rank when N > 1)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    # stdout carries exactly ONE JSON line: anything a library prints there meanwhile (NCCL's version banner, ...) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    import raytracing_jl_b200 as rt
    from raytracing_jl_b200.distributed import init_comm

    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        from raytracing_jl_b200.distributed import bind_to_gpu_numa

        bind_to_gpu_numa(local)  # pinned result buffers next to this rank's GPU: N downloads do not share one socket's memory
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    model, n_azim, delta = load_workload(args.workload, world, args.strong)
    mesh = rt.Mesh(model)
    bcs = rt.BoundaryConditions(top=rt.Reflective, bottom=rt.Reflective, right=rt.Reflective, left=rt.Reflective)
    tg = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs, device=local, shard=(rank, world))
    if world > 1:
        init_comm(tg)
    if args.pipeline is not None:
        tg.set_option("pipeline", args.pipeline)
    rt.trace_(tg)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        rt.segmentize_(tg, rtol=RTOL, check=False, fetch_volumes=False)

    for _ in range(args.warmup):
        step()
    retimed = False
    for attempt in range(2):
        sampler = ClockSampler(local, period=args.clock_period_ms * 1e-3)
        sampler.start()
        barrier()
        tg.timer_start()
        phases = []
        for it in range(args.steps):
            step()
            if it % 8 == 7 or it == args.steps - 1:  # (reading the phase stopwatches costs host time inside the timed region: sampled)
                phases.append(tg.phase_ms())
        ms = tg.timer_stop()
        barrier()
        clocks = sampler.stop()
        # The timed region is device time between two events on the library's stream, host gaps included.  A region that took
        # more than twice its own kernel phases was disturbed on the host side (another process, a driver hiccup on a fresh box):
        # it is re-measured once, and the JSON line says so.
        kern = args.steps * float(np.mean([sum(p[k] for k in ("count", "scan", "fill", "volumes")) for p in phases]))
        if attempt == 0 and world == 1 and ms > 2.0 * kern + 1.0:
            retimed = True
            continue
        break
    nseg_local = tg.n_segments
    st = tg.stats()
    tg.segment_offsets  # (also fetches tg.segment_status)
    if args.dump_outputs:
        dump_outputs(tg, args.dump_outputs, f"_rank{rank}" if world > 1 else "")
    if world > 1:
        print(f"[rank {rank}] ms/step {ms / args.steps:.3f} segments {nseg_local} phases "
              f"{ {k: round(float(np.mean([p[k] for p in phases])), 3) for k in phases[0]} }", file=sys.stderr)
    t_ms = torch.tensor([ms], dtype=torch.float64, device="cuda")
    n_all = torch.tensor([float(nseg_local), float(tg.uid_end - tg.uid_begin), float(np.count_nonzero(tg.segment_status))],
                         dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(n_all, op=dist.ReduceOp.SUM)
    ms_max = float(t_ms.item())
    nseg, ntrk, nbad = float(n_all[0].item()), float(n_all[1].item()), int(n_all[2].item())
    value = nseg * args.steps / (ms_max * 1e-3)

    # ---- roofline: SURVEY 8(d) algorithmic bytes per launch; `frac` = the dominant kernel (the evaluation), `frac_step` = the
    # whole step (count + scan + fill + volumes, host gaps included: the timed region itself)
    fill_ms = float(np.mean([p["fill"] for p in phases]))
    count_ms = float(np.mean([p["count"] for p in phases]))
    alg_bytes = 44.0 * nseg_local + 72.0 * (tg.uid_end - tg.uid_begin) + 40.0 * model.num_cells
    peak, peak_src = peaks()
    achieved = alg_bytes / (fill_ms * 1e-3) / 1e9
    achieved_step = alg_bytes / (ms / args.steps * 1e-3) / 1e9
    kern = {3: "k_eval3 (one lane per segment: records -> Segment columns)", 0: "k_walk<true> (fill pass)",
            1: "k_walk<true> (fill pass)"}[3 if args.pipeline is None else args.pipeline]
    roofline = {"bound": "hbm", "kernel": kern, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                "launch_ms": fill_ms, "count_pass_ms": count_ms, "achieved_step": achieved_step, "frac_step": achieved_step / peak,
                "note": "frac: launch_ms = the fill phase (dominant kernel + k_track_status); frac_step: the same algorithmic bytes over the "
                        "whole step (SURVEY 8d: count + scan + fill + volumes).  The count walk (k_march) is a latency-bound pointer chase "
                        "with ~4 algorithmic bytes per segment, see DESIGN.md and profiles/"}
    tr = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tr):
        try:
            roofline["traffic"] = json.load(open(tr)).get(args.workload)
        except Exception:
            pass

    # ---- e2e through the public API with host buffers
    e2e, seg = None, None
    if not args.no_e2e:
        def e2e_step():
            tg.upload_mesh()  # H2D of the flattened model + device preparation
            rt.trace_(tg)
            rt.segmentize_(tg, rtol=RTOL, check=False)  # includes the D2H of volumes
            tg.segment_offsets
            # D2H of every Segment record into pinned host buffers -- over the thin wire: q, len, element (28 B per segment) plus the
            # list of positions where p is not the preceding q; p is rebuilt on the host when it is first used (the parity block
            # below does so and compares it with the oracle)
            return tg.fetch_segments(pinned=True, compact=True)

        tg.pin_mesh()  # inputs of the step live in pinned host memory
        for _ in range(2):  # the first call allocates the pinned host buffers of the results
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        n_e2e = 3
        for _ in range(n_e2e):
            seg = e2e_step()
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        h2d = tg.mesh_h2d_bytes() + 7 * 8 * n_azim // 2
        d2h = sum(seg[k].nbytes for k in ("qx", "qy", "len", "element")) + 24 * tg.n_exceptions + tg.segment_offsets.nbytes + \
            tg.segment_status.nbytes + tg.volumes.nbytes
        # the same step with `len` left on the device too (20 B per segment; rebuilt on the host as norm(p - q), same IEEE operations)
        def e2e_step20():
            tg.upload_mesh()
            rt.trace_(tg)
            rt.segmentize_(tg, rtol=RTOL, check=False)
            tg.segment_offsets
            return tg.fetch_segments(pinned=True, compact="q")

        e2e_step20()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            seg = e2e_step20()
        torch.cuda.synchronize()
        dt20 = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(dt20, op=dist.ReduceOp.MAX)
        wire20 = {"value": nseg * n_e2e / float(dt20.item()), "ms_per_step": 1e3 * float(dt20.item()) / n_e2e,
                  "d2h_bytes_per_step": int(d2h - 8 * nseg_local), "what": "as e2e, with q + element only on the wire (len = norm(p - q) rebuilt on the host)"}
        e2e = {"value": nseg * n_e2e / float(dt.item()), "unit": "segments/s", "h2d_bytes_per_step": int(h2d), "wire20": wire20,
               "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * float(dt.item()) / n_e2e,
               "wire_bytes_per_segment": 28, "p_exceptions": int(tg.n_exceptions),
               "what": "rt_mesh_upload + rt_trace + rt_segmentize + rt_volumes + rt_segment_offsets + rt_segments_download_compact "
                       "(q, len, element + exception list; p[i] = q[i-1] rebuilt lazily on the host, bit-identical to the full download)"}

    # ---- parity in the same run: the GPU's records of sampled uid blocks against the CPU oracle, bit for bit; at N = 1 the sample
    # is the one the cpu_baseline is timed on, at N > 1 every rank checks a few small blocks of its own shard
    if seg is None:
        rt.segmentize_(tg, rtol=RTOL, check=False)
        seg = tg.fetch_segments()
    cmp_ = Compare(tg, seg)
    cpu = cpu1 = None
    if world == 1 and not args.no_cpu_baseline:
        s, t, cores, sample, otg = cpu_sample(model, n_azim, delta, compare=cmp_)
        cpu = {"value": s / t, "unit": "segments/s", "cores": cores, "kind": "port", "sample": sample,
               "note": "oracle port of the reference algorithm, OpenMP over tracks (schedule(dynamic, 1)); the Julia reference itself is single-threaded"}
        s1, t1, _, sample1, otg = cpu_sample(model, n_azim, delta, budget_segments=3.0e6, blocks=4, threads=1, otg=otg)
        cpu1 = {"value": s1 / t1, "unit": "segments/s", "cores": 1, "kind": "port", "sample": sample1,
                "note": "the reference's own execution model: one serial loop over tracks_by_uid (src/trackgenerator.jl:362)"}
    else:
        cpu_sample(model, n_azim, delta, budget_segments=4.0e5, blocks=4, compare=cmp_, uid_range=(tg.uid_begin, tg.uid_end))
    parity = cmp_.result()
    area = rt.synth.mesh_area(model)
    rt.segmentize_(tg, rtol=RTOL, check=False)  # (fetches the -- all-reduced -- volumes)
    parity["volumes_sum_over_area"] = float(tg.volumes.sum() / area)
    vol_ok = abs(parity["volumes_sum_over_area"] - 1.0) <= 1e-8 or nbad > 0
    if world > 1:
        pt = torch.tensor([float(parity["checked_tracks"]), float(parity["checked_segments"]), float(parity["mismatches"])],
                          dtype=torch.float64, device="cuda")
        dist.all_reduce(pt)
        parity.update(checked_tracks=int(pt[0].item()), checked_segments=int(pt[1].item()), mismatches=int(pt[2].item()))
        # every rank holds the same all-reduced volumes, bit for bit
        v = torch.tensor(tg.volumes, device="cuda")
        lo, hi = v.clone(), v.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        parity["ranks_hold_identical_volumes"] = bool(torch.equal(lo, hi))
        # the shards' segments add up to the unsharded count (rank 0 counts the whole track set with the sequential kernels)
        parity["segments_match_unsharded"] = None
        if rank == 0:
            whole = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs, device=local)
            rt.trace_(whole)
            rt.segmentize_(whole, rtol=RTOL, check=False, flags=rt.RT_SEG_COUNT_ONLY | rt.RT_SEG_NO_VOLUMES)
            parity["segments_unsharded"] = int(whole.n_segments)
            parity["segments_match_unsharded"] = bool(int(whole.n_segments) == int(nseg))
            whole.close()
        parity["ok"] = bool(parity["mismatches"] == 0 and parity["checked_segments"] > 0 and parity["ranks_hold_identical_volumes"]
                            and vol_ok and parity["segments_match_unsharded"] is not False)
    else:
        parity["ok"] = bool(parity["ok"] and vol_ok)
    # kernels of one steady-state call (rt_segmentize's own count) + with a communicator the k_normalise rt_volumes launches behind the all-reduce
    launches = int(st["launches"] + (1 if world > 1 else 0)) * args.steps
    fallbacks = int(tg.info("verify_fallbacks"))
    bad_status = int(tg.bad_status)

    # ---- strong scaling at the named sizes (N > 1): cfg4 sharded vs unsharded in the same run, cfg5 at N = 8
    strong = None
    if world > 1 and not args.no_strong_block and not args.strong and args.workload == "cfg3":
        tg.close()
        strong = strong_block("cfg4", rank, world, local, dist, torch)
        if world >= 8:
            strong["cfg5"] = strong_block("cfg5", rank, world, local, dist, torch, steps=2)

    if rank == 0:
        out = {"metric": "segments/sec for segmentize!", "value": value, "unit": "segments/s", "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "strong" if args.strong else "weak",
               "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args, model, n_azim, delta),
               "segments_per_step": nseg, "tracks": ntrk, "roofline": roofline, "cpu_baseline": cpu, "cpu_baseline_1thread": cpu1,
               "e2e": e2e, "parity": parity, "strong": strong, "clocks": clocks, "gpu_launches": launches,
               "phase_ms": {k: float(np.mean([p[k] for p in phases])) for k in phases[0]},
               "walk_stats": {k: st[k] for k in ("fast_transitions", "literal_iterations", "nn_queries", "knn_queries")},
               "bad_tracks": nbad, "bad_tracks_status": bad_status, "retimed": retimed, "verify_fallbacks": fallbacks}
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(out), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
