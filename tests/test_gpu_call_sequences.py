"""Seeded call sequences on ONE context against the oracle.  A transport code keeps one context per GPU for a whole run: it re-traces,
swaps the mesh, changes the segment capacity and the options, switches flags and calls the accessors in between.  Every kernel
output is already compared with the oracle on a fresh context; this module tests the state a context keeps BETWEEN calls.

The world is small and fixed: two jittered 60 x 60 meshes with the same bounding box and counts (so that a live context can swap
them), the pin cell at (16, 0.02) and (16, 0.08), a 64-angle configuration (the boundary-band rules of the chunk plan apply), three
boundary-condition sets, and a mixed quad/triangle mesh for the literal-only path.  Each (mesh, angles, spacing) has ONE oracle run.
A numpy model computes what every call must give from the oracle of the current (mesh, trace configuration) -- uid ranges are slices
of the whole-domain run -- and after every action everything observable through the C ABI is compared with it.

A failure names the seed, the step and the actions so far; ``replay(seed, upto)`` runs the same sequence up to that step.  The model
itself is tested without a GPU (test_model_*)."""
import ctypes as C
import math
import traceback
from types import SimpleNamespace

import numpy as np
import pytest

import raytracing_jl_b200 as rt
from raytracing_jl_b200 import _lib as L
from raytracing_jl_b200.api import TrackLayout, _angle_tables
from raytracing_jl_b200.distributed import plan_shards
from oracle.oracle import OracleMesh, OracleTrackGenerator
from tests.test_gpu_knobs_flags import assert_volumes_exact, expected_capped, first_segments, reference_volumes
from tests.test_gpu_parity import assert_segments_equal, assert_tracks_equal
from tests.test_gpu_sweep_outputs import numpy_areas, numpy_factors

LIT, NO_VOL, COUNT, NO_CHUNKS, SEQ = rt.RT_SEG_LITERAL, rt.RT_SEG_NO_VOLUMES, rt.RT_SEG_COUNT_ONLY, rt.RT_SEG_NO_CHUNKS, rt.RT_SEG_SEQUENTIAL
EXACT, LEN_ONLY = rt.RT_SEG_EXACT_VOLUMES, rt.RT_SEG_LENGTHS_ONLY
RT_ERR_ARG, RT_ERR_NOT_TRACED = -2, -7
KEYS = ("px", "py", "qx", "qy", "len", "element")
BCS = [(0, 0, 0, 0), (1, 1, 1, 1), (2, 2, 2, 2)]
BIG = 10_000  # MAX_ITER: no track of the world has that many segments
N_REGIONS = 3
GROUPS = 2

WORLDS = {
    "jittered": {"meshes": {"jitA": lambda pin: rt.synth.jittered_triangle_mesh(60, 60, seed=5),
                            "jitB": lambda pin: rt.synth.jittered_triangle_mesh(60, 60, seed=6)},
                 "configs": [(64, 0.02), (16, 0.02)]},
    "pincell": {"meshes": {"pin": lambda pin: pin}, "configs": [(16, 0.02), (16, 0.08)]},  # 0.08: every track starts on a node
    "mixed": {"meshes": {"mixed": lambda pin: rt.synth.mixed_quad_triangle_mesh(19, 15, 1.5, 1.1, jitter=0.2, seed=17, quad_fraction=0.5)},
              "configs": [(8, 0.04)]},
}
SEEDS = [(0, "jittered"), (1, "pincell"), (2, "jittered"), (3, "pincell"), (4, "jittered"), (5, "mixed")]
STEPS = 60


# ---- the oracle of the world, one run per (mesh, angles, spacing) ------------------------------------------------------------
class World:
    def __init__(self, name, pincell_model):
        self.name = name
        spec = WORLDS[name]
        self.models = {k: make(pincell_model) for k, make in spec["meshes"].items()}
        self.meshes = {k: rt.Mesh(m) for k, m in self.models.items()}
        self.omeshes = {k: OracleMesh.from_mesh(m) for k, m in self.meshes.items()}
        self.configs = spec["configs"]
        self.mixed = name == "mixed"
        self._seg, self._trk = {}, {}

    def oracle(self, mesh, cfg):
        """the segmentized whole-domain oracle of (mesh, n_azim, delta) with vacuum boundaries (segments do not depend on them)"""
        key = (mesh, cfg)
        if key not in self._seg:
            otg = OracleTrackGenerator(self.omeshes[mesh], cfg[0], cfg[1]).trace().segmentize(check=False, nthreads=8)
            assert not np.any(otg.seg_status == 1)  # (no "Try increasing k": any k >= 5 gives these segments)
            self._seg[key] = otg
        return self._seg[key]

    def tracks(self, mesh, cfg, bcs):
        key = (mesh, cfg, bcs)
        if key not in self._trk:
            self._trk[key] = self.oracle(mesh, cfg).tracks if bcs == BCS[0] else \
                OracleTrackGenerator(self.omeshes[mesh], cfg[0], cfg[1], bcs=bcs).trace().tracks
        return self._trk[key]


_WORLDS = {}


def world(name, pincell_model):
    if name not in _WORLDS:
        _WORLDS[name] = World(name, pincell_model)
    return _WORLDS[name]


# ---- the model: what a call on uids [u0, u1) must give, from the whole-domain oracle ---------------------------------------------
def shard_slice(otg, u0, u1, max_iter=BIG):
    """offsets (from 0), status, Segment columns and azimuthal indices of the uids [u0, u1); with max_iter the segments a capped call
    keeps.  `sure`: the tracks whose status can be predicted (a track of exactly max_iter segments: the length check decides)."""
    g0, g1 = int(otg.seg_offsets[u0 - 1]), int(otg.seg_offsets[u1 - 1])
    off = otg.seg_offsets[u0 - 1:u1] - g0
    status = otg.seg_status[u0 - 1:u1 - 1]
    cols = {k: otg.seg[k][g0:g1] for k in KEYS}
    sure = np.ones(u1 - u0, bool)
    if max_iter < BIG:
        off, keep, sure, status = expected_capped(SimpleNamespace(seg_offsets=off, seg_status=status), max_iter)
        cols = {k: v[keep] for k, v in cols.items()}
    return SimpleNamespace(u0=u0, u1=u1, off=np.asarray(off, np.int64), status=np.asarray(status, np.int32), sure=sure, cols=cols,
                           azim=otg.tracks["azim_idx"][u0 - 1:u1 - 1])


def atomic_reference(otg, sl):
    """(volumes, terms per element) of reference_volumes over the shard's segments"""
    sub = SimpleNamespace(mesh=otg.mesh, tracks={"azim_idx": sl.azim}, deltas=otg.deltas)
    return reference_volumes(sub, sl.off, sl.cols, otg.n2)


def exact_reference(otg, sl):
    """RT_SEG_EXACT_VOLUMES: delta_eff[azim] * len added in segment order (np.add.at is unbuffered, in index order), / n_azim_2"""
    acc = np.zeros(otg.mesh.n_cells)
    terms = otg.deltas[np.repeat(sl.azim - 1, np.diff(sl.off))] * sl.cols["len"]
    np.add.at(acc, sl.cols["element"].astype(np.int64) - 1, terms)
    return acc / otg.n2


def region_sums(region, values):
    """the cells of every region in ascending id, one `+` each from 0.0 (rt_region_volumes)"""
    out = np.zeros(N_REGIONS)
    np.add.at(out, np.asarray(region, np.int64) - 1, values)
    return out


def bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def uid_ranges(layout, rng):
    """the uid ranges the sequences trace: whole domain, one track, inside a 32-track block, the last tracks, one angle, empty"""
    n = layout.n_total_tracks
    i = int(rng.integers(len(layout.n_tracks)))
    u = int(rng.integers(1, n + 1))
    return [(1, n + 1), (u, u + 1), (33, 97), (n - 4, n + 1), (int(layout._base[i]) + 1, int(layout._base[i + 1]) + 1), (u, u)]


# ---- the model's self-test (no GPU) ---------------------------------------------------------------------------------------------
def test_model_on_the_oracle(pincell_model):
    """The numpy model against the oracle itself: the shard slices of a partition concatenate to the whole run; the np.add.at
    reference over the whole domain is the oracle's volumes() bit for bit, and over the slices of a partition it adds up to them
    within the bound; the capped expectations agree with expected_capped; one dropped term fails assert_volumes_exact."""
    w = world("pincell", pincell_model)
    for cfg in w.configs:
        otg = w.oracle("pin", cfg)
        n = otg.n_total_tracks
        cuts = [1, 2, 33, 97, n // 2, n - 4, n + 1]
        parts = [shard_slice(otg, a, b) for a, b in zip(cuts, cuts[1:])]
        for k in KEYS:
            assert bits_equal(np.concatenate([p.cols[k] for p in parts]), otg.seg[k])
        assert bits_equal(np.concatenate([p.off[:-1] + otg.seg_offsets[p.u0 - 1] for p in parts] + [[otg.n_segments]]), otg.seg_offsets)
        assert bits_equal(np.concatenate([p.status for p in parts]), otg.seg_status)
        whole = shard_slice(otg, 1, n + 1)
        assert bits_equal(exact_reference(otg, whole), otg.volumes())
        ref, m = atomic_reference(otg, whole)
        assert_volumes_exact(otg.volumes(), ref, m)
        assert_volumes_exact(sum(exact_reference(otg, p) for p in parts), ref, m)
        for mi in (3, 10):
            capped = shard_slice(otg, 1, n + 1, mi)
            off, keep, sure, status = expected_capped(otg, mi)
            assert bits_equal(capped.off, off) and bits_equal(capped.status[sure], status[sure]) and bits_equal(capped.sure, sure)
            assert bits_equal(capped.cols["len"], otg.seg["len"][first_segments(otg.seg_offsets, mi)])
            cref, cm = atomic_reference(otg, capped)
            assert_volumes_exact(exact_reference(otg, capped), cref, cm)
            assert cm.sum() == off[-1]
        e = int(otg.seg["element"][0]) - 1  # drop the first term of the first element crossed
        short = otg.volumes().copy()
        short[e] -= otg.deltas[otg.tracks["azim_idx"][0] - 1] * otg.seg["len"][0] / otg.n2
        with pytest.raises(AssertionError):
            assert_volumes_exact(short, ref, m)
        empty = shard_slice(otg, 7, 7)
        assert empty.off.tolist() == [0] and all(v.size == 0 for v in empty.cols.values())
        assert not np.any(exact_reference(otg, empty))


# ---- the sequence runner ------------------------------------------------------------------------------------------------------
OPTIONS = [("pipeline", 0), ("pipeline", 1), ("pipeline", 3), ("pipeline", 3), ("chunk_segments", 3), ("chunk_segments", 12),
           ("chunk_segments", 208), ("plan_cache", 0), ("plan_cache", 1), ("optimistic", 0), ("optimistic", 1), ("band_min", 0),
           ("band_min", 0.0625), ("band_div", 64), ("band_div", 8), ("order_grid", 0), ("order_grid", 32), ("order_classes", 0),
           ("order_classes", 3), ("pool_slots", 2048), ("pool_slots", 32768), ("pool_slots", 0), ("pool_slots", 0), ("pool_extra", 0), ("pool_extra", 1.25),
           ("debug_verify_fail", 1), ("debug_verify_fail", 0), ("debug_verify_fail", 0)]
ACTIONS = {"segmentize": 14, "option": 6, "capacity": 3, "retrace": 3, "swap": 1, "regions": 2, "locate": 1, "tau": 2,
           "region_volumes": 2, "element_volumes": 1, "track_view": 1, "quadrature": 1, "plan_shards": 2, "compact": 2}
CALLBACKS = ("copy", "download", "tau", "correct", "locate", "raise", "nested")


class Sequence:
    """One context driven by a seeded rng, and the model of what it holds"""

    def __init__(self, w, seed):
        self.w, self.seed = w, seed
        self.rng = np.random.default_rng(seed)
        self.mesh = next(iter(w.meshes))
        self.cfg, self.bcs = w.configs[0], BCS[0]
        self.tg = rt.TrackGenerator(w.meshes[self.mesh], *self.cfg)
        self.tg.set_option("target_walkers", 1e9)  # (chunk_segments alone sizes the chunks)
        self.log = []
        self.traced = False
        self.seg = None           # the last completed segmentize: what the context must hold
        self.has_delta = False
        self.regions = None
        self.cap = 0
        self.opts = {"pipeline": 3, "pool_slots": 0, "pool_extra": 1.25, "debug_verify_fail": 0}
        self.cancels = 0
        self.trace_range(1, self.tg.n_total_tracks + 1)

    # -- helpers
    def otg(self):
        return self.w.oracle(self.mesh, self.cfg)

    def lib(self):
        return L.lib()

    def trace_range(self, u0, u1):
        """rt_trace of the uids [u0, u1) with the current configuration, and the mirror updated as trace_ does"""
        tg = self.tg
        sin_t, cos_t, tan_t, dxe, dye = _angle_tables(tg)
        aq = tg.azimuthal_quadrature
        tg.bcs = rt.BoundaryConditions(*(rt.BoundaryType(c) for c in self.bcs))
        tg.uid_begin, tg.uid_end = u0, u1
        tg._traced = tg._segmented = False
        tg._track_data = tg._segments = tg._offsets = tg._resident = None
        L.check(tg._ctx, self.lib().rt_trace(tg._ctx, len(aq.phis), tg.n_tracks_x, tg.n_tracks_y, aq.phis, sin_t, cos_t, tan_t, dxe, dye,
                                             tg.bcs.codes(), u0, u1))
        tg._traced = True
        self.traced, self.seg, self.has_delta = True, None, False
        self.shard = (u0, u1)

    def rc_of(self, fn, *args):
        try:
            fn(*args)
            return 0
        except L.RTError as e:
            return e.code

    # -- actions
    def step(self):
        names = list(ACTIONS)
        p = np.array([ACTIONS[a] for a in names], float)
        if self.w.mixed:
            p[names.index("element_volumes")] = 0
        name = names[int(self.rng.choice(len(names), p=p / p.sum()))]
        self.note(name)
        return getattr(self, "act_" + name)()

    def note(self, desc):
        self.log[-1] = self.log[-1].split(": ")[0] + ": " + desc

    def act_option(self):
        name, value = OPTIONS[int(self.rng.integers(len(OPTIONS)))]
        self.tg.set_option(name, value)
        if name in self.opts:
            self.opts[name] = value
        return f"set_option({name!r}, {value})"

    def act_capacity(self):
        otg = self.otg()
        n = otg.n_segments
        # (the smallest: just above the longest track, which must fit in one batch)
        self.cap = int(self.rng.choice([0, 0, n // 5, n // 2, int(np.diff(otg.seg_offsets).max()) + 1]))
        L.check(self.tg._ctx, self.lib().rt_set_segment_capacity(self.tg._ctx, self.cap))
        return f"capacity({self.cap})"

    def act_retrace(self):
        what = self.rng.choice(["config", "bcs", "range", "range"])
        if what == "config":
            self.cfg = self.w.configs[int(self.rng.integers(len(self.w.configs)))]
            TrackLayout.__init__(self.tg, self.tg.mesh, *self.cfg)
        elif what == "bcs":
            self.bcs = BCS[int(self.rng.integers(len(BCS)))]
        rngs = uid_ranges(self.tg, self.rng)
        u0, u1 = rngs[0] if what != "range" else rngs[int(self.rng.integers(len(rngs)))]
        if what == "range" and self.rng.random() < 0.2:  # one part of the device planner's bounds
            b = self.plan(3)
            r = int(self.rng.integers(3))
            u0, u1 = int(b[r]), int(b[r + 1])
        self.trace_range(u0, u1)
        return f"retrace({what}: cfg={self.cfg}, bcs={self.bcs}, uids=[{u0}, {u1}))"

    def act_swap(self):
        names = list(self.w.meshes)
        self.mesh = names[(names.index(self.mesh) + 1) % len(names)]
        self.tg.mesh = self.w.meshes[self.mesh]
        self.tg.upload_mesh()
        self.traced, self.seg, self.regions = False, None, None
        return f"upload_mesh({self.mesh})"

    def act_regions(self):
        if self.rng.random() < 0.3:
            self.tg.set_regions(None)
            self.regions = None
            return "set_regions(None)"
        reg = self.rng.integers(1, N_REGIONS + 1, self.w.meshes[self.mesh].num_cells).astype(np.int32)
        self.tg.set_regions(reg, N_REGIONS)
        self.regions = reg
        return "set_regions(random)"

    def points(self, n=24):
        m = self.w.meshes[self.mesh]
        lo, hi = np.asarray(m.bb_min), np.asarray(m.bb_max)
        return lo + (hi - lo) * self.rng.uniform(-0.05, 1.05, (n, 2))

    def check_locate(self, pts, ids):
        om = self.w.omeshes[self.mesh]
        assert ids.tolist() == [om.find_element(float(x), float(y), 2) for x, y in pts]

    def act_locate(self):
        pts = self.points()
        ids, _ = self.tg.find_elements(pts, 2)
        self.check_locate(pts, ids)
        return "find_elements"

    def sigma(self, rows):
        return np.random.default_rng(rows).uniform(0.1, 2.0, (rows, GROUPS))

    def act_tau(self):
        by_region = self.regions is not None and self.rng.random() < 0.5
        sig = self.sigma(N_REGIONS if by_region else self.w.meshes[self.mesh].num_cells)
        call = self.tg.optical_lengths_by_region if by_region else self.tg.optical_lengths
        if self.seg is None:
            assert self.rc_of(call, sig) == RT_ERR_ARG
            return f"tau(by_region={by_region}) refused"
        tau, _ = call(sig)
        u0, u1, base, n = self.view()
        cols = self.expected_cols(base, n)
        table = sig[self.regions - 1] if by_region else sig
        assert bits_equal(tau, table[cols["element"] - 1] * cols["len"][:, None])
        return f"tau(by_region={by_region})"

    def act_region_volumes(self):
        traced = self.seg is not None and self.seg.vol != "none"
        exact = not self.w.mixed
        if self.regions is None:
            assert self.rc_of(self.tg.region_volumes, True, exact) == RT_ERR_ARG
            return "region_volumes refused (no map)"
        if not traced:
            assert self.rc_of(self.tg.region_volumes, True, False) == RT_ERR_ARG
        if not traced and not exact:
            return "region_volumes refused"
        t, e = self.tg.region_volumes(traced, exact)
        if traced:
            assert bits_equal(t, region_sums(self.regions, self.seg.volumes))
        if exact:
            assert bits_equal(e, region_sums(self.regions, numpy_areas(self.w.models[self.mesh])))
        return f"region_volumes(traced={traced}, exact={exact})"

    def act_element_volumes(self):
        assert bits_equal(self.tg.element_volumes(), numpy_areas(self.w.models[self.mesh]))
        return "element_volumes"

    def act_track_view(self):
        if not self.traced:
            assert self.rc_of(self.tg.track_view) == RT_ERR_NOT_TRACED
            return "track_view refused"
        v = self.tg.track_view()
        assert (v["uid_begin"], v["n_tracks"]) == (self.shard[0], self.shard[1] - self.shard[0])
        return "track_view"

    def act_quadrature(self):
        return "quadrature_device" if self.check_quadrature() else "quadrature_device refused"

    def check_quadrature(self):
        """the per-angle tables of rt_quadrature_device: those of the current trace, delta_eff once a call with volumes uploaded it"""
        if not self.traced:
            assert self.rc_of(self.tg.quadrature_device) == RT_ERR_NOT_TRACED
            return False
        import torch

        aq = self.tg.azimuthal_quadrature
        omega, view = self.tg.quadrature_device()
        dev = {k: torch.as_tensor(c, device="cuda").cpu().numpy() for k, c in view.items()}
        otg = self.otg()
        assert bits_equal(aq.weights, otg.weights) and bits_equal(aq.phis, otg.phis)
        assert bits_equal(omega, aq.weights) and bits_equal(dev["omega"], aq.weights) and bits_equal(dev["phi"], aq.phis)
        assert bits_equal(dev["sin"], [math.sin(p) for p in aq.phis]) and bits_equal(dev["cos"], [math.cos(p) for p in aq.phis])
        assert ("delta_eff" in dev) == self.has_delta
        if self.has_delta:
            assert bits_equal(dev["delta_eff"], otg.deltas) and bits_equal(aq.deltas, otg.deltas)
        return True

    def plan(self, parts):
        tg = self.tg
        _, _, tan_t, dxe, dye = _angle_tables(tg)
        b = np.zeros(parts + 1, np.int64)
        L.check(tg._ctx, self.lib().rt_plan_shards(tg._ctx, len(tg.n_tracks), tg.n_tracks_x, tg.n_tracks_y,
                                                    tg.azimuthal_quadrature.phis, tan_t, dxe, dye, parts, b))
        assert b[0] == 1 and b[-1] == tg.n_total_tracks + 1 and np.all(np.diff(b) >= 0)
        if self.traced:  # (the host planner reads rho from the context: it has the mesh's, not the shard's, only once traced)
            assert np.abs(b - plan_shards(tg, parts)).max() <= 1
        return b

    def act_plan_shards(self):
        parts = int(self.rng.choice([1, 2, 3, 7]))
        self.plan(parts)
        return f"rt_plan_shards({parts})"

    def act_compact(self):
        tg = self.tg
        if self.seg is None or self.seg.lengths_only:
            k = C.c_int64(0)
            assert self.lib().rt_segments_download_compact(tg._ctx, None, None, None, None, 0, None, None, None, C.byref(k)) == RT_ERR_ARG
            return "compact download refused"
        cols = tg.fetch_segments(compact=True)
        u0, u1, base, n = self.view()
        exp = self.expected_cols(base, n)
        for k in KEYS:
            assert bits_equal(cols[k], exp[k]), k
        tg._segments = None
        return "compact download"

    # -- segmentize_
    def draw_call(self):
        r = self.rng
        flags = 0
        for f, p in ((LIT, 0.15), (NO_CHUNKS, 0.15), (SEQ, 0.15), (COUNT, 0.1), (NO_VOL, 0.15), (EXACT, 0.3), (LEN_ONLY, 0.3)):
            if r.random() < p:
                flags |= f
        max_iter = int(r.choice([BIG, BIG, BIG, BIG, 3, 10, 40]))
        k = int(r.choice([5, 5, 5, 5, 8, 32, 33]))
        cbs = [c for c in CALLBACKS if r.random() < 0.3] if r.random() < 0.5 else []
        if self.w.mixed and "correct" in cbs:
            cbs.remove("correct")
        raise_at = int(r.integers(0, 3))
        return flags, max_iter, k, cbs, raise_at

    def act_segmentize(self):
        flags, max_iter, k, cbs, raise_at = self.draw_call()
        desc = f"segmentize(flags={flags}, max_iter={max_iter}, k={k}, on_batch={cbs}, raise_at={raise_at})"
        self.note(desc)
        tg, otg = self.tg, self.otg()
        want_vol = not flags & NO_VOL
        if not self.traced:
            with pytest.raises(RuntimeError):
                rt.segmentize_(tg, k=k, flags=flags, max_iter=max_iter, check=False)
            return desc + " refused (not traced)"
        if flags & EXACT and flags & (COUNT | NO_VOL) or k > 32:
            with pytest.raises(L.RTError) as e:
                rt.segmentize_(tg, k=k, flags=flags, max_iter=max_iter, check=False)
            assert e.value.code == RT_ERR_ARG
            self.seg = None
            return desc + " refused (arguments)"
        sl = shard_slice(otg, *self.shard, max_iter)
        prev = self.seg if (self.seg is not None and self.seg.vol != "none") else None
        lengths_only = bool(flags & LEN_ONLY) and not flags & COUNT
        batches, events = [], []
        count = {"n": 0}

        def on_batch(b):
            j = count["n"]
            count["n"] += 1
            rec = SimpleNamespace(u0=b.uid_begin, u1=b.uid_end, base=b.offset_base, n=b.n_segments, attempt=b.attempt, cols={}, f=None)
            assert tg.resident_batch() == (b.uid_begin, b.uid_end, b.offset_base, b.n_segments)
            assert (b.px is None) == lengths_only
            if "correct" in cbs:
                try:
                    rec.f = tg.correct_volumes()
                    events.append(("correct", True))
                except L.RTError as e:
                    assert e.code == RT_ERR_ARG
                    events.append(("correct", False))
            if "copy" in cbs:
                import torch

                torch.cuda.synchronize()
                for key in (("len", "element") if lengths_only else KEYS):
                    rec.cols[key] = torch.as_tensor(getattr(b, key), device="cuda")[:b.n_segments].cpu().numpy()
            if "download" in cbs:
                s = tg.fetch_segments()
                rec.dl = {key: s[key].copy() for key in s}
            if "tau" in cbs:
                sig = self.sigma(self.w.meshes[self.mesh].num_cells)
                rec.tau = (sig, tg.optical_lengths(sig)[0])
            if "locate" in cbs:
                pts = self.points(8)
                rec.loc = (pts, tg.find_elements(pts, 2)[0])
            if "nested" in cbs:
                z = C.c_int64(0)
                rc = self.lib().rt_segmentize(tg._ctx, tg.tiny_step, 5, rt.RTOL_DEFAULT, BIG, None, NO_VOL, None, None, C.byref(z), C.byref(z),
                                              C.byref(C.c_int32(0)))
                events.append(("nested", rc))
            batches.append(rec)
            if "raise" in cbs and j == raise_at:
                raise KeyError("stop at batch %d" % j)

        cb = on_batch if cbs else None
        cancels0 = tg.info("optimistic_cancels")
        try:
            rt.segmentize_(tg, k=k, flags=flags, max_iter=max_iter, check=False, on_batch=cb)
            raised = None
        except KeyError as e:
            raised = e
        if want_vol:
            self.has_delta = True
        for what, v in events:
            if what == "correct":
                assert v == (prev is not None), "rt_correct_volumes inside on_batch"
            else:
                assert v == RT_ERR_ARG
        if raised is not None:
            assert "raise" in cbs and count["n"] == raise_at + 1
            self.seg = None
            return desc + f" raised at batch {raise_at}"
        assert not ("raise" in cbs and count["n"] > raise_at)
        # the call completed: the model's record of it
        corrected = [b.f for b in batches if b.f is not None]
        seg = SimpleNamespace(sl=sl, flags=flags, lengths_only=lengths_only, count_only=bool(flags & COUNT),
                              vol="none" if not want_vol else ("exact" if flags & EXACT else "atomic"), volumes=None,
                              factors=corrected[-1] if corrected else None,
                              whole=self.cap == 0 and self.opts["pool_slots"] == 0)
        if seg.factors is not None:
            area = numpy_areas(self.w.models[self.mesh])
            assert bits_equal(seg.factors, numpy_factors(area, prev.volumes))
        self.seg = seg
        # returned scalars
        n_shard = sl.u1 - sl.u0
        assert tg.n_segments == sl.off[-1]
        # batches of the last attempt: contiguous, covering the shard, the expected columns
        if batches and not seg.count_only:
            last = max(b.attempt for b in batches)
            got = [b for b in batches if b.attempt == last]
            assert got[0].u0 == sl.u0 and got[-1].u1 == sl.u1 and all(a.u1 == b.u0 for a, b in zip(got, got[1:]))
            assert sum(b.n for b in got) == sl.off[-1]
            for b in got:
                exp = self.expected_cols(b.base, b.n)
                for key, v in b.cols.items():
                    assert bits_equal(v, exp[key]), key
                for key, v in getattr(b, "dl", {}).items():
                    assert bits_equal(v, exp[key]), key
                if hasattr(b, "tau"):
                    sig, tau = b.tau
                    assert bits_equal(tau, sig[exp["element"] - 1] * exp["len"][:, None])
                if hasattr(b, "loc"):
                    self.check_locate(*b.loc)
        # rt_info of the call
        mode = 1 if (flags & (SEQ | COUNT)) or self.w.mixed else self.opts["pipeline"]
        mode = 1 if mode == 3 and flags & LIT else mode
        # the hooks that force a fall-back: a failed verification (pipelines 3 and 0 restart in 1), a record pool that runs out or
        # whose batches cannot take one 32-track block (pipeline 3 restarts in 0; a failed verification there may follow)
        fail_hook = bool(self.opts["debug_verify_fail"]) and mode != 1 and n_shard > 0
        pool_hook = (self.opts["pool_extra"] == 0 or self.opts["pool_slots"] > 0) and mode == 3 and n_shard > 0
        vf = tg.info("verify_fallbacks")
        assert vf <= int(fail_hook) + int(pool_hook) and vf >= int(fail_hook)
        cb_n = tg.info("count_batches")
        if n_shard == 0:
            assert cb_n == 0
        elif mode in (0, 1):
            assert cb_n == 1
        else:
            assert cb_n >= 1
        cancels = tg.info("optimistic_cancels")
        assert cancels0 <= cancels <= cancels0 + 1
        if cb or self.cap or flags & EXACT:
            assert cancels == cancels0
        # volumes
        if want_vol:
            seg.volumes = tg.volumes.copy()
            if seg.vol == "exact":
                assert bits_equal(seg.volumes, exact_reference(otg, sl))
            else:
                assert_volumes_exact(seg.volumes, *atomic_reference(otg, sl))
        return desc

    def expected_cols(self, base, n):
        """the columns of the resident segments [base, base + n) of the shard, as the last call left them"""
        s = self.seg
        cols = {k: v[base:base + n] for k, v in s.sl.cols.items()}
        if s.factors is not None:
            cols["len"] = cols["len"] * s.factors[cols["element"] - 1]
        if s.lengths_only:
            cols = {k: cols[k] for k in ("len", "element")}
        return cols

    def view(self):
        v = L.rt_batch()
        L.check(self.tg._ctx, self.lib().rt_segments_device(self.tg._ctx, C.byref(v)))
        return int(v.uid_begin), int(v.uid_end), int(v.offset_base), int(v.n_segments)

    # -- everything observable through the C ABI, after every action
    def check(self):
        tg, lib, ctx = self.tg, self.lib(), self.tg._ctx
        assert tg._traced == self.traced
        if self.traced:
            tg._track_data = None
            o = self.tracks_slice()
            for key, v in tg.track_data.items():
                assert bits_equal(v, o[key]), key
        else:
            assert lib.rt_tracks_download(ctx, *([None] * 13)) == RT_ERR_NOT_TRACED
        v = L.rt_batch()
        z = np.zeros(1)
        if self.seg is None:
            assert lib.rt_segment_offsets(ctx, None, None) == RT_ERR_ARG
            assert lib.rt_segments_device(ctx, C.byref(v)) == RT_ERR_ARG
            assert lib.rt_segments_download(ctx, None, None, None, None, None, None) == RT_ERR_ARG
            assert lib.rt_volumes(ctx, L.ptr(np.zeros(tg.mesh.num_cells))) == RT_ERR_ARG
        else:
            s, sl = self.seg, self.seg.sl
            n_shard = sl.u1 - sl.u0
            off, status = np.zeros(n_shard + 1, np.int64), np.zeros(max(n_shard, 1), np.int32)
            L.check(ctx, lib.rt_segment_offsets(ctx, L.ptr(off), L.ptr(status)))
            status = status[:n_shard]
            assert bits_equal(off, sl.off) and bits_equal(status[sl.sure], sl.status[sl.sure])
            bad = np.nonzero(status)[0]
            first = (sl.u0 + int(bad[0]), int(status[bad[0]])) if bad.size else (0, 0)
            assert (tg.first_bad_uid, tg.bad_status) == first
            u0, u1, base, n = self.view()
            if s.count_only:
                assert n == 0
            else:
                assert sl.u0 <= u0 <= u1 == sl.u1 and base == sl.off[u0 - sl.u0] and n == sl.off[u1 - sl.u0] - base
                if s.whole:  # (no capacity and no record-pool limit: the shard is one batch)
                    assert u0 == sl.u0 or n == 0
            assert tg.info("segment_capacity") >= n
            exp = self.expected_cols(base, n) if not s.count_only else {}
            if s.lengths_only:
                assert lib.rt_segments_download(ctx, L.ptr(z), None, None, None, None, None) == RT_ERR_ARG
            got = {k: np.zeros(n, np.int32 if k == "element" else np.float64) for k in KEYS}
            if s.lengths_only:
                got = {k: got[k] for k in ("len", "element")}
            L.check(ctx, lib.rt_segments_download(ctx, *[L.ptr(got.get(k)) for k in KEYS]))
            for k, col in got.items():
                assert bits_equal(col, exp[k] if exp else col[:0]), k
            vol = np.zeros(tg.mesh.num_cells)
            rc = lib.rt_volumes(ctx, L.ptr(vol))
            if s.vol == "none":
                assert rc == RT_ERR_ARG
            else:
                assert rc == 0 and bits_equal(vol, s.volumes)
        if self.regions is None:  # (rt_mesh_upload clears the map)
            assert lib.rt_region_volumes(ctx, None, None) == RT_ERR_ARG
        self.check_quadrature()
        cancels = tg.info("optimistic_cancels")
        assert self.cancels <= cancels <= self.cancels + 1
        self.cancels = cancels

    def tracks_slice(self):
        t = self.w.tracks(self.mesh, self.cfg, self.bcs)
        u0, u1 = self.shard
        return {k: v[u0 - 1:u1 - 1] for k, v in t.items()}


def run_sequence(w, seed, steps=STEPS):
    seq = Sequence(w, seed)
    try:
        seq.check()
        for i in range(steps):
            seq.log.append(f"{i}: ...")
            seq.log[-1] = f"{i}: {seq.step()}"
            seq.check()
    except BaseException:
        pytest.fail(f"seed {seed} ({w.name}), step {len(seq.log) - 1}; replay({seed}, {len(seq.log)}) repeats it\n"
                    + "\n".join(seq.log) + "\n" + traceback.format_exc(), pytrace=False)
    finally:
        seq.tg.close()
    return seq


def replay(seed, upto=STEPS, pincell_model=None):
    """the sequence of `seed` up to (and including) step upto - 1, with the checks after every step (on a GPU)"""
    if pincell_model is None:
        import os

        d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pincell.npz"))
        pincell_model = rt.UnstructuredDiscreteModel(d["node_coordinates"], d["cell_ptrs"], d["cell_data"])
    rt.build()
    return run_sequence(world(dict(SEEDS)[seed], pincell_model), seed, upto)


@pytest.mark.gpu
@pytest.mark.parametrize("seed,world_name", SEEDS)
def test_call_sequence(pincell_model, seed, world_name):
    rt.build()
    seq = run_sequence(world(world_name, pincell_model), seed)
    assert len(seq.log) == STEPS


# ---- the two defects the sequences are built around, one targeted test each ----------------------------------------------------
@pytest.mark.gpu
def test_segments_device_needs_a_resident_batch(pincell_model):
    """rt_segments_device refuses (RT_ERR_ARG) unless a batch is resident: before the first segmentize, after a re-trace, after a
    mesh upload and after a failed segmentize -- a view then would pair the new shard with the previous call's columns"""
    rt.build()
    w = world("pincell", pincell_model)
    otg = w.oracle("pin", w.configs[0])
    tg = rt.TrackGenerator(w.meshes["pin"], *w.configs[0])
    lib, v = L.lib(), L.rt_batch()
    rt.trace_(tg)
    assert lib.rt_segments_device(tg._ctx, C.byref(v)) == RT_ERR_ARG
    rt.segmentize_(tg, check=False)
    assert_segments_equal(otg, tg)
    n = tg.n_total_tracks
    assert tg.resident_batch() == (1, n + 1, 0, otg.n_segments)

    def refused():
        assert lib.rt_segments_device(tg._ctx, C.byref(v)) == RT_ERR_ARG
        with pytest.raises(RuntimeError):
            tg.resident_batch()
        with pytest.raises(L.RTError) as e:
            tg.optical_lengths(np.ones((tg.mesh.num_cells, 1)))
        assert e.value.code == RT_ERR_ARG

    tg.shard = (1, 2)  # a re-trace onto the second half of the uids: the old view would start inside it with the old columns
    rt.trace_(tg)
    refused()
    rt.segmentize_(tg, check=False)
    u0, u1 = tg.uid_begin, tg.uid_end
    assert 1 < u0 < u1 == n + 1
    assert tg.resident_batch() == (u0, u1, 0, otg.n_segments - otg.seg_offsets[u0 - 1])
    tg.upload_mesh()
    refused()
    tg.shard = (0, 1)
    rt.trace_(tg)
    refused()
    with pytest.raises(L.RTError):
        rt.segmentize_(tg, k=33, check=False)
    refused()
    rt.segmentize_(tg, check=False)
    assert_segments_equal(otg, tg)
    assert tg.resident_batch() == (1, n + 1, 0, otg.n_segments)
    tg.close()


@pytest.mark.gpu
def test_plan_shards_leaves_a_traced_context_as_it_was(pincell_model):
    """rt_plan_shards is a query: on a traced and segmentized context it changes neither the trace, the segments, the volumes nor
    the per-angle tables of rt_quadrature_device, and the next segmentize still works.  rt_quadrature_device hands out only the
    tables of a completed rt_trace: it refuses after a mesh upload and after an rt_trace that failed"""
    import torch

    rt.build()
    w = world("pincell", pincell_model)
    otg = w.oracle("pin", w.configs[0])
    tg = rt.TrackGenerator(w.meshes["pin"], *w.configs[0])
    rt.segmentize_(rt.trace_(tg), check=False)
    vol = tg.volumes.copy()

    def quad():
        _, view = tg.quadrature_device()
        return {k: torch.as_tensor(c, device="cuda").cpu().numpy() for k, c in view.items()}

    before = quad()
    assert bits_equal(before["sin"], otg.sin_phi) and bits_equal(before["delta_eff"], otg.deltas)
    other = TrackLayout(tg.mesh, 32, 0.01)  # another angle count than the context's trace
    for lay in (tg, other):
        _, _, tan_t, dxe, dye = _angle_tables(lay)
        b = np.zeros(4, np.int64)
        L.check(tg._ctx, L.lib().rt_plan_shards(tg._ctx, len(lay.n_tracks), lay.n_tracks_x, lay.n_tracks_y, lay.azimuthal_quadrature.phis,
                                                tan_t, dxe, dye, 3, b))
        assert b[0] == 1 and b[-1] == lay.n_total_tracks + 1
    after = quad()
    assert before.keys() == after.keys() and all(bits_equal(before[k], after[k]) for k in before)
    tg._offsets = tg._segments = tg._resident = tg._track_data = None
    assert_tracks_equal(otg, tg)
    assert_segments_equal(otg, tg)
    out = np.zeros(tg.mesh.num_cells)
    L.check(tg._ctx, L.lib().rt_volumes(tg._ctx, L.ptr(out)))
    assert bits_equal(out, vol)
    rt.segmentize_(tg, check=False)
    assert_segments_equal(otg, tg)
    # a failed rt_trace (uid range past the end) leaves no trace, and no tables to hand out
    sin_t, cos_t, tan_t, dxe, dye = _angle_tables(tg)
    aq = tg.azimuthal_quadrature
    rc = L.lib().rt_trace(tg._ctx, len(aq.phis), tg.n_tracks_x, tg.n_tracks_y, aq.phis, sin_t, cos_t, tan_t, dxe, dye, tg.bcs.codes(),
                          1, tg.n_total_tracks + 2)
    assert rc == RT_ERR_ARG
    tg._traced = tg._segmented = False
    assert L.lib().rt_quadrature_device(tg._ctx, C.byref(L.rt_quad_view()), None) == RT_ERR_NOT_TRACED
    z = C.c_int64(0)
    assert L.lib().rt_segmentize(tg._ctx, tg.tiny_step, 5, rt.RTOL_DEFAULT, BIG, L.ptr(aq.deltas), 0, None, None, C.byref(z), C.byref(z),
                                 C.byref(C.c_int32(0))) == RT_ERR_NOT_TRACED
    rt.segmentize_(rt.trace_(tg), check=False)
    assert_segments_equal(otg, tg)
    tg.upload_mesh()
    assert L.lib().rt_quadrature_device(tg._ctx, C.byref(L.rt_quad_view()), None) == RT_ERR_NOT_TRACED
    tg.close()


@pytest.mark.gpu
def test_record_pool_too_small_for_one_block_falls_back(pincell_model):
    """pipeline 3 walks the shard in count batches of whole 32-track blocks.  When one block has more chunk slots than a batch may
    take, the call restarts in the hybrid pipeline, as when the record pool runs out, instead of failing: the oracle's bits and
    volumes, one fall-back, also with a segment capacity just above the longest track"""
    rt.build()
    w = world("jittered", pincell_model)
    cfg = w.configs[0]
    otg = w.oracle("jitA", cfg)
    tg = rt.TrackGenerator(w.meshes["jitA"], *cfg)
    rt.trace_(tg)
    tg.set_option("chunk_segments", 3)
    tg.set_option("target_walkers", 1e9)
    whole = shard_slice(otg, 1, tg.n_total_tracks + 1)
    for capacity in (0, int(np.diff(otg.seg_offsets).max()) + 1):
        L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, capacity))
        for slots, fallbacks in ((32, 1), (0, 0)):  # (32 slots: one warp unit, less than any block of these tracks needs)
            tg.set_option("pool_slots", slots)
            rt.segmentize_(tg, check=False, exact_volumes=True)
            assert tg.info("verify_fallbacks") == fallbacks
            assert bits_equal(tg.volumes, exact_reference(otg, whole))
            if capacity == 0:
                assert_segments_equal(otg, tg)
            else:
                assert tg.n_segments == otg.n_segments and np.array_equal(tg.segment_offsets, otg.seg_offsets)
    tg.close()
