"""segmentize! beyond its default settings: the tuning knobs of rt_set_option, the chunk plan kept between calls on one context, and
the RT_SEG_COUNT_ONLY / RT_SEG_NO_VOLUMES flags.  Every call is compared with the CPU oracle: tracks, offsets, status and the six
Segment columns bit for bit, volumes element by element against an exactly summed reference (reference_volumes).

GPU tests are marked one by one (pytest -m gpu); the test of the volume reference itself runs without a GPU."""
import math

import numpy as np
import pytest

import raytracing_jl_b200 as rt
from raytracing_jl_b200 import _lib as L
from oracle.oracle import OracleMesh, OracleTrackGenerator
from tests.test_gpu_parity import assert_segments_equal, assert_tracks_equal

SEQ, LIT, NO_VOL, COUNT, NO_CHUNKS = rt.RT_SEG_SEQUENTIAL, rt.RT_SEG_LITERAL, rt.RT_SEG_NO_VOLUMES, rt.RT_SEG_COUNT_ONLY, rt.RT_SEG_NO_CHUNKS
RT_ERR_ARG = -2
KEYS = ("px", "py", "qx", "qy", "len", "element")
CHUNK = 12  # chunk_segments of the knob tests: several chunks per track, boundary-band heads and tails


# ---- an exactly summed volume reference ------------------------------------------------------------------------------
def reference_volumes(otg, offsets, seg, n_azim_2, max_iter=None):
    """volumes[e] = sum of delta_eff[azim(u)] * len(s) over the segments s of element e, / n_azim_2 (src/trackgenerator.jl:371-386).
    Each term is the float64 product the kernels form (walk.cuh push, eval3.cuh: no fused multiply-add); the terms of an element
    are summed exactly (math.fsum), so the only rounding after the products is that of the sum and of the division.  With
    max_iter only the first min(max_iter, n_u) segments of each track count, as in a call capped at max_iter.
    Returns (volumes, number of terms per element)."""
    offsets = np.asarray(offsets, np.int64)
    counts = np.diff(offsets)
    n_cells = otg.mesh.n_cells
    keep = np.ones(int(offsets[-1]), bool) if max_iter is None else first_segments(offsets, max_iter)
    azim = np.repeat(otg.tracks["azim_idx"] - 1, counts)[keep]
    terms = otg.deltas[azim] * seg["len"][keep]
    elem = seg["element"][keep].astype(np.int64) - 1
    order = np.argsort(elem, kind="stable")
    elem, terms = elem[order], terms[order]
    bounds = np.searchsorted(elem, np.arange(n_cells + 1))
    ref = np.array([math.fsum(terms[bounds[e]:bounds[e + 1]]) for e in range(n_cells)]) / n_azim_2
    return ref, np.diff(bounds)


def first_segments(offsets, max_iter):
    """mask of the first min(max_iter, n_u) segments of every track"""
    counts = np.diff(offsets)
    pos = np.arange(int(offsets[-1])) - np.repeat(offsets[:-1], counts)
    return pos < max_iter


def assert_volumes_exact(v, ref, counts):
    """|v - ref| <= (2 m_e + 2) 2^-53 ref for every element e with m_e terms: the terms are positive, so this bounds any order of
    summation plus the division; an element no segment crosses is exactly 0.  One dropped or duplicated term anywhere fails."""
    v = np.asarray(v)
    assert v.shape == ref.shape
    tol = (2.0 * counts + 2.0) * 2.0 ** -53 * ref
    bad = np.nonzero(np.abs(v - ref) > tol)[0]
    assert bad.size == 0, f"{bad.size} elements off, e.g. element {bad[0] + 1}: {v[bad[0]]!r} vs {ref[bad[0]]!r} ({counts[bad[0]]} terms)"
    assert np.all(v[counts == 0] == 0.0)


def test_reference_volumes_match_oracle_volumes(pincell_model):
    """the reference against the oracle's own sequential fill_volumes, within the same per-element bound; and the bound is tight
    enough to see one missing term, and max_iter above every track's count changes nothing"""
    for model, n_azim, delta in ((pincell_model, 8, 0.02), (rt.synth.jittered_triangle_mesh(40, 40, seed=11), 16, 0.01)):
        otg = OracleTrackGenerator(OracleMesh.from_mesh(rt.Mesh(model)), n_azim, delta).trace().segmentize(check=False, nthreads=8)
        ref, m = reference_volumes(otg, otg.seg_offsets, otg.seg, otg.n2)
        assert m.sum() == otg.n_segments and (m > 0).mean() > 0.99
        assert_volumes_exact(otg.volumes(), ref, m)
        ref2, m2 = reference_volumes(otg, otg.seg_offsets, otg.seg, otg.n2, max_iter=int(np.diff(otg.seg_offsets).max()))
        assert np.array_equal(ref2, ref) and np.array_equal(m2, m)
        capped, mc = reference_volumes(otg, otg.seg_offsets, otg.seg, otg.n2, max_iter=3)
        assert mc.sum() == np.minimum(np.diff(otg.seg_offsets), 3).sum() and np.all(capped <= ref)
        u = int(np.argmax(np.diff(otg.seg_offsets)))  # drop the largest term of one element
        s = otg.seg_offsets[u]
        e = otg.seg["element"][s] - 1
        short = ref.copy()
        short[e] -= otg.deltas[otg.tracks["azim_idx"][u] - 1] * otg.seg["len"][s] / otg.n2
        with pytest.raises(AssertionError):
            assert_volumes_exact(short, ref, m)


# ---- GPU cases ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def built():
    rt.build()


class Case:
    def __init__(self, model, n_azim, delta):
        self.mesh = rt.Mesh(model)
        self.n_azim, self.delta = n_azim, delta
        self.otg = OracleTrackGenerator(OracleMesh.from_mesh(self.mesh), n_azim, delta).trace().segmentize(check=False, nthreads=8)
        self.ref, self.m = reference_volumes(self.otg, self.otg.seg_offsets, self.otg.seg, self.otg.n2)


@pytest.fixture(scope="module")
def cases(pincell_model):
    """oracle runs shared by the tests of this module (the oracle does not depend on any knob)"""
    specs = {
        # n_azim = 64: the first angles lie within 3 degrees of the axes, so the boundary-band rules of the chunk plan apply
        "jittered70": (lambda: rt.synth.jittered_triangle_mesh(70, 70, seed=31), 64, 0.01),
        "structured70": (lambda: rt.synth.jittered_triangle_mesh(70, 70, jitter=0.0), 64, 0.01),  # through vertices, along edges
        "jittered60": (lambda: rt.synth.jittered_triangle_mesh(60, 60, seed=5), 16, 0.01),
        "pincell": (lambda: pincell_model, 16, 0.02),
    }
    done = {}

    def get(name):
        if name not in done:
            make, n_azim, delta = specs[name]
            done[name] = Case(make(), n_azim, delta)
        return done[name]

    return get


def make_tg(case, chunk=CHUNK, **options):
    tg = rt.TrackGenerator(case.mesh, case.n_azim, case.delta)
    rt.trace_(tg)
    if chunk:
        tg.set_option("chunk_segments", chunk)
        tg.set_option("target_walkers", 1e9)
    for name, value in options.items():
        tg.set_option(name, value)
    return tg


def check_call(case, tg, flags=0):
    """one segmentize! on tg: the oracle's bits, exact volumes, no fall-back"""
    rt.segmentize_(tg, flags=flags, check=False)
    assert_segments_equal(case.otg, tg)
    assert_volumes_exact(tg.volumes, case.ref, case.m)
    assert tg.info("verify_fallbacks") == 0


def collect_batches(tg, flags=0):
    """segmentize! with an on_batch that copies EVERY batch of the stream (rt_set_segment_capacity) into whole columns"""
    import torch

    got, cuts = {}, []

    def on_batch(b):
        assert b.attempt == 0
        torch.cuda.synchronize()
        for k in KEYS:
            col = torch.as_tensor(getattr(b, k), device="cuda")[:b.n_segments].cpu().numpy()
            got.setdefault(k, []).append((b.offset_base, col))
        cuts.append((b.uid_begin, b.uid_end, b.n_segments))

    rt.segmentize_(tg, flags=flags, check=False, on_batch=on_batch)
    out = {}
    for k, parts in got.items():
        a = np.zeros(tg.n_segments, parts[0][1].dtype)
        for base, col in parts:
            a[base:base + col.size] = col
        out[k] = a
    assert cuts[0][0] == 1 and cuts[-1][1] == tg.n_total_tracks + 1 and all(a[1] == b[0] for a, b in zip(cuts, cuts[1:]))
    assert sum(c[2] for c in cuts) == tg.n_segments
    return out, cuts


def check_batched(case, tg, flags=0, volumes=True):
    cols, cuts = collect_batches(tg, flags)
    otg = case.otg
    assert len(cuts) > 2
    assert tg.n_segments == otg.n_segments and np.array_equal(tg.segment_offsets, otg.seg_offsets)
    assert np.array_equal(tg.segment_status, otg.seg_status) and (tg.first_bad_uid, tg.bad_status) == (otg.first_bad_uid, otg.bad_status)
    for k in KEYS:
        assert np.array_equal(cols[k], otg.seg[k]), k
    if volumes:
        assert_volumes_exact(tg.volumes, case.ref, case.m)
    assert tg.info("verify_fallbacks") == 0


def plan_shape(tg):
    st = tg.chunk_stats()
    return (st["slots"], st["units"], st["working_chunks"])


# ---- every result-neutral knob -------------------------------------------------------------------------------------------
KNOBS = [("order_grid", 0), ("order_grid", 1), ("order_grid", 3), ("order_grid", 256), ("order_classes", 0), ("order_classes", 1),
         ("order_classes", 64), ("band_chunks", 0), ("band_min", 0), ("band_min", 1e9), ("band_div", 1), ("band_div", 64),
         ("plan_cache", 0), ("optimistic", 0), ("chunk_segments", 1), ("chunk_segments", 1e6)]


@pytest.mark.gpu
@pytest.mark.parametrize("mesh", ["jittered70", "structured70"])
@pytest.mark.parametrize("name,value", KNOBS)
def test_result_neutral_knob_matches_oracle(built, cases, mesh, name, value):
    """A knob of rt_set_option off its default, with the single-walk (3) and the hybrid (0) pipeline -- and the sequential kernels
    for the chunk-plan knobs: the oracle's bits and exact volumes every time.  Each case also checks that the knob took effect:
    the band knobs change the chunk plan, one segment per chunk leaves void seeds, a million leaves one chunk per track, no plan
    cache costs launches in a repeated call, no optimistic evaluation means no cancelled one.  The launch order (order_grid,
    order_classes; 0 gives the identity order, or reuses the walk's order for the evaluation) cannot be observed through the
    ABI: those cases rest on bit-exact equality alone."""
    case = cases(mesh)
    # (the band is one longest mesh edge wide: with 12-segment chunks every track end is longer than the default band_min already,
    # so band_min = 0 only changes the plan of longer chunks)
    chunk = 100 if (name, value) == ("band_min", 0) else CHUNK
    tg = make_tg(case, chunk=chunk, **{name: value})
    plan_knob = name.startswith("band") or name == "chunk_segments"
    for pipeline, flags in [(3, 0), (0, 0)] + ([(3, SEQ)] if plan_knob else []):
        tg.set_option("pipeline", pipeline)
        check_call(case, tg, flags)
    assert_tracks_equal(case.otg, tg)
    tg.set_option("pipeline", 3)
    rt.segmentize_(tg, check=False)
    st = tg.chunk_stats()
    n_blocks = (tg.n_total_tracks + 31) // 32
    if name.startswith("band"):
        base = make_tg(case, chunk=chunk)
        rt.segmentize_(base, check=False)
        assert plan_shape(tg) != plan_shape(base)
    elif name == "chunk_segments" and value == 1:
        assert st["void_seeds"] > 0 and st["units"] > n_blocks
    elif name == "chunk_segments":
        assert st["units"] == n_blocks and st["void_seeds"] == 0
    elif name == "plan_cache":
        base = make_tg(case, pipeline=3)
        rt.segmentize_(base, check=False)
        launches = []
        for g in (tg, base):  # the second of two identical calls
            rt.segmentize_(g, check=False)
            launches.append(g.stats()["launches"])
        assert launches[0] > launches[1]  # the plan kernels ran again
    elif name == "optimistic":
        # a first call with 3 segments per track sizes the Segment columns for them; a full call then does not fit: with the
        # optimistic evaluation on it is cancelled on the device and repeated, with it off it is never launched
        cancels = []
        for g in (make_tg(case, optimistic=0), make_tg(case)):
            rt.segmentize_(g, max_iter=3, check=False)
            rt.segmentize_(g, max_iter=3, check=False)
            assert np.array_equal(g.segment_offsets, np.concatenate([[0], np.cumsum(np.minimum(np.diff(case.otg.seg_offsets), 3))]))
            check_call(case, g)
            cancels.append(g.info("optimistic_cancels"))
        assert cancels == [0, 1]


# ---- the chunk plan kept between calls ------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_plan_cache_across_calls_on_one_context(built, cases):
    """One context, chunks of ~3 segments (void seeds): the plan is reused across pipelines (the per-chunk slots then hold what
    the previous pipeline left there), rebuilt when a key changes (no chunks, band_div, order_grid, a new trace!) and reused again
    when it changes back; a batched call in between.  Every call gives the oracle's bits and exact volumes."""
    case = cases("jittered70")
    tg = make_tg(case, chunk=3)
    n_blocks = (tg.n_total_tracks + 31) // 32

    def shape():
        st = tg.chunk_stats()
        return (st["slots"], st["units"], st["void_seeds"], st["working_chunks"])

    def call(flags=0):
        check_call(case, tg, flags)
        assert tg.info("optimistic_cancels") == 0  # the columns never shrink and every call has the same total
        return shape(), tg.stats()["launches"]

    runs = []
    for pipeline in (3, 0, 1, 3):  # same key: the plan is reused
        tg.set_option("pipeline", pipeline)
        runs.append(call())
    plan = runs[0][0]
    assert plan[2] > 0 and all(r[0] == plan for r in runs)
    assert runs[3][1] < runs[0][1]  # no plan kernels in the repeated pipeline-3 call
    s, _ = call(NO_CHUNKS)  # chunk_len is part of the key
    assert s[1] == n_blocks and s[2] == 0
    assert call()[0] == plan
    tg.set_option("band_div", 64)
    assert call()[0][:2] != plan[:2]
    tg.set_option("band_div", 8)
    assert call()[0] == plan
    for grid in (0, 32):
        tg.set_option("order_grid", grid)
        assert call()[0] == plan
    rt.trace_(tg)  # a new trace generation
    assert call()[0] == plan
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, 20000))
    check_batched(case, tg)
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, 0))
    assert call()[0] == plan
    for pipeline in (0, 3):  # ... and once more across pipelines after all that
        tg.set_option("pipeline", pipeline)
        assert call()[0] == plan


# ---- RT_SEG_COUNT_ONLY ----------------------------------------------------------------------------------------------------
def expected_capped(otg, max_iter):
    """offsets, the segment mask and the status of tracks whose count can be predicted, for a call capped at max_iter"""
    counts = np.diff(otg.seg_offsets)
    capped = np.minimum(counts, max_iter)
    off = np.concatenate([[0], np.cumsum(capped)])
    sure = counts != max_iter  # (a track of exactly max_iter segments that then fails: the length check decides)
    status = np.where(counts > max_iter, 2, otg.seg_status)  # truncated tracks fail the length check (src/track.jl:171-175)
    return off, first_segments(otg.seg_offsets, max_iter), sure, status


def check_full_call(case, tg, max_iter):
    otg = case.otg
    if max_iter is None:
        assert_segments_equal(otg, tg)
        assert_volumes_exact(tg.volumes, case.ref, case.m)
        return
    off, keep, sure, status = expected_capped(otg, max_iter)
    assert tg.n_segments == off[-1] and np.array_equal(tg.segment_offsets, off)
    assert np.array_equal(tg.segment_status[sure], status[sure])
    bad = np.nonzero(tg.segment_status)[0]
    assert bad.size > 0 and (tg.first_bad_uid, tg.bad_status) == (bad[0] + 1, tg.segment_status[bad[0]])
    s = tg.segments
    for k in KEYS:
        assert np.array_equal(s[k], otg.seg[k][keep]), k
    assert_volumes_exact(tg.volumes, *reference_volumes(otg, otg.seg_offsets, otg.seg, otg.n2, max_iter))


COUNT_CASES = [("pincell", None, 3, 0), ("pincell", None, 3, LIT), ("jittered60", None, 3, 0), ("jittered60", None, 0, 0),
               ("jittered60", 5, 3, 0), ("jittered60", 5, 0, 0), ("jittered60", 5, 3, LIT)]


@pytest.mark.gpu
@pytest.mark.parametrize("max_iter", [None, 10])
@pytest.mark.parametrize("mesh,chunk,pipeline,flags", COUNT_CASES)
def test_count_only(built, cases, mesh, chunk, pipeline, flags, max_iter):
    """RT_SEG_COUNT_ONLY (the sequential count walk whatever the pipeline): the counts, offsets and status of the full call, no
    Segment records, and the volumes of exactly the segments the full call produces -- also with max_iter below the tracks'
    segment counts and with chunked tracks, where a chunk must not add the segments the per-track fix-up drops.  The full
    call after it (optimistic evaluation) is still bit-exact."""
    case = cases(mesh)
    otg = case.otg
    tg = make_tg(case, chunk=chunk, pipeline=pipeline)
    kw = {} if max_iter is None else {"max_iter": max_iter}
    rt.segmentize_(tg, flags=flags, check=False, **kw)
    check_full_call(case, tg, max_iter)
    full = (tg.n_segments, tg.segment_offsets.copy(), tg.segment_status.copy(), tg.first_bad_uid, tg.bad_status)
    rt.segmentize_(tg, flags=flags | COUNT, check=False, **kw)
    assert (tg.n_segments, tg.first_bad_uid, tg.bad_status) == (full[0], full[3], full[4])
    assert np.array_equal(tg.segment_offsets, full[1]) and np.array_equal(tg.segment_status, full[2])
    if max_iter is None:
        assert tg.n_segments == otg.n_segments and np.array_equal(tg.segment_offsets, otg.seg_offsets)
        assert np.array_equal(tg.segment_status, otg.seg_status) and (tg.first_bad_uid, tg.bad_status) == (otg.first_bad_uid, otg.bad_status)
    assert tg.resident_batch()[3] == 0
    assert all(tg.segments[k].shape == (0,) for k in KEYS)
    assert_volumes_exact(tg.volumes, *reference_volumes(otg, otg.seg_offsets, otg.seg, otg.n2, max_iter))
    rt.segmentize_(tg, flags=flags, check=False, **kw)
    check_full_call(case, tg, max_iter)
    assert tg.info("verify_fallbacks") == 0


# ---- RT_SEG_NO_VOLUMES ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("capacity", [0, 20000])
@pytest.mark.parametrize("pipeline", [3, 0, 1])
def test_no_volumes(built, cases, pipeline, capacity):
    """RT_SEG_NO_VOLUMES between two calls with volumes: the same segments; no volumes to read or to correct with; and the next
    call's accumulator starts from zero again (pipeline 3 clears it in k_seed, the two-pass pipelines with a memset)."""
    case = cases("jittered60")
    tg = make_tg(case, chunk=7, pipeline=pipeline)
    if capacity:
        L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, capacity))

    def run(flags=0):
        if capacity:
            check_batched(case, tg, flags, volumes=not flags & NO_VOL)
        elif flags & NO_VOL:
            rt.segmentize_(tg, flags=flags, check=False)
            assert_segments_equal(case.otg, tg)
            assert tg.info("verify_fallbacks") == 0
        else:
            check_call(case, tg, flags)

    run()
    run(NO_VOL)
    buf = np.zeros(case.mesh.num_cells)
    assert L.lib().rt_volumes(tg._ctx, L.ptr(buf)) == RT_ERR_ARG
    assert L.lib().rt_correct_volumes(tg._ctx, None, None) == RT_ERR_ARG
    with pytest.raises(rt.RTError):
        tg.correct_volumes()
    run()
    run()


# ---- rt_set_option refuses what it cannot use ------------------------------------------------------------------------------
REJECTED = [("order_grid", 257), ("order_classes", 65), ("band_div", 0.5), ("band_div", 65), ("chunk_segments", 0.5), ("band_min", -1),
            ("pipeline", 2), ("no_such_option", 1.0)] + \
           [(name, math.nan) for name in ("chunk_segments", "target_walkers", "order_grid", "order_classes", "pipeline", "band_min",
                                          "band_div", "band_cost", "pool_slots", "pool_extra")]


@pytest.mark.gpu
def test_set_option_rejects_out_of_range_values(built, cases):
    """Every out-of-range or NaN value (and an unknown name) is refused with RT_ERR_ARG and leaves the option as it was: the
    next call has the chunk plan of a context that never saw them, and the oracle's bits."""
    case = cases("jittered60")
    tg = make_tg(case)
    for name, value in REJECTED:
        with pytest.raises(rt.RTError) as err:
            tg.set_option(name, value)
        assert err.value.code == RT_ERR_ARG, (name, value)
    check_call(case, tg)
    fresh = make_tg(case)
    check_call(case, fresh)
    assert tg.chunk_stats() == fresh.chunk_stats()
    assert tg.stats()["launches"] == fresh.stats()["launches"]
