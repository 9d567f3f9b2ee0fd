"""RT_SEG_LENGTHS_ONLY: a call that writes only the len and element columns computes what a default call computes -- len, element,
offsets, status, first_bad_uid and volumes are the oracle's (the exact volumes bit for bit) on every mesh kind and pipeline, in
batches, inside batch callbacks, across the verification and pool fall-backs, and on one context alternating with default calls --
and the end points are absent, not wrong: every way to read them says so."""
import numpy as np
import pytest

import raytracing_jl_b200 as rt
from raytracing_jl_b200 import _lib as L
from raytracing_jl_b200.api import DeviceColumn
from oracle.oracle import OracleMesh, OracleTrackGenerator
from tests.test_gpu_exact_volumes import Case, assert_bits, set_capacity
from tests.test_gpu_parity import assert_segments_equal
from tests.test_gpu_sweep_outputs import numpy_areas, numpy_factors

pytestmark = pytest.mark.gpu
LEN_ONLY, COUNT, NO_VOL = rt.RT_SEG_LENGTHS_ONLY, rt.RT_SEG_COUNT_ONLY, rt.RT_SEG_NO_VOLUMES
RT_ERR_ARG = -2
POINT_KEYS = ("px", "py", "qx", "qy")


@pytest.fixture(scope="module")
def cases(pincell_model):
    rt.build()
    done = {}

    def get(name):
        if name not in done:
            done[name] = Case(name, pincell_model)
        return done[name]

    return get


@pytest.fixture
def make_tg(request):
    made = []
    request.addfinalizer(lambda: [tg.close() for tg in made])

    def make(case, pipeline=None, **kw):
        mesh = rt.Mesh(case.model, device_ingest=True) if case.ingest else case.mesh
        tg = rt.TrackGenerator(mesh, case.n_azim, case.delta, **kw)
        made.append(tg)
        rt.trace_(tg)
        if pipeline is not None:
            tg.set_option("pipeline", pipeline)
        return tg

    return make


def lengths_only(tg, **kw):
    tg.volumes[:] = np.nan
    rt.segmentize_(tg, check=False, lengths_only=True, **kw)
    return tg.volumes.copy()


def assert_columns(cols, otg, sl=slice(None)):
    """len and element of a lengths-only download bit-equal to the oracle's, and nothing else in it"""
    assert sorted(cols) == ["element", "len"]
    assert_bits(cols["len"], otg.seg["len"][sl])
    assert np.array_equal(cols["element"], otg.seg["element"][sl])


def assert_same_outcome(otg, tg):
    assert tg.n_segments == otg.n_segments
    assert np.array_equal(tg.segment_offsets, otg.seg_offsets)
    assert np.array_equal(tg.segment_status, otg.seg_status)
    assert (tg.first_bad_uid, tg.bad_status) == (otg.first_bad_uid, otg.bad_status)
    assert_columns(tg.segments, otg)


def assert_volumes_close(ref, v):
    assert np.abs(v - ref).max() <= 1e-10 * np.abs(ref).max()


def batch_slice(otg, b):
    return slice(int(otg.seg_offsets[b.uid_begin - 1]), int(otg.seg_offsets[b.uid_end - 1]))


# ---- the oracle's columns on every mesh kind and pipeline ----------------------------------------------------------------------
@pytest.mark.parametrize("pipeline", [3, 0, 1])
@pytest.mark.parametrize("mesh", ["pincell", "jittered", "bwr", "mixed15", "mixed100", "ingested"])
def test_bit_equal_to_the_oracle(cases, make_tg, mesh, pipeline):
    case = cases(mesh)
    tg = make_tg(case, pipeline)
    rt.segmentize_(tg, check=False)
    default = (tg.first_bad_uid, tg.bad_status)
    assert_volumes_close(case.ref, lengths_only(tg))
    assert (tg.first_bad_uid, tg.bad_status) == default
    assert_same_outcome(case.otg, tg)
    assert_bits(lengths_only(tg, exact_volumes=True), case.ref)
    assert_same_outcome(case.otg, tg)


def test_failing_tracks(cases, make_tg):
    """tracks that fail the length check: the same status, first_bad_uid and bad_status as a default call"""
    case = cases("far")
    tg = make_tg(case)
    rt.segmentize_(tg, check=False)
    default = (tg.first_bad_uid, tg.bad_status, tg.segment_status.copy())
    assert default[1] != 0
    with pytest.raises(rt.RTError) as e:
        rt.segmentize_(tg, lengths_only=True)
    assert e.value.code == -8 and f"uid` {default[0]}" in e.value.msg
    lengths_only(tg)
    assert (tg.first_bad_uid, tg.bad_status) == default[:2] and np.array_equal(tg.segment_status, default[2])
    assert_same_outcome(case.otg, tg)


# ---- batched: the callback's view, optical lengths and the volume correction of every batch ------------------------------------
@pytest.mark.parametrize("pipeline", [3, 0, 1])
def test_batched(cases, make_tg, pipeline):
    case = cases("jittered")
    otg = case.otg
    tg = make_tg(case, pipeline)
    set_capacity(tg, otg.n_segments // 5 + 1)
    sigma = np.stack([np.linspace(0.5, 2.0, case.mesh.num_cells), np.linspace(3.0, 0.1, case.mesh.num_cells)], axis=1)
    seen = []

    def on_batch(b):
        assert (b.px, b.py, b.qx, b.qy) == (None, None, None, None)
        sl = batch_slice(otg, b)
        assert b.n_segments == sl.stop - sl.start
        s = tg.segments
        assert_columns(s, otg, sl)
        with pytest.raises(KeyError, match="RT_SEG_LENGTHS_ONLY"):
            s["px"]
        tau, _ = tg.optical_lengths(sigma)
        el, ln = otg.seg["element"][sl] - 1, otg.seg["len"][sl]
        assert_bits(tau, sigma[el] * ln[:, None])
        seen.append(b.n_segments)

    assert_volumes_close(case.ref, lengths_only(tg, on_batch=on_batch))
    assert len(seen) >= 5 and sum(seen) == otg.n_segments

    # a second lengths-only call corrects every batch with the volumes of the first
    v = tg.volumes.copy()
    want_f = numpy_factors(numpy_areas(case.model), v)
    corrected = []

    def correct(b):
        assert_bits(tg.correct_volumes(), want_f)
        sl = batch_slice(otg, b)
        s = tg.segments
        assert_bits(s["len"], otg.seg["len"][sl] * want_f[otg.seg["element"][sl] - 1])
        assert np.array_equal(s["element"], otg.seg["element"][sl])
        corrected.append(s["len"].copy())

    rt.segmentize_(tg, flags=NO_VOL, check=False, on_batch=correct, lengths_only=True)
    assert len(corrected) >= 5
    assert_bits(np.concatenate(corrected), otg.seg["len"] * want_f[otg.seg["element"] - 1])


def test_volume_correction_flag(cases, make_tg):
    case = cases("jittered")
    tg = make_tg(case, volume_correction=True)
    v = lengths_only(tg, exact_volumes=True)
    assert_bits(v, case.ref)
    f = numpy_factors(numpy_areas(case.model), case.ref)
    assert_bits(tg.volume_factors, f)
    assert_bits(tg.segments["len"], case.otg.seg["len"] * f[case.otg.seg["element"] - 1])


# ---- fall-backs -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batched", [False, True])
@pytest.mark.parametrize("pipeline", [3, 0])
def test_restart_after_failed_verification(cases, make_tg, pipeline, batched):
    case = cases("jittered")
    tg = make_tg(case, pipeline)
    if batched:
        set_capacity(tg, case.otg.n_segments // 4 + 1)
    tg.set_option("debug_verify_fail", 1)
    attempts = []
    assert_bits(lengths_only(tg, exact_volumes=True, on_batch=lambda b: attempts.append(b.attempt)), case.ref)
    assert tg.info("verify_fallbacks") == 1 and attempts[-1] == 1
    if not batched:
        assert_same_outcome(case.otg, tg)


def test_pool_exhaustion_falls_back_to_the_hybrid_pipeline():
    """pipeline 3 whose record pool runs out (no spare blocks, chunks longer than one block) restarts in pipeline 0, whose fill
    walk then writes the lengths-only columns"""
    rt.build()
    model = rt.synth.jittered_triangle_mesh(130, 130, seed=21)
    mesh = rt.Mesh(model)
    otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), 16, 0.004).trace().segmentize(check=False, nthreads=8)
    tg = rt.TrackGenerator(mesh, 16, 0.004)
    try:
        rt.trace_(tg)
        tg.set_option("pipeline", 3)
        tg.set_option("pool_extra", 0)
        tg.set_option("chunk_segments", 700)
        rt.segmentize_(tg, check=False, lengths_only=True, exact_volumes=True)
        assert tg.info("verify_fallbacks") == 1
        assert_same_outcome(otg, tg)
        assert_bits(tg.volumes, otg.volumes())
    finally:
        tg.close()


# ---- one context, both layouts --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("first", ["default", "lengths"])
def test_alternating_layouts_on_one_context(cases, make_tg, first):
    """optimistic evaluation and plan cache on (the defaults): every call is right, a default call after a lengths-only one has
    its end points back, and no optimistic evaluation is cancelled (a call whose layout the columns do not serve skips it)"""
    case = cases("jittered")
    otg = case.otg
    tg = make_tg(case)
    order = ["default", "lengths"] * 3 if first == "default" else ["lengths", "default"] * 3
    for kind in order:
        if kind == "lengths":
            assert_volumes_close(case.ref, lengths_only(tg))
            assert_same_outcome(otg, tg)
            assert tg.info("segment_capacity") >= otg.n_segments
        else:
            tg.volumes[:] = np.nan
            rt.segmentize_(tg, check=False)
            assert_volumes_close(case.ref, tg.volumes)
            assert_segments_equal(otg, tg)
            view = L.rt_batch()
            L.check(tg._ctx, L.lib().rt_segments_device(tg._ctx, view))
            assert all(getattr(view, "d_" + k) for k in POINT_KEYS)
    assert tg.info("optimistic_cancels") == 0


# ---- errors ---------------------------------------------------------------------------------------------------------------------
def test_end_points_are_refused(cases, make_tg):
    case = cases("pincell")
    tg = make_tg(case)
    lengths_only(tg)
    n = tg.n_segments
    col = np.full(n, -1.0)
    lib = L.lib()
    for i in range(4):
        args = [None] * 4
        args[i] = L.ptr(col)
        assert lib.rt_segments_download(tg._ctx, *args, None, None) == RT_ERR_ARG
        assert "RT_SEG_LENGTHS_ONLY" in lib.rt_last_error(tg._ctx).decode()
        assert np.all(col == -1.0)  # (nothing copied)
    # len and element alone
    ln, el = np.zeros(n), np.zeros(n, np.int32)
    L.check(tg._ctx, lib.rt_segments_download(tg._ctx, None, None, None, None, L.ptr(ln), L.ptr(el)))
    assert_bits(ln, case.otg.seg["len"])
    k = L.C.c_int64(0)
    assert lib.rt_segments_download_compact(tg._ctx, None, None, L.ptr(ln), None, 0, None, None, None, L.C.byref(k)) == RT_ERR_ARG
    assert "RT_SEG_LENGTHS_ONLY" in lib.rt_last_error(tg._ctx).decode()
    view = L.rt_batch()
    L.check(tg._ctx, lib.rt_segments_device(tg._ctx, view))
    assert not any(getattr(view, "d_" + k) for k in POINT_KEYS) and view.d_len and view.d_element and view.n_segments == n
    # the Python accessors
    with pytest.raises(KeyError, match="RT_SEG_LENGTHS_ONLY"):
        tg.segments["qx"]
    with pytest.raises(RuntimeError, match="RT_SEG_LENGTHS_ONLY"):
        tg.fetch_segments(compact=True)
    track = tg.tracks_by_uid[1]
    assert len(track.segments) == case.otg.seg_offsets[1] - case.otg.seg_offsets[0]
    with pytest.raises(RuntimeError, match="RT_SEG_LENGTHS_ONLY"):
        track.segments[0]
    assert_columns(tg.fetch_segments(pinned=True), case.otg)


def assert_no_segments(tg):
    """a count-only call leaves no resident segment: both downloads give empty columns"""
    assert tg.resident_batch()[3] == 0
    s = tg.fetch_segments()
    assert all(s[k].shape == (0,) for k in ("px", "py", "qx", "qy", "len", "element"))
    s = tg.fetch_segments(compact=True)
    assert tg.n_exceptions == 0 and all(s[k].shape == (0,) for k in ("qx", "qy", "len", "element"))


@pytest.mark.parametrize("pipeline", [3, 1])
def test_count_only_ignores_the_flag(cases, make_tg, pipeline):
    """also as the first call of a context (no Segment columns allocated yet) and after a lengths-only call (columns without p
    and q): no segments, and nothing to refuse"""
    case = cases("jittered")
    tg = make_tg(case, pipeline)
    for flags in (COUNT | NO_VOL, COUNT):
        rt.segmentize_(tg, flags=flags, check=False)
        assert_no_segments(tg)
        ref = (tg.n_segments, tg.segment_offsets.copy(), tg.segment_status.copy(), tg.volumes.copy())
        rt.segmentize_(tg, flags=flags | LEN_ONLY, check=False)
        assert_no_segments(tg)
        assert tg.n_segments == ref[0] == case.otg.n_segments
        assert np.array_equal(tg.segment_offsets, ref[1]) and np.array_equal(tg.segment_status, ref[2])
        if not flags & NO_VOL:
            assert np.allclose(tg.volumes, ref[3], rtol=1e-12, atol=0.0)
            assert_volumes_close(case.ref, tg.volumes)
    rt.segmentize_(tg, lengths_only=True, check=False)
    rt.segmentize_(tg, flags=COUNT, check=False)
    assert_no_segments(tg)


# ---- size -----------------------------------------------------------------------------------------------------------------------
def test_cfg3_size_equals_a_default_call_on_the_device():
    import torch

    rt.build()
    model, n_azim, delta = rt.synth.workload("cfg3")
    tg = rt.TrackGenerator(rt.Mesh(model), n_azim, delta)

    def columns():
        view = L.rt_batch()
        L.check(tg._ctx, L.lib().rt_segments_device(tg._ctx, view))
        n = int(view.n_segments)
        ln = torch.as_tensor(DeviceColumn(view.d_len, n, "<f8"), device="cuda").clone()
        el = torch.as_tensor(DeviceColumn(view.d_element, n, "<i4"), device="cuda").clone()
        return ln, el

    try:
        rt.trace_(tg)
        rt.segmentize_(tg, rtol=1e-6, check=False)
        ln, el = columns()
        offs = tg.segment_offsets.copy()
        rt.segmentize_(tg, rtol=1e-6, check=False, lengths_only=True)
        ln2, el2 = columns()
        assert tg.n_segments == ln.numel() == ln2.numel() > 4e7
        assert torch.equal(ln.view(torch.int64), ln2.view(torch.int64)) and torch.equal(el, el2)
        assert np.array_equal(tg.segment_offsets, offs)
    finally:
        tg.close()
