"""The volume path of a context with an NCCL communicator, on one GPU.  A one-rank communicator (rt_comm_unique_id + rt_comm_init
with the NCCL that torch loads) takes every branch the multi-GPU path has, without a second process:
- the two accumulators b_vol / b_vol_alt that alternate from call to call, each waiting for the collective of two calls ago;
- the all-reduce of rt_volumes and the normalisation behind it, both on the collective stream;
- the volume correction, resident and inside on_batch, that waits for a collective still in flight;
- the failed-rank flag in the extra element n_cells of the accumulator, and its clearing by the next call;
- a rank whose on_batch raises, which must still join the call's all-reduce.
tests/test_multi_gpu.py covers two ranks, on a box with two GPUs.

Every fetched result is compared with the exactly summed reference of THAT call (tests.test_gpu_knobs_flags.reference_volumes).
Neighbouring calls of a sequence differ in max_iter, and the tests check that their references are told apart by the bound, so a
result one or two calls stale fails.  rt_info(ctx, "collectives") counts the all-reduces: one per segmentize! with volumes,
whatever failed, plus one per extra rt_volumes."""
import ctypes as C
import types

import numpy as np
import pytest

import raytracing_jl_b200 as rt
from raytracing_jl_b200 import _lib as L
from oracle.oracle import OracleMesh, OracleTrackGenerator
from tests.test_gpu_knobs_flags import KEYS, assert_volumes_exact, reference_volumes
from tests.test_gpu_sweep_outputs import assert_corrected_volumes, corrected_volumes, numpy_areas, numpy_factors

pytestmark = pytest.mark.gpu

NO_VOL, COUNT = rt.RT_SEG_NO_VOLUMES, rt.RT_SEG_COUNT_ONLY
RT_ERR_ARG, RT_ERR_NCCL = -2, -9
U = 2.0 ** -53  # unit roundoff of float64
PIPELINES = [3, 0, 1]
MAX_ITERS = (None, 3, 5, 7)  # None: the full walk
MESHES = {
    "pincell": (lambda pincell: pincell, 16, 0.02),  # 3910 cells
    # 2048 cells, a multiple of 256: the flag element n_cells is the first slot of a block of its own
    "jittered32": (lambda pincell: rt.synth.jittered_triangle_mesh(32, 32, seed=29), 16, 0.01),
    "coarse": (lambda pincell: pincell, 4, 0.8),  # 8 tracks: a split into more parts than tracks has empty shards
}


# ---- references -------------------------------------------------------------------------------------------------------------
class Case:
    """one mesh: the oracle's segments, the cell areas and the exact volume reference of every max_iter of MAX_ITERS"""

    def __init__(self, model, n_azim, delta):
        self.model, self.mesh = model, rt.Mesh(model)
        self.n_azim, self.delta = n_azim, delta
        otg = OracleTrackGenerator(OracleMesh.from_mesh(self.mesh), n_azim, delta).trace().segmentize(check=False, nthreads=8)
        self.otg = otg
        self.refs = {mi: reference_volumes(otg, otg.seg_offsets, otg.seg, otg.n2, mi) for mi in MAX_ITERS}
        self.area = numpy_areas(model)

    def n_segments(self, max_iter):
        counts = np.diff(self.otg.seg_offsets)
        return int(counts.sum() if max_iter is None else np.minimum(counts, max_iter).sum())

    def told_apart(self, a, b):
        """share of the elements crossed by call a or call b (max_iter a, b) where the two references differ by more than the
        sum of their bounds (assert_volumes_exact): there the volumes of one call fail the check against the other's reference"""
        (ra, ma), (rb, mb) = self.refs[a], self.refs[b]
        crossed = (ma > 0) | (mb > 0)
        apart = np.abs(ra - rb) > (2.0 * ma + 2.0) * U * ra + (2.0 * mb + 2.0) * U * rb
        return np.count_nonzero(crossed & apart) / np.count_nonzero(crossed)


@pytest.fixture(scope="module")
def cases(pincell_model):
    """the oracle runs once per mesh for the whole module"""
    done = {}

    def get(name):
        if name not in done:
            make, n_azim, delta = MESHES[name]
            done[name] = Case(make(pincell_model), n_azim, delta)
        return done[name]

    return get


def assert_factors(f, area, ref, m):
    """factors f = fl(area / V) of volumes V that assert_volumes_exact accepts against (ref, m): V = ref (1 + e) with
    |e| <= (2m + 2) u, and the division adds u, so |f ref - area| <= ((2m + 2) u + 2u) area (one u to spare for the product in
    this check and the second-order terms); f is exactly 1 where no track crosses the element (m = 0)."""
    crossed = m > 0
    tol = ((2.0 * m + 2.0) * U + 2.0 * U) * area
    bad = np.nonzero(crossed & (np.abs(f * ref - area) > tol))[0]
    assert bad.size == 0, f"{bad.size} factors off, e.g. element {bad[0] + 1}: {f[bad[0]]!r} * {ref[bad[0]]!r} vs area {area[bad[0]]!r}"
    assert np.all(f[~crossed] == 1.0)


# ---- contexts with a one-rank communicator ------------------------------------------------------------------------------------
def attach_comm(tg):
    """a one-rank NCCL communicator on tg's context.  RT_ERR_NCCL (no libnccl.so.2 to dlopen) skips only on a torch build without
    NCCL: wherever torch has NCCL, the library must find it."""
    import torch.distributed as dist

    buf = C.create_string_buffer(128)
    rc = L.lib().rt_comm_unique_id(tg._ctx, buf)
    if rc == RT_ERR_NCCL and not (dist.is_available() and dist.is_nccl_available()):
        pytest.skip("this torch build has no NCCL")
    L.check(tg._ctx, rc)
    L.check(tg._ctx, L.lib().rt_comm_init(tg._ctx, 1, 0, buf.raw))
    tg._has_comm = True


@pytest.fixture
def make_tg(request):
    """TrackGenerator factory: traced, with a one-rank communicator unless comm=False.  Every TrackGenerator is closed at the end
    of the test: rt_destroy waits for the collective stream and destroys the communicator, so no NCCL work outlives the test."""
    import torch  # noqa: F401 -- loads the NCCL that ships with torch, which the library's dlopen("libnccl.so.2") then finds

    rt.build()
    made = []
    request.addfinalizer(lambda: [tg.close() for tg in made])

    def make(case, pipeline=None, comm=True, **kw):
        tg = rt.TrackGenerator(case.mesh, case.n_azim, case.delta, **kw)
        made.append(tg)
        if comm:
            attach_comm(tg)
        rt.trace_(tg)
        if pipeline is not None:
            tg.set_option("pipeline", pipeline)
        return tg

    return make


def set_capacity(tg, n):
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, n))


def call(tg, case, max_iter=None, flags=0, fetch=True, **kw):
    """one segmentize! on tg.  With volumes: exactly one more collective if tg has a communicator, and -- when fetched -- volumes
    that pass assert_volumes_exact against the reference of this call's max_iter (tg.volumes is poisoned first, so a copy that
    did not happen fails too).  Without: no collective.  Returns the max_iter of a call with volumes, None otherwise."""
    before = tg.info("collectives")
    if fetch:
        tg.volumes[:] = np.nan
    kept = tg.volumes.copy()
    rt.segmentize_(tg, flags=flags, check=False, fetch_volumes=fetch, **({} if max_iter is None else {"max_iter": max_iter}), **kw)
    assert tg.n_segments == case.n_segments(max_iter)
    if flags & NO_VOL:
        assert tg.info("collectives") == before
        return None
    assert tg.info("collectives") == before + getattr(tg, "_has_comm", False)
    if fetch:
        assert_volumes_exact(tg.volumes, *case.refs[max_iter])
    else:
        assert np.array_equal(tg.volumes, kept)  # (the collective is left in flight; nothing is copied)
    return max_iter


# ---- 1. a call sequence on one context --------------------------------------------------------------------------------------
@pytest.mark.parametrize("pipeline", PIPELINES)
@pytest.mark.parametrize("mesh", ["pincell", "jittered32"])
def test_call_sequence_on_one_context(cases, make_tg, mesh, pipeline):
    """One context, calls of different max_iter, so that every fetched result is checked against the reference of its own call:
    - max_iter 3 right after trace! (the careful path; it sizes the Segment columns for 3 segments per track);
    - max_iter 7, which does not fit those columns: pipeline 3's optimistic evaluation is cancelled and repeated, without adding
      its sums twice;
    - the full walk with fetch_volumes=False (its collective stays in flight), then max_iter 5, whose buffer and collective are
      its own;
    - RT_SEG_NO_VOLUMES (no buffer switch, no collective), then RT_SEG_COUNT_ONLY with volumes and max_iter 3;
    - a batched full call (segment capacity 1/6 of the total);
    - pipelines 3 and 0: max_iter 7 with a failed verification, whose sequential restart clears the accumulator again;
    - rt_volumes once more for the last call: bit-identical, since a one-rank all-reduce is a copy.
    Then the count of collectives is that of the calls with volumes plus the repeat."""
    case = cases(mesh)
    tg = make_tg(case, pipeline=pipeline)
    planned = [3, 7, None, 5, 3, None] + ([7] if pipeline in (3, 0) else [])
    for i in range(1, len(planned)):  # a result one or two calls stale fails its check
        for j in (i - 1, i - 2):
            if j >= 0:
                assert planned[i] != planned[j] and case.told_apart(planned[i], planned[j]) > 0.5, (planned[i], planned[j])
    assert case.refs[None][1][-1] > 0  # (the last element is crossed: a normalisation one element short shows)

    done = [call(tg, case, 3)]
    cancels = tg.info("optimistic_cancels")
    done.append(call(tg, case, 7))
    assert tg.info("optimistic_cancels") == cancels + (pipeline == 3)
    done.append(call(tg, case, None, fetch=False))
    done.append(call(tg, case, 5))
    assert call(tg, case, None, flags=NO_VOL) is None
    done.append(call(tg, case, 3, flags=COUNT))
    assert tg.resident_batch()[3] == 0
    set_capacity(tg, case.otg.n_segments // 6 + 1)
    batches = []
    done.append(call(tg, case, None, on_batch=lambda b: batches.append(b.n_segments)))
    assert len(batches) >= 6 and sum(batches) == case.otg.n_segments
    set_capacity(tg, 0)
    assert tg.info("verify_fallbacks") == 0
    if pipeline in (3, 0):
        tg.set_option("debug_verify_fail", 1)
        done.append(call(tg, case, 7))
        assert tg.info("verify_fallbacks") == 1
        tg.set_option("debug_verify_fail", 0)
    assert done == planned
    first = tg.volumes.copy()
    again = np.full(case.mesh.num_cells, np.nan)
    L.check(tg._ctx, L.lib().rt_volumes(tg._ctx, L.ptr(again)))
    assert np.array_equal(again.view(np.uint64), first.view(np.uint64))
    assert tg.info("collectives") == len(planned) + 1


# ---- 2. the failed-rank flag --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pipeline", PIPELINES)
@pytest.mark.parametrize("mesh", ["pincell", "jittered32"])
def test_failed_rank_flag_is_cleared_by_the_next_calls(cases, make_tg, mesh, pipeline):
    """A call that fails joins the collective with a zero contribution and the failed-rank flag in element n_cells of b_vol:
    - k = 33 fails with RT_ERR_ARG before the call starts;
    - the next call's on_batch runs correct_volumes(), which has no volumes to use after a failure: the callback's RT_ERR_ARG
      is raised, and that call joins the collective too;
    - three calls with different max_iter then use both accumulators: each must clear the flag again (k_seed in pipeline 3, the
      memset of the two-pass pipelines), or its volumes are refused with RT_ERR_PEER."""
    case = cases(mesh)
    tg = make_tg(case, pipeline=pipeline)
    call(tg, case, 5)
    n = tg.info("collectives")
    with pytest.raises(rt.RTError) as err:
        rt.segmentize_(tg, k=33, check=False)
    assert err.value.code == RT_ERR_ARG and tg.info("collectives") == n + 1

    def correct(b):
        tg.correct_volumes()

    with pytest.raises(rt.RTError) as err:
        rt.segmentize_(tg, check=False, on_batch=correct)
    assert err.value.code == RT_ERR_ARG and "inside a batch callback" in err.value.msg
    assert tg.info("collectives") == n + 2
    for max_iter in (3, 7, None):
        call(tg, case, max_iter)
    assert tg.info("collectives") == n + 5


# ---- 3. on_batch raises ---------------------------------------------------------------------------------------------------------
class Stop(Exception):
    pass


class CountingLib:
    """the loaded library with its rt_volumes calls recorded"""

    def __init__(self, lib):
        self._lib, self.volumes_calls = lib, []

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def rt_volumes(self, ctx, volumes):
        self.volumes_calls.append(volumes)
        return self._lib.rt_volumes(ctx, volumes)


@pytest.mark.parametrize("pipeline", PIPELINES)
@pytest.mark.parametrize("comm", [True, False], ids=["comm", "no_comm"])
def test_raising_on_batch_joins_the_collective(cases, make_tg, monkeypatch, pipeline, comm):
    """on_batch raises in the second batch: segmentize_ raises that exception.  With a communicator the call first joins the
    all-reduce (one rt_volumes without a host pointer, one more collective), as any failed call does -- unless the call ran
    without volumes.  Without a communicator there is nothing to join and rt_volumes is not called.  The next three calls are
    exact."""
    case = cases("jittered32")
    tg = make_tg(case, pipeline=pipeline, comm=comm)
    call(tg, case, 5)
    lib = CountingLib(L.lib())
    monkeypatch.setattr(L, "_lib", lib)
    seen = []

    def stop(b):
        seen.append(b.n_segments)
        if len(seen) == 2:
            raise Stop

    set_capacity(tg, case.otg.n_segments // 6 + 1)
    n = tg.info("collectives")
    for flags in (0, NO_VOL):
        seen.clear()
        with pytest.raises(Stop):
            rt.segmentize_(tg, flags=flags, check=False, on_batch=stop)
        assert len(seen) == 2
    assert lib.volumes_calls == ([None] if comm else [])
    assert tg.info("collectives") == n + comm
    set_capacity(tg, 0)
    for max_iter in (3, 7, None):
        call(tg, case, max_iter)


# ---- 4. the resident correction -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fetch", [True, False], ids=["fetch", "in_flight"])
@pytest.mark.parametrize("mesh", ["pincell", "jittered32"])
def test_resident_correction(cases, make_tg, mesh, fetch):
    """volume_correction = true after a call of another max_iter: the factors come from this call's all-reduced volumes -- with
    fetch_volumes=False the correction waits for the event of a collective that may still be running.  Factors within
    assert_factors' bound of the exact reference (bit-equal to area / v when the volumes v were fetched), corrected lengths
    bit-equal to the oracle's len * f[element], end points and elements untouched, and the traced volumes of the corrected
    lengths equal to the areas within assert_corrected_volumes' bound."""
    case = cases(mesh)
    otg = case.otg
    tg = make_tg(case, volume_correction=True)
    call(tg, case, 7)
    call(tg, case, None, fetch=fetch)
    f = tg.volume_factors
    assert f is not None
    ref, m = case.refs[None]
    assert_factors(f, case.area, ref, m)
    if fetch:
        assert np.array_equal(f, numpy_factors(case.area, tg.volumes))
    s = tg.segments
    assert np.array_equal(s["len"], otg.seg["len"] * f[otg.seg["element"] - 1])
    for k in KEYS:
        if k != "len":
            assert np.array_equal(s[k], otg.seg[k]), k
    w, mw = corrected_volumes(otg, s["len"])
    assert_corrected_volumes(w, case.area, mw)


# ---- 5. the correction inside on_batch, behind a collective in flight --------------------------------------------------------------
@pytest.mark.parametrize("flags", [0, NO_VOL], ids=["volumes", "no_volumes"])
@pytest.mark.parametrize("pipeline", PIPELINES)
def test_correction_inside_on_batch_behind_a_collective_in_flight(cases, make_tg, pipeline, flags):
    """A full call, then call A (max_iter 7, fetch_volumes=False: its collective is left in flight), then a batched full call B
    whose on_batch corrects every batch.  The factors come from A's volumes: the same bits in every batch, within
    assert_factors' bound of A's reference and NOT of the full walk's (the two are told apart: factors from the volumes of the
    call before A, or from B's own, fail).  Every batch's lengths are the oracle's len * f[element] bit for bit."""
    case = cases("pincell")
    otg = case.otg
    tg = make_tg(case, pipeline=pipeline)
    call(tg, case, None)
    call(tg, case, 7, fetch=False)
    set_capacity(tg, otg.n_segments // 6 + 1)
    factors, cuts = [], []

    def on_batch(b):
        f = tg.correct_volumes()
        sl = slice(b.offset_base, b.offset_base + b.n_segments)
        assert np.array_equal(tg.fetch_segments()["len"], otg.seg["len"][sl] * f[otg.seg["element"][sl] - 1])
        factors.append(f)
        cuts.append(b.n_segments)

    call(tg, case, None, flags=flags, on_batch=on_batch)
    assert len(cuts) >= 6 and sum(cuts) == otg.n_segments and tg.info("verify_fallbacks") == 0
    for f in factors[1:]:
        assert np.array_equal(f.view(np.uint64), factors[0].view(np.uint64))
    assert_factors(factors[0], case.area, *case.refs[7])
    with pytest.raises(AssertionError):
        assert_factors(factors[0], case.area, *case.refs[None])


# ---- 6. shards, each with a communicator of its own ----------------------------------------------------------------------------
def shard_reference(otg, uid_begin, uid_end):
    """reference_volumes over the oracle's segments of the uids [uid_begin, uid_end)"""
    part = otg.fetch(uid_begin, uid_end)
    view = types.SimpleNamespace(mesh=otg.mesh, deltas=otg.deltas, tracks={"azim_idx": otg.tracks["azim_idx"][uid_begin - 1:uid_end - 1]})
    return reference_volumes(view, np.concatenate([[0], np.cumsum(part["counts"])]), part, otg.n2)


def test_shards_with_a_communicator_each(cases, make_tg):
    """Three uid shards on one GPU, each with a one-rank communicator of its own: every shard's volumes are exact against the
    reference of its uid range, and their sum is within (2m + 6) u of the whole reference (the shards' sums, two more additions
    and the reference's own two roundings)."""
    case = cases("pincell")
    total = np.zeros(case.mesh.num_cells)
    bounds = []
    for r in range(3):
        tg = make_tg(case, shard=(r, 3))
        assert tg.uid_begin < tg.uid_end
        bounds.append((tg.uid_begin, tg.uid_end))
        tg.volumes[:] = np.nan
        rt.segmentize_(tg, check=False)
        assert tg.info("collectives") == 1
        assert_volumes_exact(tg.volumes, *shard_reference(case.otg, tg.uid_begin, tg.uid_end))
        total += tg.volumes
    assert bounds[0][0] == 1 and bounds[-1][1] == case.otg.n_total_tracks + 1 and all(a[1] == b[0] for a, b in zip(bounds, bounds[1:]))
    ref, m = case.refs[None]
    bad = np.nonzero(np.abs(total - ref) > (2.0 * m + 6.0) * U * ref)[0]
    assert bad.size == 0, f"{bad.size} elements off, e.g. element {bad[0] + 1}: {total[bad[0]]!r} vs {ref[bad[0]]!r}"


def test_empty_shard_with_a_communicator(cases, make_tg):
    """A split of the coarse pin cell's 8 tracks into 12 parts has empty shards: such a shard's call joins the collective and
    gives volumes of exactly 0.0, without an error."""
    case = cases("coarse")
    n_parts = 12
    probe = make_tg(case, comm=False, shard=(0, n_parts))
    empty = [r for r in range(n_parts) if probe.shard_bounds[r] == probe.shard_bounds[r + 1]]
    assert empty
    tg = make_tg(case, shard=(empty[-1], n_parts))
    assert tg.uid_begin == tg.uid_end
    tg.volumes[:] = np.nan
    rt.segmentize_(tg)
    assert tg.n_segments == 0 and tg.info("collectives") == 1
    assert np.array_equal(tg.volumes.view(np.uint64), np.zeros(case.mesh.num_cells, np.uint64))
