"""RT_SEG_EXACT_VOLUMES: the volumes summed in the reference's order (fill_volumes, src/trackgenerator.jl:371-386) are bit-equal to
the oracle's volumes() -- on every mesh kind, pipeline, walk flag and knob, resident and in batches (also across a restart), on a
uid shard, with a one-rank communicator, with failing tracks -- and the flag changes nothing but the volumes.  The reference for a
uid shard is the numpy fold of tests/test_exact_volumes_cpu.py.  Two ranks: tools/check_exact_volumes.py (skipped below two GPUs)."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

import raytracing_jl_b200 as rt
from raytracing_jl_b200 import _lib as L
from oracle.oracle import OracleMesh, OracleTrackGenerator
from tests.test_exact_volumes_cpu import fold_volumes
from tests.test_gpu_comm_volumes import attach_comm
from tests.test_gpu_parity import assert_segments_equal
from tests.test_gpu_sweep_outputs import numpy_areas, numpy_factors

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXACT, COUNT, NO_VOL, NO_CHUNKS, LIT = (rt.RT_SEG_EXACT_VOLUMES, rt.RT_SEG_COUNT_ONLY, rt.RT_SEG_NO_VOLUMES, rt.RT_SEG_NO_CHUNKS,
                                        rt.RT_SEG_LITERAL)
RT_ERR_ARG = -2
KEYS = ("px", "py", "qx", "qy", "len", "element")


def model_of(name, pincell_model):
    if name == "pincell":
        return pincell_model, 16, 0.02
    if name == "jittered":
        return rt.synth.jittered_triangle_mesh(40, 30, 1.3, 0.9, 0.3, 7, x0=-0.4, y0=2.0), 16, 0.01
    if name == "far":  # far from the origin: at rtol = sqrt(eps) ten tracks fail the length check (RT_TRACK_LENGTH)
        return rt.synth.jittered_triangle_mesh(23, 17, 2.5, 1.25, 0.3, 11, x0=1e3, y0=7.5), 16, 0.01
    if name in ("bwr", "ingested"):
        model, n_azim, delta = rt.synth.workload("cfg2")
        return model, n_azim, delta
    if name.startswith("mixed"):
        return rt.synth.mixed_quad_triangle_mesh(31, 23, 1.5, 1.1, jitter=0.22, seed=17, quad_fraction=float(name[5:]) / 100,
                                                 x0=-0.3, y0=0.7), 8, 0.02
    raise ValueError(name)


class Case:
    def __init__(self, name, pincell_model):
        self.model, self.n_azim, self.delta = model_of(name, pincell_model)
        self.ingest = name == "ingested"
        self.mesh = rt.Mesh(self.model)
        self.otg = OracleTrackGenerator(OracleMesh.from_mesh(self.mesh), self.n_azim, self.delta).trace().segmentize(check=False, nthreads=8)
        self.ref = self.otg.volumes()


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

    def make(case, pipeline=None, comm=False, **kw):
        mesh = rt.Mesh(case.model, device_ingest=True) if case.ingest else case.mesh
        tg = rt.TrackGenerator(mesh, case.n_azim, case.delta, **kw)
        made.append(tg)
        if comm:
            attach_comm(tg)
        rt.trace_(tg)
        if pipeline is not None:
            tg.set_option("pipeline", pipeline)
        return tg

    return make


def exact(tg, flags=0, **kw):
    tg.volumes[:] = np.nan
    rt.segmentize_(tg, flags=flags, check=False, exact_volumes=True, **kw)
    return tg.volumes.copy()


def assert_bits(v, ref):
    bad = np.nonzero(v.view(np.int64) != ref.view(np.int64))[0]
    assert bad.size == 0, f"{bad.size} elements differ, e.g. element {bad[0] + 1}: {v[bad[0]]!r} vs {ref[bad[0]]!r}"


def set_capacity(tg, n):
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, int(n)))


# ---- bit equality with the oracle ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pipeline", [3, 0, 1])
@pytest.mark.parametrize("mesh", ["pincell", "jittered", "bwr", "mixed15", "mixed100", "ingested"])
def test_bit_equal_to_the_oracle(cases, make_tg, mesh, pipeline):
    case = cases(mesh)
    tg = make_tg(case, pipeline)
    assert_bits(exact(tg), case.ref)
    assert_segments_equal(case.otg, tg)
    assert tg.info("exact_vol_ms") > 0.0


@pytest.mark.parametrize("flags", [NO_CHUNKS, LIT, NO_CHUNKS | LIT])
@pytest.mark.parametrize("mesh", ["pincell", "jittered"])
def test_walk_flags(cases, make_tg, mesh, flags):
    case = cases(mesh)
    tg = make_tg(case)
    assert_bits(exact(tg, flags), case.ref)
    assert_segments_equal(case.otg, tg)


# ---- reproducible -------------------------------------------------------------------------------------------------------------
def test_same_bits_across_calls_and_knobs(cases, make_tg):
    case = cases("jittered")
    tg = make_tg(case)
    for _ in range(3):
        assert_bits(exact(tg), case.ref)
    for name, values in (("order_grid", (0, 32)), ("chunk_segments", (12, 64, 208)), ("target_walkers", (1e3, 148 * 2048 * 4)),
                         ("plan_cache", (0, 1))):
        for value in values:
            tg.set_option(name, value)
            assert_bits(exact(tg), case.ref)


# ---- batched ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("callback", [None, "download", "tau"])
@pytest.mark.parametrize("batches", [2, 7, "track"])
@pytest.mark.parametrize("pipeline", [3, 0, 1])
def test_batched(cases, make_tg, pipeline, batches, callback):
    case = cases("pincell")
    tg = make_tg(case, pipeline)
    counts = np.diff(case.otg.seg_offsets)
    total = int(counts.sum())
    cap = int(counts.max()) if batches == "track" else max(-(-total // batches), int(counts.max()))
    set_capacity(tg, cap)
    seen = []
    sigma = np.linspace(0.5, 2.0, case.mesh.num_cells)

    def on_batch(b):
        seen.append((b.uid_begin, b.uid_end, b.n_segments))
        if callback == "download":
            s = tg.segments
            lo, hi = case.otg.seg_offsets[b.uid_begin - 1], case.otg.seg_offsets[b.uid_end - 1]
            for k in KEYS:
                assert np.array_equal(s[k], case.otg.seg[k][lo:hi]), k
        elif callback == "tau":
            tau, _ = tg.optical_lengths(sigma[:, None])
            assert tau.shape == (b.n_segments, 1)

    assert_bits(exact(tg, on_batch=on_batch), case.ref)
    assert sum(n for _, _, n in seen) == total
    assert len(seen) >= -(-total // cap) and (batches == "track" or len(seen) >= batches)


@pytest.mark.parametrize("batched", [False, True])
@pytest.mark.parametrize("pipeline", [3, 0])
def test_restart_after_failed_verification(cases, make_tg, pipeline, batched):
    case = cases("jittered")
    tg = make_tg(case, pipeline)
    if batched:
        set_capacity(tg, case.otg.n_segments // 5 + 1)
    tg.set_option("debug_clear_pool", 1)
    tg.set_option("debug_verify_fail", 1)
    attempts = []
    assert_bits(exact(tg, on_batch=lambda b: attempts.append(b.attempt)), case.ref)
    assert tg.info("verify_fallbacks") == 1 and attempts[-1] == 1
    tg.set_option("debug_verify_fail", 0)
    assert_bits(exact(tg), case.ref)


# ---- a uid shard of one context ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("part", [0, 1, 2])
def test_uid_shard(cases, make_tg, part):
    case = cases("jittered")
    tg = make_tg(case, shard=(part, 3))
    v = exact(tg)
    got = case.otg.fetch(tg.uid_begin, tg.uid_end)
    ref = fold_volumes(case.otg, np.concatenate([[0], np.cumsum(got["counts"])]), got, case.mesh.num_cells, tg.uid_begin)
    assert_bits(v, ref)


# ---- a one-rank NCCL communicator ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pipeline", [3, 1])
def test_one_rank_communicator(cases, make_tg, pipeline):
    """the rank-order chain with one rank: no NCCL call ("collectives" unchanged), the same bits resident and batched, and the
    default all-reduce of the next call still counts one collective"""
    case = cases("pincell")
    tg = make_tg(case, pipeline, comm=True)
    before = tg.info("collectives")
    assert_bits(exact(tg), case.ref)
    set_capacity(tg, case.otg.n_segments // 3 + 1)
    assert_bits(exact(tg), case.ref)
    rt.segmentize_(tg, check=False, fetch_volumes=False, exact_volumes=True)  # (left in flight)
    assert_bits(exact(tg), case.ref)
    assert tg.info("collectives") == before
    rt.segmentize_(tg, check=False)
    assert tg.info("collectives") == before + 1
    assert np.allclose(tg.volumes, case.ref, rtol=1e-12, atol=0.0)


# ---- failing tracks -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pipeline", [3, 0, 1])
def test_failing_tracks_contribute(cases, make_tg, pipeline):
    """in one batch and in several: the failing tracks' segments are summed, and the first failing track is the oracle's"""
    case = cases("far")
    assert np.count_nonzero(case.otg.seg_status == 2) > 0
    tg = make_tg(case, pipeline)
    for capacity in (0, case.otg.n_segments // 4 + 1):
        set_capacity(tg, capacity)
        assert_bits(exact(tg), case.ref)
        assert np.array_equal(tg.segment_status, case.otg.seg_status)
        assert (tg.first_bad_uid, tg.bad_status) == (case.otg.first_bad_uid, case.otg.bad_status)


# ---- only the volumes change ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pipeline", [3, 0, 1])
def test_only_the_volumes_change(cases, make_tg, pipeline):
    case = cases("jittered")
    tg = make_tg(case, pipeline)
    rt.segmentize_(tg, check=False)
    default = tg.volumes.copy()
    segs, offs, status = tg.segments, tg.segment_offsets.copy(), tg.segment_status.copy()
    v = exact(tg)
    assert np.array_equal(tg.segment_offsets, offs) and np.array_equal(tg.segment_status, status)
    for k in KEYS:
        assert np.array_equal(tg.segments[k], segs[k]), k
    assert_bits(v, case.ref)
    assert np.allclose(default, v, rtol=1e-12, atol=0.0)


# ---- volume correction --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batched", [False, True])
def test_volume_correction(cases, make_tg, batched):
    case = cases("jittered")
    factors = numpy_factors(numpy_areas(case.model), case.ref)
    corrected = case.otg.seg["len"] * factors[case.otg.seg["element"] - 1]
    if not batched:
        tg = make_tg(case, volume_correction=True)
        exact(tg)
        assert_bits(tg.volume_factors, factors)
        assert_bits(tg.segments["len"], corrected)
        return
    tg = make_tg(case)
    set_capacity(tg, case.otg.n_segments // 4 + 1)
    exact(tg)
    got_f, got_len = [], []

    def on_batch(b):
        got_f.append(tg.correct_volumes())
        got_len.append(tg.segments["len"].copy())

    rt.segmentize_(tg, flags=NO_VOL, check=False, on_batch=on_batch)
    assert len(got_len) >= 4
    for f in got_f:
        assert_bits(f, factors)
    assert_bits(np.concatenate(got_len), corrected)


# ---- errors ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flag,name", [(COUNT, "RT_SEG_COUNT_ONLY"), (NO_VOL, "RT_SEG_NO_VOLUMES")])
def test_flag_conflicts(cases, make_tg, flag, name):
    case = cases("pincell")
    tg = make_tg(case)
    with pytest.raises(rt.RTError) as e:
        rt.segmentize_(tg, flags=flag, exact_volumes=True)
    assert e.value.code == RT_ERR_ARG and "RT_SEG_EXACT_VOLUMES together with " + name in e.value.msg
    assert_bits(exact(tg), case.ref)  # (the context is usable again)


# ---- size -----------------------------------------------------------------------------------------------------------------------
def test_cfg3_size():
    rt.build()
    model, n_azim, delta = rt.synth.workload("cfg3")
    mesh = rt.Mesh(model)
    otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), n_azim, delta).trace().segmentize(
        rtol=1e-6, check=False, fetch=False, nthreads=os.cpu_count() or 8)
    ref = otg.volumes()
    tg = rt.TrackGenerator(mesh, n_azim, delta)
    try:
        rt.trace_(tg)
        v = exact(tg, rtol=1e-6)
        assert tg.n_segments == otg.n_segments
        assert_bits(v, ref)
    finally:
        tg.close()


# ---- two ranks ------------------------------------------------------------------------------------------------------------------
def test_two_ranks():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(ROOT, "tools", "check_exact_volumes.py")], capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "exact volumes ok: 2 ranks" in r.stdout
