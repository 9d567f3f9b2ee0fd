"""Material regions on the device: rt_set_regions (the region of every cell, checked and ordered by region), the optical lengths
from per-region cross sections (rt_optical_lengths_by_region, k_tau<true>) and the per-region sums of the traced volumes and the
cell areas (rt_region_volumes).

tau is one IEEE product per value, so it is compared bit for bit with sigma_r[region[element] - 1] * len computed in numpy from the
oracle's columns, and with rt_optical_lengths given the per-cell table expanded from the per-region one.  The region sums add the
cells of a region in ascending id with one `+` each from 0.0, which is np.add.at over the cells in id order: bit for bit again."""
import ctypes as C
import math

import numpy as np
import pytest

import raytracing_jl_b200 as rt
from raytracing_jl_b200 import _lib as L
from raytracing_jl_b200 import api
from oracle.oracle import OracleMesh, OracleTrackGenerator
from tests.test_gpu_comm_volumes import attach_comm
from tests.test_gpu_exact_volumes import Case, assert_bits, set_capacity
from tests.test_gpu_sweep_outputs import U, corrected_volumes

pytestmark = pytest.mark.gpu
RT_ERR_ARG = -2
GROUPS = [1, 7, 33, 70]
MESHES = ["pincell", "jittered", "bwr", "mixed15", "mixed100", "ingested"]
N_REGIONS = 3


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


def region_map(n_cells, n_regions=N_REGIONS, seed=0):
    """every region used, cells of a region scattered over the id range"""
    r = np.random.default_rng(seed).integers(1, n_regions + 1, size=n_cells).astype(np.int32)
    r[:n_regions] = np.arange(1, n_regions + 1)
    return r


def sigma_r(groups, n_regions=N_REGIONS):
    return np.random.default_rng(2000 + groups).uniform(0.01, 10.0, size=(n_regions, groups))


def check_tau(tg, region, sig, length, element):
    """tau by region in both layouts, host copy and device column, bit-equal to the numpy products and to the per-cell call with
    the expanded table"""
    import torch

    ref = sig[region[element - 1] - 1] * length[:, None]
    expanded = sig[region - 1]
    for layout, want in ((0, ref), (1, ref.T)):
        host, dev = tg.optical_lengths_by_region(sig, layout=layout)
        assert host.shape == want.shape
        assert_bits(host.reshape(-1), np.ascontiguousarray(want).reshape(-1))
        assert_bits(torch.as_tensor(dev, device="cuda").cpu().numpy(), np.ascontiguousarray(want).reshape(-1))
        cell, _ = tg.optical_lengths(expanded, layout=layout)
        assert_bits(host.reshape(-1), cell.reshape(-1))


def add_at(region, values, n_regions=N_REGIONS):
    out = np.zeros(n_regions)
    np.add.at(out, region - 1, values)
    return out


# ---- optical lengths by region ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("groups", GROUPS)
@pytest.mark.parametrize("mesh", MESHES)
def test_tau_by_region(cases, make_tg, mesh, groups):
    case = cases(mesh)
    tg = make_tg(case)
    rt.segmentize_(tg, check=False)
    region = region_map(case.model.num_cells)
    tg.set_regions(region)
    assert tg.n_regions == N_REGIONS
    cols = tg.segments
    assert np.array_equal(cols["element"], case.otg.seg["element"]) and np.array_equal(cols["len"], case.otg.seg["len"])
    check_tau(tg, region, sigma_r(groups), case.otg.seg["len"], case.otg.seg["element"])
    assert tg.info("tau_ms") >= 0.0


@pytest.mark.parametrize("where", ["shard", "lengths_only", "max_iter0"])
def test_tau_by_region_calls(cases, make_tg, where):
    """on the middle uid shard of three, after a lengths-only call, and with no segment (tau of shape (0, G), no error)"""
    case = cases("jittered")
    tg = make_tg(case, shard=(1, 3) if where == "shard" else (0, 1))
    region = region_map(case.model.num_cells, seed=4)
    tg.set_regions(region)  # (before segmentize_: the map belongs to the mesh, not to a call)
    otg = case.otg
    if where == "max_iter0":
        rt.segmentize_(tg, max_iter=0, check=False)
        assert tg.n_segments == 0
        for layout, shape in ((0, (0, 7)), (1, (7, 0))):
            host, dev = tg.optical_lengths_by_region(sigma_r(7), layout=layout)
            assert host.shape == shape and dev.__cuda_array_interface__["shape"] == (0,)
        return
    rt.segmentize_(tg, check=False, lengths_only=where == "lengths_only")
    if where == "shard":
        assert 1 < tg.uid_begin < tg.uid_end < tg.n_total_tracks + 1
        otg = OracleTrackGenerator(OracleMesh.from_mesh(case.mesh), case.n_azim, case.delta).trace()
        otg.segmentize(uid_begin=tg.uid_begin, uid_end=tg.uid_end, check=False, nthreads=8)
    assert np.array_equal(tg.segments["len"], otg.seg["len"])
    for groups in (1, 7, 70):
        check_tau(tg, region, sigma_r(groups), otg.seg["len"], otg.seg["element"])


@pytest.mark.parametrize("pipeline", [3, 0, 1])
def test_tau_by_region_of_every_batch(cases, make_tg, pipeline):
    """inside on_batch with a small segment capacity: every batch's slice of the oracle's columns; the batch, its segments and the
    stats are the same before and after the region calls"""
    case = cases("jittered")
    otg = case.otg
    tg = make_tg(case, pipeline=pipeline)
    set_capacity(tg, otg.n_segments // 6)
    region = region_map(case.model.num_cells, seed=1)
    tg.set_regions(region)
    cuts = []

    def on_batch(b):
        assert b.attempt == 0
        sl = slice(int(otg.seg_offsets[b.uid_begin - 1]), int(otg.seg_offsets[b.uid_end - 1]))
        before = (tg.resident_batch(), {k: v.copy() for k, v in tg.fetch_segments().items()}, tg.stats())
        for groups in (1, 7, 33):
            check_tau(tg, region, sigma_r(groups), otg.seg["len"][sl], otg.seg["element"][sl])
        tg.set_regions(region)  # (allowed inside a callback: it touches neither the batch nor the volumes)
        with pytest.raises(rt.RTError) as e:
            tg.region_volumes()
        assert e.value.code == RT_ERR_ARG and "batch callback" in e.value.msg
        tg._resident = None
        after = (tg.resident_batch(), tg.fetch_segments(), tg.stats())
        assert before[0] == after[0] and before[2] == after[2]
        for k, v in before[1].items():
            assert np.array_equal(v, after[1][k]), k
        cuts.append((b.uid_begin, b.uid_end, b.n_segments))

    rt.segmentize_(tg, check=False, on_batch=on_batch)
    assert len(cuts) > 2 and sum(c[2] for c in cuts) == tg.n_segments == otg.n_segments
    assert tg.info("verify_fallbacks") == 0


def test_tau_by_region_beyond_2_32_values():
    """cfg3 at its named size with n_segments * G > 2^32: compared with torch's products in slices (layout 0) and group by group
    (layout 1), as for rt_optical_lengths"""
    import torch

    rt.build()
    model, n_azim, delta = rt.synth.workload("cfg3")
    tg = rt.TrackGenerator(rt.Mesh(model, device_ingest=True), n_azim, delta)
    rt.trace_(tg)
    rt.segmentize_(tg, check=False, flags=rt.RT_SEG_NO_VOLUMES)
    n = tg.n_segments
    groups = max(96, 2 ** 32 // n + 1)
    assert n > 40_000_000 and n * groups > 2 ** 32
    region = region_map(model.num_cells, seed=3)
    tg.set_regions(region)
    sig = sigma_r(groups)
    view = L.rt_batch()
    L.check(tg._ctx, L.lib().rt_segments_device(tg._ctx, C.byref(view)))
    batch = api.SegmentBatch(view)
    length = torch.as_tensor(batch.len, device="cuda")
    reg = torch.from_numpy(region).cuda().long()[torch.as_tensor(batch.element, device="cuda").long() - 1] - 1
    sig_d = torch.from_numpy(sig).cuda()
    sig_t = sig_d.t().contiguous()
    step = 1 << 22
    for layout in (0, 1):
        host, dev = tg.optical_lengths_by_region(sig, layout=layout, fetch=False)
        assert host is None
        tau = torch.as_tensor(dev, device="cuda")
        assert tau.numel() == n * groups
        if layout == 0:
            tau = tau.view(n, groups)
            for s0 in range(0, n, step):
                assert torch.equal(tau[s0:s0 + step], sig_d[reg[s0:s0 + step]] * length[s0:s0 + step, None]), s0
        else:
            tau = tau.view(groups, n)
            for g in range(groups):
                assert torch.equal(tau[g], sig_t[g][reg] * length), g
        del tau
    tg.close()


# ---- region volumes ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mesh", ["pincell", "jittered", "bwr", "ingested"])
def test_region_volumes(cases, make_tg, mesh):
    """traced: np.add.at over the device's own volumes; exact: np.add.at over element_volumes(), summing to the domain area"""
    case = cases(mesh)
    tg = make_tg(case)
    rt.segmentize_(tg, check=False)
    region = region_map(case.model.num_cells, seed=2)
    tg.set_regions(region)
    traced, exact = tg.region_volumes()
    assert_bits(traced, add_at(region, tg.volumes))
    assert_bits(exact, add_at(region, tg.element_volumes()))
    assert math.isclose(exact.sum(), rt.synth.mesh_area(case.model), rel_tol=1e-12)
    t2, e2 = tg.region_volumes(exact=False)
    assert e2 is None and np.array_equal(t2, traced)


@pytest.mark.parametrize("comm", [False, True])
def test_region_volumes_exact(cases, make_tg, comm):
    """RT_SEG_EXACT_VOLUMES: the traced region volumes are np.add.at over the oracle's volumes, bit for bit, also with a one-rank
    communicator; the default volumes with the communicator: np.add.at over the all-reduced ones, also when rt_volumes only
    enqueued the collective"""
    case = cases("jittered")
    tg = make_tg(case, comm=comm)
    region = region_map(case.model.num_cells, seed=5)
    tg.set_regions(region)
    rt.segmentize_(tg, check=False, exact_volumes=True)
    traced, _ = tg.region_volumes(exact=False)
    assert_bits(traced, add_at(region, case.ref))
    rt.segmentize_(tg, check=False, fetch_volumes=False)
    traced, _ = tg.region_volumes(exact=False)
    vol = np.zeros(case.model.num_cells)
    L.check(tg._ctx, L.lib().rt_volumes(tg._ctx, L.ptr(vol)))
    assert_bits(traced, add_at(region, vol))


def test_region_volumes_after_correction(cases, make_tg):
    """after volume_correction the traced volumes of the corrected lengths equal the areas within the bound of
    assert_corrected_volumes, summed per region (plus the rounding of the two region sums)"""
    case = cases("pincell")
    tg = make_tg(case, volume_correction=True)
    region = region_map(case.model.num_cells, seed=6)
    tg.set_regions(region)
    rt.segmentize_(tg, check=False)
    assert tg.volume_factors is not None
    w, m = corrected_volumes(case.otg, tg.segments["len"].copy())
    _, exact = tg.region_volumes(traced=False)
    area = tg.element_volumes()
    counts = np.bincount(region - 1, minlength=N_REGIONS)
    crossed = m > 0
    assert np.all(w[~crossed] == 0.0)
    tol = add_at(region, np.where(crossed, (2.0 * m + 12.0) * U * area, 0.0)) + 2.0 * counts * U * exact
    wr, ar = add_at(region, w), add_at(region, np.where(crossed, area, 0.0))
    assert np.all(np.abs(wr - ar) <= tol), (wr, ar, tol)


# ---- errors and state -------------------------------------------------------------------------------------------------------
def test_bad_maps_keep_the_previous_one(cases, make_tg):
    case = cases("pincell")
    tg = make_tg(case)
    rt.segmentize_(tg, check=False)
    region = region_map(case.model.num_cells)
    tg.set_regions(region)
    sig = sigma_r(7)
    good, _ = tg.optical_lengths_by_region(sig)
    for bad_value, cell in ((0, 17), (N_REGIONS + 1, 5), (-4, 1234)):
        bad = region.copy()
        bad[cell - 1] = bad_value
        bad[cell + 10] = 0  # (a later bad cell: the message names the first)
        with pytest.raises(rt.RTError) as e:
            tg.set_regions(bad, n_regions=N_REGIONS)
        assert e.value.code == RT_ERR_ARG and f"cell {cell} has region {bad_value}," in e.value.msg, e.value.msg
        tg._n_regions = N_REGIONS  # (the binding records the map only on success; the library kept the old one)
        again, _ = tg.optical_lengths_by_region(sig)
        assert_bits(again.reshape(-1), good.reshape(-1))
    rc = L.lib().rt_set_regions(tg._ctx, 0, L.ptr(region))
    assert rc == RT_ERR_ARG and "n_regions = 0" in L.lib().rt_last_error(tg._ctx).decode()
    tg.set_regions(None)
    with pytest.raises(rt.RTError) as e:
        L.check(tg._ctx, L.lib().rt_region_volumes(tg._ctx, L.ptr(np.zeros(3)), None))
    assert e.value.code == RT_ERR_ARG and "no region map" in e.value.msg


def test_tau_by_region_needs_a_map_of_this_mesh(cases, make_tg):
    case = cases("pincell")
    tg = make_tg(case)
    rt.segmentize_(tg, check=False)
    d = C.c_void_p()

    def call():
        sig = sigma_r(2).reshape(-1)
        return L.lib().rt_optical_lengths_by_region(tg._ctx, 2, sig, 0, C.byref(d), None)

    assert call() == RT_ERR_ARG and "no region map" in L.lib().rt_last_error(tg._ctx).decode()
    tg.set_regions(region_map(case.model.num_cells))
    assert call() == 0
    tg.upload_mesh()  # a new rt_mesh_upload clears the map
    rt.trace_(tg)
    rt.segmentize_(tg, check=False)
    assert call() == RT_ERR_ARG and "no region map" in L.lib().rt_last_error(tg._ctx).decode()


def test_region_volumes_preconditions(cases, make_tg):
    """before rt_volumes, after a call without volumes, and exact areas on a mixed mesh are refused; the three calls leave the
    segments, offsets, volumes and stats as they are"""
    case = cases("pincell")
    tg = make_tg(case)
    region = region_map(case.model.num_cells)
    tg.set_regions(region)
    n, bad, st = C.c_int64(0), C.c_int64(0), C.c_int32(0)
    L.check(tg._ctx, L.lib().rt_segmentize(tg._ctx, tg.tiny_step, 5, rt.RTOL_DEFAULT, rt.MAX_ITER, L.ptr(tg.azimuthal_quadrature.deltas),
                                           0, None, None, C.byref(n), C.byref(bad), C.byref(st)))
    with pytest.raises(rt.RTError) as e:
        tg.region_volumes()
    assert e.value.code == RT_ERR_ARG and "rt_volumes first" in e.value.msg
    _, exact = tg.region_volumes(traced=False)  # (the areas need no volumes)
    vol = np.zeros(case.model.num_cells)
    L.check(tg._ctx, L.lib().rt_volumes(tg._ctx, L.ptr(vol)))
    tg._segmented = True
    segs = {k: v.copy() for k, v in tg.fetch_segments().items()}
    offsets, stats, phases = tg.segment_offsets.copy(), tg.stats(), tg.phase_ms()
    traced, exact2 = tg.region_volumes()
    assert_bits(traced, add_at(region, vol))
    assert_bits(exact2, exact)
    tg.optical_lengths_by_region(sigma_r(7))
    tg.set_regions(region)
    vol2 = np.zeros_like(vol)
    L.check(tg._ctx, L.lib().rt_volumes(tg._ctx, L.ptr(vol2)))
    assert_bits(vol2, vol)
    for k, v in tg.fetch_segments().items():
        assert np.array_equal(v, segs[k]), k
    tg._offsets = None
    assert np.array_equal(tg.segment_offsets, offsets) and tg.stats() == stats and tg.phase_ms() == phases
    rt.segmentize_(tg, check=False, flags=rt.RT_SEG_NO_VOLUMES)
    with pytest.raises(rt.RTError) as e:
        tg.region_volumes()
    assert e.value.code == RT_ERR_ARG

    mixed = cases("mixed15")
    tg = make_tg(mixed)
    region = region_map(mixed.model.num_cells)
    tg.set_regions(region)
    rt.segmentize_(tg, check=False)
    with pytest.raises(rt.RTError) as e:
        tg.region_volumes()
    assert e.value.code == RT_ERR_ARG and "triangle meshes only" in e.value.msg
    traced, _ = tg.region_volumes(exact=False)
    assert_bits(traced, add_at(region, tg.volumes))
