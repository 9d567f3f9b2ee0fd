"""What a transport sweep reads besides the Segment records: optical lengths tau = sigma_t[element] * len (rt_optical_lengths,
k_tau), the azimuthal weights (rt_quadrature_device, k_weights), the track views of a shard (rt_tracks_device), the exact cell
areas (rt_element_volumes, k_element_volumes) and the volume correction (rt_correct_volumes, k_volume_factors, k_scale_lengths).
They are checked with all segments resident, batch by batch from inside on_batch (rt_set_segment_capacity), on a uid shard, on a
mixed quadrilateral / triangle mesh and with zero segments.

Every reference is plain float64 (numpy on the host, torch on the device) built from the CPU oracle's Segment columns.  tau,
areas, factors and scaled lengths are single IEEE operations (the library is built with -fmad=false), so they are compared bit
for bit; only sums get a bound (assert_corrected_volumes).  GPU tests are marked one by one (pytest -m gpu); the test of that
bound runs without a GPU."""
import ctypes as C
import math

import numpy as np
import pytest

import raytracing_jl_b200 as rt
from raytracing_jl_b200 import _lib as L
from raytracing_jl_b200 import api
from oracle.oracle import OracleMesh, OracleTrackGenerator
from tests.test_gpu_knobs_flags import KEYS, assert_volumes_exact, reference_volumes
from tests.test_gpu_parity import assert_segments_equal, bcs_of

NO_VOL = rt.RT_SEG_NO_VOLUMES
RT_ERR_ARG = -2
U = 2.0 ** -53  # unit roundoff of float64
GROUPS = [1, 7, 33, 70]
PIPELINES = [3, 0, 1]
CAPACITY = 20000  # resident segments of the batched cases: about six batches of jittered60


# ---- float64 references ---------------------------------------------------------------------------------------------------
def numpy_areas(model):
    """element_volume = 1/2 * abs((x2 - x1) x (x3 - x1)) (src/trackgenerator.jl:402-411), the operations of k_element_volumes"""
    xy = model.node_coordinates
    tri = model.triangles0()
    x1, x2, x3 = xy[tri[:, 0]], xy[tri[:, 1]], xy[tri[:, 2]]
    ax, ay, bx, by = x2[:, 0] - x1[:, 0], x2[:, 1] - x1[:, 1], x3[:, 0] - x1[:, 0], x3[:, 1] - x1[:, 1]
    return 0.5 * np.abs(ax * by - ay * bx)


def numpy_factors(area, volumes):
    """area / volume where a track crosses the element, exactly 1 where none does"""
    return np.where(volumes > 0, area / np.where(volumes > 0, volumes, 1.0), 1.0)


def assert_corrected_volumes(w, area, m):
    """The traced volumes w of corrected lengths (reference_volumes: products summed with math.fsum) against the exact areas A.

    For an element with m > 0 segments, to first order in u = 2^-53:
    - the traced volume V of the first call sums m rounded positive products delta * len in some order and divides by n_azim_2:
      |V - V*| <= (m + 1) u V*, where V* is the exact value of the same sum;
    - the factor f = fl(A / V) adds u;
    - every corrected length fl(len * f) adds u, and every term fl(delta * len') of w another u.  The terms are positive, so these
      bound the relative error of their sum by 2u (not 2mu);
    - w itself is summed exactly and rounded once (u), then divided by n_azim_2 (u).
    So w = A (1 + r) with |r| <= (m + 1) u + u + 2u + 2u = (m + 6) u.  The check allows twice that, (2m + 12) u, which also covers
    the second-order terms.  An element that no track crosses has no term: w is exactly 0."""
    w, m = np.asarray(w), np.asarray(m)
    crossed = m > 0
    tol = (2.0 * m + 12.0) * U * area
    bad = np.nonzero(crossed & (np.abs(w - area) > tol))[0]
    assert bad.size == 0, f"{bad.size} elements off, e.g. element {bad[0] + 1}: {w[bad[0]]!r} vs area {area[bad[0]]!r} ({m[bad[0]]} terms)"
    assert np.all(w[~crossed] == 0.0)


def corrected_volumes(otg, length):
    """(w, m) of reference_volumes for the oracle's segments with the lengths `length`"""
    return reference_volumes(otg, otg.seg_offsets, {"len": length, "element": otg.seg["element"]}, otg.n2)


def shuffled_volumes(otg, seed):
    """traced volumes summed term by term in a random order, as the device's atomics may sum them"""
    counts = np.diff(otg.seg_offsets)
    terms = otg.deltas[np.repeat(otg.tracks["azim_idx"] - 1, counts)] * otg.seg["len"]
    order = np.random.default_rng(seed).permutation(terms.size)
    v = np.zeros(otg.mesh.n_cells)
    np.add.at(v, otg.seg["element"][order].astype(np.int64) - 1, terms[order])
    return v / otg.n2


def test_correction_bound_on_oracle_segments(pincell_model):
    """assert_corrected_volumes on the oracle's segments, corrected on the host with volumes summed in a shuffled order: the
    traced volumes of the corrected lengths are within the bound of the areas, elements no track crosses keep factor 1 and
    volume 0.  One segment left unscaled, one factor computed from a volume one term short, or the lengths of one element off by
    twice the bound's allowance, is caught."""
    for model, n_azim, delta in ((pincell_model, 16, 0.02), (pincell_model, 4, 0.8), (rt.synth.jittered_triangle_mesh(40, 40, seed=11), 16, 0.01)):
        otg = OracleTrackGenerator(OracleMesh.from_mesh(rt.Mesh(model)), n_azim, delta).trace().segmentize(check=False, nthreads=8)
        area = numpy_areas(model)
        e = otg.seg["element"] - 1
        for seed in range(3):
            f = numpy_factors(area, shuffled_volumes(otg, seed))
            corrected = otg.seg["len"] * f[e]
            w, m = corrected_volumes(otg, corrected)
            assert_corrected_volumes(w, area, m)
            assert np.all(f[m == 0] == 1.0)
        c = int(np.argmax(m))  # (the widest allowance)
        bumped = corrected * np.where(e == c, 1.0 + (4.0 * m[c] + 24.0) * U, 1.0)
        w, m2 = corrected_volumes(otg, bumped)
        with pytest.raises(AssertionError):
            assert_corrected_volumes(w, area, m2)
        s = int(np.argmax(np.abs(f[e] - 1.0)))
        unscaled = corrected.copy()
        unscaled[s] = otg.seg["len"][s]
        w, m = corrected_volumes(otg, unscaled)
        with pytest.raises(AssertionError):
            assert_corrected_volumes(w, area, m)
        v = shuffled_volumes(otg, 0)
        v[e[s]] -= otg.deltas[otg.tracks["azim_idx"][np.searchsorted(otg.seg_offsets, s, side="right") - 1] - 1] * otg.seg["len"][s] / otg.n2
        w, m = corrected_volumes(otg, otg.seg["len"] * numpy_factors(area, v)[e])
        with pytest.raises(AssertionError):
            assert_corrected_volumes(w, area, m)


# ---- GPU cases ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def built():
    rt.build()


class Case:
    def __init__(self, model, n_azim, delta):
        self.model, self.mesh = model, rt.Mesh(model)
        self.n_azim, self.delta = n_azim, delta
        self.otg = OracleTrackGenerator(OracleMesh.from_mesh(self.mesh), n_azim, delta).trace().segmentize(check=False, nthreads=8)
        self.ref, self.m = reference_volumes(self.otg, self.otg.seg_offsets, self.otg.seg, self.otg.n2)


@pytest.fixture(scope="module")
def cases(pincell_model):
    """oracle runs shared by the tests of this module"""
    specs = {
        "pincell": (lambda: pincell_model, 16, 0.02),
        "coarse": (lambda: pincell_model, 4, 0.8),  # 8 tracks, 490 segments: most elements are crossed by no track
        "jittered60": (lambda: rt.synth.jittered_triangle_mesh(60, 60, seed=5), 16, 0.01),
        "mixed": (lambda: rt.synth.mixed_quad_triangle_mesh(31, 23, 1.5, 1.1, jitter=0.22, seed=17, quad_fraction=0.5, x0=-0.3, y0=0.7), 16, 0.02),
    }
    done = {}

    def get(name):
        if name not in done:
            make, n_azim, delta = specs[name]
            done[name] = Case(make(), n_azim, delta)
        return done[name]

    return get


def make_tg(case, pipeline=None, capacity=0, **kw):
    tg = rt.TrackGenerator(case.mesh, case.n_azim, case.delta, **kw)
    rt.trace_(tg)
    if pipeline is not None:
        tg.set_option("pipeline", pipeline)
    if capacity:
        L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, capacity))
    return tg


def sigma_t(num_cells, groups):
    return np.random.default_rng(1000 + groups).uniform(0.01, 10.0, size=(num_cells, groups))


def batch_slice(b):
    return slice(b.offset_base, b.offset_base + b.n_segments)


def assert_batch_equal(cols, otg, sl, keys=KEYS):
    """one batch of Segment columns bit-equal to its slice of the oracle's (assert_segments_equal compares whole calls)"""
    for k in keys:
        assert np.array_equal(cols[k], otg.seg[k][sl]), k


def check_cuts(tg, cuts, batched):
    """the batches of one call tile the uid range and the segments, in order, without a fall-back"""
    assert len(cuts) > 2 if batched else len(cuts) == 1
    assert cuts[0][0] == 1 and cuts[-1][1] == tg.n_total_tracks + 1 and all(a[1] == b[0] for a, b in zip(cuts, cuts[1:]))
    assert sum(c[2] for c in cuts) == tg.n_segments
    assert tg.info("verify_fallbacks") == 0


def check_tau(tg, sigma, length, element):
    """tau in both layouts, the host copy and the device column, bit-equal to sigma[element - 1] * len in float64"""
    import torch

    ref = sigma[element - 1] * length[:, None]
    for layout, want in ((0, ref), (1, ref.T)):
        host, dev = tg.optical_lengths(sigma, layout=layout)
        assert host.shape == want.shape and np.array_equal(host, want), layout
        assert np.array_equal(torch.as_tensor(dev, device="cuda").cpu().numpy(), want.reshape(-1)), layout


# ---- a. optical lengths ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("groups", GROUPS)
@pytest.mark.parametrize("where", ["whole", "shard", "mixed", "corrected", "max_iter0"])
def test_optical_lengths(built, cases, where, groups):
    """tau of the resident segments: the whole pin cell, the middle uid shard of three, a mixed quadrilateral / triangle mesh,
    the lengths after correct_volumes(), and a call with max_iter = 0 that leaves no segment (tau of shape (0, G), no error)."""
    case = cases("mixed" if where == "mixed" else "pincell")
    otg = case.otg
    sigma = sigma_t(case.mesh.num_cells, groups)
    tg = make_tg(case, shard=(1, 3) if where == "shard" else (0, 1))
    if where == "max_iter0":
        rt.segmentize_(tg, max_iter=0, check=False)
        assert tg.n_segments == 0 and tg.resident_batch()[3] == 0
        for layout, shape in ((0, (0, groups)), (1, (groups, 0))):
            host, dev = tg.optical_lengths(sigma, layout=layout)
            assert host.shape == shape and dev.__cuda_array_interface__["shape"] == (0,)
        return
    rt.segmentize_(tg, check=False)
    if where == "shard":  # the oracle on the shard's uid range
        assert 1 < tg.uid_begin < tg.uid_end < tg.n_total_tracks + 1
        otg = OracleTrackGenerator(OracleMesh.from_mesh(case.mesh), case.n_azim, case.delta).trace()
        otg.segmentize(uid_begin=tg.uid_begin, uid_end=tg.uid_end, check=False, nthreads=8)
    assert_segments_equal(otg, tg)
    length, element = otg.seg["len"], otg.seg["element"]
    if where == "corrected":
        f = tg.correct_volumes()
        assert np.count_nonzero(f != 1.0) > 0.9 * f.size
        length = length * f[element - 1]
    check_tau(tg, sigma, length, element)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", PIPELINES)
def test_optical_lengths_of_every_batch(built, cases, pipeline):
    """tau taken inside on_batch for every batch of a call whose segments do not fit at once: the batch's slice of the oracle's
    columns, every group count, both layouts, device column and host copy."""
    case = cases("jittered60")
    otg = case.otg
    tg = make_tg(case, pipeline=pipeline, capacity=CAPACITY)
    sigmas = [sigma_t(case.mesh.num_cells, g) for g in GROUPS]
    cuts = []

    def on_batch(b):
        assert b.attempt == 0
        assert tg.resident_batch() == (b.uid_begin, b.uid_end, b.offset_base, b.n_segments)
        sl = batch_slice(b)
        for sigma in sigmas:
            check_tau(tg, sigma, otg.seg["len"][sl], otg.seg["element"][sl])
        cuts.append((b.uid_begin, b.uid_end, b.n_segments))

    rt.segmentize_(tg, check=False, on_batch=on_batch)
    check_cuts(tg, cuts, batched=True)


@pytest.mark.gpu
def test_optical_lengths_beyond_2_32_values(built, record_property):
    """cfg3 at its named size (~5e7 segments) with enough groups that n_segments * G > 2^32: the flat index of k_tau passes 2^32
    in both layouts.  tau (~38 GB) stays on the device and is compared with torch's float64 products in slices of segments
    (layout 0) or one group at a time (layout 1), so that the reference adds a few GB at most."""
    import torch

    model, n_azim, delta = rt.synth.workload("cfg3")
    tg = rt.TrackGenerator(rt.Mesh(model, device_ingest=True), n_azim, delta)
    rt.trace_(tg)
    rt.segmentize_(tg, check=False, flags=NO_VOL)
    n = tg.n_segments
    groups = max(96, 2 ** 32 // n + 1)
    assert n > 40_000_000 and n * groups > 2 ** 32
    sigma = sigma_t(model.num_cells, groups)
    view = L.rt_batch()
    L.check(tg._ctx, L.lib().rt_segments_device(tg._ctx, C.byref(view)))
    batch = api.SegmentBatch(view)
    assert batch.n_segments == n
    length = torch.as_tensor(batch.len, device="cuda")
    element = torch.as_tensor(batch.element, device="cuda").long() - 1
    sig = torch.from_numpy(sigma).cuda()
    sig_t = sig.t().contiguous()
    free, total = torch.cuda.mem_get_info()
    least_free = free
    step = 1 << 22
    for layout in (0, 1):
        host, dev = tg.optical_lengths(sigma, layout=layout, fetch=False)
        assert host is None
        tau = torch.as_tensor(dev, device="cuda")
        assert tau.numel() == n * groups
        if layout == 0:
            tau = tau.view(n, groups)
            for s0 in range(0, n, step):
                assert torch.equal(tau[s0:s0 + step], sig[element[s0:s0 + step]] * length[s0:s0 + step, None]), s0
                least_free = min(least_free, torch.cuda.mem_get_info()[0])
        else:
            tau = tau.view(groups, n)
            for g in range(groups):
                assert torch.equal(tau[g], sig_t[g][element] * length), g
            least_free = min(least_free, torch.cuda.mem_get_info()[0])
        del tau
    record_property("n_segments", n)
    record_property("groups", groups)
    record_property("tau_bytes", n * groups * 8)
    record_property("torch_peak_reserved_bytes", torch.cuda.max_memory_reserved())
    record_property("device_peak_used_bytes", total - least_free)
    tg.close()


# ---- b. azimuthal weights -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_azim", [4, 8, 16, 64, 128])
def test_quadrature_weights_on_the_device(built, pincell_model, n_azim):
    """k_weights before and after the first segmentize_: omega bit-equal to the host init_weights! (equal to the oracle's),
    symmetric and positive; the per-angle tables as passed to rt_trace; delta_eff absent before segmentize_ and equal to the
    effective spacings after it.  n_azim = 4 is the case where the first and the last angle of (0, pi/2) coincide."""
    import torch

    tg = rt.TrackGenerator(pincell_model, n_azim, 0.1)
    rt.trace_(tg)
    aq = tg.azimuthal_quadrature
    otg = OracleTrackGenerator(OracleMesh.from_mesh(tg.mesh), n_azim, 0.1).trace()
    assert np.array_equal(aq.phis, otg.phis) and np.array_equal(aq.weights, otg.weights)
    for stage in ("traced", "segmentized"):
        omega, view = tg.quadrature_device()
        dev = {k: torch.as_tensor(c, device="cuda").cpu().numpy() for k, c in view.items()}
        assert omega.shape == (n_azim // 2,) and np.array_equal(omega, aq.weights) and np.array_equal(dev["omega"], omega)
        assert np.array_equal(omega, omega[::-1]) and np.all(omega > 0)
        assert np.array_equal(dev["phi"], aq.phis)
        assert np.array_equal(dev["sin"], [math.sin(p) for p in aq.phis]) and np.array_equal(dev["cos"], [math.cos(p) for p in aq.phis])
        if stage == "traced":
            assert "delta_eff" not in view
            rt.segmentize_(tg, check=False)
        else:
            assert np.array_equal(dev["delta_eff"], aq.deltas)


# ---- c. track views of a shard --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_track_views_of_shards(built, pincell_model):
    """track_view() of every shard of three: its uid range, every column bit-equal to the matching slice of the whole domain's
    track table, and the links to the next tracks as global uids (some of them point into other shards)."""
    import torch

    bcs = bcs_of((0, 1, 2, 1))
    whole = rt.TrackGenerator(pincell_model, 16, 0.02, bcs=bcs)
    rt.trace_(whole)
    t, n_total = whole.track_data, whole.n_total_tracks
    ends, outside = [], 0
    for r in range(3):
        tg = rt.TrackGenerator(pincell_model, 16, 0.02, bcs=bcs, shard=(r, 3))
        rt.trace_(tg)
        v = tg.track_view()
        assert v["uid_begin"] == tg.uid_begin and v["n_tracks"] == tg.uid_end - tg.uid_begin > 0
        ends.append((tg.uid_begin, tg.uid_end))
        sl = slice(tg.uid_begin - 1, tg.uid_end - 1)
        want = {"px": t["p"][sl, 0], "py": t["p"][sl, 1], "qx": t["q"][sl, 0], "qy": t["q"][sl, 1], "len": t["len"][sl],
                "a": t["abc"][sl, 0], "b": t["abc"][sl, 1], "c": t["abc"][sl, 2], "azim": t["azim_idx"][sl] - 1}
        want.update({k: t[k][sl] for k in ("track_idx", "next_fwd", "next_bwd", "bc_fwd", "bc_bwd", "dir_fwd", "dir_bwd")})
        dev = {k: torch.as_tensor(c, device="cuda").cpu().numpy() for k, c in v.items() if isinstance(c, api.DeviceColumn)}
        assert set(dev) == set(want)
        for k in want:
            assert np.array_equal(dev[k], want[k]), k
        links = np.concatenate([dev["next_fwd"], dev["next_bwd"]])
        assert links.min() >= 1 and links.max() <= n_total
        outside += np.count_nonzero((links < tg.uid_begin) | (links >= tg.uid_end))
        tg.close()
    assert ends[0][0] == 1 and ends[-1][1] == n_total + 1 and all(a[1] == b[0] for a, b in zip(ends, ends[1:]))
    assert outside > 0


# ---- d. element areas -----------------------------------------------------------------------------------------------------
def clockwise_mesh():
    """a jittered mesh with every third triangle stored clockwise (negative cross product)"""
    m = rt.synth.jittered_triangle_mesh(24, 18, 1.2, 0.9, 0.3, 13)
    tri = m.triangles0().copy()
    tri[::3] = tri[::3, ::-1]
    return rt.UnstructuredDiscreteModel.from_triangles(m.node_coordinates, tri, sort_nodes=False)


AREA_MESHES = {
    "pin_lattice": (lambda: rt.synth.pin_lattice_mesh(2, 1.26, 0.4096, 0.0655, 0.05, seed=3), False),
    "far_offset": (lambda: rt.synth.jittered_triangle_mesh(30, 20, 0.75, 0.5, 0.3, 7, x0=1e3, y0=-2.5e3), False),
    "clockwise": (clockwise_mesh, False),
    "device_ingest": (lambda: rt.synth.jittered_triangle_mesh(23, 17, 2.5, 1.25, 0.3, 11, x0=1e3, y0=7.5), True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("which", list(AREA_MESHES))
def test_element_areas(built, which):
    """element_volumes() bit-equal to numpy's 0.5 * abs(ax*by - ay*bx): a pin lattice, a mesh far from the origin (large
    coordinates, small differences), a mesh with clockwise triangles, and a mesh ingested on the device."""
    make, device_ingest = AREA_MESHES[which]
    model = make()
    if which == "clockwise":
        xy, tri = model.node_coordinates, model.triangles0()
        a, b = xy[tri[:, 1]] - xy[tri[:, 0]], xy[tri[:, 2]] - xy[tri[:, 0]]
        cross = a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]
        assert np.count_nonzero(cross < 0) > 0.3 * cross.size and np.count_nonzero(cross > 0) > 0.3 * cross.size
    tg = rt.TrackGenerator(rt.Mesh(model, device_ingest=device_ingest), 8, 0.05)
    area = numpy_areas(model)
    assert np.all(area > 0) and math.isclose(area.sum(), rt.synth.mesh_area(model), rel_tol=1e-12)
    assert np.array_equal(tg.element_volumes(), area)


# ---- e. volume correction, resident and batched -----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("second_flags", [0, NO_VOL])
@pytest.mark.parametrize("pipeline", PIPELINES)
@pytest.mark.parametrize("mesh,capacity", [("jittered60", CAPACITY), ("coarse", 128), ("coarse", 0)])
def test_volume_correction_inside_on_batch(built, cases, mesh, capacity, pipeline, second_flags):
    """One call with volumes, then a correcting call whose on_batch runs correct_volumes() on every batch (with or without
    RT_SEG_NO_VOLUMES): factors bit-equal to area / v of the first call's volumes v (exactly 1 where no track crosses), every
    batch's corrected lengths bit-equal to the oracle's len * f[element], end points and elements untouched, and the traced
    volumes of the corrected lengths equal to the areas within assert_corrected_volumes' bound.  volume_correction = true with
    batched segments corrects nothing and leaves no factors."""
    case = cases(mesh)
    otg = case.otg
    tg = make_tg(case, pipeline=pipeline, capacity=capacity, volume_correction=bool(capacity))
    rt.segmentize_(tg, check=False)
    assert tg.volume_factors is None
    v = tg.volumes.copy()
    assert_volumes_exact(v, case.ref, case.m)
    area = numpy_areas(case.model)
    want_f = numpy_factors(area, v)
    corrected = np.full(otg.n_segments, np.nan)
    cuts = []

    def on_batch(b):
        assert b.attempt == 0
        assert np.array_equal(tg.correct_volumes(), want_f)
        sl = batch_slice(b)
        s = tg.fetch_segments()
        assert np.array_equal(s["len"], otg.seg["len"][sl] * want_f[otg.seg["element"][sl] - 1])
        assert_batch_equal(s, otg, sl, ("px", "py", "qx", "qy", "element"))
        corrected[sl] = s["len"]
        cuts.append((b.uid_begin, b.uid_end, b.n_segments))

    rt.segmentize_(tg, flags=second_flags, check=False, on_batch=on_batch)
    check_cuts(tg, cuts, batched=bool(capacity))
    assert tg.volume_factors is None
    if second_flags & NO_VOL:  # a correcting call without volumes leaves none to read
        assert L.lib().rt_volumes(tg._ctx, L.ptr(np.zeros(case.mesh.num_cells))) == RT_ERR_ARG
    else:  # summed before the callback ran: the volumes of the lengths before correction
        assert_volumes_exact(tg.volumes, case.ref, case.m)
    w, m = corrected_volumes(otg, corrected)
    assert np.array_equal(m, case.m)
    assert_corrected_volumes(w, area, m)
    if mesh == "coarse":
        assert np.count_nonzero(m == 0) > 1000 and np.all(want_f[m == 0] == 1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", PIPELINES)
def test_volume_correction_flag_with_batched_segments(built, cases, pipeline):
    """volume_correction = true corrects the segments of a call only when they are all resident -- also when an earlier call on
    the context allocated columns for all of them and a segment capacity then cuts the next call into batches."""
    case = cases("jittered60")
    otg = case.otg
    tg = make_tg(case, pipeline=pipeline, volume_correction=True)
    rt.segmentize_(tg, check=False)
    f = tg.volume_factors
    assert f is not None and np.array_equal(f, numpy_factors(numpy_areas(case.model), tg.volumes))
    assert np.array_equal(tg.segments["len"], otg.seg["len"] * f[otg.seg["element"] - 1])
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, CAPACITY))
    rt.segmentize_(tg, check=False)
    assert tg.volume_factors is None
    n = tg.resident_batch()[3]
    assert 0 < n < tg.n_segments
    assert_batch_equal(tg.segments, otg, slice(otg.n_segments - n, None))


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", PIPELINES)
def test_correction_inside_on_batch_needs_volumes(built, cases, pipeline):
    """Inside on_batch, correct_volumes() uses the volumes of the call before: without any (a fresh context, a call with
    RT_SEG_NO_VOLUMES) it raises RT_ERR_ARG and the call stops; after a call with volumes it corrects.  Outside callbacks the
    refusal after RT_SEG_NO_VOLUMES stands."""
    case = cases("jittered60")
    otg = case.otg
    tg = make_tg(case, pipeline=pipeline, capacity=CAPACITY)

    def correct(b):
        tg.correct_volumes()

    for first_flags in (None, NO_VOL):
        if first_flags is not None:
            rt.segmentize_(tg, flags=first_flags, check=False)
        with pytest.raises(rt.RTError) as err:
            rt.segmentize_(tg, check=False, on_batch=correct)
        assert err.value.code == RT_ERR_ARG
        assert b"asked to stop" in L.lib().rt_last_error(tg._ctx)
    rt.segmentize_(tg, flags=NO_VOL, check=False)
    with pytest.raises(rt.RTError):
        tg.correct_volumes()
    rt.segmentize_(tg, check=False)
    rt.segmentize_(tg, flags=NO_VOL, check=False, on_batch=correct)
    assert_batch_equal(tg.segments, otg, slice(otg.n_segments - tg.resident_batch()[3], None), ("px", "py", "qx", "qy", "element"))


# ---- f. downloads inside the callback ---------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", PIPELINES)
def test_downloads_inside_on_batch(built, cases, pipeline):
    """fetch_segments(), full and compact, inside on_batch: the batch's slice of the oracle's columns bit for bit; after the
    call tg.segments is the last batch, not a copy cached inside a callback."""
    case = cases("jittered60")
    otg = case.otg
    tg = make_tg(case, pipeline=pipeline, capacity=CAPACITY)
    cuts = []

    def on_batch(b):
        assert b.attempt == 0
        sl = batch_slice(b)
        for cols in (tg.fetch_segments(), tg.fetch_segments(compact=True), tg.segments):
            assert_batch_equal(cols, otg, sl)
        cuts.append((b.uid_begin, b.uid_end, b.n_segments))

    rt.segmentize_(tg, check=False, on_batch=on_batch)
    check_cuts(tg, cuts, batched=True)
    assert_batch_equal(tg.segments, otg, slice(otg.n_segments - cuts[-1][2], None))
