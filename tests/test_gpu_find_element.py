"""rt_find_elements (k_find_elements, locate.cuh): find_element(mesh, x, k) (src/mesh.jl:103-146) for batches of points on the
device, pinned bit for bit on the CPU oracle's find_element run over the batch (tests/locate_oracle.c) -- on the pin cell, a jittered mesh, the BWR
lattice, mixed meshes with 15 % and 100 % quadrilaterals and a device-ingested mesh, for k = 1, 2, 5 and 32, with the point
families of tests/test_find_element_cpu.py (nodes, edge midpoints, shared edges, points at and just outside the bounding box,
far points), and for 1e6 random points on a cfg3-size mesh.  Also: argument errors, n = 0, a sharded context, cell_raster, and
that a call after segmentize_ or inside its on_batch leaves the segments, volumes and stats as a run without it leaves them (the
volumes of two runs agree up to the order of the device's atomic sums; the device buffer itself is left bit for bit)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import raytracing_jl_b200 as rt  # noqa: E402
from raytracing_jl_b200 import _lib  # noqa: E402
from oracle.oracle import OracleMesh  # noqa: E402
from tests.locate_oracle import find_elements as oracle_find_elements  # noqa: E402
from tests.test_find_element_cpu import point_families  # noqa: E402

RT_ERR_ARG = -2
KS = (1, 2, 5, 32)
STAT_COUNTS = ("launches", "fast_transitions", "literal_iterations", "nn_queries", "knn_queries")
KEYS = ("px", "py", "qx", "qy", "len", "element")


@pytest.fixture(scope="module", autouse=True)
def _built():
    rt.build()


def bcs_reflective():
    return rt.BoundaryConditions(top=rt.Reflective, bottom=rt.Reflective, right=rt.Reflective, left=rt.Reflective)


def all_points(mesh, seed=0, n_random=20000):
    return np.concatenate(list(point_families(mesh, seed, n_random).values()))


def model_of(name, pincell_model):
    if name == "pincell":
        return pincell_model
    if name == "jittered":
        return rt.synth.jittered_triangle_mesh(40, 30, 1.3, 0.9, 0.3, 7, x0=-0.4, y0=2.0)
    if name == "bwr":
        return rt.synth.workload("cfg2")[0]
    if name.startswith("mixed"):
        return rt.synth.mixed_quad_triangle_mesh(31, 23, 1.5, 1.1, jitter=0.22, seed=17, quad_fraction=float(name[5:]) / 100,
                                                 x0=-0.3, y0=0.7)
    raise ValueError(name)


@pytest.mark.parametrize("name", ["pincell", "jittered", "bwr", "mixed15", "mixed100", "ingested"])
def test_ids_equal_the_oracle(pincell_model, name):
    model = model_of("bwr" if name == "ingested" else name, pincell_model)
    host = rt.Mesh(model)
    tg = rt.TrackGenerator(rt.Mesh(model, device_ingest=True) if name == "ingested" else host, 4, 0.5)
    om = OracleMesh.from_mesh(host)
    pts = all_points(host)
    for k in KS:
        want, n_knn = oracle_find_elements(om, host, pts, k)
        ids, _ = tg.find_elements(pts, k)
        bad = np.nonzero(ids != want)[0]
        assert bad.size == 0, (name, k, bad.size, pts[bad[:3]], ids[bad[:3]], want[bad[:3]])
        assert tg.info("locate_knn") == n_knn
        assert tg.info("locate_ms") > 0.0
    one = pts[:: max(1, pts.shape[0] // 40)]
    assert [rt.find_element(tg, p) for p in one] == [om.find_element(float(x), float(y), 2) for x, y in one]


def test_knn_branch_runs_on_the_jittered_mesh(pincell_model):
    model = model_of("jittered", pincell_model)
    mesh = rt.Mesh(model)
    tg = rt.TrackGenerator(mesh, 4, 0.5)
    rng = np.random.default_rng(5)
    inside = mesh.bb_min + rng.uniform(0.0, 1.0, size=(200000, 2)) * (mesh.bb_max - mesh.bb_min)
    ids, _ = tg.find_elements(inside)
    want, n_knn = oracle_find_elements(OracleMesh.from_mesh(mesh), mesh, inside)
    assert np.array_equal(ids, want)
    assert tg.info("locate_knn") == n_knn > 0  # the fallback of src/mesh.jl:123 runs, and finds the cell
    assert np.all(ids[(inside > mesh.bb_min).all(1) & (inside < mesh.bb_max).all(1)] > 0)


def test_a_million_points_on_a_cfg3_size_mesh():
    model, _, _ = rt.synth.workload("cfg3")
    mesh = rt.Mesh(model)
    tg = rt.TrackGenerator(mesh, 4, 0.5)
    pts = np.random.default_rng(11).uniform(-0.01, 1.01, size=(1_000_000, 2))
    ids, col = tg.find_elements(pts)
    want, n_knn = oracle_find_elements(OracleMesh.from_mesh(mesh), mesh, pts)
    assert np.array_equal(ids, want) and tg.info("locate_knn") == n_knn
    import torch

    assert np.array_equal(torch.as_tensor(col, device="cuda").cpu().numpy(), ids)  # the device buffer holds the same ids
    none, _ = tg.find_elements(pts[:10], fetch=False)
    assert none is None


def test_argument_errors_and_empty_calls(pincell_model, pincell_mesh):
    L = _lib.lib()
    h = C.c_void_p()
    assert L.rt_create(C.byref(h), 0) == 0
    try:
        assert L.rt_find_elements(h, 1, np.zeros(2), 2, None, None) == RT_ERR_ARG  # before rt_mesh_upload
        assert b"upload" in L.rt_last_error(h)
    finally:
        L.rt_destroy(h)
    tg = rt.TrackGenerator(pincell_model, 8, 0.02)
    pts = np.full((5, 2), 0.8)
    for k in (0, 33):
        with pytest.raises(rt.RTError) as e:
            tg.find_elements(pts, k)
        assert e.value.code == RT_ERR_ARG
    for bad in (np.nan, np.inf, -np.inf):
        p = pts.copy()
        p[3, 1] = bad
        with pytest.raises(rt.RTError) as e:
            tg.find_elements(p)
        assert e.value.code == RT_ERR_ARG and "point 3 " in e.value.msg
    assert L.rt_find_elements(tg._ctx, -1, np.zeros(2), 2, None, None) == RT_ERR_ARG
    ids, _ = tg.find_elements(np.zeros((0, 2)))
    assert ids.size == 0 and tg.info("locate_knn") == 0
    ids, _ = tg.find_elements(pts, 32)
    assert np.all(ids == oracle_find_elements(OracleMesh.from_mesh(pincell_mesh), pincell_mesh, pts, 32)[0])


def test_sharded_context_gives_the_same_ids(pincell_model):
    pts = all_points(rt.Mesh(pincell_model))
    whole = rt.TrackGenerator(pincell_model, 16, 0.02, bcs=bcs_reflective())
    shard = rt.TrackGenerator(pincell_model, 16, 0.02, bcs=bcs_reflective(), shard=(1, 3))
    rt.trace_(shard)
    assert shard.uid_begin > 1
    for k in (2, 5):
        assert np.array_equal(shard.find_elements(pts, k)[0], whole.find_elements(pts, k)[0])


def device_volumes(tg):
    v = np.zeros(tg.mesh.num_cells)
    _lib.check(tg._ctx, _lib.lib().rt_volumes(tg._ctx, _lib.ptr(v)))
    return v


def assert_volumes_agree(v, ctrl):
    """the volumes of two runs of the same segmentize_: equal up to the order in which the device's atomics add the terms"""
    assert np.abs(v - ctrl).max() <= 1e-12 * np.abs(ctrl).max()


def test_call_between_segmentize_and_fetch_leaves_the_results(pincell_model, pincell_mesh):
    pts = all_points(rt.Mesh(pincell_model))
    want = oracle_find_elements(OracleMesh.from_mesh(pincell_mesh), pincell_mesh, pts)[0]
    ctrl = rt.TrackGenerator(pincell_model, 16, 0.02, bcs=bcs_reflective())
    rt.segmentize_(rt.trace_(ctrl))
    tg = rt.TrackGenerator(pincell_model, 16, 0.02, bcs=bcs_reflective())
    rt.segmentize_(rt.trace_(tg))
    assert np.array_equal(tg.find_elements(pts)[0], want)  # before anything of the segmentize_ has been read back
    assert np.array_equal(tg.segment_offsets, ctrl.segment_offsets) and tg.resident_batch() == ctrl.resident_batch()
    for key in KEYS:
        assert np.array_equal(tg.segments[key], ctrl.segments[key]), key
    v = device_volumes(tg)
    assert np.array_equal(v, tg.volumes)  # as segmentize_ copied them before the call
    assert_volumes_agree(v, ctrl.volumes)
    s, c = tg.stats(), ctrl.stats()
    assert [s[k] for k in STAT_COUNTS] == [c[k] for k in STAT_COUNTS]
    ph = tg.phase_ms()
    tg.find_elements(pts, 5)
    assert tg.stats() == s and tg.phase_ms() == ph  # the timings of the segmentize_ too
    assert np.array_equal(tg.fetch_segments(compact=True)["px"], ctrl.segments["px"])


def test_call_inside_on_batch_leaves_the_batches(pincell_model, pincell_mesh):
    pts = all_points(rt.Mesh(pincell_model))
    want = oracle_find_elements(OracleMesh.from_mesh(pincell_mesh), pincell_mesh, pts)[0]

    def run(locate):
        tg = rt.TrackGenerator(pincell_model, 16, 0.02, bcs=bcs_reflective())
        rt.trace_(tg)
        _lib.lib().rt_set_segment_capacity(tg._ctx, 3000)
        batches, ids = [], []

        def on_batch(b):
            if locate:
                ids.append(tg.find_elements(pts)[0])
            s = tg.fetch_segments()
            batches.append((b.uid_begin, b.uid_end, b.attempt, {k: s[k].copy() for k in KEYS}))

        rt.segmentize_(tg, on_batch=on_batch)
        return tg, batches, ids

    ctrl, cb, _ = run(False)
    tg, tb, ids = run(True)
    assert len(tb) == len(cb) > 1 and len(ids) == len(tb)
    for a, b in zip(tb, cb):
        assert a[:3] == b[:3]
        for key in KEYS:
            assert np.array_equal(a[3][key], b[3][key]), key
    assert all(np.array_equal(i, want) for i in ids)
    assert_volumes_agree(tg.volumes, ctrl.volumes)
    s, c = tg.stats(), ctrl.stats()
    assert [s[k] for k in STAT_COUNTS] == [c[k] for k in STAT_COUNTS]


def test_cell_raster_equals_the_oracle_raster(pincell_model):
    mesh = rt.Mesh(pincell_model)
    tg = rt.TrackGenerator(mesh, 8, 0.02)
    nx, ny = 200, 150
    values = np.random.default_rng(2).uniform(1.0, 2.0, mesh.num_cells)
    x, y, z = rt.plotdata.cell_raster(tg, nx, ny, values)
    xs = mesh.bb_min[0] + (np.arange(nx) + 0.5) * (mesh.width / nx)
    ys = mesh.bb_min[1] + (np.arange(ny) + 0.5) * (mesh.height / ny)
    gx, gy = np.meshgrid(xs, ys)
    ids = oracle_find_elements(OracleMesh.from_mesh(mesh), mesh, np.stack([gx.reshape(-1), gy.reshape(-1)], 1))[0].reshape(ny, nx)
    assert np.array_equal(x, gx) and np.array_equal(y, gy)
    assert np.array_equal(z, np.where(ids > 0, values[ids - 1], np.nan), equal_nan=True)
    _, _, zid = rt.plotdata.cell_raster(tg, nx, ny)
    assert np.array_equal(zid, np.where(ids > 0, ids, np.nan), equal_nan=True)
