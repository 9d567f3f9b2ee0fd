"""GPU parity tests (run on the B200 box: pytest -m gpu).  Every call goes through the C ABI
(librt_b200.so via ctypes) and is compared with the CPU oracle on the same seeded inputs:
track/segment counts, element ids and segment order bit-exact; p/q/len bit-exact (the bar in
BASELINE.json is 1e-12 relative, the kernels are built to reproduce the reference's IEEE ops exactly);
volumes to 1e-10 relative (atomics reorder the sum)."""
import math
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import raytracing_jl_b200 as rt  # noqa: E402
from raytracing_jl_b200 import api  # noqa: E402
from oracle.oracle import OracleMesh, OracleTrackGenerator  # noqa: E402
from tests.golden import runtests_goldens as G  # noqa: E402

P_TOL = 1e-12  # relative tolerance named by BASELINE.json:north_star for p/q/len


@pytest.fixture(scope="module", autouse=True)
def _built():
    rt.build()


def bcs_of(codes):
    t, b, r, l = (rt.BoundaryType(c) for c in codes)
    return rt.BoundaryConditions(top=t, bottom=b, right=r, left=l)


def run_both(model, n_azim, delta, bcs=(0, 0, 0, 0), flags=0, k=5, capacity=0, chunk_segments=None, pipeline=None):
    mesh = rt.Mesh(model)
    otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), n_azim, delta, bcs=bcs)
    otg.trace()
    otg.segmentize(k=k, check=False, nthreads=8)
    tg = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs_of(bcs))
    rt.trace_(tg)
    if chunk_segments:
        tg.set_option("chunk_segments", chunk_segments)
        tg.set_option("target_walkers", 1e9)
    if pipeline is not None:
        tg.set_option("pipeline", pipeline)
    if capacity:
        from raytracing_jl_b200 import _lib
        _lib.lib().rt_set_segment_capacity(tg._ctx, capacity)
    rt.segmentize_(tg, k=k, flags=flags, check=False)
    return otg, tg


def assert_tracks_equal(otg, tg):
    t, o = tg.track_data, otg.tracks
    assert tg.n_total_tracks == otg.n_total_tracks
    assert np.array_equal(tg.n_tracks_x, otg.n_tracks_x) and np.array_equal(tg.n_tracks_y, otg.n_tracks_y)
    aq = tg.azimuthal_quadrature
    assert np.array_equal(aq.phis, otg.phis) and np.array_equal(aq.deltas, otg.deltas) and np.array_equal(aq.weights, otg.weights)
    for key in ("azim_idx", "track_idx", "bc_fwd", "bc_bwd", "dir_fwd", "dir_bwd", "next_fwd", "next_bwd"):
        assert np.array_equal(t[key], o[key]), key
    for key in ("p", "q", "phi", "len", "abc"):
        assert np.array_equal(t[key], o[key]), key  # bit-exact


def assert_segments_equal(otg, tg, whole=True):
    assert tg.n_segments == otg.n_segments
    assert np.array_equal(tg.segment_offsets, otg.seg_offsets)
    assert np.array_equal(tg.segment_status, otg.seg_status)
    assert (tg.first_bad_uid, tg.bad_status) == (otg.first_bad_uid, otg.bad_status)
    if whole:
        s, o = tg.segments, otg.seg
        assert np.array_equal(s["element"], o["element"])
        for key in ("px", "py", "qx", "qy", "len"):
            assert np.array_equal(s[key], o[key]), key
            scale = np.maximum(np.abs(o[key]), 1e-300)
            assert (np.abs(s[key] - o[key]) / scale).max(initial=0.0) <= P_TOL


def assert_volumes_close(otg, tg):
    vo, vg = otg.volumes(), tg.volumes
    assert np.abs(vg - vo).max() <= 1e-10 * np.abs(vo).max()


# ---- trace! ------------------------------------------------------------------------------------------
def test_trace_goldens_through_host_api(pincell_model):  # test/runtests.jl:10-27
    tg = rt.TrackGenerator(pincell_model, G.MAIN["n_azim"], G.MAIN["delta"])
    rt.trace_(tg)
    assert tg.n_total_tracks == G.MAIN["n_total_tracks"]
    assert tg.n_tracks_x.tolist() == G.MAIN["n_tracks_x"] and tg.n_tracks_y.tolist() == G.MAIN["n_tracks_y"]
    assert tg.n_tracks.tolist() == G.MAIN["n_tracks"]
    aq = tg.azimuthal_quadrature
    assert (rt.nazim(aq), rt.nazim2(aq), rt.nazim4(aq)) == (8, 4, 2)
    assert all(math.isclose(d, G.MAIN["delta_eff"], rel_tol=rt.RTOL_DEFAULT) for d in aq.deltas)
    assert np.allclose(aq.phis, G.MAIN["phis"], rtol=rt.RTOL_DEFAULT, atol=0)


@pytest.mark.parametrize("n_azim,table", [(4, G.LINKS_4), (8, G.LINKS_8)])
def test_reflection_goldens_through_host_api(pincell_model, n_azim, table):  # test/runtests.jl:46-335
    bcs = rt.BoundaryConditions(**{k: getattr(rt, v) for k, v in G.REFLECTION_BCS.items()})
    tg = rt.TrackGenerator(pincell_model, n_azim, 0.8, bcs=bcs)
    rt.trace_(tg)
    for uid, (bf, bb, nf, nb, df, db) in table.items():
        tr = tg.tracks_by_uid[uid]
        assert int(rt.bc_fwd(tr)) == G.BC_CODE[bf] and int(rt.bc_bwd(tr)) == G.BC_CODE[bb]
        assert tr.next_track_fwd.uid == nf and tr.next_track_bwd.uid == nb
        assert int(rt.dir_next_track_fwd(tr)) == G.DIR_CODE[df] and int(rt.dir_next_track_bwd(tr)) == G.DIR_CODE[db]


@pytest.mark.parametrize("n_azim,delta,bcs", [(8, 0.02, (0, 0, 0, 0)), (16, 0.08, (1, 1, 1, 1)), (32, 0.013, (2, 2, 2, 2)),
                                             (4, 0.8, (0, 1, 0, 1)), (64, 0.05, (2, 1, 0, 2))])
def test_trace_matches_oracle_bitwise(pincell_model, n_azim, delta, bcs):
    mesh = rt.Mesh(pincell_model)
    otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), n_azim, delta, bcs=bcs).trace()
    tg = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs_of(bcs))
    rt.trace_(tg)
    assert_tracks_equal(otg, tg)


# ---- segmentize! -------------------------------------------------------------------------------------
SEQ = rt.RT_SEG_SEQUENTIAL


@pytest.mark.parametrize("flags,chunk", [(0, None), (rt.RT_SEG_LITERAL, None), (rt.RT_SEG_NO_CHUNKS, None),
                                         (rt.RT_SEG_LITERAL | rt.RT_SEG_NO_CHUNKS, None), (0, 4), (0, 1), (rt.RT_SEG_LITERAL, 3),
                                         (SEQ, None), (SEQ | rt.RT_SEG_LITERAL, None), (SEQ | rt.RT_SEG_NO_CHUNKS, None), (SEQ, 4),
                                         (SEQ, 1)])
@pytest.mark.parametrize("n_azim,delta", [(8, 0.02), (16, 0.08), (32, 0.01), (4, 0.8)])
def test_pincell_segments_match_oracle(pincell_model, n_azim, delta, flags, chunk):
    otg, tg = run_both(pincell_model, n_azim, delta, flags=flags, chunk_segments=chunk)
    assert_tracks_equal(otg, tg)
    assert_segments_equal(otg, tg)
    assert_volumes_close(otg, tg)
    assert otg.bad_status == 0
    if not flags & SEQ:  # the hybrid pipeline (sign-test count walk + geometric fill walk); the default (3) ran above
        for pipeline in (0,):
            otg, tg = run_both(pincell_model, n_azim, delta, flags=flags, chunk_segments=chunk, pipeline=pipeline)
            assert_segments_equal(otg, tg)
            assert_volumes_close(otg, tg)
            assert tg.info("verify_fallbacks") == 0


def test_reference_invariants_on_gpu_result(pincell_model):  # test/runtests.jl:30-43
    tg = rt.TrackGenerator(pincell_model, 8, 0.02)
    rt.segmentize_(rt.trace_(tg))

    def approx(a, b):
        return np.linalg.norm(a - b) <= rt.RTOL_DEFAULT * max(np.linalg.norm(a), np.linalg.norm(b))

    for track in tg.tracks_by_uid:
        segs = track.segments
        assert approx(track.p, segs[0].p) and approx(track.q, segs[-1].q)
        assert math.isclose(track.ell, sum(rt.ell(s) for s in segs), rel_tol=rt.RTOL_DEFAULT)
    assert math.isclose(tg.volumes.sum(), 2.56, rel_tol=1e-9)


@pytest.mark.parametrize("seed,n,n_azim,delta", [(1234, 60, 16, 0.01), (7, 37, 32, 0.004), (99, 90, 8, 0.003)])
def test_jittered_mesh_matches_oracle(seed, n, n_azim, delta):
    model = rt.synth.jittered_triangle_mesh(n, n, seed=seed)
    otg, tg = run_both(model, n_azim, delta)
    assert_segments_equal(otg, tg)
    assert_volumes_close(otg, tg)
    st = tg.stats()
    assert st["fast_transitions"] > 0.8 * tg.n_segments
    assert tg.info("verify_fallbacks") == 0
    otg, tg = run_both(model, n_azim, delta, chunk_segments=5)  # many tiny chunks: exercises every hand-off rule
    assert_segments_equal(otg, tg)
    assert_volumes_close(otg, tg)
    otg, tg = run_both(model, n_azim, delta, flags=SEQ, chunk_segments=5)  # the sequential kernels on the same input
    assert_segments_equal(otg, tg)
    assert_volumes_close(otg, tg)
    walk_counters = ("fast_transitions", "literal_iterations", "nn_queries", "knn_queries")
    counters = {(3, None): [st[c] for c in walk_counters]}
    for pipeline, chunk in ((0, 5), (0, None), (3, 5), (3, 600)):  # hybrid pipeline; single walk with tiny / with multi-block chunks
        otg, tg = run_both(model, n_azim, delta, chunk_segments=chunk, pipeline=pipeline)
        assert_segments_equal(otg, tg)
        assert_volumes_close(otg, tg)
        assert tg.info("verify_fallbacks") == 0
        counters[pipeline, chunk] = [tg.stats()[c] for c in walk_counters]
    for chunk in (5, None):  # the count pass of the hybrid pipeline is the single walk's walk: same decisions, same counters
        assert counters[0, chunk] == counters[3, chunk]


def test_offset_domain_and_rectangle():
    """non-zero bb_min and a non-square domain (not covered by any reference test)"""
    model = rt.synth.jittered_triangle_mesh(40, 25, lx=2.0, ly=1.25, seed=5, x0=-3.5, y0=10.0)
    otg, tg = run_both(model, 16, 0.02, bcs=(1, 1, 1, 1))
    assert_tracks_equal(otg, tg)
    assert_segments_equal(otg, tg)


def test_pin_lattice_matches_oracle():
    model = rt.synth.pin_lattice_mesh(2, 1.26, 0.4096, 0.0655, 0.05, seed=3)
    otg, tg = run_both(model, 32, 0.004, bcs=(1, 1, 1, 1))
    assert_segments_equal(otg, tg)
    assert_volumes_close(otg, tg)


def test_cfg2_bwr_matches_oracle():
    model, n_azim, delta = rt.synth.workload("cfg2")
    otg, tg = run_both(model, n_azim, delta, bcs=(1, 1, 1, 1))
    assert_segments_equal(otg, tg)
    otg, tg = run_both(model, n_azim, 0.002, bcs=(1, 1, 1, 1))  # the delta test/bwr-gmsh.jl:151 itself uses
    assert_segments_equal(otg, tg)


def test_commensurate_boundary_vertex_hits(pincell_model):
    """delta=0.08 makes every track start and end on a boundary mesh node (SURVEY B.1): n_int=3 paths."""
    otg, tg = run_both(pincell_model, 16, 0.08)
    assert otg.stats()["n_int_ge3"] > 100
    assert_segments_equal(otg, tg)


def test_structured_mesh_exact_vertex_crossings():
    """unjittered structured mesh: tracks through vertices / along edges, and error statuses must agree too"""
    model = rt.synth.jittered_triangle_mesh(16, 16, jitter=0.0)
    otg, tg = run_both(model, 8, 0.0625)
    assert_segments_equal(otg, tg)


@pytest.mark.parametrize("pipeline", [0, 1, 3])
@pytest.mark.parametrize("chunk", [None, 7])
def test_batched_fill_equals_single_shot(pincell_model, chunk, pipeline):
    otg, tg = run_both(pincell_model, 32, 0.01, capacity=20000, chunk_segments=chunk, pipeline=pipeline)
    assert tg.n_segments == otg.n_segments and np.array_equal(tg.segment_offsets, otg.seg_offsets)
    # only the last batch is resident: compare it with the tail of the oracle's arrays
    s = tg.segments
    n = s["px"].shape[0]
    assert 0 < n <= 20000
    for key in ("px", "py", "qx", "qy", "len", "element"):
        assert np.array_equal(s[key], otg.seg[key][-n:])
    assert_volumes_close(otg, tg)
    last = tg.tracks_by_uid[tg.n_total_tracks].segments
    assert len(last) == otg.seg_counts[-1]


def test_idempotent_and_max_iter(pincell_model):
    tg = rt.TrackGenerator(pincell_model, 8, 0.05)
    rt.segmentize_(rt.trace_(tg))
    a = {k: v.copy() for k, v in tg.segments.items()}
    a_off = tg.segment_offsets.copy()
    v0 = tg.volumes.copy()
    rt.segmentize_(tg)
    assert all(np.array_equal(a[k], tg.segments[k]) for k in a)
    assert np.abs(tg.volumes - v0).max() <= 1e-12
    # MAX_ITER cap (src/track.jl:104,119): tracks stop at max_iter segments and fail the length check
    rt.segmentize_(tg, max_iter=10, check=False)
    assert np.diff(tg.segment_offsets).max() == 10 and tg.bad_status == 2
    tg.set_option("chunk_segments", 3)
    tg.set_option("target_walkers", 1e9)
    rt.segmentize_(tg, max_iter=10, check=False)
    assert np.diff(tg.segment_offsets).max() == 10 and tg.bad_status == 2
    off = tg.segment_offsets
    for u in (0, len(off) // 2, len(off) - 2):  # capped tracks keep the FIRST max_iter segments of the full walk
        n_u = off[u + 1] - off[u]
        assert n_u == min(10, a_off[u + 1] - a_off[u])
        assert np.array_equal(tg.segments["element"][off[u]:off[u + 1]], a["element"][a_off[u]:a_off[u] + n_u])


def test_optimistic_evaluation_cancelled_on_the_device_is_repeated():
    """The steady-state call launches the evaluation behind the walk without reading the segment total back (DESIGN.md section 6);
    the scan's guard cancels it on the device when the batch does not fit the Segment columns of the previous call, and the call
    is repeated on the careful path: same bits as the oracle, one cancellation counted."""
    mesh = rt.Mesh(rt.synth.jittered_triangle_mesh(60, 60, seed=5))
    otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), 16, 0.01).trace().segmentize(check=False, nthreads=8)
    tg = rt.TrackGenerator(mesh, 16, 0.01)
    rt.trace_(tg)
    rt.segmentize_(tg, max_iter=3, check=False)  # first call after trace!: careful path, Segment columns sized for 3 segments per track
    small = tg.n_segments
    rt.segmentize_(tg, max_iter=3, check=False)  # optimistic, fits
    assert tg.n_segments == small and tg.info("optimistic_cancels") == 0
    rt.segmentize_(tg, check=False)  # ~20x the segments: does not fit
    assert tg.info("optimistic_cancels") == 1 and tg.n_segments > 5 * small and tg.info("verify_fallbacks") == 0
    assert_segments_equal(otg, tg)
    assert_volumes_close(otg, tg)
    rt.segmentize_(tg, check=False)  # the careful call re-fitted the columns: optimistic again, and it fits
    assert tg.info("optimistic_cancels") == 1
    assert_segments_equal(otg, tg)
    assert_volumes_close(otg, tg)


def test_error_paths(pincell_model):
    tg = rt.TrackGenerator(pincell_model, 8, 0.05)
    with pytest.raises(RuntimeError):
        rt.segmentize_(tg)  # src/trackgenerator.jl:360-361
    for args in [(0, 0.1), (6, 0.1), (8, 0.0)]:
        with pytest.raises(rt.DomainError):
            rt.TrackGenerator(pincell_model, *args)


def test_neighbour_table(pincell_model):
    tg = rt.TrackGenerator(pincell_model, 4, 0.8)
    nb = tg.neighbours()
    tri = pincell_model.triangles0()
    edges = {}
    for c, t in enumerate(tri):
        for k in range(3):
            edges.setdefault(frozenset((t[k], t[(k + 1) % 3])), []).append(c)
    for c, t in enumerate(tri):
        for k in range(3):
            cs = [x for x in edges[frozenset((t[k], t[(k + 1) % 3]))] if x != c]
            assert nb[c, k] == (cs[0] + 1 if cs else 0)


@pytest.mark.parametrize("which", ["pincell", "lattice", "offset"])
def test_device_side_ingestion(pincell_model, which):
    """SURVEY 8f-3: vertex->cells table and bounding box built on the device (rt_mesh_upload with NULL tables) equal the host
    ones (Gridap order: ascending cell id around every node; exact min/max), and the whole path gives the same bits."""
    if which == "pincell":
        model, n_azim, delta = pincell_model, 8, 0.02
    elif which == "lattice":
        model, n_azim, delta = rt.synth.pin_lattice_mesh(3, 1.26, 0.4096, 0.0655, 0.09, 5), 16, 0.03
    else:
        model, n_azim, delta = rt.synth.jittered_triangle_mesh(23, 17, 2.5, 1.25, 0.3, 11, x0=-3.25, y0=7.5), 8, 0.04
    host = rt.Mesh(model)
    dev = rt.Mesh(model, device_ingest=True)
    assert dev.bb_min is None and dev._node_cells is None
    tg = rt.TrackGenerator(dev, n_azim, delta, bcs=bcs_of((1, 1, 1, 1)))
    assert np.array_equal(dev.bb_min, host.bb_min) and np.array_equal(dev.bb_max, host.bb_max)
    ptrs, data = tg.device_node_cells()
    assert np.array_equal(ptrs, host.node_cells[0]) and np.array_equal(data, host.node_cells[1])
    rt.segmentize_(rt.trace_(tg))
    otg = OracleTrackGenerator(OracleMesh.from_mesh(host), n_azim, delta, bcs=(1, 1, 1, 1)).trace().segmentize()
    assert_segments_equal(otg, tg)
    assert_volumes_close(otg, tg)


def test_sweep_facing_device_views(pincell_model):
    """SURVEY 8f-1: what a transport sweep consumes stays on the device -- track linkage (rt_tracks_device), azimuthal weights
    computed on the device (rt_quadrature_device) and per-segment optical lengths tau = sigma_t[element] * len
    (rt_optical_lengths, the Segment.tau field the reference leaves empty)."""
    import torch

    bcs = (0, 1, 2, 1)
    tg = rt.TrackGenerator(pincell_model, 16, 0.05, bcs=bcs_of(bcs))
    rt.segmentize_(rt.trace_(tg))
    # linkage: the device arrays equal the downloaded track table, which equals the oracle's (test_trace_matches_oracle_bitwise)
    v, t = tg.track_view(), tg.track_data
    assert v["uid_begin"] == 1 and v["n_tracks"] == tg.n_total_tracks
    dev = {k: torch.as_tensor(c, device="cuda").cpu().numpy() for k, c in v.items() if isinstance(c, api.DeviceColumn)}
    assert np.array_equal(dev["px"], t["p"][:, 0]) and np.array_equal(dev["qy"], t["q"][:, 1]) and np.array_equal(dev["len"], t["len"])
    assert np.array_equal(np.stack([dev["a"], dev["b"], dev["c"]], 1), t["abc"])
    assert np.array_equal(dev["azim"] + 1, t["azim_idx"]) and np.array_equal(dev["track_idx"], t["track_idx"])
    for k in ("next_fwd", "next_bwd", "bc_fwd", "bc_bwd", "dir_fwd", "dir_bwd"):
        assert np.array_equal(dev[k], t[k]), k
    # weights: bit-identical to init_weights! on the host (src/azimuthal_quad.jl:35-53; the reference's formula as it stands)
    omega, qv = tg.quadrature_device()
    assert np.array_equal(omega, tg.azimuthal_quadrature.weights) and np.all(omega > 0) and np.array_equal(omega, omega[::-1])
    assert np.array_equal(torch.as_tensor(qv["omega"], device="cuda").cpu().numpy(), omega)
    assert np.array_equal(torch.as_tensor(qv["delta_eff"], device="cuda").cpu().numpy(), tg.azimuthal_quadrature.deltas)
    # optical lengths, both layouts, 7 groups (C5G7)
    rng = np.random.default_rng(3)
    sigma = rng.uniform(0.1, 2.0, size=(pincell_model.num_cells, 7))
    s = tg.segments
    ref = sigma[s["element"] - 1] * s["len"][:, None]
    tau0, d0 = tg.optical_lengths(sigma, layout=0)
    assert np.array_equal(tau0, ref)
    assert np.array_equal(torch.as_tensor(d0, device="cuda").cpu().numpy().reshape(-1, 7), ref)
    tau1, _ = tg.optical_lengths(sigma, layout=1)
    assert np.array_equal(tau1, ref.T)


def test_shard_planner_matches_device(pincell_model):
    from raytracing_jl_b200 import _lib
    from raytracing_jl_b200.api import _angle_tables
    from raytracing_jl_b200.distributed import plan_shards

    tg = rt.TrackGenerator(pincell_model, 32, 0.01)
    _, _, tan_t, dxe, dye = _angle_tables(tg)
    for parts in (2, 3, 8):
        host = plan_shards(tg, parts)
        dev = np.zeros(parts + 1, np.int64)
        _lib.check(tg._ctx, _lib.lib().rt_plan_shards(tg._ctx, 16, tg.n_tracks_x, tg.n_tracks_y, tg.azimuthal_quadrature.phis,
                                                      tan_t, dxe, dye, parts, dev))
        assert dev[0] == 1 and dev[-1] == tg.n_total_tracks + 1
        assert np.abs(dev - host).max() <= 1  # summation order may move a split by one track


def test_sharded_union_equals_whole(pincell_model):
    """uid-range shards on one GPU: the union of the shards' segments is the single-context result"""
    whole = rt.TrackGenerator(pincell_model, 16, 0.02, bcs=bcs_of((1, 1, 1, 1)))
    rt.segmentize_(rt.trace_(whole))
    parts, vol = [], np.zeros_like(whole.volumes)
    for r in range(3):
        tg = rt.TrackGenerator(pincell_model, 16, 0.02, bcs=bcs_of((1, 1, 1, 1)), shard=(r, 3))
        rt.segmentize_(rt.trace_(tg))
        parts.append(tg)
        vol += tg.volumes
    assert parts[0].uid_begin == 1 and parts[-1].uid_end == whole.n_total_tracks + 1
    for key in ("px", "py", "qx", "qy", "len", "element"):
        assert np.array_equal(np.concatenate([p.segments[key] for p in parts]), whole.segments[key])
    assert np.abs(vol - whole.volumes).max() <= 1e-12
    assert np.array_equal(np.concatenate([p.track_data["next_fwd"] for p in parts]), whole.track_data["next_fwd"])


# ---- size-independent properties at a larger size -------------------------------------------------------
def test_properties_at_scale():
    model, n_azim, delta = rt.synth.workload("cfg3", scale=0.25)  # ~250 k triangles
    tg = rt.TrackGenerator(model, n_azim, 4 * delta, bcs=bcs_of((1, 1, 1, 1)))
    rt.segmentize_(rt.trace_(tg), check=False)
    off, s, t = tg.segment_offsets, tg.segments, tg.track_data
    ok = tg.segment_status == 0
    assert ok.mean() > 0.999
    seg_sum = np.add.reduceat(s["len"], off[:-1])
    assert np.all(np.abs(seg_sum[ok] - t["len"][ok]) <= rt.RTOL_DEFAULT * t["len"][ok])
    # contiguity q_k == p_{k+1} inside a track (bit-identical on generic transitions, close otherwise)
    inner = np.ones(s["px"].shape[0], bool)
    inner[off[1:-1]] = False
    d = np.hypot(s["qx"][:-1] - s["px"][1:], s["qy"][:-1] - s["py"][1:])[inner[1:]]
    assert d.max() < 1e-6 and (d == 0).mean() > 0.99
    assert s["element"].min() >= 1 and s["element"].max() <= model.num_cells
    assert math.isclose(tg.volumes.sum(), 1.0, rel_tol=1e-6)
    # idempotence of the checksum
    chk = (float(s["len"].sum()), int(s["element"].astype(np.int64).sum()))
    rt.segmentize_(tg, check=False)
    s2 = tg.segments
    assert chk == (float(s2["len"].sum()), int(s2["element"].astype(np.int64).sum()))


def test_cfg4_full_size_pipelines_agree():
    """BASELINE.json configs[3] at its FULL size (3.7 M cells, 3.5 M tracks, 7.9e9 segments, batched fill over a recycled
    buffer).  Size-independent properties: the three independently coded pipelines produce the same stream of Segment records
    (order- and bit-sensitive per-batch checksums computed on the device), the traced volumes add up to the mesh area, and
    the tracks that fail the reference's own checks are the same in every pipeline.  Spot checks against the oracle: uid
    ranges spread over the shard, plus every failing track, are compared bit for bit."""
    import torch

    from raytracing_jl_b200 import _lib as L

    model, n_azim, delta = rt.synth.workload("cfg4")
    mesh = rt.Mesh(model)
    tg = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs_of((1, 1, 1, 1)))
    rt.trace_(tg)
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, 1_500_000_000))
    area = rt.synth.mesh_area(model)
    n = tg.n_total_tracks
    ranges = [(int(u), int(u) + 40) for u in np.linspace(1, n - 40, 7)]
    keys = ("px", "py", "qx", "qy", "len", "element")
    M64 = (1 << 64) - 1
    results = []
    for pipeline in (0, 1, 3):
        tg.set_option("pipeline", pipeline)
        chk, slices, sums = [], {}, {}

        def on_batch(b, chk=chk, slices=slices, sums=sums):
            torch.cuda.synchronize()
            cols = {k: torch.as_tensor(getattr(b, k), device="cuda") for k in keys}
            off = torch.as_tensor(api.DeviceColumn(b.d_offsets, n + 1, "<i8"), device="cuda")
            row = [b.uid_begin, b.uid_end, b.n_segments]
            step = 1 << 27
            for lo in range(0, b.n_segments, step):
                hi = min(b.n_segments, lo + step)
                # weights from the GLOBAL segment position: the sums do not depend on how a pipeline cuts the batches
                w = (torch.arange(lo, hi, device="cuda", dtype=torch.int64) + int(b.offset_base)) % 1021 + 1
                # (the device sums wrap modulo 2^64, so the totals are kept modulo 2^64 too: independent of the batch cuts)
                sums["element"] = (sums.get("element", 0) + int((cols["element"][lo:hi].to(torch.int64) * w).sum())) & M64
                for k in keys[:5]:  # bit patterns, so that any differing bit changes the sum
                    sums[k] = (sums.get(k, 0) + int((cols[k][lo:hi].view(torch.int64) & 0xFFFFFFFF).mul_(w).sum())) & M64
            chk.append(tuple(row))
            for (u0, u1) in ranges:
                if b.uid_begin <= u0 and u1 <= b.uid_end:
                    o = off[u0 - 1:u1].cpu().numpy() - b.offset_base
                    slices[(u0, u1)] = (o - o[0], {k: cols[k][int(o[0]):int(o[-1])].cpu().numpy() for k in keys})
            torch.cuda.synchronize()

        rt.segmentize_(tg, rtol=1e-6, check=False, on_batch=on_batch)
        assert tg.info("verify_fallbacks") == 0
        assert tg.n_segments > 7_000_000_000 and len(chk) >= 4
        assert sum(r[2] for r in chk) == tg.n_segments
        assert math.isclose(tg.volumes.sum(), area, rel_tol=1e-8)
        assert [r[0] for r in chk[1:]] == [r[1] for r in chk[:-1]] and chk[0][0] == 1 and chk[-1][1] == n + 1  # batches tile the uids
        results.append((tg.n_segments, sums, tg.segment_offsets.copy(), tg.segment_status.copy(), slices))
    for other in results[1:]:
        assert other[0] == results[0][0], (other[0], results[0][0])
        assert other[1] == results[0][1], (other[1], results[0][1])
        assert np.array_equal(other[2], results[0][2]) and np.array_equal(other[3], results[0][3])
    # ---- the oracle on the sampled uid ranges and on every failing track
    off, status, slices = results[0][2], results[0][3], results[0][4]
    bad = np.nonzero(status)[0] + 1
    assert 0 < bad.size < 1e-5 * n  # the reference's own end-of-track / length-check failures (DESIGN.md, "Error behaviour")
    otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), n_azim, delta, bcs=(1, 1, 1, 1)).trace()
    checked = 0
    for (u0, u1), (o, cols) in slices.items():
        otg.segmentize(rtol=1e-6, uid_begin=u0, uid_end=u1, fetch=True, check=False)
        assert np.array_equal(otg.seg_offsets, o)
        for k in keys:
            assert np.array_equal(otg.seg[k], cols[k]), (u0, k)
        assert np.array_equal(otg.seg_status, status[u0 - 1:u1 - 1])
        checked += int(o[-1])
        otg.free_segments()
    assert len(slices) >= 5 and checked > 100_000
    for uid in bad:
        otg.segmentize(rtol=1e-6, uid_begin=int(uid), uid_end=int(uid) + 1, fetch=False, check=False)
        assert otg.seg_status[0] == status[uid - 1] and otg.seg_counts[0] == off[uid] - off[uid - 1], uid
        otg.free_segments()


def test_cfg3_named_size_every_segment_matches_oracle_for_all_bcs():
    """BASELINE.json configs[2] AT ITS NAMED SIZE (the workload bench.py times): 1.0 M cells, n_phi = 64, delta = 1e-3, and the
    config's "vacuum/periodic/reflective sweep".  Every track record and every one of the ~5e7 Segment records is compared
    with the oracle bit for bit, with the reference's default rtol (88 tracks fail its length check, src/track.jl:171-175:
    same uids, same status) -- boundary conditions only enter trace! (src/trackgenerator.jl:231-265), the walk never reads them."""
    model, n_azim, delta = rt.synth.workload("cfg3")
    mesh = rt.Mesh(model)
    omesh = OracleMesh.from_mesh(mesh)
    threads = os.cpu_count() or 8
    tg = None
    for bcs in ((0, 0, 0, 0), (2, 2, 2, 2), (1, 1, 1, 1)):
        otg = OracleTrackGenerator(omesh, n_azim, delta, bcs=bcs).trace()
        otg.segmentize(check=False, nthreads=threads)
        if tg is not None:
            tg.close()
        tg = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs_of(bcs))
        rt.trace_(tg)
        rt.segmentize_(tg, check=False)
        assert tg.n_total_tracks > 40_000 and tg.n_segments > 45_000_000
        assert_tracks_equal(otg, tg)
        assert_segments_equal(otg, tg)
        assert_volumes_close(otg, tg)
        assert tg.info("verify_fallbacks") == 0
        assert 0 < np.count_nonzero(tg.segment_status) < 200 and set(np.unique(tg.segment_status)) == {0, 2}
        # ... and with the rtol bench.py passes (the remedy the reference's error message suggests) every track completes
        otg.free_segments()
        del otg
    rt.segmentize_(tg, rtol=1e-6, check=True)
    assert np.count_nonzero(tg.segment_status) == 0
    tg.close()


def test_cfg5_named_size_sampled_against_oracle():
    """BASELINE.json configs[4] at its FULL size on one GPU (18 M cells, 52 M tracks, 2.6e11 segments through the batched
    evaluation): uid ranges spread over the whole track set and a sample of every failing-status class are compared with the
    oracle bit for bit; the traced volumes add up to the mesh area; the batches tile the uid range."""
    import torch

    from raytracing_jl_b200 import _lib as L

    model, n_azim, delta = rt.synth.workload("cfg5")
    mesh = rt.Mesh(model)
    tg = rt.TrackGenerator(mesh, n_azim, delta, bcs=bcs_of((1, 1, 1, 1)))
    rt.trace_(tg)
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, 2_000_000_000))
    area = rt.synth.mesh_area(model)
    n = tg.n_total_tracks
    assert n > 50_000_000
    rng = np.random.default_rng(5)
    starts = np.unique(np.concatenate([np.linspace(1, n - 24, 10).astype(np.int64), rng.integers(1, n - 24, 6)]))
    ranges = [(int(u), int(u) + 24) for u in starts]
    keys = ("px", "py", "qx", "qy", "len", "element")
    rows, slices = [], {}

    def on_batch(b):
        torch.cuda.synchronize()
        rows.append((b.uid_begin, b.uid_end, b.n_segments))
        hit = [(u0, u1) for (u0, u1) in ranges if b.uid_begin <= u0 and u1 <= b.uid_end]
        if not hit:
            return
        cols = {k: torch.as_tensor(getattr(b, k), device="cuda") for k in keys}
        off = torch.as_tensor(api.DeviceColumn(b.d_offsets, n + 1, "<i8"), device="cuda")
        for (u0, u1) in hit:
            o = off[u0 - 1:u1].cpu().numpy() - b.offset_base
            slices[(u0, u1)] = (o - o[0], {k: cols[k][int(o[0]):int(o[-1])].cpu().numpy() for k in keys})
        torch.cuda.synchronize()

    rt.segmentize_(tg, rtol=1e-6, check=False, on_batch=on_batch)
    assert tg.info("verify_fallbacks") == 0
    assert tg.n_segments > 2.5e11 and sum(r[2] for r in rows) == tg.n_segments
    assert [r[0] for r in rows[1:]] == [r[1] for r in rows[:-1]] and rows[0][0] == 1 and rows[-1][1] == n + 1
    assert math.isclose(tg.volumes.sum(), area, rel_tol=1e-8)
    off, status = tg.segment_offsets, tg.segment_status
    tr = tg.tracks_by_uid[1]
    with pytest.raises(LookupError):  # only the last batch is resident
        tr.segments
    otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), n_azim, delta, bcs=(1, 1, 1, 1)).trace()
    checked = 0
    for (u0, u1), (o, cols) in slices.items():
        otg.segmentize(rtol=1e-6, uid_begin=u0, uid_end=u1, fetch=True, check=False, nthreads=8)
        assert np.array_equal(otg.seg_offsets, o), (u0, u1)
        for k in keys:
            assert np.array_equal(otg.seg[k], cols[k]), (u0, k)
        assert np.array_equal(otg.seg_status, status[u0 - 1:u1 - 1])
        checked += int(o[-1])
        otg.free_segments()
    assert len(slices) >= 8 and checked > 500_000
    # the reference's own failures (DESIGN.md "Error behaviour"): same uids, same status, same number of segments before the stop
    classes = [int(c) for c in np.unique(status) if c != 0]
    assert classes and 0 < np.count_nonzero(status) < 0.02 * n
    for c in classes:
        uids = np.nonzero(status == c)[0] + 1
        for uid in rng.choice(uids, size=min(48, uids.size), replace=False):
            otg.segmentize(rtol=1e-6, uid_begin=int(uid), uid_end=int(uid) + 1, fetch=False, check=False)
            assert otg.seg_status[0] == c and otg.seg_counts[0] == off[uid] - off[uid - 1], (c, uid)
            otg.free_segments()
    tg.close()


def test_compact_download_is_bit_identical(pincell_model):
    """rt_segments_download_compact: q, len, element + the exception list rebuild exactly the columns of the full download --
    on a mesh with many literal records (pincell: every track starts and ends on a boundary node for delta = 0.08), with tiny
    chunks, with a batched evaluation (only the last batch is resident), and track by track (p_range)."""
    from raytracing_jl_b200 import _lib as L

    cases = [(pincell_model, 16, 0.08, None, 0), (pincell_model, 32, 0.01, 5, 0), (rt.synth.jittered_triangle_mesh(60, 60, seed=3), 16, 0.01, None, 0),
             (pincell_model, 32, 0.01, None, 20000)]
    for model, n_azim, delta, chunk, cap in cases:
        tg = rt.TrackGenerator(model, n_azim, delta, bcs=bcs_of((1, 0, 2, 2)))
        rt.trace_(tg)
        if chunk:
            tg.set_option("chunk_segments", chunk)
            tg.set_option("target_walkers", 1e9)
        if cap:
            L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, cap))
        rt.segmentize_(tg, check=False)
        full = {k: v.copy() for k, v in tg.fetch_segments().items()}
        for pinned in (False, True):
            comp = tg.fetch_segments(pinned=pinned, compact=True)
            assert comp.compact and 0 < tg.n_exceptions < max(64, 0.2 * full["px"].size)
            u0, u1, base, n = tg.resident_batch()
            off = tg.segment_offsets - base
            for uid in (u0, (u0 + u1) // 2, u1 - 1):  # track by track, before the whole columns are rebuilt
                lo, hi = int(off[uid - tg.uid_begin]), int(off[uid - tg.uid_begin + 1])
                px, py = comp.p_range(lo, hi)
                assert np.array_equal(px, full["px"][lo:hi]) and np.array_equal(py, full["py"][lo:hi])
                segs = tg.tracks_by_uid[uid].segments
                if len(segs):
                    assert np.array_equal(segs[0].p, [full["px"][lo], full["py"][lo]]) and np.array_equal(segs[-1].p, [full["px"][hi - 1], full["py"][hi - 1]])
            for k in api.SegmentColumns.KEYS:
                assert np.array_equal(comp[k], full[k]), k
        small = tg.fetch_segments(compact=True, max_exceptions=8)  # too small a list: the call reports the count and is repeated
        assert all(np.array_equal(small[k], full[k]) for k in api.SegmentColumns.KEYS)
        small = tg.fetch_segments(compact="q")  # 20 bytes per segment: len rebuilt as norm(p - q) too
        assert "len" not in small._cols
        assert all(np.array_equal(small[k], full[k]) for k in api.SegmentColumns.KEYS)
        tg.close()


@pytest.mark.parametrize("frac,n_azim,delta,bcs", [(0.5, 16, 0.02, (1, 1, 1, 1)), (1.0, 8, 0.03, (0, 2, 0, 2)), (0.15, 32, 0.011, (2, 2, 1, 1))])
def test_mixed_quad_triangle_mesh_matches_oracle(frac, n_azim, delta, bcs):
    """SURVEY 8(f)-4: meshes that mix triangles and 4-node quadrilaterals (all quadrilaterals for frac = 1).  Cells are located
    with the reference's point_in_quadrangle (src/mesh.jl:184-201), chords come from its 4-edge intersections()
    (src/intersection.jl:42-44, 81-95): only the literal walk runs on such a mesh, and it reproduces the oracle bit for bit."""
    model = rt.synth.mixed_quad_triangle_mesh(31, 23, 1.5, 1.1, jitter=0.22, seed=17, quad_fraction=frac, x0=-0.3, y0=0.7)
    assert model.has_quads
    otg, tg = run_both(model, n_azim, delta, bcs=bcs)
    assert_tracks_equal(otg, tg)
    assert_segments_equal(otg, tg)
    assert_volumes_close(otg, tg)
    assert otg.bad_status == 0 and tg.stats()["fast_transitions"] == 0  # every step re-located like src/track.jl:122
    quad_ids = np.nonzero(model.cell_sizes == 4)[0] + 1
    assert np.isin(tg.segments["element"], quad_ids).mean() > 0.3 * frac  # (a quadrilateral is crossed about as often as the two triangles it replaces)
    comp = tg.fetch_segments(compact=True)
    full = tg.fetch_segments()
    assert all(np.array_equal(comp[k], full[k]) for k in api.SegmentColumns.KEYS)
    sx, sy, sz = rt.plotdata.segment_lines(tg, uid=[1, tg.n_total_tracks])  # src/plot_recipes.jl:50-74 on two tracks
    n1 = len(tg.tracks_by_uid[1].segments)
    assert sx.shape[0] == 2 and sx.shape[1] == n1 + len(tg.tracks_by_uid[tg.n_total_tracks].segments)
    assert np.array_equal(sx[0, :n1], full["px"][:n1]) and np.array_equal(sz[0, :n1], full["element"][:n1])
    tx, ty = rt.plotdata.track_lines(tg)
    assert tx.shape == (2, tg.n_total_tracks) and np.array_equal(tx[1], tg.track_data["q"][:, 0])
    with pytest.raises(rt.RTError):
        tg.neighbours()
    with pytest.raises(rt.RTError):
        tg.element_volumes()


def test_resident_batch_guards_and_k_limit(pincell_model):
    """Track.segments refuses tracks whose batch is not resident (instead of indexing another batch's columns); k beyond
    RT_MAX_K is rejected instead of being clamped; k within it reaches the kNN fallback unchanged."""
    from raytracing_jl_b200 import _lib as L

    tg = rt.TrackGenerator(pincell_model, 16, 0.02)
    rt.trace_(tg)
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, 20000))
    rt.segmentize_(tg)
    u0, u1, base, nres = tg.resident_batch()
    assert u0 > 1 and u1 == tg.n_total_tracks + 1 and 0 < nres <= 20000
    with pytest.raises(LookupError):
        tg.tracks_by_uid[1].segments
    with pytest.raises(LookupError):
        tg.tracks_by_uid[u0 - 1].segments
    assert len(tg.tracks_by_uid[u0].segments) == tg.segment_offsets[u0] - tg.segment_offsets[u0 - 1]
    assert tg.tracks_by_uid[u1 - 1].segments[-1].element >= 1
    a = tg.fetch_segments()  # copies by default: a later run does not change them
    keep = {k: v.copy() for k, v in a.items()}
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, 0))
    rt.segmentize_(tg)
    assert tg.resident_batch()[0] == 1 and len(tg.tracks_by_uid[1].segments) > 0
    assert all(np.array_equal(a[k], keep[k]) for k in a)
    with pytest.raises(rt.RTError):
        rt.segmentize_(tg, k=33)
    otg = OracleTrackGenerator(OracleMesh.from_mesh(rt.Mesh(pincell_model)), 16, 0.02).trace().segmentize(k=32)
    rt.segmentize_(tg, k=32)
    assert_segments_equal(otg, tg)


@pytest.mark.parametrize("exp_span", [0, 3, 40, 400, 520, 1022])
def test_shared_reciprocal_division_is_ieee(pincell_model, exp_span):
    """geom.cuh div_shared(x, recip_prepare(d)) == x / d bit for bit (2.7e8 quotients per span, incl. hard cases)"""
    import ctypes as C

    from raytracing_jl_b200 import _lib

    tg = rt.TrackGenerator(pincell_model, 4, 0.8)
    bad = C.c_int64(-1)
    _lib.check(tg._ctx, _lib.lib().rt_selftest_division(tg._ctx, 1 << 22, 12345 + exp_span, exp_span, C.byref(bad)))
    assert bad.value == 0


def test_self_verifying_pipelines_fall_back_to_sequential(pincell_model):
    """a failed verification in k_eval3 / k_walk<true> restarts the call with the sequential kernels; the result is the same"""
    mesh = rt.Mesh(pincell_model)
    otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), 16, 0.02).trace().segmentize(check=False, nthreads=8)
    tg = rt.TrackGenerator(mesh, 16, 0.02)
    rt.trace_(tg)
    rt.segmentize_(tg, check=False)
    assert_segments_equal(otg, tg)
    for pipeline in (0, 3):
        tg.set_option("pipeline", pipeline)
        tg.set_option("debug_verify_fail", 0)
        rt.segmentize_(tg, check=False)
        assert tg.info("verify_fallbacks") == 0
        assert_segments_equal(otg, tg)
        tg.set_option("debug_verify_fail", 1)
        rt.segmentize_(tg, check=False)
        assert tg.info("verify_fallbacks") == 1
        assert_segments_equal(otg, tg)
        assert_volumes_close(otg, tg)
    tg.set_option("debug_verify_fail", 0)
    tg.set_option("pipeline", 1)
    rt.segmentize_(tg, check=False)
    assert tg.info("verify_fallbacks") == 0
    assert_segments_equal(otg, tg)


def test_single_walk_pipeline_batches_and_pool_exhaustion():
    """pipeline 3 (k_march + k_eval3): uid batches of the count walk when the record pool is small, sub-batches of the
    evaluation when the Segment columns are small, chunks longer than one pool block, and the fall-back to the hybrid pipeline
    when the pool runs out -- always the oracle's bits."""
    model = rt.synth.jittered_triangle_mesh(130, 130, seed=21)
    mesh = rt.Mesh(model)
    otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), 16, 0.004).trace().segmentize(check=False, nthreads=8)
    tg = rt.TrackGenerator(mesh, 16, 0.004)
    rt.trace_(tg)
    tg.set_option("pipeline", 3)
    tg.set_option("chunk_segments", 700)  # one walker per track: up to ~370 segments = two pool blocks (walk.cuh kRecBlock = 256)
    rt.segmentize_(tg, check=False)
    assert tg.info("verify_fallbacks") == 0 and tg.info("count_batches") == 1
    assert_segments_equal(otg, tg)
    assert_volumes_close(otg, tg)
    off_all = tg.segment_offsets.copy()
    tg.set_option("chunk_segments", 40)
    tg.set_option("pool_slots", 2048)  # many count batches
    rt.segmentize_(tg, check=False)
    assert tg.info("verify_fallbacks") == 0 and tg.info("count_batches") > 3
    assert np.array_equal(tg.segment_offsets, off_all) and tg.n_segments == otg.n_segments
    s = tg.segments  # the last count batch is resident
    n = s["px"].shape[0]
    assert 0 < n < otg.n_segments
    for key in ("px", "py", "qx", "qy", "len", "element"):
        assert np.array_equal(s[key], otg.seg[key][-n:])
    assert_volumes_close(otg, tg)
    from raytracing_jl_b200 import _lib as L
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, 5000))  # ... and evaluation sub-batches inside each of them
    import torch

    got = {key: np.zeros_like(otg.seg[key]) for key in ("px", "py", "qx", "qy", "len", "element")}
    cuts = []

    def on_batch(b):  # EVERY batch of the stream, not only the resident last one
        for key in got:
            got[key][b.offset_base:b.offset_base + b.n_segments] = torch.as_tensor(getattr(b, key), device="cuda")[:b.n_segments].cpu().numpy()
        cuts.append((b.uid_begin, b.uid_end))

    rt.segmentize_(tg, check=False, on_batch=on_batch)
    assert tg.info("count_batches") > 3 and len(cuts) > 3 * tg.info("count_batches")
    assert cuts[0][0] == 1 and cuts[-1][1] == tg.n_total_tracks + 1 and all(a[1] == b[0] for a, b in zip(cuts, cuts[1:]))
    for key in got:
        assert np.array_equal(got[key], otg.seg[key]), key
    assert tg.info("verify_fallbacks") == 0 and np.array_equal(tg.segment_offsets, off_all)
    n = tg.segments["px"].shape[0]
    assert 0 < n <= 5000
    for key in ("px", "py", "qx", "qy", "len", "element"):
        assert np.array_equal(tg.segments[key], otg.seg[key][-n:])
    assert_volumes_close(otg, tg)
    L.check(tg._ctx, L.lib().rt_set_segment_capacity(tg._ctx, 0))
    tg.set_option("pool_slots", 0)
    tg.set_option("pool_extra", 0)  # no spare blocks: chunks longer than one block exhaust the pool
    tg.set_option("chunk_segments", 700)
    rt.segmentize_(tg, check=False)
    assert tg.info("verify_fallbacks") == 1
    assert_segments_equal(otg, tg)
    assert_volumes_close(otg, tg)


def test_element_volumes_and_volume_correction(pincell_model):
    """SURVEY 8f-2: element_volume (src/trackgenerator.jl:402-411) on the device, bit-equal to the reference's formula, and the
    volume correction the reference only announces (:388-397): lengths scaled by area/volume per element, after which the
    traced volumes (src/trackgenerator.jl:371-386) of the corrected segments equal the exact areas."""
    for model, n_azim, delta in ((pincell_model, 8, 0.02), (rt.synth.jittered_triangle_mesh(40, 33, 2.0, 1.5, 0.3, 17, x0=-1.0, y0=4.0), 16, 0.01)):
        tg = rt.TrackGenerator(model, n_azim, delta, volume_correction=True)
        xy = np.asarray(model.node_coordinates, dtype=np.float64).reshape(-1, 2)
        tri = model.triangles0()
        x1, x2, x3 = xy[tri[:, 0]], xy[tri[:, 1]], xy[tri[:, 2]]
        ax, ay, bx, by = x2[:, 0] - x1[:, 0], x2[:, 1] - x1[:, 1], x3[:, 0] - x1[:, 0], x3[:, 1] - x1[:, 1]
        area = 1 / 2 * np.abs(ax * by - ay * bx)  # 1 / 2 * abs((x2 - x1) x (x3 - x1))
        assert np.array_equal(tg.element_volumes(), area)
        assert math.isclose(area.sum(), rt.synth.mesh_area(model), rel_tol=1e-12)
        rt.trace_(tg)
        tg.volume_correction = False
        rt.segmentize_(tg)
        raw = {k: v.copy() for k, v in tg.segments.items()}
        tg.volume_correction = True
        rt.segmentize_(tg)
        vol = tg.volumes.copy()  # the traced volumes of THIS call (atomic accumulation: the last bits differ from call to call)
        f = tg.volume_factors
        assert np.array_equal(f, np.where(vol > 0, area / np.where(vol > 0, vol, 1.0), 1.0))
        s = tg.segments
        e = raw["element"] - 1
        assert np.array_equal(s["len"], raw["len"] * f[e])  # lengths scaled ...
        assert all(np.array_equal(s[k], raw[k]) for k in ("px", "py", "qx", "qy", "element"))  # ... end points untouched
        azim = np.repeat(np.array([t.azim_idx for t in tg.tracks_by_uid]) - 1, np.diff(tg.segment_offsets))
        traced = np.bincount(e, weights=tg.azimuthal_quadrature.deltas[azim] * s["len"], minlength=area.size) / (n_azim // 2)
        crossed = vol > 0
        assert crossed.mean() > 0.99 and np.allclose(traced[crossed], area[crossed], rtol=1e-12, atol=0.0)
