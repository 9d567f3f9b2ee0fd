"""SURVEY 8(f)-4 on the CPU: the oracle's restatement of point_in_quadrangle (src/mesh.jl:184-201) and of the 4-edge
intersections (src/intersection.jl:42-44, 81-95) on quadrilateral cells, mixed-mesh host tables, and the plot-friendly views of
src/plot_recipes.jl."""
import os

import numpy as np
import pytest

import raytracing_jl_b200 as rt
from oracle.oracle import OracleError, OracleMesh, OracleTrackGenerator


def unit_quads():
    # two unit squares side by side, nodes stored as a counter-clockwise cycle; and the same squares cut into triangles
    xy = np.array([[0, 0], [1, 0], [2, 0], [0, 1], [1, 1], [2, 1]], float)
    quads = rt.UnstructuredDiscreteModel.from_cells(xy, [(0, 1, 4, 3), (1, 2, 5, 4)])
    tris = rt.UnstructuredDiscreteModel.from_cells(xy, [(0, 1, 4), (0, 4, 3), (1, 2, 5), (1, 5, 4)])
    return quads, tris


def test_point_in_quadrangle_and_four_edge_chords():
    quads, _ = unit_quads()
    om = OracleMesh.from_mesh(rt.Mesh(quads))
    assert om.point_in_element(1, 0.9, 0.1) and om.point_in_element(1, 0.1, 0.9)  # both halves of the square, whatever triangle holds them
    assert om.point_in_element(1, 1.0, 0.5) and om.point_in_element(2, 1.0, 0.5)  # the shared edge belongs to both (tolerant test)
    assert not om.point_in_element(1, 1.5, 0.5) and om.point_in_element(2, 1.5, 0.5)
    assert om.find_element(0.25, 0.75) == 1 and om.find_element(1.75, 0.25) == 2
    # a horizontal line y = 0.5: general form of (0, .5) -> (2, .5)
    abc = np.zeros(3)
    from oracle.oracle import lib
    lib().orc_general_form(0.0, 0.5, 2.0, 0.5, abc)
    rc, pq, ed, n = om.intersections(1, abc, 0.0)
    assert rc == 0 and n == 2 and np.allclose(pq, [0, .5, 1, .5]) and sorted(ed.tolist()) == [1, 3]  # right and left edge of the cycle
    # the diagonal y = x crosses square 1 through two of its corners: four edge hits, the farthest pair wins (src/intersection.jl:81-95)
    lib().orc_general_form(0.0, 0.0, 1.0, 1.0, abc)
    rc, pq, ed, n = om.intersections(1, abc, np.pi / 4)
    assert rc == 0 and n == 4 and np.allclose(pq, [0, 0, 1, 1])


def test_mixed_mesh_walk_covers_the_area_and_matches_its_triangulation_in_length():
    model = rt.synth.mixed_quad_triangle_mesh(9, 7, 1.8, 1.4, jitter=0.2, seed=5, quad_fraction=0.5)
    assert model.has_quads and set(model.cell_sizes.tolist()) == {3, 4}
    mesh = rt.Mesh(model)
    ptrs, data = mesh.node_cells
    assert ptrs[-1] - 1 == model.cell_data.size  # every (cell, node) incidence once
    otg = OracleTrackGenerator(OracleMesh.from_mesh(mesh), 16, 0.03, bcs=(1, 1, 1, 1)).trace().segmentize()
    assert otg.bad_status == 0 and np.all(otg.seg_status == 0)
    area = rt.synth.mesh_area(model)
    assert np.isclose(area, 1.8 * 1.4, rtol=1e-12)
    assert np.isclose(otg.volumes().sum(), area, rtol=2e-3)  # the tracked volumes approximate the areas, cell by cell
    # reference invariants (test/runtests.jl:30-43): first p, last q, sum of lengths
    off, t = otg.seg_offsets, otg.tracks
    for u in range(otg.n_total_tracks):
        a, b = off[u], off[u + 1]
        assert b > a
        assert np.allclose([otg.seg["px"][a], otg.seg["py"][a]], t["p"][u], rtol=0, atol=1e-7)
        assert np.allclose([otg.seg["qx"][b - 1], otg.seg["qy"][b - 1]], t["q"][u], rtol=0, atol=1e-7)
        assert np.isclose(otg.seg["len"][a:b].sum(), t["len"][u], rtol=1.5e-8)
    quad_ids = np.nonzero(model.cell_sizes == 4)[0] + 1
    assert np.isin(otg.seg["element"], quad_ids).mean() > 0.3  # the walk does cross the quadrilaterals


def test_k_limit_is_an_error_not_a_clamp():
    d = rt.synth.jittered_triangle_mesh(6, 6, seed=2)
    otg = OracleTrackGenerator(OracleMesh.from_mesh(rt.Mesh(d)), 4, 0.2).trace()
    otg.segmentize(k=32)
    with pytest.raises(OracleError):
        otg.segmentize(k=33)


def test_plot_views_match_the_recipes():
    quads, tris = unit_quads()
    x, y = rt.plotdata.mesh_lines(rt.Mesh(quads))  # src/plot_recipes.jl:76-107: (nn + 1) x n_cells, closed cycles
    assert x.shape == (5, 2) and np.array_equal(x[:, 0], [0, 1, 1, 0, 0]) and np.array_equal(y[:, 1], [0, 0, 1, 1, 0])
    x, y = rt.plotdata.mesh_lines(rt.Mesh(tris))
    assert x.shape == (4, 4) and np.array_equal(x[0], x[-1])
    mixed = rt.synth.mixed_quad_triangle_mesh(3, 2, seed=1)
    with pytest.raises(ValueError):
        rt.plotdata.mesh_lines(rt.Mesh(mixed))  # the reference's `error("error")` for cells of different sizes
    fx, fy = rt.plotdata.flat_mesh_edges(rt.Mesh(mixed))
    assert np.isnan(fx).sum() == mixed.num_cells - 1 and fx.size == mixed.cell_data.size + 2 * mixed.num_cells - 1
    cols = dict(px=np.array([0., 1.]), py=np.array([0., 0.]), qx=np.array([1., 2.]), qy=np.array([0., 1.]), element=np.array([7, 9], np.int32))
    sx, sy, sz = rt.plotdata.segment_lines(cols)  # src/plot_recipes.jl:26-48
    assert np.array_equal(sx, [[0, 1], [1, 2]]) and np.array_equal(sz, [[7, 9], [7, 9]])
    fx, fy, fz = rt.plotdata.flat_polyline(sx, sy, sz)
    assert np.array_equal(fx[[0, 1, 3, 4]], [0, 1, 1, 2]) and np.isnan(fx[2]) and fx.size == 5 and np.array_equal(fz[[0, 1, 3, 4]], [7, 7, 9, 9])


def _write_gridap_json(path, xy, ptrs, data):
    import json

    with open(path, "w") as fh:
        json.dump({"grid": {"Dp": 2, "node_coordinates": xy.tolist(), "cell_node_ids": {"ptrs": ptrs.tolist(), "data": data.tolist()}}}, fh)


def _write_msh41(path, xy, tri0, seed=7):
    """MSH 4.1 ASCII laid out the way Gmsh writes a 2-D mesh: node blocks per geometric entity in no particular tag order, tags
    with gaps, a node no triangle uses, point and line elements before the triangles, triangle nodes not in ascending order."""
    rng = np.random.default_rng(seed)
    tags = 2 * np.arange(xy.shape[0] + 1) + 2
    coords = np.vstack([xy, [[0.123, 0.456]]])  # the last node is referenced by the point element only
    tags[-1] = 1
    blocks = np.array_split(rng.permutation(coords.shape[0]), 3)
    out = ["$MeshFormat", "4.1 0 8", "$EndMeshFormat", "$Nodes", f"{len(blocks)} {coords.shape[0]} 1 {tags.max()}"]
    for dim, b in enumerate(blocks):
        out.append(f"{dim} {dim + 1} 0 {b.size}")
        out += [str(tags[i]) for i in b] + [f"{float(coords[i, 0])!r} {float(coords[i, 1])!r} 0" for i in b]
    out.append("$EndNodes")
    rot = np.roll(tags[tri0], 1, axis=1)
    halves = np.array_split(np.arange(rot.shape[0]), 2)
    out += ["$Elements", f"{2 + len(halves)} {1 + 2 + rot.shape[0]} 1 {3 + rot.shape[0]}", "0 1 15 1", f"1 {tags[-1]}",
            "1 1 1 2", f"2 {tags[tri0[0, 0]]} {tags[tri0[0, 1]]}", f"3 {tags[tri0[1, 0]]} {tags[tri0[1, 1]]}"]
    for s, h in enumerate(halves):
        out.append(f"2 {s + 1} 2 {h.size}")
        out += [f"{4 + e} {a} {b} {c}" for e, (a, b, c) in zip(h, rot[h])]
    out.append("$EndElements")
    with open(path, "w") as fh:
        fh.write("\n".join(out) + "\n")


def test_mesh_readers_on_the_reference_files(tmp_path):
    """The readers for the two formats the reference ships its quick-start mesh in (demo/pincell.json: Gridap JSON, loaded by
    test/runtests.jl:5-6; demo/pincell.msh: MSH 4.1) give back the committed fixture tests/golden/pincell.npz, which was read
    from those files.  The reference's files are not part of this repository: the fixture is written in both formats here."""
    import raytracing_jl_b200 as rt

    d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pincell.npz"))
    xy, ptrs, data = d["node_coordinates"], d["cell_ptrs"], d["cell_data"]
    _write_gridap_json(tmp_path / "pincell.json", xy, ptrs, data)
    _write_msh41(tmp_path / "pincell.msh", xy, data.reshape(-1, 3).astype(np.int64) - 1)
    for m in (rt.DiscreteModelFromFile(str(tmp_path / "pincell.json")), rt.GmshDiscreteModel(str(tmp_path / "pincell.msh"))):
        assert np.array_equal(m.node_coordinates, xy)
        assert np.array_equal(m.cell_ptrs, ptrs) and np.array_equal(m.cell_data, data)
