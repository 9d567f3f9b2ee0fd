"""Material regions read from the two model formats: UnstructuredDiscreteModel.cell_regions gives every cell the 1-based position of
the first listed name whose tag holds the cell's entity, for Gridap JSON (labeling names / tags / entities_2) and MSH 4.1 physical
groups.  The files are written here from synthetic meshes with a known assignment."""
import json
import os
import re

import numpy as np
import pytest

import raytracing_jl_b200 as rt
from raytracing_jl_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gridap_json(path, model, entities, names, tags):
    d = {"grid": {"node_coordinates": model.node_coordinates.reshape(-1).tolist(), "Dp": 2,
                  "cell_node_ids": {"ptrs": model.cell_ptrs.tolist(), "data": model.cell_data.tolist()}},
         "labeling": {"names": names, "tags": tags, "entities_2": [int(e) for e in entities]}}
    with open(path, "w") as fh:
        json.dump(d, fh)


@pytest.fixture(scope="module")
def labelled(tmp_path_factory):
    """a jittered mesh whose cells carry entities 1..5; tags a = {1, 2}, b = {2, 3} (entity 2 in both), c = {4, 5}, and a
    boundary name that tags no cell"""
    model = rt.synth.jittered_triangle_mesh(12, 9, seed=3)
    ent = 1 + np.random.default_rng(5).integers(0, 5, size=model.num_cells)
    path = str(tmp_path_factory.mktemp("json") / "model.json")
    gridap_json(path, model, ent, ["boundary", "a", "b", "c"], [[9], [1, 2], [2, 3], [4, 5]])
    return rt.DiscreteModelFromFile(path), ent


def test_json_regions(labelled):
    model, ent = labelled
    r = model.cell_regions(["a", "b", "c"])
    assert r.dtype == np.int32 and r.shape == (model.num_cells,)
    assert np.array_equal(r, np.select([np.isin(ent, [1, 2]), ent == 3], [1, 2], 3))
    # overlapping tags: the first listed name wins
    r = model.cell_regions(["b", "a", "c"])
    assert np.array_equal(r, np.select([np.isin(ent, [2, 3]), ent == 1], [1, 2], 3))
    assert np.array_equal(model.cell_regions(["c", "boundary", "b", "a"]), np.select([ent >= 4, np.isin(ent, [2, 3])], [1, 3], 4))


def test_json_region_errors(labelled):
    model, ent = labelled
    with pytest.raises(ValueError, match="unknown label 'fuel'"):
        model.cell_regions(["a", "fuel"])
    missing = np.flatnonzero(~np.isin(ent, [1, 2, 3]))
    with pytest.raises(ValueError, match=rf"^{missing.size} cells are in none of the tags \['a', 'b'\]; the first is cell {missing[0] + 1} "):
        model.cell_regions(["a", "b"])
    with pytest.raises(ValueError, match="no cell labeling"):
        rt.synth.jittered_triangle_mesh(3, 3).cell_regions(["a"])


def write_msh(path, model, blocks, seed=0):
    """MSH 4.1 ASCII of a triangle model: node tags shuffled, sparse and with one unused node (the reader renumbers), boundary
    line elements on curve 7, and the triangles in `blocks` = [(surface tag, cell ids), ...] in that order.  Physical groups:
    "outer" (dim 1, tag 1), "fuel" (dim 2, tag 1: the same number as the curve group), "moderator" (dim 2, tag 2), "all" (dim 2,
    tag 3, on every surface)."""
    rng = np.random.default_rng(seed)
    n = model.num_nodes
    tags = rng.permutation(n + 1)[:n] * 3 + 5  # node i -> tag
    unused = int(tags.max() + 4)
    tri = model.triangles0()
    xy = model.node_coordinates
    lines = ["$MeshFormat", "4.1 0 8", "$EndMeshFormat", "$PhysicalNames", "4", '1 1 "outer"', '2 1 "fuel"', '2 2 "moderator"',
             '2 3 "all"', "$EndPhysicalNames", "$Entities", f"0 1 {len(blocks)} 0", "7 0 0 0 1 1 0 1 1 0"]
    for j, (s, _) in enumerate(blocks):  # surface: box, 2 physical tags (fuel or moderator, and all), 1 bounding curve
        lines.append(f"{s} 0 0 0 1 1 0 2 {1 if j == 0 else 2} 3 1 7")
    lines.append("$EndEntities")
    order = rng.permutation(n)
    lines += ["$Nodes", f"1 {n + 1} 1 {unused}", f"2 1 0 {n + 1}"]
    lines += [str(int(tags[i])) for i in order] + [str(unused)]
    lines += [f"{float(xy[i, 0])!r} {float(xy[i, 1])!r} 0" for i in order] + ["0.5 0.5 0"]
    lines.append("$EndNodes")
    bnd = [(tags[a], tags[b]) for a, b in ((tri[0, 0], tri[0, 1]), (tri[1, 1], tri[1, 2]))]
    n_el = len(bnd) + sum(len(c) for _, c in blocks)
    lines += ["$Elements", f"{1 + len(blocks)} {n_el} 1 {n_el}", f"1 7 1 {len(bnd)}"]
    k = 1
    for a, b in bnd:
        lines.append(f"{k} {a} {b}")
        k += 1
    for s, cells in blocks:
        lines.append(f"2 {s} 2 {len(cells)}")
        for c in cells:
            lines.append(f"{k} " + " ".join(str(int(tags[v])) for v in tri[c][::-1]))
            k += 1
    lines.append("$EndElements")
    with open(path, "w") as fh:
        fh.write("\n".join(lines) + "\n")


def test_msh_regions(tmp_path):
    """two triangle entities (surface 20 written first, then 10), boundary line elements, node tags shuffled and renumbered: the
    cells come in file order with their surface's groups"""
    src = rt.synth.jittered_triangle_mesh(10, 8, seed=9)
    cells = np.arange(src.num_cells)
    first, second = cells[cells % 3 == 0], cells[cells % 3 != 0]
    path = str(tmp_path / "m.msh")
    write_msh(path, src, [(20, first), (10, second)])
    model = rt.GmshDiscreteModel(path)
    assert model.num_cells == src.num_cells and model.num_nodes == src.num_nodes
    # geometry: the cells in file order, node ids ascending within a cell
    order = np.concatenate([first, second])
    got = model.node_coordinates[model.triangles0()]
    want = np.sort(src.triangles0()[order], axis=1)
    assert np.array_equal(np.sort(got.view(np.complex128)[..., 0], axis=1), np.sort(src.node_coordinates[want].view(np.complex128)[..., 0], axis=1))
    assert model.labels["names"] == ["outer", "fuel", "moderator", "all"]
    assert model.labels["entities_2"] == [20] * first.size + [10] * second.size
    expect = np.r_[np.ones(first.size, np.int32), np.full(second.size, 2, np.int32)]
    assert np.array_equal(model.cell_regions(["fuel", "moderator"]), expect)
    assert np.array_equal(model.cell_regions(["moderator", "fuel"]), 3 - expect)
    assert np.array_equal(model.cell_regions(["fuel", "all"]), expect)  # overlap: the first listed name wins
    assert np.all(model.cell_regions(["all", "fuel"]) == 1)
    with pytest.raises(ValueError, match=rf"{second.size} cells are in none of the tags \['outer', 'fuel'\]; the first is cell {first.size + 1} "):
        model.cell_regions(["outer", "fuel"])
    # the same file without renumbering keeps the unused node, and the same cells and regions
    raw = rt.GmshDiscreteModel(path, renumber=False)
    assert raw.num_nodes == src.num_nodes + 1
    assert np.array_equal(raw.cell_regions(["fuel", "moderator"]), expect)


def test_region_calls_are_bound():
    """the three region calls are declared in the header, in the ctypes table and called by the Julia glue"""
    hdr = open(os.path.join(ROOT, "include", "rt_b200.h")).read()
    jl = open(os.path.join(ROOT, "julia", "RayTracingB200.jl")).read()
    for name in ("rt_set_regions", "rt_optical_lengths_by_region", "rt_region_volumes"):
        assert re.search(rf"\bint {name}\(", hdr) and name in _lib.SYMBOLS and f"(:{name}, LIBRT_B200)" in jl, name
