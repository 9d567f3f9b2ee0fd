"""find_element(mesh, x, k) (src/mesh.jl:103-146) for batches of points, without a GPU: the oracle's find_element
run over a batch (tests/locate_oracle.c) against the pure-Python brute force of tests/pyref.py on the point families that exercise it -- random points,
every node, edge midpoints (exact nearest-node distance ties), points on shared edges, points just outside the bounding box within
and beyond the tolerance of the barycentric test, points far away -- and plotdata.cell_raster against hand-built matrices.  The
families are shared with tests/test_gpu_find_element.py, which pins the device on the oracle."""
import numpy as np

import raytracing_jl_b200 as rt
from oracle.oracle import OracleMesh
from tests.locate_oracle import find_elements as oracle_find_elements
from tests.pyref import RTOL, PyRef


def cell_edges(mesh):
    """(a, b) 0-based node pairs of every cell edge (consecutive stored nodes, like intersections), each undirected edge once,
    and whether it is shared by two cells"""
    ptrs, data = (a.astype(np.int64) - 1 for a in mesh.cell_nodes)
    sizes = np.diff(ptrs)
    nxt = np.arange(data.size) + 1
    nxt[ptrs[1:] - 1] = ptrs[:-1]
    e = np.sort(np.stack([data, data[nxt]], 1), axis=1)
    assert e.shape[0] == sizes.sum()
    uniq, counts = np.unique(e, axis=0, return_counts=True)
    return uniq, counts == 2


def point_families(mesh, seed=0, n_random=2000):
    """{family: (n, 2) points} over the mesh's bounding box"""
    rng = np.random.default_rng(seed)
    xy = mesh.model.node_coordinates
    lo, hi = np.asarray(mesh.bb_min, float), np.asarray(mesh.bb_max, float)
    w = hi - lo
    edges, shared = cell_edges(mesh)
    a, b = xy[edges[:, 0]], xy[edges[:, 1]]
    t = rng.uniform(size=(int(shared.sum()), 1))
    # a boundary point pushed out of the box by d (in units of the box size) across the side it lies on
    on_side = np.concatenate([np.stack([rng.uniform(lo[0], hi[0], 200), np.full(200, y)], 1) for y in (lo[1], hi[1])] +
                             [np.stack([np.full(200, x), rng.uniform(lo[1], hi[1], 200)], 1) for x in (lo[0], hi[0])])
    outward = np.repeat(np.array([[0, -1], [0, 1], [-1, 0], [1, 0]], float), 200, axis=0)
    h = np.sqrt(w[0] * w[1] / mesh.num_cells)  # a typical cell size: the barycentric tolerance is about RTOL * h in distance
    return {
        "random": lo + rng.uniform(-0.02, 1.02, size=(n_random, 2)) * w,
        "nodes": xy.copy(),
        "edge_midpoints": 0.5 * (a + b),
        "shared_edges": a[shared] + t * (b[shared] - a[shared]),
        "on_box": on_side,
        "outside_within_tol": on_side + outward * (0.01 * RTOL * h),
        "outside_beyond_tol": on_side + outward * (100.0 * RTOL * h),
        "far": lo + rng.uniform(-1.0, 1.0, size=(200, 2)) * 50.0 * w,
    }


def jittered(nx=12, ny=9, seed=3):
    return rt.Mesh(rt.synth.jittered_triangle_mesh(nx, ny, 1.3, 0.9, 0.3, seed, x0=-0.4, y0=2.0))


def test_oracle_batch_equals_pure_python(pincell_mesh):
    for mesh in (pincell_mesh, jittered(), rt.Mesh(rt.synth.mixed_quad_triangle_mesh(7, 5, 1.4, 1.0, seed=2, quad_fraction=0.5))):
        om, ref = OracleMesh.from_mesh(mesh), PyRef(mesh)
        for name, pts in point_families(mesh, n_random=600).items():
            # the knn branch is entered where no cell around the nearest node passes
            knn_want = sum(not any(ref.pie(c, p) for c in ref.node_cells(ref.nearest(p, 1)[0])) for p in pts)
            for k in (1, 2, 5):
                ids, n_knn = oracle_find_elements(om, mesh, pts, k)
                want = np.array([ref.find_element(p, k) for p in pts], np.int32)
                assert np.array_equal(ids, want), (name, k, np.nonzero(ids != want)[0][:5])
                assert n_knn == knn_want, (name, k)
                # the batch is the per-point call in a loop
                one = np.array([om.find_element(float(x), float(y), k) for x, y in pts[:50]], np.int32)
                assert np.array_equal(ids[:50], one)


def test_families_cover_what_they_name(pincell_mesh):
    mesh = jittered()
    om = OracleMesh.from_mesh(mesh)
    fam = point_families(mesh)
    ids = {name: oracle_find_elements(om, mesh, p)[0] for name, p in fam.items()}
    for name in ("random", "nodes", "edge_midpoints", "shared_edges", "on_box", "outside_within_tol"):
        assert np.all(ids[name][(fam[name] >= mesh.bb_min).all(1) & (fam[name] <= mesh.bb_max).all(1)] > 0), name
    assert np.all(ids["outside_within_tol"] > 0)  # the tolerant test accepts them
    assert np.all(ids["outside_beyond_tol"] == -1) and np.all(ids["far"] == -1)
    # the midpoint of an edge is as far from both its nodes: at least some of them are exact distance ties
    assert sum(om_tied(om, p) for p in fam["edge_midpoints"][:300]) > 0
    # the k-nearest fallback (src/mesh.jl:123) is taken inside the domain too, where it finds the cell
    inside = fam["random"][(fam["random"] > mesh.bb_min).all(1) & (fam["random"] < mesh.bb_max).all(1)]
    ids_in, n_knn = oracle_find_elements(om, mesh, inside)
    assert n_knn > 0 and np.all(ids_in > 0)


def om_tied(om, p):
    from oracle.oracle import lib

    return bool(lib().orc_nn_is_tied(om._h, float(p[0]), float(p[1])))


class _Located:
    """stands in for a TrackGenerator: the bounding box and the ids find_elements returns are given"""

    def __init__(self, bb_min, bb_max, ids):
        self.mesh = type("M", (), {"bb_min": np.array(bb_min, float), "bb_max": np.array(bb_max, float)})()
        self.ids, self.points = np.asarray(ids, np.int32), None

    def find_elements(self, xy, k=2):
        self.points = xy
        return self.ids.copy(), None


def test_cell_raster_assembles_the_heatmap():
    # 3 x 2 pixels over [0, 3] x [1, 2]: centres x = 0.5, 1.5, 2.5 and y = 1.25, 1.75; pixel (row j, column i) is point j*3 + i
    tg = _Located([0, 1], [3, 2], [4, -1, 2, 1, 1, -1])
    x, y, z = rt.plotdata.cell_raster(tg, 3, 2)
    assert np.array_equal(x, [[0.5, 1.5, 2.5], [0.5, 1.5, 2.5]]) and np.array_equal(y, [[1.25] * 3, [1.75] * 3])
    assert np.array_equal(tg.points, np.stack([x.reshape(-1), y.reshape(-1)], 1))
    assert np.array_equal(z, [[4, np.nan, 2], [1, 1, np.nan]], equal_nan=True)
    values = np.array([10.0, 20.0, 30.0, 40.0])
    _, _, z = rt.plotdata.cell_raster(tg, 3, 2, values)
    assert np.array_equal(z, [[40, np.nan, 20], [10, 10, np.nan]], equal_nan=True)
