"""The reference order of fill_volumes (src/trackgenerator.jl:371-386), restated in numpy: np.add.at adds unbuffered and in index
order, so adding delta_eff[azim] * len over the oracle's segments (uid order, walk order) and dividing by n_azim_2 is the
reference's loop.  It must be bit-equal to the oracle's volumes(); the GPU tests of RT_SEG_EXACT_VOLUMES use it as the reference
for uid shards and batches, where the oracle has no volumes of its own."""
import numpy as np
import pytest

import raytracing_jl_b200 as rt
from oracle.oracle import OracleMesh, OracleTrackGenerator


def fold_volumes(otg, offsets, seg, n_cells, uid_begin=1):
    """volumes[e] += delta_eff[azim(u)] * len(s) over the segments s of the tracks u from uid_begin on, in order; then / n_azim_2.
    offsets / seg: the segments of those tracks (the oracle's seg_offsets / seg, or a fetch of a uid range)."""
    offsets = np.asarray(offsets, np.int64)
    n_tracks = offsets.size - 1
    azim = otg.tracks["azim_idx"][uid_begin - 1:uid_begin - 1 + n_tracks] - 1
    terms = otg.deltas[np.repeat(azim, np.diff(offsets))] * seg["len"]  # each product rounded on its own
    v = np.zeros(n_cells)
    np.add.at(v, seg["element"].astype(np.int64) - 1, terms)
    return v / otg.n2


MESHES = {
    "pincell": None,
    "jittered": (lambda: rt.synth.jittered_triangle_mesh(24, 18, 1.3, 0.9, 0.25, 7), 16, 0.02),
    "mixed": (lambda: rt.synth.mixed_quad_triangle_mesh(19, 15, 1.5, 1.1, jitter=0.2, seed=17, quad_fraction=0.5), 8, 0.04),
}


@pytest.mark.parametrize("mesh", list(MESHES))
def test_numpy_fold_is_the_oracles_volumes(pincell_model, mesh):
    if MESHES[mesh] is None:
        model, n_azim, delta = pincell_model, 16, 0.02
    else:
        make, n_azim, delta = MESHES[mesh]
        model = make()
    m = rt.Mesh(model)
    otg = OracleTrackGenerator(OracleMesh.from_mesh(m), n_azim, delta).trace().segmentize(check=False, nthreads=4)
    v = fold_volumes(otg, otg.seg_offsets, otg.seg, m.num_cells)
    ref = otg.volumes()
    assert v.tobytes() == ref.tobytes()
    # not trivially so: summed in another order, the last bits of some elements differ
    perm = np.random.default_rng(0).permutation(otg.n_segments)
    shuffled = {k: otg.seg[k][perm] for k in ("len", "element")}
    azim = np.repeat(otg.tracks["azim_idx"] - 1, np.diff(otg.seg_offsets))[perm]
    w = np.zeros(m.num_cells)
    np.add.at(w, shuffled["element"].astype(np.int64) - 1, otg.deltas[azim] * shuffled["len"])
    assert np.any(w / otg.n2 != ref) and np.allclose(w / otg.n2, ref, rtol=1e-12, atol=0.0)
