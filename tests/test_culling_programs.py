"""Programs built by tests/programs.py for the culling tests (test_gpu_culling_budget.py), on the CPU.

* Every generated program is what it is meant to be for the loader: an assembly of so many bounded parts
  with (or without) a column split, or a union forest of so many primitives, deeper than the forest kernel's
  first launch provides.
* A float64 restatement of the same geometry agrees with the oracle near the origin and up to 1e6 away: the
  builder's sign and transform conventions put the scene where the tests think it is.
* The edge-group skip of polygon2d (cc_ops.cuh, restated in the oracle) gives the reference formulation's bits
  on polygons of 9 to 2000 vertices up to 1e6 from the origin, at points aimed at its near-ties.
"""
import numpy as np
import pytest

import oracle
import programs as P
from codecad_b200 import _lib

OFFSETS = [0.0, 1e3, 1e4, 1e5, 1e6]
# |float32 - float64| of a distance, in ulp of the largest coordinate in its arithmetic: a few dozen
# float32 operations deep, each rounding by half an ulp of at most that
TOL_ULPS = 16
# decisions (max / min operands, blend conditions, crossing parity) closer than this, in the same ulps, may go
# the other way in float32: such points are left out
MARGIN_ULPS = 64


@pytest.mark.parametrize("offset", OFFSETS)
@pytest.mark.parametrize("carried_by", ["vertices", "translation"])
def test_near_tie_assembly_is_an_assembly_with_columns(offset, carried_by):
    info, _ = _lib.decode_program(P.program(P.near_tie_assembly(offset, carried_by=carried_by)))
    assert info.n_parts == info.n_parts_bounded == 3
    assert info.n_forest_leaves == 0
    assert info.column_invariant_percent == 60 and info.column_axis == 2     # the polygons under a z extrusion


@pytest.mark.parametrize("offset", [0.0, 1e5])
def test_oblique_assembly_has_no_column_split(offset):
    info, _ = _lib.decode_program(P.program(P.oblique_assembly(offset)))
    assert info.n_parts == info.n_parts_bounded == 3
    assert info.column_invariant_percent == 0


def forest(rng, n, offset, r, size=1.0, spread=30.0):
    """n primitives around (offset, offset, offset): combs of 6 (stack depth 6) under a balanced tree"""
    prims = P.primitive_cloud(rng, n, (offset, offset, offset), spread, size)
    return P.balanced([P.comb(prims[i:i + 6], r) for i in range(0, n, 6)], r)


@pytest.mark.parametrize("n,offset,r", [(200, 0.0, -1.0), (300, 1e4, 0.5), (1000, 1e5, 1.0), (2000, 1e3, -1.0)])
def test_forests_are_forests(n, offset, r):
    info, _ = _lib.decode_program(P.program(forest(np.random.default_rng(n), n, offset, r)))
    assert info.n_forest_leaves == info.n_fused == n
    assert info.forest_depth > 4           # deeper than the first launch's stack (cc_forest.cu CCF_STACK_CAP)
    assert info.n_parts == 0


def _compare(tree, words, pts, vertex_max):
    d, _, margin, _ = P.evaluate(tree, pts.astype(np.float64))
    got = oracle.evaluate_points(words, pts)[:, 3].astype(np.float64)
    unit = P.ulp32(np.maximum(np.abs(pts).max(axis=1), vertex_max))
    keep = margin > MARGIN_ULPS * unit
    assert keep.mean() > 0.9, "too few points away from the branch decisions"
    err = np.abs(got - d)[keep] / unit[keep]
    assert err.max() <= TOL_ULPS, "%d points differ by more than %d ulps (worst %.1f)" % (int((err > TOL_ULPS).sum()), TOL_ULPS, err.max())


@pytest.mark.parametrize("offset", OFFSETS)
@pytest.mark.parametrize("carried_by", ["vertices", "translation", "oblique"])
def test_assembly_float64_reference_agrees_with_the_oracle(offset, carried_by):
    rng = np.random.default_rng(7)
    if carried_by == "oblique":
        tree, centre = P.oblique_assembly(offset), P.oblique_centre(offset)
    else:
        tree, centre = P.near_tie_assembly(offset, carried_by=carried_by), np.array([offset, offset, 0.0])
    words = P.program(tree)
    vmax = max(p.max_coordinate() for p in P.leaves(tree)) + 25.0
    box = (centre + rng.uniform(-22, 22, (30000, 3)) * [1, 1, 0.3]).astype(np.float32)
    # and on the medial surfaces: between neighbouring quads, where the parts nearly tie
    if carried_by == "oblique":
        medial = box
    else:
        s = rng.uniform(-20, 20, 5000)
        across = np.array([-np.sin(P.TILT), np.cos(P.TILT), 0.0])
        along = np.array([np.cos(P.TILT), np.sin(P.TILT), 0.0])
        medial = (centre + s[:, None] * along + rng.choice([-0.5, 0.5], 5000)[:, None] * across
                  + rng.uniform(-6, 6, 5000)[:, None] * [0, 0, 1]).astype(np.float32)
    pts = np.concatenate([box, medial])
    _compare(tree, words, pts, vmax)


@pytest.mark.parametrize("n,offset,r", [(200, 0.0, -1.0), (200, 1e3, 0.5), (300, 1e4, 1.0), (300, 1e5, 0.3), (200, 1e6, -1.0)])
def test_forest_float64_reference_agrees_with_the_oracle(n, offset, r):
    """(far away the primitives grow with the offset, 1e-4 of it: blends stay many ulps wide; r is relative
    to their size)"""
    rng = np.random.default_rng(int(n + offset) % 1000)
    size = max(1.0, 1e-4 * offset)
    tree = forest(rng, n, offset, r * size if r >= 0 else r, size=size, spread=30.0 * size)
    words = P.program(tree)
    pts = (np.array([offset] * 3) + rng.uniform(-34, 34, (20000, 3)) * size).astype(np.float32)
    _compare(tree, words, pts, abs(offset) + 34.0 * size)


def test_polygon_edge_group_skip_is_bit_identical():
    """oracle_set_polygon_formulation(1) (the product's loop with its edge-group skip) against (0)"""
    rng = np.random.default_rng(23)
    L = oracle.lib()
    for name, v in P.test_polygons(rng):
        words = P.polygon_program(v)
        pts = np.concatenate([P.near_edge_points(rng, v, 10000), P.near_tie_points(rng, v, 2000)])
        try:
            want = oracle.evaluate_points(words, pts)
            L.oracle_set_polygon_formulation(1)
            got = oracle.evaluate_points(words, pts)
        finally:
            L.oracle_set_polygon_formulation(0)
        diff = np.any(got.view(np.uint32) != want.view(np.uint32), axis=1)
        assert not diff.any(), "%s: %d points differ, e.g. %s" % (name, int(diff.sum()), pts[np.argmax(diff)])
