"""The assembly mass properties (DESIGN.md 4.11, cc_assembly_mass_properties_exact) against the true integrals
(tests/exact_mass.py): every part and every pair of groups of aligned boxes against exact Fractions, and curved and
rotated parts against a dense float64 count over every leaf cell, which knows nothing of the hierarchy, the part masks,
the pair rule or the accumulator.

The bars.  Volume: s^3 times a cell count, exact in float64 and in the accumulator, so to the bit.  The other nine
integrals: within 1e-13 B_i (B_i the accumulator's bound, exact_mass.bounds).  For aligned boxes with a dyadic
resolution the index sums, the cell corners and b n, b t are exact; what rounds per block is s^2/12 and the float64
products and sums around it, a few ulp (< 1e-15) of the block's value, and the truncation to the quantum 2^-97 B_i.  The
blocks' values of one integral are bounded in sum by B_i (second moments: xx >= 0, |xy| <= (xx + yy)/2), so a level
adds under 1e-15 B_i, and a plan has at most five levels.  The dense reference is the float64 of the exact sum over its
cells (one rounding)."""
import importlib
import time

import numpy as np
import pytest

import exact_mass as E
from exact_mass import buffers, integrals, plan
from test_gpu_assembly import cb, jit  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

mpm = importlib.import_module("codecad_b200.mass_properties")

# name -> (group builder, its size in leaf cells, resolution, grid)
ALIGNED = {
    "lattice32_grid16": (E.lattice32, 32, 1 / 64, 16),
    "lattice32_grid4": (E.lattice32, 32, 1 / 64, 4),   # four levels; the counter budget cuts the level of 4-cell blocks
    "nested": (E.nested, 48, 1 / 64, 4),
    "far": (E.far, 16, 1 / 64, 16),
}


def _aligned(name):
    make, size, res, grid = ALIGNED[name]
    parts, boxes, box_a, box_b = make(res, size)
    a, _, bs = plan(box_a, box_b, res, grid)
    return parts, boxes, a, res, bs


def _assert_exact(got, rows, box_a, res, bs, what=""):
    want = E.as_float(rows)
    assert got.shape == want.shape
    wrong = np.argwhere(got[:, 0] != want[:, 0]).ravel()
    assert not len(wrong), "%s volumes of sets %s differ: %s vs %s" % (what, wrong[:8], got[wrong[:8], 0], want[wrong[:8], 0])
    bad = np.abs(got - want) > 1e-13 * E.bounds(box_a, res, bs)
    assert not bad.any(), "%s (set, integral) %s" % (what, np.argwhere(bad)[:8].tolist())


def _assert_finish(got, rows, box_a):
    m = max(abs(float(v)) for v in box_a)
    for k, row in enumerate(rows):
        want = E.finish_exact(row)
        mp = mpm.finish(got[k])
        if want is None:
            assert mp.volume == 0
            continue
        vol, c, inertia = want
        I = np.array([[float(v) for v in r] for r in inertia])
        assert mp.volume == float(vol), k
        assert np.allclose(tuple(mp.centroid), [float(v) for v in c], rtol=0, atol=1e-12 * m), k
        assert np.abs(mp.inertia_tensor - I).max() <= 1e-12 * np.abs(I).max(), k


@pytest.mark.parametrize("group", sorted(ALIGNED))
def test_aligned_boxes_are_exact(cb, group):
    """every part and every pair (all 496 for the lattice) against the exact integrals; pairs that touch or do not meet
    have all-zero limbs"""
    parts, boxes, a, res, bs = _aligned(group)
    limbs, exps, st = mpm.assembly_limbs(buffers([E.P.program(p) for p in parts]), a, res, bs)
    if group.endswith("grid4"):
        assert st["launches"] > st["levels"], "no level was cut: %s" % st
    rows = E.exact_sets(boxes)
    got = integrals(limbs, exps)
    _assert_exact(got, rows, a, res, bs)
    empty = [k for k, row in enumerate(rows) if row[0] == 0]
    assert empty and not limbs[empty].any()
    assert len(empty) < len(rows) - len(parts)
    if group != "far":  # (at 2^11 the finish formula itself cancels catastrophically)
        _assert_finish(got, rows, a)


@pytest.mark.parametrize("group", ["lattice32_grid16", "nested", "far"])
def test_standalone_parts_are_exact(cb, jit, group):
    """mass_limbs of each part on both tiers: z-extruded boxes take the column split of the specialised kernel"""
    parts, boxes, a, res, bs = _aligned(group)
    got = []
    for p in buffers([E.P.program(p) for p in parts]):
        limbs, exps, _ = mpm.mass_limbs(p, a, res, bs)
        got.append(integrals(limbs, exps)[0])
    _assert_exact(np.array(got), [E.box_integrals(*b) for b in boxes], a, res, bs, "jit mode %d:" % jit)


def test_shares_add_up_to_the_exact_answers(cb):
    parts, boxes, a, res, bs = _aligned("lattice32_grid16")
    progs = buffers([E.P.program(p) for p in parts])
    total, exps = None, None
    for rank in range(3):
        limbs, exps, _ = mpm.assembly_limbs(progs, a, res, bs, rank, 3)
        total = limbs if total is None else total + limbs
    _assert_exact(integrals(total, exps), E.exact_sets(boxes), a, res, bs)


@pytest.mark.parametrize("group", sorted(E.CURVED))
def test_curved_parts_match_the_dense_reference(cb, group):
    """rotated boxes and cylinders with offsets: every set within 1e-12 B_i of the dense float64 count, whose marginal
    cells the fp32 oracle decides at the library's fp32 cell coordinates (tests/test_exact_mass.py pins how many)"""
    parts, box_a, box_b, res, grid = E.curved_group(group)
    a, _, bs = plan(box_a, box_b, res, grid)
    t0 = time.perf_counter()
    ref = E.dense_reference(parts, a, res, bs)
    host = time.perf_counter() - t0
    limbs, exps, _ = mpm.assembly_limbs(buffers([E.P.program(p) for p in parts]), a, res, bs)
    got = integrals(limbs, exps)
    B = E.bounds(a, res, bs)
    # one leaf cell more or less moves a volume by res^3, far outside the bar: the count must be the same cells
    assert res ** 3 > 1e3 * 1e-12 * B[0]
    bad = np.abs(got - ref.sets) > 1e-12 * B
    assert not bad.any(), "(set, integral) %s; dense reference: %d marginal cells, %d decided by the oracle, %.1f s" % (
        np.argwhere(bad)[:8].tolist(), ref.marginal, ref.disagreements, host)
    assert (ref.sets[len(parts):, 0] > 0).any()
    print("%s: %d marginal cells, %d disagreements, dense reference %.2f s" % (group, ref.marginal, ref.disagreements, host))
