"""CPU tests of the exact answers behind the assembly mass properties (tests/exact_mass.py): the Fraction integrals of
boxes, the dense float64 reference, and the CPU restatement of the hierarchy (tests/assembly_oracle.py) against both.
Bars: the volume to the bit (s^3 times a cell count is exact in float64), the other integrals within 1e-13 B_i."""
from fractions import Fraction

import numpy as np
import pytest

import exact_mass as E
from assembly_oracle import assembly_mass_properties as oracle_assembly, pair_index


def _assert_exact(got, rows, box_a, resolution, block_sizes):
    want = E.as_float(rows)
    assert got.shape == want.shape
    assert np.array_equal(got[:, 0], want[:, 0]), np.argwhere(got[:, 0] != want[:, 0]).ravel()
    bad = np.abs(got - want) > 1e-13 * E.bounds(box_a, resolution, block_sizes)
    assert not bad.any(), np.argwhere(bad)


def test_box_integrals():
    got = E.box_integrals((0, 0, 0), (1, 2, 3))
    # int over [0,1]x[0,2]x[0,3] of 1, x, y, z, x^2, y^2, z^2, xy, xz, yz
    assert got == [6, 3, 6, 9, 2, 8, 18, 3, Fraction(9, 2), 9]
    assert E.box_integrals((0, 0, 0), (1, 0, 1)) == [0] * 10
    assert E.box_intersection(((0, 0, 0), (2, 2, 2)), ((1, -1, 2), (3, 1, 4))) == ((1, 0, 2), (2, 1, 2))
    vol, c, inertia = E.finish_exact(E.box_integrals((1, 2, 3), (3, 6, 9)))
    # a 2 x 4 x 6 box: I_xx = V (4^2 + 6^2) / 12 about its centre, no products of inertia
    assert vol == 48 and c == [2, 4, 6]
    assert inertia == [[208, 0, 0], [0, 160, 0], [0, 0, 80]]
    assert E.finish_exact([0] * 10) is None


def test_lattice32_has_the_overlaps_it_claims():
    """face neighbours that touch, overlap by 1 cell and by several; edge and corner neighbours overlapping in small
    boxes; overlapping pairs among the parts >= 16 and with part 31"""
    res = 1 / 8
    parts, boxes, _, _ = E.lattice32(res)
    assert len(parts) == 32
    kinds = set()
    live = []
    for i in range(32):
        for j in range(i + 1, 32):
            lo, hi = E.box_intersection(boxes[i], boxes[j])
            ov = sorted(round((h - l) / res) for l, h in zip(lo, hi))
            if ov[0] < 0:
                continue
            steps = sum(a != b for a, b in zip(E._lattice(8)[i][0], E._lattice(8)[j][0]))
            kinds.add(("touch" if ov[0] == 0 else "1" if ov[0] == 1 else "several", steps))
            if ov[0] > 0:
                live.append((i, j))
    assert {("touch", 1), ("1", 1), ("several", 1), ("1", 2), ("1", 3)} <= kinds, kinds
    assert any(i >= 16 for i, _ in live) and any(j == 31 for _, j in live)


def test_nested_counts_the_triple_region_in_each_pair():
    parts, boxes, _, _ = E.nested(1 / 8)
    rows = E.exact_sets(boxes)
    n = len(parts)
    inner = rows[3]                                                   # inside the inner box, inside L
    assert rows[pair_index(n, 0, 3)] == rows[pair_index(n, 1, 3)] == inner
    assert rows[pair_index(n, 1, 4)] == rows[1] and rows[pair_index(n, 0, 1)] == rows[1]   # [A, A]; A inside L
    assert 0 < rows[pair_index(n, 0, 2)][0] < rows[2][0]             # straddles L's face
    assert boxes[1][1][0] == boxes[0][1][0]                          # the inner box touches L's inner face


ALIGNED = {
    "nested": (E.nested, 1 / 8),
    "lattice32": (E.lattice32, 1 / 8),
    "far": (E.far, 1 / 64),
}


@pytest.mark.parametrize("group", sorted(ALIGNED))
def test_dense_reference_is_exact_on_aligned_boxes(group):
    make, res = ALIGNED[group]
    parts, boxes, box_a, box_b = make(res)
    _, _, bs = E.plan(box_a, box_b, res, 4)
    got = E.dense_reference(parts, box_a, res, bs)
    _assert_exact(got.sets, E.exact_sets(boxes), box_a, res, bs)
    assert got.disagreements == 0


RESTATED = {
    "nested": (E.nested, 1 / 8, 4),
    "corner8": (E.corner8, 1 / 8, 4),
    "lattice32": (E.lattice32, 1 / 8, 4),   # pair rows with p >= 16 and the pairs of part 31
}


@pytest.mark.parametrize("group", sorted(RESTATED))
def test_restatement_is_exact_on_aligned_boxes(group):
    """the hierarchy restatement that the GPU tests compare pairs with, pinned to the true integrals: a coarse grid so
    that the parts of a pair are decided at different levels"""
    make, res, grid = RESTATED[group]
    parts, boxes, box_a, box_b = make(res)
    _, _, bs = E.plan(box_a, box_b, res, grid)
    assert len(bs) >= 3
    got = oracle_assembly([E.P.program(p) for p in parts], box_a, box_b, res, grid)
    _assert_exact(got, E.exact_sets(boxes), box_a, res, bs)


@pytest.mark.parametrize("group", sorted(E.CURVED))
def test_dense_reference_margins(group):
    """the fp32 oracle decides the cells whose float64 distance is within the margin; how many there are and how many
    it decides differently are part of the reference, so that a change of margin or of scene shows here"""
    parts, box_a, box_b, res, grid = E.curved_group(group)
    _, _, bs = E.plan(box_a, box_b, res, grid)
    got = E.dense_reference(parts, box_a, res, bs)
    marginal, disagreements = E.CURVED[group]
    assert (got.marginal, got.disagreements) == (marginal, disagreements)
    assert (got.sets[len(parts):, 0] > 0).any()
