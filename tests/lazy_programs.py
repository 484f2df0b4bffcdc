"""Small column scenes for the lazy gradient of the column brick kernel (DESIGN.md 4.10): CSG of extruded boxes whose
winners tie on a mirror plane, a hole whose gradient comes out negated, and a row of many thin boxes (many winners in
one warp)."""
import numpy as np

from programs import Part, ins, quat


def _box(hw, hh, h):
    """an extruded rectangle with a polygon profile (eight vertices): the profile is the costly part, so the column pass
    takes it"""
    v = [(hw, 0), (hw, hh), (0, hh), (-hw, hh), (-hw, 0), (-hw, -hh), (0, -hh), (hw, -hh)]
    return Part.polygon(v, h)


def _words(op, a, b):
    return np.array(a.words(0) + ins("_store", 0) + b.words(1) + ins(op, 0, -1.0) + ins("_return"), np.float32)


def mirrored_boxes(op):
    """two equal boxes mirrored about the plane x = 0 (one turned by 90 degrees about z, so that their gradients differ
    there), combined by `op` (union, intersection): on that plane both distances are equal"""
    q = quat((0, 0, 1), np.pi / 2)
    a = Part.placed(_box(3.0, 3.0, 4.0), (2.0, 0.0, 0.0))
    b = Part.placed(_box(3.0, 3.0, 4.0), (-2.0, 0.0, 0.0), q=q)
    return _words(op, a, b)


def _hole():
    return Part.placed(_box(2.5, 2.0, 5.0), (1.0, 0.5, 0.0))


def holed_box():
    """a box minus a narrower, taller box through it: inside the hole the subtrahend wins, its gradient negated.  (The
    running value is the minuend: the subtrahend is the stored operand.)"""
    return _words("subtraction", _hole(), _box(6.0, 5.0, 3.0))


def hole():
    """the subtrahend of holed_box() on its own"""
    return np.array(_hole().words(0) + ins("_return"), np.float32)


def box_row(n=12):
    """n thin boxes side by side along x, unions in a comb: the cells of one warp are won by several of them"""
    words = []
    for k in range(n):
        words += Part.placed(_box(0.2, 4.0, 3.0 + 0.25 * k), (0.5 * k - 3.0, 0.0, 0.0)).words(k)
        if k < n - 1:
            words += ins("_store", k)
    for k in reversed(range(n - 1)):
        words += ins("union", k, -1.0)
    return np.array(words + ins("_return"), np.float32)


BOX = ((-8.0, -8.0, -8.0), (8.0, 8.0, 8.0))
PROGRAMS = {"mirrored_union": lambda: mirrored_boxes("union"), "mirrored_intersection": lambda: mirrored_boxes("intersection"),
            "holed_box": holed_box, "box_row": box_row}
