"""The column brick kernel's sweep with min / max extrusions (CC_SWEEP_MINMAX, DESIGN.md 4.10).  Must not change a bit:
against the CPU oracle and against the build with the selects (CC_SWEEP_MINMAX=0), on cells where an
extrusion's az and profile distance are both exactly zero (the warp must fall back), where only one of them is, on a
+0 / -0 tie between two leaves, on odd grids that end mid-brick, and on planetary.  Every launch writes into a grid
filled with 0xff bytes first."""
import numpy as np
import pytest

import oracle
from lazy_programs import BOX, PROGRAMS, _box, _words
from programs import Part, ins
from test_gpu_lazy_gradient import _eval, cb  # noqa: F401  (the module's fixture)

pytestmark = pytest.mark.gpu

BASE = "CC_SWEEP_MINMAX=0"


def _slab():
    """a 6 x 4 polygon box extruded by 4 about the origin: its faces and edges lie on grid planes of step 1/4"""
    return np.array(_box(3.0, 2.0, 4.0).words(0) + ins("_return"), np.float32)


def _notch():
    """a box minus a box that reaches its side wall x = 6 with its own: on that wall the box's distance is +0 and the
    subtrahend's, negated, -0"""
    return _words("subtraction", Part.placed(_box(2.0, 2.0, 5.0), (4.0, 0.0, 0.0)), _box(6.0, 5.0, 3.0))


def _compare(cb, words, corner, step, dims, what, defines=None):  # noqa: F811  (the fixture's value)
    from codecad_b200 import CompiledScene, _lib
    src = _lib.specialize_source(words, 2, sink_mask=1 << 8)
    assert "struct SceneSweep" in src, what
    make = lambda: CompiledScene(words, 3, BOX[0], BOX[1])  # noqa: E731
    got, fallbacks = _eval(cb, make, corner, step, dims, defines)
    base, base_fallbacks = _eval(cb, make, corner, step, dims, BASE)
    want = oracle.grid_eval(words, corner, step, dims)
    assert np.array_equal(got, want, equal_nan=True), "%s: %d values differ from the oracle" % (what, int((got != want).sum()))
    assert got.tobytes() == base.tobytes(), "%s: differs from the build with the selects" % what
    assert fallbacks == base_fallbacks, "%s: %d warps fell back, the other build %d" % (what, fallbacks, base_fallbacks)
    return got, fallbacks


def test_both_zero_falls_back(cb):
    """x = 3 and z = 4 are grid planes: along that line az = w = 0, s = 0, and the warps must take the full walk"""
    corner, step, dims = np.array([-5.0, -4.0, -6.0], np.float32), np.float32(0.25), (41, 33, 50)
    got, fallbacks = _compare(cb, _slab(), corner, step, dims, "slab on grid planes")
    assert fallbacks > 0
    assert got[32, 16, 40, 3] == 0.0  # (x 3, y 0, z 4)


@pytest.mark.parametrize("shift", [(0.125, 0.125, 0.0), (0.0, 0.0, 0.125)])
def test_one_zero_does_not_flag(cb, shift):
    """only the faces z = +-4 (az = 0), or only the profile's edges (w = 0), on grid planes: nothing flags, and max / min
    must give the selects' bits"""
    corner = np.array([-5.0, -4.0, -6.0], np.float32) - np.array(shift, np.float32)
    step, dims = np.float32(0.25), (41, 33, 50)
    got, fallbacks = _compare(cb, _slab(), corner, step, dims, "slab shifted by %s" % (shift,))
    assert fallbacks == 0
    assert np.any(got[..., 3] == 0.0)


def test_signed_zero_tie(cb):
    """on the wall x = 6 the box (+0) and the negated subtrahend (-0) tie: the leaf that wins, and its gradient, must
    be the selects'"""
    corner, step, dims = np.array([-7.0, -6.0, -4.0], np.float32), np.float32(0.25), (61, 49, 33)
    got, _ = _compare(cb, _notch(), corner, step, dims, "notch")
    wall = got[52]  # x = -7 + 52 * 0.25 = 6
    assert np.any(wall[..., 3] == 0.0)


@pytest.mark.parametrize("name", sorted(PROGRAMS))
def test_lazy_programs_with_the_replay_check(cb, name):
    """the lazy gradient's own cases, on an odd grid that ends mid-brick, with CC_LAZY_CHECK=1 (a cell whose replayed .w
    differs from the sweep's gets a poisoned gradient)"""
    corner, step, dims = np.array([-7.0, -6.0, -4.0], np.float32), np.float32(0.1875), (75, 61, 43)
    _compare(cb, PROGRAMS[name](), corner, step, dims, name, "CC_LAZY_CHECK=1")


def test_planetary_256(cb, scenes):
    s = scenes["cfg_planetary"]
    corner, step = s.grid(256)
    dims = (256, 256, 256)
    got, fallbacks = _eval(cb, s.compiled, corner, step, dims)
    base, base_fallbacks = _eval(cb, s.compiled, corner, step, dims, BASE)
    assert got.tobytes() == base.tobytes()
    assert fallbacks == base_fallbacks == 0
    for x0 in (0, 131, 255):
        want = oracle.grid_eval(s.words, corner, step, (1, 256, 256), x0)
        assert np.array_equal(got[x0:x0 + 1], want, equal_nan=True), "x-plane %d" % x0
