"""The lazy gradient of the column brick kernel (DESIGN.md 4.10): the per-cell body carries distances and leaf ids, and
the winning leaf of each cell is replayed for its gradient.  Must not change a bit: against the CPU oracle and against
the eager body (CC_LAZY_GRADIENT=0) — on ties between CSG operands with different gradients, on holes whose gradient
comes out negated, on warps with many different winners, and on grids where every warp falls back to the full walk.
Every launch writes into a grid filled with a sentinel first."""
import os

import numpy as np
import pytest

import oracle
from lazy_programs import BOX, PROGRAMS, hole

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cb():
    import codecad_b200
    from codecad_b200 import _lib
    _lib.init(0)
    L = _lib.lib()
    old_jit = _lib.check(L.cc_set_jit_mode(2))
    _lib.check(L.cc_set_columns_mode(1))
    yield codecad_b200
    _lib.check(L.cc_set_jit_mode(old_jit))


def _f4(arr):
    return np.stack([arr["x"], arr["y"], arr["z"], arr["w"]], axis=-1)


def _eval(cb, make_scene, corner, step, dims, defines=None):
    """(grid, warps that fell back) of one launch into a device grid filled with 0xff bytes first"""
    from codecad_b200 import _lib
    from codecad_b200.cl_util import Buffer
    from codecad_b200.geometry import FLOAT4
    old = os.environ.get("CODECAD_B200_JIT_DEFINES")
    if defines is not None:
        os.environ["CODECAD_B200_JIT_DEFINES"] = defines
    buf = Buffer(FLOAT4, dims)
    try:
        scene = make_scene()
        cb.grid_eval(scene, corner, step, dims)      # (compiles the units)
        _lib.check(_lib.lib().cc_memset_async(buf.device_ptr, 0xFF, buf.size, None))
        _lib.lib().cc_reset_counters()
        cb.grid_eval(scene, corner, step, dims, device_out=buf)
        return _f4(np.array(buf.read())), _lib.check_fallbacks()
    finally:
        buf.release()
        if old is None:
            os.environ.pop("CODECAD_B200_JIT_DEFINES", None)
        else:
            os.environ["CODECAD_B200_JIT_DEFINES"] = old


def _check(cb, words, corner, step, dims, what):
    from codecad_b200 import CompiledScene, _lib
    assert "struct SceneSweep" in _lib.specialize_source(words, 2, sink_mask=1 << 8), what
    make = lambda: CompiledScene(words, 3, BOX[0], BOX[1])  # noqa: E731
    got, fallbacks = _eval(cb, make, corner, step, dims)
    eager, eager_fallbacks = _eval(cb, make, corner, step, dims, "CC_LAZY_GRADIENT=0")
    want = oracle.grid_eval(words, corner, step, dims)
    assert np.array_equal(got, want, equal_nan=True), "%s: %d values differ from the oracle" % (what, int((got != want).sum()))
    assert got.tobytes() == eager.tobytes(), "%s: differs from the eager body" % what
    assert fallbacks == eager_fallbacks, "%s: %d warps fell back, the eager body %d" % (what, fallbacks, eager_fallbacks)
    return got, fallbacks


@pytest.mark.parametrize("name", ["mirrored_union", "mirrored_intersection"])
def test_ties_on_the_mirror_plane(cb, name):
    """cells whose x is exactly 0 (a power-of-two step, the grid's corner on a multiple of it): both operands have
    the same distance there and different gradients; the one the eager body keeps must be the one replayed"""
    words = PROGRAMS[name]()
    corner, step, dims = np.array([-8.0, -7.5, -6.0], np.float32), np.float32(0.25), (65, 61, 49)
    got, _ = _check(cb, words, corner, step, dims, name)
    plane = got[32]        # x = -8 + 32 * 0.25 = 0
    assert np.any(plane[..., 0] != 0) and np.any(plane[..., 1] != 0), "%s: no tie with two different gradients" % name


def test_subtrahend_wins_with_negated_gradient(cb):
    words = PROGRAMS["holed_box"]()
    corner, step, dims = np.array([-7.0, -6.0, -4.0], np.float32), np.float32(0.125), (113, 97, 65)
    got, _ = _check(cb, words, corner, step, dims, "holed_box")
    # in the hole (x 1, y 1.5, z 0) its wall at y = 2.5 is the nearest surface: the hole's distance and gradient, negated
    c = got[64, 60, 32]
    h = oracle.grid_eval(hole(), np.array([1.0, 1.5, 0.0], np.float32), step, (1, 1, 1)).reshape(4)
    assert c[3] > 0 and c[1] != 0 and np.array_equal(c, -h), (c, h)


@pytest.mark.parametrize("dims", [(41, 13, 35), (96, 24, 40)])
def test_many_winners_in_a_warp(cb, dims):
    words = PROGRAMS["box_row"]()
    corner, step = np.array([-4.5, -5.0, -5.5], np.float32), np.float32(0.1875)
    _check(cb, words, corner, step, dims, "box_row %s" % (dims,))


@pytest.mark.parametrize("name", ["holed_box", "box_row"])
def test_far_grids_fall_back(cb, name):
    """far from the origin every extrusion's range test fails: every warp takes the full walk, none replays"""
    words = PROGRAMS[name]()
    corner, step, dims = np.array([4e19, -3e19, 5e19], np.float32), np.float32(1e17), (16, 16, 33)
    _, fallbacks = _check(cb, words, corner, step, dims, name + " far away")
    assert fallbacks > 0


def test_replayed_distance_equals_the_sweeps(cb, scenes):
    """CC_LAZY_CHECK=1: a cell whose replayed .w differs in any bit from the sweep's gets a poisoned gradient"""
    s = scenes["cfg_planetary"]
    corner, step = s.grid(96)
    dims = (96, 96, 96)
    got, _ = _eval(cb, s.compiled, corner, step, dims, "CC_LAZY_CHECK=1")
    eager, _ = _eval(cb, s.compiled, corner, step, dims, "CC_LAZY_GRADIENT=0")
    assert got.tobytes() == eager.tobytes()
