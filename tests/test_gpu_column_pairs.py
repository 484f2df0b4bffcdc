"""The column brick kernel (DESIGN.md 4.10) with a thread's two cells in one column and one deferred range check per
warp.  Must not change a bit: against the CPU oracle, against the same library with the column kernels switched off,
and against the kernel built with both changes switched off (CC_COL_PAIR=0, CC_DEFER_CHECKS=0) — on odd grids that
straddle bricks along every column axis, and on grids where the deferred ops see operands outside their fast path's
range, so that warps must fall back to the full walk."""
import os

import numpy as np
import pytest

import oracle
from scenes import COLUMN_NAMES

COLUMN_SCENES = ["cfg_planetary", "cfg_airfoil", "x_gear3d", "dsdf2d_gear", "dsdf2d_mirror_2d"] + COLUMN_NAMES

pytestmark = pytest.mark.gpu
OFF = "CC_COL_PAIR=0,CC_DEFER_CHECKS=0"


@pytest.fixture(scope="module")
def cb():
    import codecad_b200
    from codecad_b200 import _lib
    _lib.init(0)
    L = _lib.lib()
    old_jit = _lib.check(L.cc_set_jit_mode(2))
    yield codecad_b200
    _lib.check(L.cc_set_columns_mode(1))
    _lib.check(L.cc_set_jit_mode(old_jit))


def _f4(arr):
    return np.stack([arr["x"], arr["y"], arr["z"], arr["w"]], axis=-1)


def _three_ways(cb, s, corner, step, dims, x_offset=0):
    """(the new kernel, the kernel with both changes off, the other kernels) on one grid, and the new kernel's fallbacks"""
    from codecad_b200 import _lib
    L = _lib.lib()
    _lib.check(L.cc_set_columns_mode(1))
    scene = s.compiled()
    cb.grid_eval(scene, corner, step, dims, x_offset=x_offset)   # (compiles the units)
    L.cc_reset_counters()
    got = _f4(cb.grid_eval(scene, corner, step, dims, x_offset=x_offset))
    fallbacks = _lib.check_fallbacks()
    old = os.environ.get("CODECAD_B200_JIT_DEFINES")
    os.environ["CODECAD_B200_JIT_DEFINES"] = OFF
    try:
        parent = _f4(cb.grid_eval(s.compiled(), corner, step, dims, x_offset=x_offset))
    finally:
        if old is None:
            del os.environ["CODECAD_B200_JIT_DEFINES"]
        else:
            os.environ["CODECAD_B200_JIT_DEFINES"] = old
    _lib.check(L.cc_set_columns_mode(0))
    other = _f4(cb.grid_eval(s.compiled(), corner, step, dims, x_offset=x_offset))
    _lib.check(L.cc_set_columns_mode(1))
    return got, parent, other, fallbacks


def _same(a, b):
    return a.tobytes() == b.tobytes()


@pytest.mark.parametrize("name", COLUMN_SCENES)
def test_pairs_on_odd_grids(cb, scenes, name):
    s = scenes[name]
    corner, step = s.grid(24)
    for dims, x_offset in (((13, 11, 9), 0), ((10, 9, 17), 3), ((9, 19, 41), 5)):
        got, parent, other, _ = _three_ways(cb, s, corner, step, dims, x_offset)
        want = oracle.grid_eval(s.words, corner, step, dims, x_offset)
        assert np.array_equal(got, want, equal_nan=True), "%s %s: %d values differ from the oracle" % (name, dims, int((got != want).sum()))
        assert _same(got, parent), "%s %s: differs from the kernel with both changes off" % (name, dims)
        assert _same(got, other), "%s %s: differs from the other kernels" % (name, dims)


@pytest.mark.parametrize("name", ["cfg_planetary", "x_gear3d", "col_assembly", "colr_05"])
def test_out_of_range_operands_fall_back(cb, scenes, name):
    """Far from the origin every extrusion's s = az^2 + w^2 overflows: every warp must take the full walk.  On the
    coordinate planes (a power-of-two step) cap planes and profile edges fall on cell centres.  (Scenes whose
    per-cell body defers its checks.)"""
    from codecad_b200 import _lib
    s = scenes[name]
    assert "deferred = CC_DEFER_CHECKS != 0" in _lib.specialize_source(s.words, 2, sink_mask=1 << 8)
    size = max(b - a for a, b in zip(s.box_a, s.box_b))
    st = np.float32(2.0 ** np.floor(np.log2(size / 40)))
    grids = [(np.array([4e19, -3e19, 5e19], np.float32), np.float32(1e17), (16, 16, 33), True),
             (np.array([-20 * st, -16 * st, -24 * st], np.float32), st, (40, 32, 49), False)]
    for corner, step, dims, must_fall_back in grids:
        got, parent, other, fallbacks = _three_ways(cb, s, corner, step, dims)
        want = oracle.grid_eval(s.words, corner, step, dims)
        assert np.array_equal(got, want, equal_nan=True), "%s: %d values differ from the oracle" % (name, int((got != want).sum()))
        assert _same(got, parent) and _same(got, other)
        print("%s corner %s: %d warps fell back" % (name, corner, fallbacks))
        if must_fall_back:
            assert fallbacks > 0


def test_planetary_256(cb, scenes):
    s = scenes["cfg_planetary"]
    corner, step = s.grid(256)
    got, parent, other, fallbacks = _three_ways(cb, s, corner, step, (256, 256, 256))
    assert _same(got, parent) and _same(got, other)
    # the oracle on a sample of the x-planes
    for x0 in (0, 101, 255):
        want = oracle.grid_eval(s.words, corner, step, (1, 256, 256), x0)
        assert np.array_equal(got[x0:x0 + 1], want, equal_nan=True), "x-plane %d" % x0
    print("planetary 256^3: %d of %d warps fell back" % (fallbacks, 256 ** 3 // 64))
