"""The column brick kernel (DESIGN.md 4.10) with a CTA walking a run of bricks along the columns' axis.  Must not change
a bit: against the CPU oracle, against one brick per CTA (CODECAD_B200_BRICK_RUN=1), and against the same library
with the column kernels switched off — on odd grids whose stacks of bricks end in short runs along every column axis,
with runs longer than the stacks, on grids whose columns fail the per-column check (every brick of their runs takes the
full walk), and on grids where every warp falls back to the full walk.  Every launch writes into a grid filled with a
sentinel first, so a cell the kernels skip cannot pass for a value of an earlier launch."""
import os

import numpy as np
import pytest

import oracle
from scenes import COLUMN_NAMES

pytestmark = pytest.mark.gpu
RUN_SCENES = ["cfg_planetary", "cfg_airfoil", "x_gear3d"] + COLUMN_NAMES
# the scene whose columns fail the per-column check on the coordinate-plane grid below (75 bricks with one brick per
# CTA; x_gear3d, col_star_x and col_crossed_extrusions flag none there)
FLAGGED_SCENES = ["cfg_planetary"]


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


def _with_run(run, fn):
    old = os.environ.get("CODECAD_B200_BRICK_RUN")
    os.environ["CODECAD_B200_BRICK_RUN"] = str(run)
    try:
        return fn()
    finally:
        if old is None:
            del os.environ["CODECAD_B200_BRICK_RUN"]
        else:
            os.environ["CODECAD_B200_BRICK_RUN"] = old


def _eval(cb, scene, corner, step, dims, x_offset):
    """one launch into a device grid filled with 0xff bytes first: a cell the kernels leave unwritten keeps that pattern,
    a NaN no kernel stores, and cannot inherit an earlier launch's value"""
    from codecad_b200 import _lib
    from codecad_b200.cl_util import Buffer
    from codecad_b200.geometry import FLOAT4
    buf = Buffer(FLOAT4, dims)
    try:
        _lib.check(_lib.lib().cc_memset_async(buf.device_ptr, 0xFF, buf.size, None))
        cb.grid_eval(scene, corner, step, dims, x_offset=x_offset, device_out=buf)
        return _f4(np.array(buf.read()))
    finally:
        buf.release()


def _three_ways(cb, s, corner, step, dims, runs, x_offset=0):
    """{run: grid} of the column kernels at each run length, the grid of the other kernels, and {run: (warps that fell
    back, bricks that flagged columns sent to the full walk)}"""
    from codecad_b200 import _lib
    L = _lib.lib()
    _lib.check(L.cc_set_columns_mode(1))
    scene = s.compiled()
    cb.grid_eval(scene, corner, step, dims, x_offset=x_offset)   # (compiles the units)
    got, counts = {}, {}
    for run in runs:
        L.cc_reset_counters()
        got[run] = _with_run(run, lambda: _eval(cb, scene, corner, step, dims, x_offset))
        counts[run] = (_lib.check_fallbacks(), _lib.flagged_bricks())
    _lib.check(L.cc_set_columns_mode(0))
    other = _eval(cb, s.compiled(), corner, step, dims, x_offset)
    _lib.check(L.cc_set_columns_mode(1))
    return got, other, counts


def _same(a, b):
    return a.tobytes() == b.tobytes()


@pytest.mark.parametrize("name", RUN_SCENES)
def test_runs_on_odd_grids(cb, scenes, name):
    """Stacks of 1, 2, 3 and 5 bricks along each axis: with runs of 2 every stack of 3 or 5 ends in a run of one brick,
    runs of 4 end a stack of 5 with one brick, and runs of 64 are longer than every stack."""
    s = scenes[name]
    corner, step = s.grid(24)
    for dims, x_offset in (((13, 11, 33), 0), ((21, 19, 41), 3), ((33, 9, 17), 5), ((9, 37, 70), 2)):
        got, other, counts = _three_ways(cb, s, corner, step, dims, (1, 2, 4, 64), x_offset)
        want = oracle.grid_eval(s.words, corner, step, dims, x_offset)
        assert np.array_equal(other, want, equal_nan=True), "%s %s: the other kernels differ from the oracle" % (name, dims)
        for run in (1, 2, 4, 64):
            assert _same(got[run], other), "%s %s: runs of %d differ from the other kernels in %d values" % (
                name, dims, run, int((got[run].view(np.uint32) != other.view(np.uint32)).sum()))
            assert counts[run][1] == counts[1][1], "%s %s: runs of %d flag other bricks" % (name, dims, run)


@pytest.mark.parametrize("name", FLAGGED_SCENES)
def test_flagged_columns_send_their_runs_to_the_full_walk(cb, scenes, name):
    """Cell centres on the coordinate planes (a power-of-two step): a transform whose coefficient along the columns is
    rounding residue sees that coordinate there, the per-column check flags the column, and every brick of its runs must
    be evaluated by the full walk: as many bricks as with one brick per CTA, and every cell written."""
    s = scenes[name]
    size = max(b - a for a, b in zip(s.box_a, s.box_b))
    st = np.float32(2.0 ** np.floor(np.log2(size / 40)))
    corner, dims = np.array([-20 * st, -16 * st, -24 * st], np.float32), (40, 32, 72)
    got, other, counts = _three_ways(cb, s, corner, step=st, dims=dims, runs=(1, 3, 16))
    want = oracle.grid_eval(s.words, corner, st, dims)
    assert np.array_equal(other, want, equal_nan=True), "%s: the other kernels differ from the oracle" % name
    flagged = counts[1][1]
    print("%s: %d bricks sent to the full walk" % (name, flagged))
    assert flagged > 0, "%s: no column was flagged on the coordinate planes" % name
    for run in (1, 3, 16):
        assert _same(got[run], other), "%s: runs of %d differ from the other kernels" % (name, run)
        assert counts[run][1] == flagged, "%s: runs of %d sent %d bricks to the full walk, not %d" % (name, run, counts[run][1], flagged)


@pytest.mark.parametrize("name", ["cfg_planetary", "x_gear3d"])
def test_out_of_range_operands_fall_back(cb, scenes, name):
    """Far from the origin every extrusion's s = az^2 + w^2 overflows: every warp of every brick of a run must take the
    full walk."""
    s = scenes[name]
    corner, step, dims = np.array([4e19, -3e19, 5e19], np.float32), np.float32(1e17), (16, 16, 70)
    got, other, counts = _three_ways(cb, s, corner, step, dims, (1, 8))
    want = oracle.grid_eval(s.words, corner, step, dims)
    assert np.array_equal(other, want, equal_nan=True), "%s: the other kernels differ from the oracle" % name
    assert _same(got[1], other) and _same(got[8], other)
    assert counts[8][0] > 0


def test_planetary_256(cb, scenes):
    s = scenes["cfg_planetary"]
    corner, step = s.grid(256)
    got, other, counts = _three_ways(cb, s, corner, step, (256, 256, 256), (1, 16))
    assert _same(got[16], other) and _same(got[1], other)
    for x0 in (0, 77, 255):
        want = oracle.grid_eval(s.words, corner, step, (1, 256, 256), x0)
        assert np.array_equal(got[16][x0:x0 + 1], want, equal_nan=True), "x-plane %d" % x0
    print("planetary 256^3, runs of 16: %d warps fell back" % counts[16][0])
