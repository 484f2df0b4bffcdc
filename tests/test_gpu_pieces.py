"""The calls that cut one request into several launches, at sizes that make them cut: cc_grid_eval's x-pieces of at most
2^30 cells (and one-plane launches of up to 2^31), the to-host pipeline's slabs through the device ring, the PyMCubes
copy-out in 64 MiB pieces, the hierarchy level loops' chunks of kChunkCells = 2^27 cells, cc_polygon_blocks' chunks and
cc_evaluate_points' launches of 2^30 points.  Every case first shows that the cut happened (launch counts, the mass
statistics, or the piece arithmetic), then compares with the CPU oracle or, where the whole is too big for it, every
byte with the same grid evaluated as explicit single-piece launches, and the oracle on both sides of each seam.

Device grids are filled with 0xff bytes before a launch: a cell that no piece writes keeps that pattern (a NaN no
kernel stores) and cannot pass for a value of an earlier launch.  The big grids use a power-of-two step and a corner
that is a multiple of it, every coordinate below 2^24 steps: corner + step * i is then exact, and a row anywhere in
the grid is the oracle's grid with the corner moved to it."""
import contextlib
import ctypes
import math
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import oracle
from oracle import host

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GiB = 1 << 30
F4, PYMC = 0, 1                 # LAYOUT_INDEX3_FLOAT4, LAYOUT_PYMCUBES_FLOAT
CHUNK_CELLS = 1 << 27           # kChunkCells of the level loops


@pytest.fixture(scope="module")
def cb():
    import codecad_b200
    from codecad_b200 import _lib
    _lib.init(0)
    L = _lib.lib()
    old = [_lib.check(L.cc_set_jit_mode(2)), _lib.check(L.cc_set_columns_mode(1)), _lib.check(L.cc_set_parts_mode(1)),
           _lib.check(L.cc_set_forest_mode(1))]
    yield codecad_b200
    _lib.check(L.cc_set_jit_mode(old[0]))
    _lib.check(L.cc_set_columns_mode(old[1]))
    _lib.check(L.cc_set_parts_mode(old[2]))
    _lib.check(L.cc_set_forest_mode(old[3]))


_PROGRAMS = {}


def _prog(scene):
    from codecad_b200.cl_util.buffer import ProgramBuffer
    if scene.name not in _PROGRAMS:
        _PROGRAMS[scene.name] = ProgramBuffer(scene.words)
    return _PROGRAMS[scene.name]


# the dense routes: (scene, jit mode, columns mode, parts mode, forest mode, brick run)
ROUTES = {
    "interpreter": ("cfg_planetary", 0, 0, 0, 0, None),
    "columns": ("cfg_planetary", 2, 1, 1, 0, "8"),
    "parts": ("cfg_planetary", 2, 0, 1, 0, None),
    "forest": ("cfg_synthetic500", 2, 1, 1, 1, None),
}


@contextlib.contextmanager
def _route(name, prog):
    """The modes of route `name` for the program `prog`.  A program that has loaded a specialised kernel uses it whatever
    the JIT mode (the kernels of a small grid's launch are compiled even where the column and part paths decline it), so
    the interpreter route also switches the program's specialised kernels off."""
    from codecad_b200 import _lib
    L = _lib.lib()
    _, jit, columns, parts, forest, run = ROUTES[name]
    if jit == 0:
        assert not prog.use_specialized(False)
    old = [_lib.check(L.cc_set_jit_mode(jit)), _lib.check(L.cc_set_columns_mode(columns)),
           _lib.check(L.cc_set_parts_mode(parts)), _lib.check(L.cc_set_forest_mode(forest))]
    old_run = os.environ.get("CODECAD_B200_BRICK_RUN")
    if run is not None:
        os.environ["CODECAD_B200_BRICK_RUN"] = run
    try:
        yield
    finally:
        if run is not None:
            if old_run is None:
                del os.environ["CODECAD_B200_BRICK_RUN"]
            else:
                os.environ["CODECAD_B200_BRICK_RUN"] = old_run
        _lib.check(L.cc_set_jit_mode(old[0]))
        _lib.check(L.cc_set_columns_mode(old[1]))
        _lib.check(L.cc_set_parts_mode(old[2]))
        _lib.check(L.cc_set_forest_mode(old[3]))
        if jit == 0:
            prog.use_specialized(True)


# kernels per call of each route on a grid of at least 4096 cells with 8 cells along the columns: the interpreter and the
# forest kernel are one launch, part culling a brick-centre pass and the culled kernel, the column route the brick centres,
# the column pass, the brick kernel and the flagged bricks' full walk
ROUTE_LAUNCHES = {"interpreter": 1, "columns": 4, "parts": 2, "forest": 1}


def _launches():
    from codecad_b200 import _lib
    return _lib.counters()[0]


def _need_device_memory(gib):
    """The big cases allocate tens of GB on a device other jobs share: skip, saying why, when it is not free."""
    import torch
    free, _ = torch.cuda.mem_get_info(0)
    if free < gib * GiB:
        pytest.skip("needs %.0f GiB of free device memory, %.1f GiB free" % (gib, free / GiB))


def _peak_gib():
    """the peak of the device buffers this test allocated (torch's allocator; the library's own scratch is not in it)"""
    import torch
    return torch.cuda.max_memory_allocated() / GiB


def _reset_peak():
    import torch
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()


def _filled(shape):
    """a device int32 tensor of 0xff bytes"""
    import torch
    return torch.full(shape, -1, dtype=torch.int32, device="cuda")


def _grid(prog, corner, step, dims, x_offset, layout, out, byte_offset=0):
    """cc_grid_eval into the torch tensor `out` (from `byte_offset` on), synchronised"""
    import torch
    from codecad_b200 import _lib
    L = _lib.lib()
    nx, ny, nz = (int(d) for d in dims)
    torch.cuda.synchronize()        # (torch's fill runs on its own stream)
    _lib.check(L.cc_grid_eval(prog.handle, _lib.f3(corner), float(step), nx, ny, nz, int(x_offset), layout,
                              ctypes.c_void_p(out.data_ptr() + byte_offset), None))
    _lib.check(L.cc_synchronize())


def _dyadic(corner, step, dy=0, dz=0):
    """the corner moved by (0, dy, dz) steps: exact for a power-of-two step and a corner on its multiples"""
    c = np.asarray(corner, np.float32).copy()
    c[1] = c[1] + np.float32(dy) * np.float32(step)
    c[2] = c[2] + np.float32(dz) * np.float32(step)
    assert float(c[1]) == float(corner[1]) + dy * float(step) and float(c[2]) == float(corner[2]) + dz * float(step)
    return c


def _same_as_single_launches(prog, corner, step, dims, x_offset, got):
    """Every byte of the float4 grid `got` (device, [nx][ny][nz][4] int32) against explicit calls of at most 2^27 cells,
    each one launch: slabs of whole planes, or runs of rows where a plane is larger.  -> number of calls"""
    import torch
    nx, ny, nz = dims
    sy = ny if ny * nz <= CHUNK_CELLS else max(1, CHUNK_CELLS // nz)
    sx = max(1, CHUNK_CELLS // (sy * nz))
    scratch = torch.empty(min(sx, nx) * sy * nz * 4, dtype=torch.int32, device="cuda")
    calls = 0
    for x0 in range(0, nx, sx):
        for y0 in range(0, ny, sy):
            d = (min(sx, nx - x0), min(sy, ny - y0), nz)
            part = scratch[:d[0] * d[1] * d[2] * 4].view(d + (4,))
            part.fill_(-1)
            _grid(prog, _dyadic(corner, step, dy=y0), step, d, x_offset + x0, F4, part)
            calls += 1
            assert torch.equal(got[x0:x0 + d[0], y0:y0 + d[1]], part), \
                "planes %d.. rows %d..: differ from an explicit launch of the same cells" % (x0, y0)
    del scratch
    return calls


def _f4(t):
    """device int32 [..][4] -> host float32 [..][4]"""
    return t.cpu().numpy().view(np.float32)


def _rows_match_oracle(words, corner, step, got, x_offset, planes, rows):
    """rows `rows` of the x-planes `planes` of the float4 grid `got` (device) against the oracle, row by row"""
    nz = got.shape[2]
    for x in planes:
        for y in rows:
            want = oracle.grid_eval(words, _dyadic(corner, step, dy=y), step, (1, 1, nz), x_offset + x)[0, 0]
            assert np.array_equal(_f4(got[x, y]), want, equal_nan=True), "plane %d row %d differs from the oracle" % (x, y)


# ---- 1. cc_grid_eval's x-pieces ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("route", list(ROUTES))
def test_x_pieces_of_a_plane_that_does_not_divide_2_30(cb, scenes, route):
    """1080 x 1000 x 1000: pieces of 1073 planes (2^30 // 10^6), so the second piece starts mid-brick (1073 = 8 * 134 + 1)
    with nx = 7."""
    _need_device_memory(24)
    import torch
    s = scenes[ROUTES[route][0]]
    prog = _prog(s)
    dims, x_offset = (1080, 1000, 1000), 0
    plane = dims[1] * dims[2]
    max_x = (1 << 30) // plane
    assert max_x == 1073 and dims[0] > max_x
    step = np.float32(0.125)
    corner = np.array([-64.0, -64.0, -56.0], np.float32)
    t0 = time.time()
    _reset_peak()
    with _route(route, prog):
        got = _filled(dims + (4,))
        # the two pieces as explicit calls, for their launch counts
        n0 = _launches()
        _grid(prog, corner, step, (max_x, dims[1], dims[2]), x_offset, F4, got)
        n1 = _launches()
        _grid(prog, corner, step, (dims[0] - max_x, dims[1], dims[2]), x_offset + max_x, F4, got, max_x * plane * 16)
        n2 = _launches()
        got.fill_(-1)
        _grid(prog, corner, step, dims, x_offset, F4, got)
        n3 = _launches()
        assert n1 - n0 == n2 - n1 == ROUTE_LAUNCHES[route], "the %s route takes %d + %d launches" % (route, n1 - n0, n2 - n1)
        assert n3 - n2 == (n1 - n0) + (n2 - n1), \
            "one call: %d launches, its two pieces: %d + %d" % (n3 - n2, n1 - n0, n2 - n1)
        calls = _same_as_single_launches(prog, corner, step, dims, x_offset, got)
        peak = _peak_gib()
    # the oracle on planes 1064..1079 (both pieces' brick layers at the seam) and on planes elsewhere
    rows = (0, 1, 499, 998, 999) if route == "forest" else (0, 1, 250, 499, 500, 777, 998, 999)
    _rows_match_oracle(s.words, corner, step, got, x_offset, range(1064, 1080), rows)
    _rows_match_oracle(s.words, corner, step, got, x_offset, (0, 7, 8, 536, 1063), (0, 500, 999))
    if route != "forest":
        for x in (1072, 1073):
            want = oracle.grid_eval(s.words, corner, step, (1, dims[1], dims[2]), x_offset + x)[0]
            assert np.array_equal(_f4(got[x]), want, equal_nan=True), "plane %d differs from the oracle" % x
    del got
    torch.cuda.empty_cache()
    print("%s %s: 2 pieces (%d + %d planes), %d + %d launches, %d single-launch calls compared; test buffers peak %.1f GiB, %.1f s"
          % (route, dims, max_x, dims[0] - max_x, n1 - n0, n2 - n1, calls, peak, time.time() - t0))


def test_pymcubes_launch_of_2_31_cells(cb, scenes):
    """1 x 32768 x 65536: the largest launch the host allows, in the y-flipped PyMCubes layout."""
    _need_device_memory(10)
    import torch
    s = scenes["cfg_planetary"]
    prog = _prog(s)
    dims = (1, 32768, 65536)
    assert dims[0] * dims[1] * dims[2] == 1 << 31
    step = np.float32(2.0 ** -8)
    corner = np.array([0.5, -64.0, -96.0], np.float32)
    t0 = time.time()
    _reset_peak()
    got = _filled((dims[1], dims[0], dims[2]))
    n0 = _launches()
    _grid(prog, corner, step, dims, 0, PYMC, got)
    launches = _launches() - n0
    peak = _peak_gib()
    ny, nz = dims[1], dims[2]
    # row r of the flipped layout is y = ny - 1 - r
    for r in (0, 1, 2, 4095, 16383, 16384, 27000, ny - 2, ny - 1):
        want = oracle.grid_eval_pymcubes(s.words, _dyadic(corner, step, dy=ny - 1 - r), step, (1, 1, nz))[0, 0]
        assert np.array_equal(got[r, 0].cpu().numpy().view(np.float32), want, equal_nan=True), "row %d" % r
    assert not bool((got == -1).any()), "cells left unwritten"
    del got
    torch.cuda.empty_cache()
    print("PyMCubes %s: one launch of 2^31 cells (%d kernel launches); test buffers peak %.1f GiB, %.1f s"
          % (dims, launches, peak, time.time() - t0))


def test_one_plane_launches_above_2_30_cells(cb, scenes):
    """3 x 32768 x 32769: a plane of 2^30 + 32768 cells, so max_x = 1 and the grid is three launches of one plane."""
    _need_device_memory(56)
    import torch
    s = scenes["cfg_planetary"]
    prog = _prog(s)
    dims = (3, 32768, 32769)
    plane = dims[1] * dims[2]
    assert plane > 1 << 30 and max(1, (1 << 30) // plane) == 1
    step = np.float32(2.0 ** -8)
    corner = np.array([-1.0, -64.0, -60.0], np.float32)
    t0 = time.time()
    _reset_peak()
    got = _filled(dims + (4,))
    n0 = _launches()
    _grid(prog, corner, step, (1, dims[1], dims[2]), 0, F4, got)
    one = _launches() - n0
    got.fill_(-1)
    n0 = _launches()
    _grid(prog, corner, step, dims, 0, F4, got)
    launches = _launches() - n0
    assert launches == 3 * one, "three one-plane launches of %d kernels each, not %d" % (one, launches)
    calls = _same_as_single_launches(prog, corner, step, dims, 0, got)
    peak = _peak_gib()
    _rows_match_oracle(s.words, corner, step, got, 0, range(3), (0, 1, 16383, 16384, 32766, 32767))
    del got
    torch.cuda.empty_cache()
    print("float4 %s: 3 one-plane launches, %d kernel launches, %d single-launch calls compared; test buffers peak %.1f GiB, %.1f s"
          % (dims, launches, calls, peak, time.time() - t0))


# ---- 2. the to-host slabs at the default slab size ---------------------------------------------------------------------

def _slabs(dims, slab_mib):
    """grid_to_host_share's slabs: (x0, planes)"""
    nx, ny, nz = dims
    plane = ny * nz * 16
    sx = max(1, (slab_mib << 20) // plane)
    if ((sx + 7) & ~7) * plane <= 512 << 20:
        sx = (sx + 7) & ~7
    sx = min(sx, nx)
    return [(x0, min(sx, nx - x0)) for x0 in range(0, nx, sx)]


def _to_host(prog, corner, step, dims, x_offset):
    """cc_grid_eval_to_host into a host array of 0xff bytes -> (float4 array as int32 [..][4], launches)"""
    from codecad_b200 import _lib
    out = np.full(tuple(dims) + (4,), -1, np.int32)
    n0 = _launches()
    _lib.check(_lib.lib().cc_grid_eval_to_host(prog.handle, _lib.f3(corner), float(step), *(int(d) for d in dims),
                                               int(x_offset), F4, out.ctypes.data))
    return out, _launches() - n0


def _to_host_matches(prog, words, corner, step, dims, x_offset, slab_mib, oracle_rows=None):
    """the to-host grid: slab count and launches, every byte against the device-resident grid, and the oracle on the
    planes on both sides of every slab seam (rows `oracle_rows` of them, or whole planes)"""
    slabs = _slabs(dims, slab_mib)
    host, launches = _to_host(prog, corner, step, dims, x_offset)
    dev = _filled(tuple(dims) + (4,))
    per_slab = 0
    for x0, n in slabs:
        n0 = _launches()
        _grid(prog, corner, step, (n,) + tuple(dims[1:]), x_offset + x0, F4, dev, x0 * dims[1] * dims[2] * 16)
        per_slab += _launches() - n0
    assert launches == per_slab, "to host: %d launches, its %d slabs as device calls: %d" % (launches, len(slabs), per_slab)
    dev.fill_(-1)
    _grid(prog, corner, step, dims, x_offset, F4, dev)
    same = host.tobytes() == dev.cpu().numpy().tobytes()
    assert same, "the to-host grid differs from the device-resident one"
    del dev
    seams = sorted({x for x0, _ in slabs[1:] for x in (x0 - 1, x0)})
    f = host.view(np.float32)
    for x in seams:
        if oracle_rows is None:
            want = oracle.grid_eval(words, corner, step, (1,) + tuple(dims[1:]), x_offset + x)[0]
            assert np.array_equal(f[x], want, equal_nan=True), "plane %d differs from the oracle" % x
        else:
            for y in oracle_rows:
                want = oracle.grid_eval(words, _dyadic(corner, step, dy=y), step, (1, 1, dims[2]), x_offset + x)[0, 0]
                assert np.array_equal(f[x, y], want, equal_nan=True), "plane %d row %d differs from the oracle" % (x, y)
    return len(slabs), launches


def test_to_host_slabs_wrap_the_ring(cb, scenes):
    """200 x 512 x 512 with x_offset 13: 4 MiB planes, 16-plane slabs, 13 slabs through the ring of 4 (it wraps three
    times), the last one of 8 planes.  Then planes above 64 MiB: 5 x 2048 x 2049, one-plane slabs (8 would exceed 512
    MiB).  A small call before and after the large ones, on whatever ring the process holds (the ring is kept for the
    process: its growth from a fresh one is the 1 MiB child's case)."""
    import torch
    p, c = scenes["cfg_planetary"], scenes["cfg_csg_example"]
    t0 = time.time()
    with _route("columns", _prog(p)):
        small = ((37, 45, 70), np.array([-8.0, -16.0, -4.0], np.float32), np.float32(0.5), 5)
        big = ((200, 512, 512), np.array([-64.0, -64.0, -8.0], np.float32), np.float32(0.25), 13)
        got = []
        for dims, corner, step, x_offset in (small, big, small):
            rows = None if dims == small[0] else range(0, 512, 37)
            got.append(_to_host_matches(_prog(p), p.words, corner, step, dims, x_offset, 64, rows))
        assert got[0][0] == 1 and got[1][0] == 13 and _slabs(big[0], 64)[-1] == (192, 8)
        wide = (5, 2048, 2049)
        assert [n for _, n in _slabs(wide, 64)] == [1] * 5
        got.append(_to_host_matches(_prog(c), c.words, np.array([-64.0, -64.0, -64.0], np.float32), np.float32(0.0625),
                                    wide, 1000, 64))
    torch.cuda.empty_cache()
    print("to host (slabs, launches): small %s, 200x512x512 %s, small again %s, 5x2048x2049 %s; %.1f s"
          % (got[0], got[1], got[2], got[3], time.time() - t0))


# ---- 3. the to-host slabs at 1 MiB, in a child process ------------------------------------------------------------------

CHILD = r"""
import os, sys, time
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests")
import numpy as np
from codecad_b200 import _lib
from scenes import load_scenes
import oracle
import test_gpu_pieces as t
_lib.init(0)
S = load_scenes()
t0 = time.time()
# (scene, dims, x_offset, corner, step); the first grid is small: the ring grows at the next ones and is re-used by the last
GRIDS = [("cfg_planetary", (5, 16, 16), 3), ("cfg_planetary", (37, 45, 70), 5), ("cfg_planetary", (61, 33, 129), 3),
         ("cfg_planetary", (29, 100, 211), 11), ("cfg_synthetic500", (37, 45, 70), 6), ("cfg_synthetic500", (61, 33, 129), 1),
         ("cfg_planetary", (5, 16, 16), 3)]
for name, dims, x_offset in GRIDS:
    s = S[name]
    corner, step = np.array([-56.0, -56.0, -8.0], np.float32), np.float32(0.5)
    want = oracle.grid_eval(s.words, corner, step, dims, x_offset)
    slabs = t._slabs(dims, 1)
    for route in (["forest"] if name == "cfg_synthetic500" else ["interpreter", "columns", "parts"]):
        with t._route(route, t._prog(s)):
            host, launches = t._to_host(t._prog(s), corner, step, dims, x_offset)
            per_slab = 0
            dev = t._filled(tuple(dims) + (4,))
            for x0, n in slabs:
                n0 = t._launches()
                t._grid(t._prog(s), corner, step, (n,) + dims[1:], x_offset + x0, 0, dev, x0 * dims[1] * dims[2] * 16)
                per_slab += t._launches() - n0
        assert launches == per_slab, (name, dims, route, launches, per_slab)
        if dims[1] * dims[2] * min(n for _, n in slabs) >= 4096:
            assert launches == len(slabs) * t.ROUTE_LAUNCHES[route], (name, dims, route, launches, "not this route's kernels")
        assert host.tobytes() == dev.cpu().numpy().tobytes(), (name, dims, route, "differs from its slabs as device calls")
        assert np.array_equal(host.view(np.float32), want, equal_nan=True), (name, dims, route, "differs from the oracle")
        print("%%s %%s x_offset %%d %%s: %%d slabs %%s, %%d launches" %% (name, dims, x_offset, route, len(slabs),
                                                                [n for _, n in slabs], launches))
print("child ok %%.1f s" %% (time.time() - t0))
"""


def test_to_host_one_mib_slabs_on_every_dense_route(cb):
    """CODECAD_B200_SLAB_MIB is read once per process: a child with 1 MiB slabs evaluates odd grids with x offsets on
    every dense route, many slabs per call, slab ends falling inside runs of bricks and column stacks.  The ring starts
    empty in the child: it grows from the first, small grid to the larger ones and is re-used by the small one at the end."""
    assert len(_slabs((61, 33, 129), 1)) == 4 and len(_slabs((29, 100, 211), 1)) == 4
    env = dict(os.environ, CODECAD_B200_SLAB_MIB="1")
    t0 = time.time()
    r = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT}], capture_output=True, text=True, timeout=900,
                       env=env, cwd=ROOT)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "child ok" in r.stdout
    print("child: %.1f s" % (time.time() - t0))


# ---- 4. the PyMCubes copy-out in 64 MiB pieces ----------------------------------------------------------------------

def test_pymcubes_to_host_in_pieces(cb, scenes):
    """300 x 256 x 256 floats are 75 MiB: two pieces of the copy, the seam 64 MiB in, at flipped row 218, x = 136."""
    from codecad_b200 import _lib
    s = scenes["cfg_planetary"]
    prog = _prog(s)
    dims = (300, 256, 256)
    nx, ny, nz = dims
    nbytes = nx * ny * nz * 4
    piece = 64 << 20
    assert piece < nbytes <= 2 * piece
    seam_row, rest = divmod(piece // 4, nx * nz)
    assert (seam_row, rest) == (218, 136 * nz)
    step = np.float32(0.5)
    corner = np.array([-75.0, -64.0, -48.0], np.float32)
    host = np.full((ny, nx, nz), -1, np.int32)
    _lib.check(_lib.lib().cc_grid_eval_to_host(prog.handle, _lib.f3(corner), float(step), nx, ny, nz, 0, PYMC,
                                               host.ctypes.data))
    dev = _filled((ny, nx, nz))
    _grid(prog, corner, step, dims, 0, PYMC, dev)
    same = host.tobytes() == dev.cpu().numpy().tobytes()
    assert same, "the to-host PyMCubes grid differs from the device-resident one"
    f4 = _filled(dims + (4,))
    _grid(prog, corner, step, dims, 0, F4, f4)
    w = f4[..., 3].cpu().numpy()
    same = host.tobytes() == np.ascontiguousarray(np.transpose(w, (1, 0, 2))[::-1]).tobytes()
    assert same, "the PyMCubes grid is not the y-flipped, transposed float4 grid's distances"
    for r in (seam_row - 1, seam_row, seam_row + 1):
        want = oracle.grid_eval_pymcubes(s.words, _dyadic(corner, step, dy=ny - 1 - r), step, (nx, 1, nz))[0]
        assert np.array_equal(host[r].view(np.float32), want, equal_nan=True), "flipped row %d" % r
    print("PyMCubes to host %s: %d bytes, 2 pieces of the copy" % (dims, nbytes))


# ---- 5. the hierarchy level loops above kChunkCells -----------------------------------------------------------------------

def _plan(scene, resolution, grid, overlap, expand):
    from codecad_b200.geometry import BoundingBox, as_vector
    from codecad_b200.subdivision import calculate_block_sizes
    box = BoundingBox(as_vector(scene.box_a), as_vector(scene.box_b))
    if expand:
        box = box.expanded_additive(resolution / 2)
    return box, calculate_block_sizes(box, scene.dimension, resolution, grid, overlap)


def _chunks(blocks, dims):
    cells = dims[0] * dims[1] * dims[2]
    per = max(1, CHUNK_CELLS // cells)
    return -(-blocks // per)


def test_mass_leaf_level_in_chunks_matches_oracle(cb, scenes):
    """The unit sphere at resolution 0.0026, grid 64: a top level of 13^3 and 776 leaf blocks of 64^3, two chunks of
    at most 512 blocks.  Against the oracle, and the same doubles from the interpreter and the specialised tile units."""
    import importlib
    from codecad_b200 import _lib
    mpm = importlib.import_module("codecad_b200.mass_properties")
    s = scenes["mp_sphere"]
    res, grid = 0.0026, 64
    t0 = time.time()
    st = {}
    got = cb.mass_properties(s.compiled(), res, grid, stats=st)
    leaf = st["dealt_blocks"]                    # the leaf level's blocks (dealt level n - 2 = 0 hands them out)
    assert st["levels"] == 2 and leaf > CHUNK_CELLS // grid ** 3
    assert st["launches"] == 1 + _chunks(leaf, (grid,) * 3) > st["levels"], st
    w_vol, w_cen, w_inertia = host.mass_properties(s.words, s.box_a, s.box_b, res, grid)
    assert got.volume == pytest.approx(w_vol, rel=1e-12)
    assert tuple(got.centroid) == pytest.approx(tuple(w_cen), rel=1e-9, abs=1e-9 * max(1.0, abs(w_vol)) ** (1 / 3))
    assert np.allclose(got.inertia_tensor, w_inertia, rtol=1e-9, atol=1e-9 * np.abs(w_inertia).max())
    box, plan = _plan(s, res, grid, False, False)
    prog = s.compiled().program_buffer()
    L = _lib.lib()
    old = _lib.check(L.cc_set_jit_mode(0))
    try:
        interp = mpm.mass_limbs(prog, box.a, res, plan)
    finally:
        _lib.check(L.cc_set_jit_mode(old))
    tiles = mpm.mass_limbs(prog, box.a, res, plan)
    assert np.array_equal(interp[0], tiles[0]) and interp[2]["launches"] == tiles[2]["launches"]
    print("mass sphere %g grid %d: %d leaf blocks, %d launches; %.1f s" % (res, grid, leaf, st["launches"], time.time() - t0))


def test_mass_shares_with_the_dealt_level_in_chunks(cb, scenes):
    """The unit sphere at resolution 0.00012, grid 8: five levels, the dealt one (n - 2) of ~370 000 blocks of 8^3 (two
    chunks), the leaf of ~24 M blocks (90 chunks).  Shares of 2 and 3 add up to the unsharded accumulator limb for limb."""
    import importlib
    mpm = importlib.import_module("codecad_b200.mass_properties")
    s = scenes["mp_sphere"]
    res, grid = 0.00012, 8
    box, plan = _plan(s, res, grid, False, False)
    prog = s.compiled().program_buffer()
    t0 = time.time()
    whole, exps, st = mpm.mass_limbs(prog, box.a, res, plan)
    dealt = mpm.mass_limbs(prog, box.a, res, plan[:-1])[2]["dealt_blocks"]   # the blocks of level n - 2
    n = len(plan)
    assert n == 5 and dealt * grid ** 3 > CHUNK_CELLS, (plan, dealt)
    assert st["launches"] > st["levels"] and st["launches"] >= _chunks(dealt, plan[-2][1]) + _chunks(st["dealt_blocks"], plan[-1][1])
    vol = mpm.limbs_to_integrals(whole, exps)[0]
    assert vol == pytest.approx(4 * math.pi / 3, rel=1e-3)
    for world in (2, 3):
        total = np.zeros(40, dtype=np.int64)
        for rank in range(world):
            limbs, e, _ = mpm.mass_limbs(prog, box.a, res, plan, rank, world)
            assert np.array_equal(e, exps)
            total += limbs
        assert np.array_equal(total, whole), "%d shares do not add up to the unsharded accumulator" % world
    print("mass shares sphere %g grid %d: dealt level %d blocks (%d chunks), leaf %d blocks, %d launches; %.1f s"
          % (res, grid, dealt, _chunks(dealt, plan[-2][1]), st["dealt_blocks"], st["launches"], time.time() - t0))


def _oracle_leaf_corners(words, box_a, box_b, dimension, resolution, overlap, grid):
    """oracle.host.subdivision's leaf int corners, restated level by level with numpy: its plan, origin, per-block corners,
    thresholds and oracle.subdivision_step, and its block order, without its Python tuple per leaf block (minutes for
    the 12 M blocks below) -> (plan, corners int64 [n][3], blocks per level)"""
    a = tuple(c - resolution / 2 for c in box_a)
    b = tuple(c + resolution / 2 for c in box_b)
    if dimension == 2:
        a, b = (a[0], a[1], 0), (b[0], b[1], 0)
    plan = host.calculate_block_sizes(a, b, dimension, resolution, grid, overlap)
    corners = np.zeros((1, 3), np.int64)
    counts = []
    for cs, dims in plan[:-1]:
        counts.append(len(corners))
        box_step = cs * resolution
        thr = box_step * math.sqrt(dimension) / 2
        shift = np.array([cs / 2, cs / 2, cs / 2 if dimension == 3 else 0])
        out = []
        for c in corners:
            corner = ((c + shift) * resolution + np.array(a, np.float64)).astype(np.float32)
            hits = oracle.subdivision_step(words, corner, box_step, thr, dims)
            out.append(c + hits[:, :3].astype(np.int64) * cs)
        corners = np.concatenate(out) if out else np.zeros((0, 3), np.int64)
    counts.append(len(corners))
    return plan, corners, counts


def test_subdivision_level_in_chunks_matches_oracle(cb, scenes):
    """The unit sphere at resolution 0.00009, grid 16: level n - 2 has more than 32 768 blocks of 16^3 (two chunks).
    The leaf corners are the oracle's; shares of 3 ranks merge into the unsharded array."""
    import importlib
    sub = importlib.import_module("codecad_b200.subdivision")
    s = scenes["mp_sphere"]
    # the restatement is oracle.host.subdivision's block list where that one is quick to build
    plan, small, _ = _oracle_leaf_corners(s.words, s.box_a, s.box_b, 3, 0.01, True, 8)
    assert len(plan) == 3 and np.array_equal(small, [blk[3] for blk in host.subdivision(s.words, s.box_a, s.box_b, 3, 0.01, True, 8)[1]])
    res, grid = 0.00009, 16
    box, plan = _plan(s, res, grid, True, True)
    prog = s.compiled().program_buffer()
    t0 = time.time()
    whole = sub.subdivide_int_corners(prog, box.a, res, plan, 3)
    want_plan, want, counts = _oracle_leaf_corners(s.words, s.box_a, s.box_b, 3, res, True, grid)
    assert [(int(c), tuple(int(d) for d in dims)) for c, dims in plan] == [(c, tuple(d)) for c, d in want_plan]
    assert counts[-2] > CHUNK_CELLS // grid ** 3, counts
    assert np.array_equal(whole, want), "%d leaf blocks, the oracle %d" % (len(whole), len(want))
    parts = [sub.subdivide_int_corners(prog, box.a, res, plan, 3, r, 3) for r in range(3)]
    assert np.array_equal(sub.sort_leaf_corners(np.concatenate(parts), plan), whole)
    print("subdivision sphere %g grid %d: blocks per level %s, level n-2 in %d chunks; %.1f s"
          % (res, grid, counts, _chunks(counts[-2], plan[-2][1]), time.time() - t0))


def test_assembly_levels_in_chunks_with_and_without_tile_masks(cb, scenes):
    """Planetary: mass at 0.12 (grid 64) with the leaf level in chunks, subdivision at 0.0025 (grid 64) with level 1 in
    chunks; the part masks of the tile units (rounding budget from the hierarchy's coordinate bound) change nothing."""
    import importlib
    from codecad_b200 import _lib
    mpm = importlib.import_module("codecad_b200.mass_properties")
    sub = importlib.import_module("codecad_b200.subdivision")
    s = scenes["cfg_planetary"]
    prog = s.compiled().program_buffer()
    L = _lib.lib()
    t0 = time.time()
    mbox, mplan = _plan(s, 0.12, 64, False, False)
    sbox, splan = _plan(s, 0.0025, 64, True, True)
    assert len(splan) == 3
    cs, dims = splan[0]
    top = ((np.array([cs / 2] * 3) * 0.0025 + np.array([sbox.a.x, sbox.a.y, sbox.a.z])).astype(np.float32))
    level1 = len(oracle.subdivision_step(s.words, top, cs * 0.0025, cs * 0.0025 * math.sqrt(3) / 2, dims))
    assert level1 > CHUNK_CELLS // 64 ** 3
    got = {}
    for parts in (1, 0):
        old = _lib.check(L.cc_set_parts_mode(parts))
        try:
            got[parts] = (mpm.mass_limbs(prog, mbox.a, 0.12, mplan), sub.subdivide_int_corners(prog, sbox.a, 0.0025, splan, 3))
        finally:
            _lib.check(L.cc_set_parts_mode(old))
    (limbs1, _, st), corners1 = got[1]
    (limbs0, _, _), corners0 = got[0]
    assert st["dealt_blocks"] > CHUNK_CELLS // 64 ** 3 and st["launches"] > st["levels"], st
    assert np.array_equal(limbs1, limbs0), "the mass sums change with the tile masks"
    assert np.array_equal(corners1, corners0), "the leaf blocks change with the tile masks"
    print("planetary: mass leaf %d blocks, %d launches; subdivision level 1 %d blocks (%d chunks), %d leaves; %.1f s"
          % (st["dealt_blocks"], st["launches"], level1, _chunks(level1, (64,) * 3), len(corners1), time.time() - t0))


# ---- 6. cc_polygon_blocks' chunks -------------------------------------------------------------------------------------

def test_polygon_blocks_in_chunks(cb, scenes):
    """The gear's square covered by 34 x 34 boxes of 256 x 256 samples: more than 2^26 / 65536 = 1024 boxes, two chunks.
    The boxes the outline crosses are put around the seam; each box there is the oracle's evaluation and
    process_polygon, vertex for vertex."""
    from codecad_b200.rendering import polygon2d
    s = scenes["dsdf2d_gear"]
    prog = _prog(s)
    g, n = 256, 34
    res = 11.0 / (n * (g - 1))
    ij = np.stack(np.meshgrid(np.arange(n), np.arange(n), indexing="ij"), -1).reshape(-1, 2)
    corners = np.zeros((n * n, 3))
    corners[:, :2] = -5.5 + ij * (g - 1) * res
    centre = corners[:, :2] + (g - 1) * res / 2
    order = np.argsort(np.abs(np.hypot(centre[:, 0], centre[:, 1]) - 4.5), kind="stable")
    chunk = (1 << 26) // (g * g)
    assert len(corners) > chunk
    place = np.empty(len(corners), np.int64)
    near = list(range(chunk - 64, chunk + 64))
    place[order[:len(near)]] = near
    place[order[len(near):]] = [i for i in range(len(corners)) if not chunk - 64 <= i < chunk + 64]
    boxes = np.empty_like(corners)
    boxes[place] = corners
    t0 = time.time()
    n0 = _launches()
    vertices, links, starts, counts = polygon2d.polygon_blocks(prog, (g, g), boxes, res)
    launches = _launches() - n0
    assert launches == 3 * 2, "two chunks of one evaluation and two outline launches each, not %d launches" % launches
    crossed = 0
    for b in near + [len(boxes) - 1]:
        c32 = boxes[b].astype(np.float32)
        field = oracle.grid_eval(s.words, c32, np.float32(res), (g, g, 1))[:, :, 0, :]
        want_v, want_l, want_s = oracle.process_polygon(c32[:2], np.float32(res), field)
        assert np.array_equal(vertices[b], want_v) and np.array_equal(links[b], want_l), "box %d" % b
        assert int(counts[b]) == len(want_s) and np.array_equal(starts[b][:len(want_s)], want_s), "box %d" % b
        crossed += bool(np.any(want_v))
    assert crossed >= 8, "the boxes at the seam should carry the outline"
    print("polygon blocks: %d boxes of %d^2 samples, chunks of %d, %d launches; %d seam boxes crossed; %.1f s"
          % (len(boxes), g, chunk, launches, crossed, time.time() - t0))


def _oracle_outlines(words, boxes, g):
    """the outlines of oracle.host.subdivision's boxes `boxes` of g x g samples: each box through the oracle's grid_eval
    and process_polygon, chained by the native assembler"""
    from codecad_b200.rendering import polygon2d
    n, cells = len(boxes), 2 * (g - 1) ** 2
    vertices, links = np.zeros((n, cells, 2), np.float32), np.zeros((n, cells), np.uint32)
    starts, counts = np.zeros((n, 2 * (g - 1)), np.uint32), np.zeros(n, np.uint32)
    for i, (_, corner, step, _, _) in enumerate(boxes):
        c32 = np.array(corner, np.float64).astype(np.float32)
        field = oracle.grid_eval(words, c32, step, (g, g, 1))[:, :, 0, :]
        vertices[i], links[i], st = oracle.process_polygon(c32[:2], step, field)
        starts[i, :len(st)], counts[i] = st, len(st)
    int_corners = np.array([blk[3] for blk in boxes], np.int64)
    return polygon2d.assemble(vertices, links, starts, counts, int_corners, boxes[0][4] * (g - 1))


def test_polygon_in_chunks_matches_oracle(cb, scenes):
    """polygon() of the gear at feature size / 704 with boxes of 256^2 samples: 1223 boxes, two chunks of
    cc_polygon_blocks.  The reference is oracle.host.polygon's procedure on the oracle's boxes and per-box kernels, with
    the chains joined by the native assembler, which tests/test_gpu_polygon.py holds to oracle.host.polygon: at this
    size host.polygon would build a Python tuple for each of the 2^27 triangles' vertices, minutes of run time."""
    from codecad_b200 import CompiledScene
    from codecad_b200.rendering import polygon2d
    from test_polygon_oracle import canonical
    s = scenes["dsdf2d_gear"]
    small = host.subdivision(s.words, s.box_a, s.box_b, 2, s.feature_size / 32, True, 32)[1]
    assert canonical(_oracle_outlines(s.words, small, 32)) == canonical(host.polygon(s.words, s.box_a, s.box_b, s.feature_size / 16, 32))
    g, feature = 256, s.feature_size / 704
    t0 = time.time()
    got = list(polygon2d.polygon(CompiledScene(s.words, 2, s.box_a, s.box_b, feature, s.name), g))
    dims, boxes = host.subdivision(s.words, s.box_a, s.box_b, 2, feature / 2, True, g)
    chunk = (1 << 26) // (g * g)
    assert tuple(dims) == (g, g, 1) and len(boxes) > chunk, (dims, len(boxes))
    want = _oracle_outlines(s.words, boxes, g)
    assert len(got) == len(want) and canonical(got) == canonical(want)
    print("polygon(): %d boxes of %d^2 samples, %d chunks, %d outlines of %d vertices; %.1f s"
          % (len(boxes), g, -(-len(boxes) // chunk), len(got), sum(map(len, got)), time.time() - t0))


# ---- 7. cc_evaluate_points across 2^30 ----------------------------------------------------------------------------------

def test_evaluate_points_across_2_30(cb, scenes):
    """2^30 + 4099 points in one call: two launches.  The 8192 results around index 2^30 (distinct points) equal a
    separate small call on them and the oracle; so do the first and the last points."""
    _need_device_memory(36)
    import torch
    from codecad_b200 import _lib
    L = _lib.lib()
    s = scenes["cfg_planetary"]
    prog = _prog(s)
    n = (1 << 30) + 4099
    rng = np.random.default_rng(11)
    a, b = np.array(s.box_a), np.array(s.box_b)

    def points(k):
        p = np.zeros((k, 4), np.float32)
        p[:, :3] = a + (b - a) * (rng.random((k, 3)) * 1.2 - 0.1)
        return p

    pattern = points(4096)
    seam = points(8192)
    t0 = time.time()
    _reset_peak()
    pts = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    full = (n // 4096) * 4096
    pts[:full].view(-1, 4096, 4).copy_(torch.from_numpy(pattern).cuda().expand(n // 4096, 4096, 4))
    pts[full:] = torch.from_numpy(pattern[:n - full]).cuda()
    lo = (1 << 30) - 4096
    torch.cuda.synchronize()        # the pattern's copies (torch's stream) before the seam's (the library's)
    _lib.check(L.cc_memcpy_h2d_async(ctypes.c_void_p(pts.data_ptr() + lo * 16), seam.ctypes.data, seam.nbytes, None))
    out = _filled((n, 4))
    _lib.check(L.cc_synchronize())
    torch.cuda.synchronize()
    n0 = _launches()
    _lib.check(L.cc_evaluate_points(prog.handle, ctypes.c_void_p(pts.data_ptr()), n, ctypes.c_void_p(out.data_ptr()), None))
    _lib.check(L.cc_synchronize())
    launches = _launches() - n0
    peak = _peak_gib()
    del pts

    def small(p):
        d_in = torch.from_numpy(p).cuda()
        d_out = _filled((len(p), 4))
        torch.cuda.synchronize()
        n0 = _launches()
        _lib.check(L.cc_evaluate_points(prog.handle, ctypes.c_void_p(d_in.data_ptr()), len(p),
                                        ctypes.c_void_p(d_out.data_ptr()), None))
        _lib.check(L.cc_synchronize())
        return d_out.cpu().numpy(), _launches() - n0

    want_seam, one = small(seam)
    assert launches == 2 * one, "2^30 + 4099 points: %d launches, a small call %d" % (launches, one)
    got_seam = out[lo:lo + 8192].cpu().numpy()
    same = got_seam.tobytes() == want_seam.tobytes()
    assert same, "results around index 2^30 differ from a separate call"
    assert np.array_equal(got_seam.view(np.float32), oracle.evaluate_points(s.words, seam[:, :3]), equal_nan=True)
    want_pattern, _ = small(pattern)
    same = out[:4096].cpu().numpy().tobytes() == want_pattern.tobytes()
    assert same, "the first points differ from a separate call"
    same = out[full:].cpu().numpy().tobytes() == want_pattern[:n - full].tobytes()
    assert same, "the last points differ from a separate call"
    same = out[lo - 4096:lo].cpu().numpy().tobytes() == want_pattern.tobytes()
    assert same, "the pattern's last copy before the seam points differs from a separate call"
    del out
    torch.cuda.empty_cache()
    print("evaluate_points: %d points, %d launches (a small call: %d); test buffers peak %.1f GiB, %.1f s"
          % (n, launches, one, peak, time.time() - t0))
