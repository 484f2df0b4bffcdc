"""Which kernels serve each entry point.  Every route through the library gives the same bits, so a change of route
does not show in any result; it shows in the (launches, points) that cc_get_counters reports.  This pins them for every
entry point, per scene and mode: a union forest, an assembly with a column split, an extrusion with columns and no
parts, a scene with none of the three structures, and the assembly again as a segmented program (which has no column
or specialised part kernels, but keeps the interpreter's part culling)."""
import ctypes
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# (scene, CODECAD_B200_JIT_SEGMENT_OPS or None, jit mode, forest, parts, columns); a switch the scene has no
# structure for stays on
CASES = []
for _jit in (2, 0):
    CASES += [("cfg_synthetic32", None, _jit, f, 1, 1) for f in (1, 0)]
    CASES += [("cfg_planetary", None, _jit, 1, p, c) for p in (1, 0) for c in (1, 0)]
    CASES += [("x_gear3d", None, _jit, 1, 1, c) for c in (1, 0)]
    CASES += [("cfg_csg_example", None, _jit, 1, 1, 1)]
    CASES += [("cfg_planetary", "40", _jit, 1, p, c) for p in (1, 0) for c in (1, 0)]

ENTRIES = ("grid_eval", "grid_eval_pymcubes", "evaluate_points", "subdivision_step", "mass_properties_step",
           "subdivision", "mass_properties", "mesh", "cost_profile")


def case_id(case):
    name, seg, jit, forest, parts, columns = case
    return "%s%s-jit%d-forest%d-parts%d-columns%d" % (name, "-seg" + seg if seg else "", jit, forest, parts, columns)


# case -> (launches, points) of each entry point in ENTRIES order, then cc_program_specialize_wait's count for the
# four grid sinks
EXPECTED = {
    "cfg_synthetic32-jit2-forest1-parts1-columns1":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 262152), (9, 753691), (0, 0), 4],
    "cfg_synthetic32-jit2-forest0-parts1-columns1":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 262152), (9, 753691), (0, 0), 4],
    "cfg_planetary-jit2-forest1-parts1-columns1":
        [(4, 30720), (1, 30720), (1, 3000), (3, 3840), (3, 3840), (3, 48), (9, 131076), (13, 31753344), (2, 0), 9],
    "cfg_planetary-jit2-forest1-parts1-columns0":
        [(2, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (2, 0), 8],
    "cfg_planetary-jit2-forest1-parts0-columns1":
        [(3, 30720), (1, 30720), (1, 3000), (2, 3840), (2, 3840), (3, 48), (8, 131076), (11, 31753344), (0, 0), 8],
    "cfg_planetary-jit2-forest1-parts0-columns0":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (0, 0), 4],
    "x_gear3d-jit2-forest1-parts1-columns1":
        [(2, 30720), (1, 30720), (1, 3000), (2, 3840), (2, 3840), (3, 16), (8, 131076), (10, 131076), (0, 0), 8],
    "x_gear3d-jit2-forest1-parts1-columns0":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 16), (7, 131076), (9, 131076), (0, 0), 4],
    "cfg_csg_example-jit2-forest1-parts1-columns1":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 64), (7, 262152), (6, 343), (0, 0), 4],
    "cfg_planetary-seg40-jit2-forest1-parts1-columns1":
        [(2, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (2, 0), 4],
    "cfg_planetary-seg40-jit2-forest1-parts1-columns0":
        [(2, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (2, 0), 4],
    "cfg_planetary-seg40-jit2-forest1-parts0-columns1":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (0, 0), 4],
    "cfg_planetary-seg40-jit2-forest1-parts0-columns0":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (0, 0), 4],
    "cfg_synthetic32-jit0-forest1-parts1-columns1":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 262152), (9, 753691), (0, 0), 4],
    "cfg_synthetic32-jit0-forest0-parts1-columns1":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 262152), (9, 753691), (0, 0), 4],
    "cfg_planetary-jit0-forest1-parts1-columns1":
        [(2, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (2, 0), 9],
    "cfg_planetary-jit0-forest1-parts1-columns0":
        [(2, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (2, 0), 8],
    "cfg_planetary-jit0-forest1-parts0-columns1":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (0, 0), 8],
    "cfg_planetary-jit0-forest1-parts0-columns0":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (0, 0), 4],
    "x_gear3d-jit0-forest1-parts1-columns1":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 16), (7, 131076), (9, 131076), (0, 0), 8],
    "x_gear3d-jit0-forest1-parts1-columns0":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 16), (7, 131076), (9, 131076), (0, 0), 4],
    "cfg_csg_example-jit0-forest1-parts1-columns1":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 64), (7, 262152), (6, 343), (0, 0), 4],
    "cfg_planetary-seg40-jit0-forest1-parts1-columns1":
        [(2, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (2, 0), 4],
    "cfg_planetary-seg40-jit0-forest1-parts1-columns0":
        [(2, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (2, 0), 4],
    "cfg_planetary-seg40-jit0-forest1-parts0-columns1":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (0, 0), 4],
    "cfg_planetary-seg40-jit0-forest1-parts0-columns0":
        [(1, 30720), (1, 30720), (1, 3000), (1, 3840), (1, 3840), (3, 48), (7, 131076), (9, 31753344), (0, 0), 4],
}


def measure(scenes, case):
    """Runs every entry point once on a fresh program of the case's scene under its modes."""
    import codecad_b200 as cb
    from codecad_b200 import _lib
    from codecad_b200.cl_util import Buffer, opencl_manager
    from codecad_b200.cl_util.buffer import ProgramBuffer
    from codecad_b200.geometry import UCHAR4, Vector
    from codecad_b200.rendering import mesh
    name, seg, jit, forest, parts, columns = case
    L = _lib.lib()
    s = scenes[name]
    old_seg = os.environ.get("CODECAD_B200_JIT_SEGMENT_OPS")
    if seg:
        os.environ["CODECAD_B200_JIT_SEGMENT_OPS"] = seg
    old = (_lib.check(L.cc_set_jit_mode(jit)), _lib.check(L.cc_set_forest_mode(forest)),
           _lib.check(L.cc_set_parts_mode(parts)), _lib.check(L.cc_set_columns_mode(columns)))
    try:
        scene = s.compiled()
        prog = scene.program_buffer()
        size = max(b - a for a, b in zip(s.box_a, s.box_b))
        corner, step = s.grid(40)
        dims = (40, 24, 32)
        rng = np.random.default_rng(5)
        points = (np.array(s.box_a) + (np.array(s.box_b) - np.array(s.box_a)) * rng.uniform(-0.1, 1.1, (3000, 3))).astype(np.float32)
        sdims = (16, 12, 20)
        thr = np.float32(step * np.sqrt(3) / 2)
        res = size / 48

        def step_buffers():
            counter, lst = Buffer(np.uint32, 1), Buffer(UCHAR4, sdims[0] * sdims[1] * sdims[2])
            counter.enqueue_zero_fill_compatible()
            return counter, lst

        def subdivision_step():
            counter, lst = step_buffers()
            ev = opencl_manager.k.subdivision_step(sdims, None, prog, Vector(*corner).as_float4(), step, thr, counter, lst)
            counter.read(wait_for=[ev])

        def mass_properties_step():
            counter, lst = step_buffers()
            sums = Buffer(np.uint32, 10)
            sums.enqueue_zero_fill_compatible()
            ev = opencl_manager.k.mass_properties(sdims, None, prog, Vector(*corner).as_float4(), step, thr, sums, counter, lst)
            counter.read(wait_for=[ev])

        def cost_profile():
            n = (64, 40, 48)
            cost = (ctypes.c_double * 8)()
            _lib.check(L.cc_grid_eval_cost_profile(prog.handle, _lib.f3(corner), float(step), n[0], n[1], n[2], 0, cost, 8))

        calls = {
            "grid_eval": lambda: cb.grid_eval(scene, corner, step, dims),
            "grid_eval_pymcubes": lambda: cb.grid_eval_pymcubes(scene, corner, step, dims),
            "evaluate_points": lambda: cb.evaluate_points(scene, points),
            "subdivision_step": subdivision_step,
            "mass_properties_step": mass_properties_step,
            "subdivision": lambda: cb.subdivision(scene, res, grid_size=16),
            "mass_properties": lambda: cb.mass_properties(scene, res, 32),
            "mesh": lambda: mesh.mesh_arrays(scene, 32),
            "cost_profile": cost_profile,
        }
        got = []
        for entry in ENTRIES:
            n0 = _lib.counters()
            calls[entry]()
            n1 = _lib.counters()
            got.append((n1[0] - n0[0], n1[1] - n0[1]))
        sinks = ProgramBuffer.SINK_FLOAT4 | ProgramBuffer.SINK_PYMCUBES | ProgramBuffer.SINK_CLASSIFY | ProgramBuffer.SINK_MASS
        got.append(prog.wait_specialized(sinks)[0])
        return got
    finally:
        _lib.check(L.cc_set_jit_mode(old[0]))
        _lib.check(L.cc_set_forest_mode(old[1]))
        _lib.check(L.cc_set_parts_mode(old[2]))
        _lib.check(L.cc_set_columns_mode(old[3]))
        if old_seg is None:
            os.environ.pop("CODECAD_B200_JIT_SEGMENT_OPS", None)
        else:
            os.environ["CODECAD_B200_JIT_SEGMENT_OPS"] = old_seg


@pytest.fixture(scope="module")
def lib():
    from codecad_b200 import _lib
    _lib.init(0)
    return _lib


def test_structures_of_the_scenes(scenes):
    from codecad_b200 import _lib
    info = {n: _lib.decode_program(scenes[n].words)[0] for n in ("cfg_synthetic32", "cfg_planetary", "x_gear3d", "cfg_csg_example")}
    assert info["cfg_synthetic32"].n_forest_leaves > 0
    assert info["cfg_planetary"].n_parts > 0 and info["cfg_planetary"].column_invariant_percent > 0
    assert info["x_gear3d"].n_parts == 0 and info["x_gear3d"].column_invariant_percent > 0
    i = info["cfg_csg_example"]
    assert i.n_forest_leaves == 0 and i.n_parts == 0 and i.column_invariant_percent == 0


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_launch_and_point_counts(lib, scenes, case):
    got = measure(scenes, case)
    assert got == EXPECTED[case_id(case)], "got %s" % got
