"""The rounding budget of the exact shortcuts (part masks, DESIGN.md 4.9; union forests, 4.7) away from the
origin, on scenes built by tests/programs.py.

The budget (`slack`) bounds |computed - exact| of a part's fp32 value over a launch; it must cover every
magnitude in that arithmetic: the grid's coordinates (for launches over blocks: the blocks' corners) and the
part's constants (translations, vertices, sizes).  The central scene is a near-tie assembly — thin parallel
quads one unit apart, tilted off the grid axes, so that the medial surface between two parts crosses bricks and
tiles at every offset within a cell — with its offset carried (a) by the polygons' vertices and (b) by the
translation of its transforms.  A budget short of the rounding drops a part at a cell where the full walk picks
it, and the cell's bits change.
"""
import ctypes

import numpy as np
import pytest

import oracle
import programs as P

pytestmark = pytest.mark.gpu

OFFSETS = [1e3, 1e4, 1e5, 1e6]
# cell size of the hierarchy sinks per offset: leaf blocks of 16 cells are ~250 ulp(offset) wide far out
# (closer in, the size of the scene bounds the cell count)
RESOLUTION = {1e3: 0.1, 1e4: 0.1, 1e5: 0.12, 1e6: 1.0}


@pytest.fixture(scope="module")
def cb():
    import codecad_b200
    from codecad_b200 import _lib
    _lib.init(0)
    L = _lib.lib()
    old_jit = _lib.check(L.cc_set_jit_mode(2))     # compile at first use and wait: the part kernels are NVRTC kernels
    old_forest = _lib.check(L.cc_set_forest_mode(0))
    old_parts = _lib.check(L.cc_set_parts_mode(1))
    old_columns = _lib.check(L.cc_set_columns_mode(1))
    yield codecad_b200
    _lib.check(L.cc_set_columns_mode(old_columns))
    _lib.check(L.cc_set_parts_mode(old_parts))
    _lib.check(L.cc_set_forest_mode(old_forest))
    _lib.check(L.cc_set_jit_mode(old_jit))


class modes:
    """set library switches for a block, restore them after"""

    def __init__(self, **kw):
        self.kw = kw

    def __enter__(self):
        from codecad_b200 import _lib
        L = _lib.lib()
        self.old = {k: _lib.check(getattr(L, "cc_set_%s_mode" % k)(v)) for k, v in self.kw.items()}

    def __exit__(self, *exc):
        from codecad_b200 import _lib
        L = _lib.lib()
        for k, v in self.old.items():
            _lib.check(getattr(L, "cc_set_%s_mode" % k)(v))


def _f4(arr):
    return np.stack([arr["x"], arr["y"], arr["z"], arr["w"]], axis=-1)


def scene_of(tree, centre, half, feature_size, name):
    from codecad_b200 import CompiledScene
    words = P.program(tree)
    a = tuple(float(c - h) for c, h in zip(centre, half))
    b = tuple(float(c + h) for c, h in zip(centre, half))
    return words, CompiledScene(words, 3, a, b, float(feature_size), name), a, b


def near_tie_scene(offset, variant, feature_size=1.0):
    if variant == "oblique":
        tree, centre = P.oblique_assembly(offset), P.oblique_centre(offset)
        half = (24.0, 24.0, 24.0)
    else:
        tree, centre = P.near_tie_assembly(offset, carried_by=variant), (offset, offset, 0.0)
        half = (21.0, 21.0, 6.0)
    return scene_of(tree, centre, half, feature_size, "near_tie_%s_%g" % (variant, offset))


# ---- hierarchy sinks: part masks per tile over blocks (prepare_part_masks with a.blocks) ----

def _hierarchy_results(cb, scene, res):
    from codecad_b200 import _lib
    from codecad_b200.rendering import mesh
    n0 = _lib.counters()[0]
    mp = cb.mass_properties(scene, res, 32)
    sub = cb.subdivision(scene, res, grid_size=16)
    vertices, block, _ = mesh.mesh_arrays(scene, 32)
    launches = _lib.counters()[0] - n0
    return launches, (mp.volume, tuple(mp.centroid), np.array(mp.inertia_tensor).tobytes(),
                      [tuple(map(tuple, (blk[0], blk[1], blk[3]))) + (blk[2], blk[4]) for blk in sub[2]],
                      np.array(vertices).tobytes(), np.array(block).tobytes())


@pytest.mark.parametrize("offset", OFFSETS)
@pytest.mark.parametrize("variant", ["vertices", "translation", "oblique"])
def test_hierarchy_sinks_far_assembly_identical_with_and_without_masks(cb, offset, variant):
    """mass_properties (volume, centroid, inertia bits), subdivision (the ordered leaf list) and the mesh (vertex
    and block bytes) of the near-tie assembly with the per-tile part masks and without; the column-split
    variants with the column kernels on, the oblique one (no split) with the plain tile units"""
    from codecad_b200 import _lib
    from codecad_b200.cl_util.buffer import ProgramBuffer
    res = RESOLUTION[offset]
    words, scene, _, _ = near_tie_scene(offset, variant, feature_size=2 * res)
    info = _lib.decode_program(words)[0]
    assert info.n_parts == 3 and (info.column_invariant_percent == 0) == (variant == "oblique")
    scene.program_buffer().wait_specialized(ProgramBuffer.SINK_MASS | ProgramBuffer.SINK_CLASSIFY | ProgramBuffer.SINK_PYMCUBES)
    out = {}
    for parts in (1, 0):
        with modes(parts=parts):
            out[parts] = _hierarchy_results(cb, scene, res)
    assert out[1][0] > out[0][0], "the tile-centre passes did not run"
    names = ("volume", "centroid", "inertia", "leaf blocks", "mesh vertices", "mesh blocks")
    for k in range(6):
        if out[1][1][k] != out[0][1][k]:
            extra = ""
            if k == 3:
                extra = " (%d vs %d leaves)" % (len(out[1][1][3]), len(out[0][1][3]))
            elif k == 4:
                a, b = np.frombuffer(out[1][1][4], np.float64), np.frombuffer(out[0][1][4], np.float64)
                extra = " (%d vs %d coordinates, %d differ)" % (a.size, b.size, int((a != b).sum()) if a.size == b.size else -1)
            pytest.fail("%s %g: %s differs with the part masks%s" % (variant, offset, names[k], extra))
    assert out[1][1][0] > 0 and len(out[1][1][3]) > 0


def test_hierarchy_sinks_far_assembly_match_the_oracle(cb):
    """one small size against the host oracle: mass sums (float64 order aside) and the leaf list"""
    from oracle import host
    offset, res = 1e5, 0.25
    words, scene, a, b = near_tie_scene(offset, "vertices", feature_size=2 * res)
    with modes(parts=1):
        got = cb.mass_properties(scene, res, 32)
        _, got_dims, got_sub = cb.subdivision(scene, res, True, 16)
    w_vol, w_cen, w_inertia = host.mass_properties(words, a, b, res, 32)
    assert got.volume == pytest.approx(w_vol, rel=1e-12)
    assert tuple(got.centroid) == pytest.approx(tuple(w_cen), rel=1e-12)
    assert np.allclose(got.inertia_tensor, w_inertia, rtol=1e-9, atol=1e-9 * np.abs(w_inertia).max())
    want_dims, want_sub = host.subdivision(words, a, b, 3, res, True, 16)
    assert tuple(got_dims) == tuple(want_dims)
    key = lambda blk: tuple(blk[3])
    assert [tuple(blk[3]) for blk in sorted(got_sub, key=key)] == [tuple(blk[3]) for blk in sorted(want_sub, key=key)]
    assert len(got_sub) > 0


# ---- dense grids: specialised parts kernels, interpreter tier, columns + parts ----

PATHS = {"parts": dict(jit=2, columns=0), "interpreter": dict(jit=0, columns=0), "columns": dict(jit=2, columns=1)}


def far_ring(distance, n=3, length=40.0, width=0.3, h=5.0):
    """`n` thin quads whose vertices are `distance` from the origin at equal angles, each across its radius:
    from around the origin their distances nearly tie along the bisectors"""
    parts = []
    for k in range(n):
        ang = 2 * np.pi * k / n + 0.05
        radial, tangent = np.array([np.cos(ang), np.sin(ang)]), np.array([-np.sin(ang), np.cos(ang)])
        quad = P.tilted_quad(radial * distance, tangent, radial, length, width)
        parts.append(P.Part.polygon(quad, h))
    return P.balanced(parts)


def dense_cases():
    cases = []
    for offset in OFFSETS:
        words = P.program(P.near_tie_assembly(offset))
        cases.append(("near_tie_%g" % offset, words, np.array([offset, offset, 0.0]), 4 * float(np.spacing(np.float32(offset)))))
    for distance in (1e5, 1e6):
        cases.append(("far_ring_%g" % distance, P.program(far_ring(distance)), np.zeros(3), 0.02))
    return cases


DENSE = dense_cases()


def _window_steps(offset_step):
    return [np.float32(max(offset_step, s)) for s in (0.005, 0.05, 0.4)]


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("case", range(len(DENSE)), ids=[c[0] for c in DENSE])
def test_dense_grids_far_parts_bit_exact_vs_oracle(cb, path, case):
    from codecad_b200 import CompiledScene
    from codecad_b200.cl_util.buffer import ProgramBuffer
    name, words, centre, min_step = DENSE[case]
    scene = CompiledScene(words, 3, tuple(centre - 25), tuple(centre + 25), 1.0, name)
    scene.program_buffer().wait_specialized(ProgramBuffer.SINK_FLOAT4)
    rng = np.random.default_rng(case)
    cfg = PATHS[path]
    with modes(jit=cfg["jit"], columns=cfg["columns"], parts=1):
        for step in _window_steps(min_step):
            for dims in ((40, 33, 48), (24, 40, 64)):
                # windows across the medial surfaces: the centre of the tie region, jittered
                c = centre + rng.uniform(-3, 3, 3) * [1, 1, 0.5]
                corner = (c - step * np.array(dims) / 2).astype(np.float32)
                want = oracle.grid_eval(words, corner, step, dims)
                got = _f4(cb.grid_eval(scene, corner, step, dims))
                assert np.array_equal(got, want, equal_nan=True), "%s %s step %g: %d values differ" % (
                    name, path, step, int(np.any(got != want, axis=-1).sum()))


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("case", range(len(DENSE)), ids=[c[0] for c in DENSE])
def test_dense_grids_far_parts_equal_the_full_walk(cb, path, case):
    from codecad_b200 import CompiledScene
    from codecad_b200.cl_util.buffer import ProgramBuffer
    name, words, centre, min_step = DENSE[case]
    scene = CompiledScene(words, 3, tuple(centre - 25), tuple(centre + 25), 1.0, name)
    scene.program_buffer().wait_specialized(ProgramBuffer.SINK_FLOAT4)
    cfg = PATHS[path]
    for step, dims, x_offset in ((0.4, (128, 128, 40), 0), (max(min_step, 0.03), (130, 70, 90), 5)):
        step = np.float32(step)
        corner = (centre - step * np.array(dims) / 2).astype(np.float32)
        with modes(jit=cfg["jit"], columns=cfg["columns"], parts=1):
            got = np.array(cb.grid_eval(scene, corner, step, dims, x_offset=x_offset))
        with modes(jit=cfg["jit"], columns=cfg["columns"], parts=0):
            want = np.array(cb.grid_eval(scene, corner, step, dims, x_offset=x_offset))
        if got.tobytes() != want.tobytes():
            g, w = _f4(got), _f4(want)
            pytest.fail("%s %s step %g: %d cells differ" % (name, path, step, int(np.any(g != w, axis=-1).sum())))


# ---- union forests far away and crowded ----

def forest_cases():
    rng = np.random.default_rng(31)
    cases = []
    for n, offset, r, size in ((200, 0.0, -1.0, 1.0), (600, 1e3, 0.5, 1.0), (300, 1e4, 1.0, 1.0), (1000, 1e5, 0.5, 10.0), (400, 1e5, -1.0, 10.0)):
        prims = P.primitive_cloud(rng, n, (offset,) * 3, 30.0 * size, size)
        tree = P.balanced([P.comb(prims[i:i + 6], r * size if r >= 0 else r) for i in range(0, n, 6)], r * size if r >= 0 else r)
        cases.append(("forest%d_%g_r%g" % (n, offset, r), P.program(tree), np.array([offset] * 3), size, False))
    # a dense cluster: 400 primitives within one super-tile (32 cells), stack depth 6: the second launch
    prims = P.primitive_cloud(rng, 400, (0.0, 0.0, 0.0), 3.0, 0.5)
    tree = P.balanced([P.comb(prims[i:i + 8], 0.2) for i in range(0, 400, 8)], 0.2)
    cases.append(("cluster400", P.program(tree), np.zeros(3), 0.1, True))
    return cases


FORESTS = forest_cases()


@pytest.mark.parametrize("case", range(len(FORESTS)), ids=[c[0] for c in FORESTS])
def test_forest_far_and_crowded(cb, case):
    from codecad_b200 import CompiledScene, _lib
    name, words, centre, size, cluster = FORESTS[case]
    span = 34.0 * size if not cluster else 3.5
    scene = CompiledScene(words, 3, tuple(centre - span), tuple(centre + span), size, name)
    buf = scene.program_buffer()
    assert buf.info.n_forest_leaves > 0
    fi = (ctypes.c_uint32 * 4)()
    assert _lib.lib().cc_program_get_forest_info(buf.handle, fi) == 1
    assert fi[2] > 4, "no deeper than the first launch's stack"
    if cluster:
        assert fi[3] > 256, "no more events than the first launch provides"
    rng = np.random.default_rng(case)
    # against the oracle on windows (one across the whole scene, smaller ones inside)
    for frac, dims in ((1.0, (40, 33, 48)), (0.2, (48, 40, 33)), (0.03, (33, 48, 40))):
        step = np.float32(2 * span * frac / 40)
        c = centre + rng.uniform(-0.3, 0.3, 3) * span * (1 - frac)
        corner = (c - step * np.array(dims) / 2).astype(np.float32)
        want = oracle.grid_eval(words, corner, step, dims)
        with modes(forest=1):
            got = _f4(cb.grid_eval(scene, corner, step, dims))
        assert np.array_equal(got, want, equal_nan=True), "%s frac %g: %d values differ" % (name, frac, int(np.any(got != want, axis=-1).sum()))
    # against the walk without the forest on larger grids (the 1000 primitives' walk against the oracle instead,
    # on grids half as wide)
    walk = buf.info.n_forest_leaves <= 600
    step = np.float32(2 * span / 128)
    for dims, x_offset in (((128, 128, 128), 0), ((130, 70, 90), 5)):
        if not walk:
            dims = tuple(d // 2 for d in dims)
        corner = (centre - step * np.array(dims) / 2).astype(np.float32)
        with modes(forest=1):
            got = np.array(cb.grid_eval(scene, corner, step, dims, x_offset=x_offset))
        if walk:
            with modes(forest=0, parts=0):
                want = np.array(cb.grid_eval(scene, corner, step, dims, x_offset=x_offset))
            assert got.tobytes() == want.tobytes(), "%s: forest kernel differs from the full walk" % name
        else:
            want = oracle.grid_eval(words, corner, step, dims, x_offset=x_offset)
            assert np.array_equal(_f4(got), want, equal_nan=True), "%s: forest kernel differs from the oracle" % name


# ---- polygon edge groups on the GPU ----

POLYGONS = [(n, v) for n, v in P.test_polygons(np.random.default_rng(23), scales=(1e2, 1e6))
            if not n.startswith("star9@") and not n.startswith("sliver10@")]


@pytest.mark.parametrize("tier", ["specialised", "interpreter"])
@pytest.mark.parametrize("case", range(len(POLYGONS)), ids=[p[0] for p in POLYGONS])
def test_polygon_groups_bit_exact_vs_oracle(cb, case, tier):
    """the polygons as 2-D scenes and extruded, by evaluate_points (near-edge and near-tie points) and grid_eval"""
    from codecad_b200 import CompiledScene
    from codecad_b200.cl_util.buffer import ProgramBuffer
    name, v = POLYGONS[case]
    rng = np.random.default_rng(case)
    lo, hi = v.min(0).astype(np.float64), v.max(0).astype(np.float64)
    ext = max(float((hi - lo).max()), 1e-3)
    words2 = P.polygon_program(v)
    words3 = P.program(P.Part.polygon(v, 0.3 * ext))
    pts = np.concatenate([P.near_edge_points(rng, v, 20000), P.near_tie_points(rng, v, 2000)])
    pts3 = pts.copy()
    pts3[:, 2] = (rng.uniform(-0.4, 0.4, len(pts)) * ext).astype(np.float32)
    for dim, words, p in ((2, words2, pts), (3, words3, pts3)):
        a = tuple(lo - 0.1 * ext) + (-0.4 * ext,)
        b = tuple(hi + 0.1 * ext) + (0.4 * ext,)
        scene = CompiledScene(words, dim, a, b, ext / 50, "%s_%dd" % (name, dim))
        if tier == "specialised":
            scene.program_buffer().wait_specialized(ProgramBuffer.SINK_FLOAT4 | ProgramBuffer.SINK_POINTS)
        with modes(jit=2 if tier == "specialised" else 0):
            got = np.asarray(cb.evaluate_points(scene, p))
            want = oracle.evaluate_points(words, p)
            got = got if got.ndim == 2 else _f4(got)
            diff = np.any(got.view(np.uint32) != want.view(np.uint32), axis=1)
            assert not diff.any(), "%s %dd %s: %d points differ" % (name, dim, tier, int(diff.sum()))
            step = np.float32(1.2 * ext / 40)
            corner = ((lo + hi) / 2 - step * 20).tolist() + [-step * 8]
            corner = np.array(corner, np.float32)
            dims = (40, 37, 16 if dim == 3 else 1)
            want = oracle.grid_eval(words, corner, step, dims)
            got = _f4(cb.grid_eval(scene, corner, step, dims))
            assert np.array_equal(got, want, equal_nan=True), "%s %dd %s grid: %d values differ" % (
                name, dim, tier, int(np.any(got != want, axis=-1).sum()))
