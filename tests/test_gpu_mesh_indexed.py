"""Welded mesh export on the GPU (cc_mesh_blocks_indexed behind codecad_b200.rendering.indexed_mesh):
bit-exact against the contract's CPU restatement (tests/indexed_mesh_oracle.py) on the same blocks,
closed by index with no tolerance, equal to the triangle soup where blocks agree on shared samples,
the same in the resident and chunked paths, input checks, and the 3MF file."""
import numpy as np
import pytest

import oracle
from oracle import host, mc_oracle as mc

import indexed_mesh_oracle as imo

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cb():
    import codecad_b200
    from codecad_b200 import _lib
    _lib.init(0)
    return codecad_b200


def _size(s):
    return max(b - a for a, b in zip(s.box_a, s.box_b))


def _scene_at(s, res):
    """The scene with feature_size / 2 = res, so that indexed_mesh and mesh_arrays mesh at res."""
    from codecad_b200 import CompiledScene
    return CompiledScene(s.words, 3, s.box_a, s.box_b, 2 * res, "%s@%r" % (s.name, res))


def _oracle_blocks(s, res, grid_size):
    dims, blocks = host.subdivision(s.words, s.box_a, s.box_b, s.dimension, res, True, grid_size)
    fields = []
    for box_size, box_corner, box_resolution, *_ in blocks:
        corner32 = np.array(box_corner, np.float64).astype(np.float32)
        field = oracle.grid_eval_pymcubes(s.words, corner32, np.float32(box_resolution), box_size)
        fields.append(field.reshape(-1).reshape(tuple(int(d) for d in dims)))  # mesh.py:20
    corners = np.array([b[1] for b in blocks], np.float64).reshape(-1, 3)
    int_corners = np.array([b[3] for b in blocks], np.int64).reshape(-1, 3)
    return fields, corners, int_corners


def _differing_shared_planes(corners, int_corners, n, res):
    """Face-neighbour pairs whose shared plane of samples gets different coordinates in the two blocks:
    fp32 sample coordinate (fp32(corner) + step * i) or float64 vertex coordinate (mesh.py:68-71)."""
    m = n - 1
    where = {tuple(c): b for b, c in enumerate(int_corners.tolist())}
    step = np.float32(res)
    count = 0
    for a, ca in enumerate(int_corners.tolist()):
        for ax in range(3):
            nb = list(ca)
            nb[ax] += m
            b = where.get(tuple(nb))
            if b is None:
                continue
            # block a's last sample layer along world axis ax is block b's first
            if ax == 1:   # y is flipped: a's layer is array row i = 0, b's is row i = m
                f32_a, f32_b = np.float32(corners[a][1]) + step * np.float32(m), np.float32(corners[b][1])
                f64_a, f64_b = -0.0 * res + corners[a][1], -float(m) * res + corners[b][1]
            else:
                f32_a, f32_b = np.float32(corners[a][ax]) + step * np.float32(m), np.float32(corners[b][ax])
                f64_a, f64_b = float(m) * res + corners[a][ax], 0.0 * res + corners[b][ax]
            count += bool(f32_a != f32_b or f64_a != f64_b)
    return count


SCENES = ["sub_box10", "dsdf3d_sphere", "dsdf3d_torus", "x_shell_sphere"]


@pytest.mark.parametrize("resolution", ["feature", "size/37"])
@pytest.mark.parametrize("grid_size", [2, 12, 16])
@pytest.mark.parametrize("name", SCENES)
def test_bit_exact_against_the_oracle(cb, scenes, name, grid_size, resolution):
    from codecad_b200.rendering import indexed_mesh
    s = scenes[name]
    res = s.feature_size / 2 if resolution == "feature" else _size(s) / 37
    fields, corners, int_corners = _oracle_blocks(s, res, grid_size)
    if resolution == "size/37":   # not dyadic: neighbours place some shared planes differently
        assert len(fields) > 1
        assert _differing_shared_planes(corners, int_corners, fields[0].shape[0], res) > 0
    v, t, b, boxes = indexed_mesh(_scene_at(s, res), grid_size)
    assert np.array_equal(np.asarray(boxes.corners if hasattr(boxes, "corners") else [x[1] for x in boxes], np.float64),
                          corners)
    want_v, want_t, want_b = imo.indexed_mesh(fields, corners, int_corners, res)
    assert len(want_t) > 0
    assert v.shape == want_v.shape and t.shape == want_t.shape
    assert np.array_equal(v, want_v)
    assert np.array_equal(t, want_t)
    assert np.array_equal(b, want_b)


@pytest.mark.parametrize("name, euler", [("sub_box10", 2), ("dsdf3d_sphere", 2), ("dsdf3d_torus", 0), ("x_shell_sphere", 4)])
def test_closed_manifold_by_index(cb, scenes, name, euler):
    from codecad_b200.rendering import indexed_mesh
    s = scenes[name]
    v, t, _, boxes = indexed_mesh(_scene_at(s, _size(s) / 96), 32)
    assert len(boxes) > 1
    rep = imo.index_manifold_report(t, len(v))
    assert rep == {"repeated_edges": 0, "unpaired_edges": 0, "unreferenced_vertices": 0, "euler": euler}, rep
    assert mc.signed_volume(v[t]) > 0


@pytest.mark.parametrize("name, res, grid_size", [("cfg_csg_example", 100.0 / 128, 16), ("cfg_planetary", None, 32)])
def test_closed_on_many_blocks(cb, scenes, name, res, grid_size):
    from codecad_b200.rendering import indexed_mesh
    s = scenes[name]
    res = res or _size(s) / 128
    v, t, _, boxes = indexed_mesh(_scene_at(s, res), grid_size)
    assert len(boxes) > 1 and len(t) > 10000
    rep = imo.index_manifold_report(t, len(v))
    assert rep["repeated_edges"] == 0 and rep["unpaired_edges"] == 0 and rep["unreferenced_vertices"] == 0, rep


def test_equal_to_the_soup(cb, scenes):
    from codecad_b200.rendering import indexed_mesh, mesh_arrays
    scene = _scene_at(scenes["sub_box10"], 5.0)
    for grid_size in (2, 3):
        soup, soup_b, boxes = mesh_arrays(scene, grid_size)
        v, t, b, _ = indexed_mesh(scene, grid_size)
        assert len(boxes) > 1 and len(t) > 0
        assert np.array_equal(v[t], soup) and np.array_equal(b, soup_b)


@pytest.mark.parametrize("mode", ["pipelined chunks", "one field buffer"])
def test_chunked_paths_give_the_same_mesh(cb, scenes, mode, monkeypatch):
    from codecad_b200.rendering import indexed_mesh
    scene = _scene_at(scenes["cfg_csg_example"], 100.0 / 128)
    want_v, want_t, want_b, boxes = indexed_mesh(scene, 16)
    assert len(boxes) > 40 and len(want_t) > 10000
    want_v, want_t, want_b = want_v.copy(), want_t.copy(), want_b.copy()
    block_bytes = 16 ** 3 * 4
    monkeypatch.setenv("CODECAD_B200_MESH_CHUNK_BYTES", str(7 * block_bytes))
    if mode == "one field buffer":
        monkeypatch.setenv("CODECAD_B200_MESH_FIELD_BUDGET", str(20 * block_bytes))
    v, t, b, _ = indexed_mesh(scene, 16)
    assert np.array_equal(v, want_v) and np.array_equal(t, want_t) and np.array_equal(b, want_b)


def test_invalid_inputs(cb, scenes):
    from codecad_b200 import _lib
    from codecad_b200.rendering import indexed_mesh_blocks
    from codecad_b200.subdivision import subdivision
    program, _, _ = subdivision(scenes["sub_box10"].compiled(), 2.5, grid_size=8)
    corners = np.zeros((2, 3))
    bad = [((8, 8, 9), [[0, 0, 0], [7, 0, 0]]),                 # several blocks, not cubic
           ((8, 8, 8), [[0, 0, 0], [5, 0, 0]]),                 # off the lattice of n - 1
           ((8, 8, 8), [[7, 0, 0], [7, 0, 0]]),                 # the same corner twice
           ((8, 8, 8), [[0, 0, 0], [0, 0, 7 << 21]])]           # wider than the block table
    for dims, ic in bad:
        with pytest.raises(_lib.CodecadB200Error, match="code -4"):
            indexed_mesh_blocks(program, dims, corners, np.array(ic, np.int64), 1.0)
    v, t, b = indexed_mesh_blocks(program, (8, 8, 8), np.zeros((0, 3)), np.zeros((0, 3), np.int64), 1.0)
    assert v.shape == (0, 3) and t.shape == (0, 3) and b.shape == (0,)


def test_render_3mf_round_trip(cb, scenes, tmp_path):
    from codecad_b200.rendering import indexed_mesh, render_3mf
    from test_mesh_indexed_oracle import read_3mf
    scene = scenes["dsdf3d_sphere"].compiled()
    path = tmp_path / "sphere.3mf"
    n = render_3mf(scene, str(path))
    v, t, _, _ = indexed_mesh(scene)
    got_v, got_t = read_3mf(str(path))
    assert n == len(t) > 0
    assert np.array_equal(got_v, v) and np.array_equal(got_t, t)
