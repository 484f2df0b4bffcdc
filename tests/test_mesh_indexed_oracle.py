"""The welded-mesh restatement (tests/indexed_mesh_oracle.py) on hand-made blocks, and the PLY / 3MF
writers of codecad_b200.rendering (host only)."""
import xml.etree.ElementTree as ET
import zipfile

import numpy as np
import pytest

from oracle import mc_oracle as mc

import indexed_mesh_oracle as imo


def _sphere_blocks(int_corners, n, centre, radius):
    """float32 PYMCUBES blocks of a sphere, sampled at the lattice points (X + j, Y + n-1-i, Z + k)."""
    i, j, k = np.meshgrid(np.arange(n), np.arange(n), np.arange(n), indexing="ij")
    out = []
    for x, y, z in int_corners:
        p = np.stack([x + j, y + n - 1 - i, z + k], axis=-1).astype(np.float64)
        out.append((np.linalg.norm(p - np.array(centre), axis=-1) - radius).astype(np.float32))
    return out


def test_one_block_expands_to_block_mesh():
    rng = np.random.default_rng(7)
    block = rng.standard_normal((6, 7, 5)).astype(np.float32)   # every case, ambiguous ones included
    block[2, 3, 1] = 0.0                                         # a sample exactly on the surface
    corner, res = (1.25, -3.5, 0.75), 0.3
    v, t, b = imo.indexed_mesh([block], [corner], [(4, 5, 6)], res)
    want = mc.block_mesh(block, corner, res)
    assert len(t) == len(want) > 50
    assert np.array_equal(v[t], want)
    assert np.array_equal(b, np.zeros(len(t), np.uint32))
    assert len(np.unique(t)) == len(v)


def test_second_block_takes_the_first_blocks_shared_face():
    n, res = 9, 0.5
    ic = [(0, 0, 0), (n - 1, 0, 0)]                     # neighbours along x: block 1's j = 0 is block 0's j = n-1
    corners = [tuple(c * res for c in p) for p in ic]
    fields = _sphere_blocks(ic, n, (8.0, 4.0, 4.0), 3.3)
    disturbed = [fields[0], fields[1].copy()]
    disturbed[1][:, 0, :] = -disturbed[1][:, 0, :] + np.float32(0.25)   # deliberately different values
    assert not np.array_equal(disturbed[1][:, 0, :], fields[0][:, n - 1, :])
    v, t, b = imo.indexed_mesh(disturbed, corners, ic, res)
    # the same mesh as when block 1 had evaluated its face like block 0
    agreed = [fields[0], disturbed[1].copy()]
    agreed[1][:, 0, :] = fields[0][:, n - 1, :]
    v2, t2, b2 = imo.indexed_mesh(agreed, corners, ic, res)
    assert np.array_equal(v, v2) and np.array_equal(t, t2) and np.array_equal(b, b2)
    assert set(b.tolist()) == {0, 1}
    # block 0 alone is unchanged, block 1's triangles are its soup on the agreed field
    assert np.array_equal(v[t[b == 0]], mc.block_mesh(fields[0], corners[0], res))
    assert np.array_equal(v[t[b == 1]], mc.block_mesh(agreed[1], corners[1], res))
    rep = imo.index_manifold_report(t, len(v))
    assert rep == {"repeated_edges": 0, "unpaired_edges": 0, "unreferenced_vertices": 0, "euler": 2}, rep


def _closed_mesh():
    n, res = 7, 0.5
    ic = [(0, 0, 0)]
    v, t, _ = imo.indexed_mesh(_sphere_blocks(ic, n, (3.0, 3.0, 3.0), 2.2), [(0.0, 0.0, 0.0)], ic, res)
    assert imo.index_manifold_report(t, len(v))["unpaired_edges"] == 0 and len(t) > 20
    return v, t


def test_write_ply_round_trip(tmp_path):
    from codecad_b200.rendering import write_ply
    v, t = _closed_mesh()
    path = tmp_path / "m.ply"
    assert write_ply(str(path), v, t) == len(t)
    raw = path.read_bytes()
    end = raw.index(b"end_header\n") + len(b"end_header\n")
    header = raw[:end].decode("ascii").splitlines()
    assert header[:2] == ["ply", "format binary_little_endian 1.0"]
    assert "element vertex %d" % len(v) in header and "element face %d" % len(t) in header
    got_v = np.frombuffer(raw, "<f8", 3 * len(v), end).reshape(-1, 3)
    faces = np.frombuffer(raw, np.dtype([("n", "u1"), ("v", "<u4", 3)]), len(t), end + 24 * len(v))
    assert end + 24 * len(v) + 13 * len(t) == len(raw)
    assert np.array_equal(got_v, v) and np.all(faces["n"] == 3) and np.array_equal(faces["v"], t)


def read_3mf(path):
    """(vertices float64 [v][3], triangles [t][3]) of a 3MF file with one mesh object."""
    ns = {"m": "http://schemas.microsoft.com/3dmanufacturing/core/2015/02"}
    with zipfile.ZipFile(path) as z:
        names = set(z.namelist())
        assert {"[Content_Types].xml", "_rels/.rels", "3D/3dmodel.model"} <= names
        assert "3D/3dmodel.model" in z.read("_rels/.rels").decode()
        root = ET.fromstring(z.read("3D/3dmodel.model"))
    assert root.get("unit") == "millimeter"
    assert len(root.findall("m:resources/m:object", ns)) == 1 and len(root.findall("m:build/m:item", ns)) == 1
    mesh = root.find("m:resources/m:object/m:mesh", ns)
    v = np.array([[float(e.get(a)) for a in "xyz"] for e in mesh.find("m:vertices", ns)], np.float64).reshape(-1, 3)
    t = np.array([[int(e.get(a)) for a in ("v1", "v2", "v3")] for e in mesh.find("m:triangles", ns)]).reshape(-1, 3)
    return v, t


def test_write_3mf_round_trip(tmp_path):
    from codecad_b200.rendering import write_3mf
    v, t = _closed_mesh()
    path = tmp_path / "m.3mf"
    assert write_3mf(str(path), v, t) == len(t)
    got_v, got_t = read_3mf(str(path))
    assert np.array_equal(got_v, v) and np.array_equal(got_t, t)


def test_writers_reject_indices_out_of_range(tmp_path):
    from codecad_b200.rendering import write_3mf, write_ply
    v = np.zeros((3, 3))
    for write in (write_ply, write_3mf):
        with pytest.raises(ValueError):
            write(str(tmp_path / "bad"), v, [[0, 1, 3]])
