"""Triangular mesh of a 3-D shape — same entry point as the reference's
/root/reference/codecad/rendering/mesh.py:10-74 `triangular_mesh(obj, subdivision_grid_size=None,
debug_subdivision_boxes=False)`: a generator of (vertices, triangles) pieces, one per leaf block of
`subdivision(obj, obj.feature_size() / 2)`.

The reference evaluates one block at a time (grid_eval_pymcubes launch, blocking 8 MiB copy) and
runs PyMCubes' marching cubes on the CPU (mesh.py:53-63).  Here `cc_mesh_blocks` does all blocks
on the device and returns the triangles in world coordinates, already carrying the reference's
post-transform (mesh.py:68-72).  Differences a caller can see: every piece is a triangle soup
(three fresh vertices per triangle, float64) instead of PyMCubes' shared-vertex arrays — the
consumers in the reference (`render_stl` expands to a soup, tests merge duplicate vertices) are
indifferent to it — and ambiguous faces are resolved by a fixed rule that keeps neighbouring cells
consistent (tools/make_mc_tables.py).

`indexed_mesh` (not in the reference) returns the same surface welded: shared vertices, triangles as
vertex indices, watertight by index (`cc_mesh_blocks_indexed`, DESIGN.md 4.4), for PLY / 3MF export.
"""
import ctypes

import numpy as np

from . import _compat  # noqa: F401  (kept tiny: shape protocol helpers)
from .. import _lib
from ..geometry import Vector
from ..subdivision import LeafBlocks, block_corners, subdivision


def _check_3d(obj):
    if hasattr(obj, "check_dimension"):
        obj.check_dimension(required=3)
    else:
        assert obj.dimension() == 3, "triangular_mesh needs a 3D shape"


def mesh_blocks(program_buffer, box_size, corners, resolution):
    """Marching cubes over equally sized blocks.  corners: float64 [n][3] (box_corner).
    Returns (vertices float64 [t][3][3], block index uint32 [t])."""
    corners = np.ascontiguousarray(corners, dtype=np.float64).reshape(-1, 3)
    out_v = ctypes.POINTER(ctypes.c_double)()
    out_b = ctypes.POINTER(ctypes.c_uint32)()
    n = ctypes.c_uint64()
    _lib.check(_lib.lib().cc_mesh_blocks(program_buffer.handle, corners.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                         float(resolution), int(box_size[0]), int(box_size[1]), int(box_size[2]),
                                         len(corners), ctypes.byref(out_v), ctypes.byref(out_b), ctypes.byref(n)))
    t = int(n.value)
    if t == 0:
        return np.zeros((0, 3, 3), np.float64), np.zeros((0,), np.uint32)
    # wrap the library's buffers without copying; they are released when the arrays die
    return _adopt(out_v, (t, 3, 3)), _adopt(out_b, (t,))


def indexed_mesh_blocks(program_buffer, box_size, corners, int_corners, resolution):
    """Welded marching cubes over the same blocks as mesh_blocks; int_corners: int64 [n][3]
    (LeafBlocks.int_corners).  Shared samples and vertices come from the first block that holds
    them, so the mesh is watertight by index.  Returns (vertices float64 [v][3], triangles uint32
    [t][3], block index uint32 [t]); vertices[triangles] is mesh_blocks' soup where neighbouring
    blocks evaluate their shared samples alike."""
    corners = np.ascontiguousarray(corners, dtype=np.float64).reshape(-1, 3)
    int_corners = np.ascontiguousarray(int_corners, dtype=np.int64).reshape(-1, 3)
    if len(int_corners) != len(corners):
        raise ValueError("corners and int_corners differ in length")
    out_v = ctypes.POINTER(ctypes.c_double)()
    out_t = ctypes.POINTER(ctypes.c_uint32)()
    out_b = ctypes.POINTER(ctypes.c_uint32)()
    nv, nt = ctypes.c_uint64(), ctypes.c_uint64()
    _lib.check(_lib.lib().cc_mesh_blocks_indexed(
        program_buffer.handle, corners.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
        int_corners.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), float(resolution),
        int(box_size[0]), int(box_size[1]), int(box_size[2]), len(corners),
        ctypes.byref(out_v), ctypes.byref(nv), ctypes.byref(out_t), ctypes.byref(out_b), ctypes.byref(nt)))
    v, t = int(nv.value), int(nt.value)
    if t == 0:
        return np.zeros((0, 3), np.float64), np.zeros((0, 3), np.uint32), np.zeros((0,), np.uint32)
    return _adopt(out_v, (v, 3)), _adopt(out_t, (t, 3)), _adopt(out_b, (t,))


class _Owner:
    """Keeps a malloc'ed library buffer alive for the numpy array built on top of it."""

    def __init__(self, pointer):
        self.pointer = pointer

    def __del__(self):
        if self.pointer and _lib._lib is not None:
            _lib._lib.cc_free(self.pointer)
            self.pointer = None


def _adopt(pointer, shape):
    owner = _Owner(pointer)
    arr = np.ctypeslib.as_array(pointer, shape=shape)
    holder = np.ndarray.__new__(_Held, shape=arr.shape, dtype=arr.dtype, buffer=arr)
    holder._owner = owner
    return holder


class _Held(np.ndarray):
    """ndarray that carries its buffer's owner (views inherit it through __array_finalize__)."""

    _owner = None

    def __array_finalize__(self, obj):
        if obj is not None:
            self._owner = getattr(obj, "_owner", None)


def mesh_arrays(obj, subdivision_grid_size=None):
    """All triangles of the shape at once: (vertices float64 [t][3][3], block index [t], boxes)."""
    _check_3d(obj)
    program_buffer, max_box_size, boxes = subdivision(obj, obj.feature_size() / 2, grid_size=subdivision_grid_size)
    if not len(boxes):
        return np.zeros((0, 3, 3), np.float64), np.zeros((0,), np.uint32), boxes
    corners = block_corners(boxes)
    # every leaf block has the same size and resolution (subdivision.py:97-111)
    vertices, block = mesh_blocks(program_buffer, max_box_size, corners, boxes[0][2])
    return vertices, block, boxes


def indexed_mesh(obj, subdivision_grid_size=None):
    """The shape's welded mesh, on the blocks mesh_arrays uses: (vertices float64 [v][3],
    triangles uint32 [t][3], block index uint32 [t], boxes)."""
    _check_3d(obj)
    program_buffer, max_box_size, boxes = subdivision(obj, obj.feature_size() / 2, grid_size=subdivision_grid_size)
    if not len(boxes):
        return np.zeros((0, 3), np.float64), np.zeros((0, 3), np.uint32), np.zeros((0,), np.uint32), boxes
    if isinstance(boxes, LeafBlocks):
        int_corners = boxes.int_corners
    else:  # a single-level plan: one block
        int_corners = np.array([[int(c) for c in b[3]] for b in boxes], dtype=np.int64).reshape(-1, 3)
    vertices, triangles, block = indexed_mesh_blocks(program_buffer, max_box_size, block_corners(boxes), int_corners,
                                                     boxes[0][2])
    return vertices, triangles, block, boxes


def triangular_mesh(obj, subdivision_grid_size=None, debug_subdivision_boxes=False):
    """Generate a triangular mesh representing the surface of a 3D shape.
    Yields tuples (vertices, indices) — rendering/mesh.py:10-74."""
    _check_3d(obj)
    if debug_subdivision_boxes:
        _, _, boxes = subdivision(obj, obj.feature_size() / 2, grid_size=subdivision_grid_size)
        for box_size, box_corner, box_resolution, *_ in boxes:  # mesh.py:28-50: the outline of each block
            size = Vector(*box_size)
            vertices = [Vector(i * size.x, j * size.y, k * size.z) * box_resolution + box_corner
                        for k in range(2) for j in range(2) for i in range(2)]
            triangles = [[0, 3, 1], [0, 2, 3], [1, 3, 5], [3, 7, 5], [4, 5, 6], [5, 7, 6],
                         [0, 6, 2], [0, 4, 6], [0, 1, 5], [0, 5, 4], [3, 2, 6], [3, 6, 7]]
            yield vertices, triangles
        return
    vertices, block, boxes = mesh_arrays(obj, subdivision_grid_size)
    if not len(block):
        return
    # triangles come back grouped by block, in block order
    starts = np.flatnonzero(np.r_[True, block[1:] != block[:-1]])
    ends = np.r_[starts[1:], len(block)]
    for s, e in zip(starts, ends):  # blocks without triangles are skipped, like mesh.py:65-66
        v = vertices[s:e].reshape(-1, 3)
        yield v, np.arange(len(v), dtype=np.int64).reshape(-1, 3)
