"""CPU restatement of the welded mesh of cc_mesh_blocks_indexed (DESIGN.md 4.4) — TEST INFRASTRUCTURE
ONLY, independent of codecad_b200.  Built on the marching-cubes restatement of oracle/mc_oracle.py
(same case table, corner and edge numbering, interpolation and post-transform), it restates the
welded mesh's contract literally: a dict over lattice points in which the first holder wins, marching
cubes per block with each vertex's lattice edge, and vertices numbered in contract order with their
positions taken from the owner block."""
import numpy as np

from oracle.mc_oracle import CORNERS, EDGES, TABLE


def triangle_edges(block):
    """marching_cubes' triangles as the cell edges their vertices lie on: int [t][3][4] = (i, j, k, axis)
    of each vertex's edge, (i, j, k) its lower end; same triangle and vertex order."""
    block = np.asarray(block, dtype=np.float32)
    d0, d1, d2 = block.shape
    inside = block <= np.float32(0.0)
    out = []
    for i in range(d0 - 1):
        for j in range(d1 - 1):
            for k in range(d2 - 1):
                case = 0
                for m, (a, b, c) in enumerate(CORNERS):
                    if inside[i + a, j + b, k + c]:
                        case |= 1 << m
                for tri in TABLE[case]:
                    edges = []
                    for e in tri:
                        ca, cb = EDGES[e]
                        low = [base + off for base, off in zip((i, j, k), CORNERS[ca])]
                        axis = [x != y for x, y in zip(CORNERS[ca], CORNERS[cb])].index(True)
                        edges.append(low + [axis])
                    out.append(edges)
    return np.array(out, dtype=np.int64).reshape(-1, 3, 4)


def indexed_mesh(fields, corners, int_corners, resolution):
    """The welded mesh of cc_mesh_blocks_indexed, restated from its contract.
    fields: float32 [n][d0][d1][d2] (the PYMCUBES blocks), corners float64 [n][3], int_corners [n][3].
    Returns (vertices float64 [v][3], triangles uint32 [t][3], triangle_block uint32 [t])."""
    fields = [np.asarray(f, dtype=np.float32) for f in fields]
    corners = [tuple(float(c) for c in p) for p in corners]
    int_corners = [tuple(int(c) for c in p) for p in int_corners]
    if not fields:
        return np.zeros((0, 3), np.float64), np.zeros((0, 3), np.uint32), np.zeros((0,), np.uint32)
    d0, d1, d2 = fields[0].shape
    ii, jj, kk = np.meshgrid(np.arange(d0), np.arange(d1), np.arange(d2), indexing="ij")

    def lattice(b):
        """lattice point of every sample of block b: array index (i, j, k) -> (X + j, Y + d0-1-i, Z + k)"""
        x, y, z = int_corners[b]
        return zip((x + jj).ravel().tolist(), (y + d0 - 1 - ii).ravel().tolist(), (z + kk).ravel().tolist())

    # 1. every sample takes the value of the first block in input order that holds it
    first = {}
    for b, f in enumerate(fields):
        for point, value in zip(lattice(b), f.ravel().tolist()):
            first.setdefault(point, value)
    rec = [np.array([first[p] for p in lattice(b)], dtype=np.float32).reshape(d0, d1, d2) for b in range(len(fields))]

    # 2. the owner of an edge is the first block holding both ends; the reconciled fields agree on
    # every shared sample, so that is the first block in which the edge is crossed
    def crossed(b):
        inside = rec[b] <= np.float32(0.0)
        found = []
        for axis in range(3):
            lo = [slice(None)] * 3
            hi = [slice(None)] * 3
            lo[axis], hi[axis] = slice(0, -1), slice(1, None)
            for i, j, k in zip(*np.nonzero(inside[tuple(lo)] != inside[tuple(hi)])):
                found.append((int(i), int(j), int(k), axis))
        return sorted(found)  # contract order: lower end in (i, j, k) order, then axis

    def key(b, i, j, k, axis):
        x, y, z = int_corners[b]
        return (x + j, y + d0 - 1 - i, z + k, axis)

    owner = {}
    for b in range(len(fields)):
        for e in crossed(b):
            owner.setdefault(key(b, *e), (b, e))

    # 3. vertices numbered by owner block, then edge; positions from the owner block
    index, vertices = {}, []
    for b in range(len(fields)):
        for e in crossed(b):
            kk_ = key(b, *e)
            if owner[kk_][0] != b:
                continue
            i, j, k, axis = e
            p = [float(i), float(j), float(k)]
            a1 = p[axis]
            a2 = a1 + 1.0
            f1, f2 = float(rec[b][i, j, k]), float(rec[b][(i + (axis == 0), j + (axis == 1), k + (axis == 2))])
            p[axis] = a1 + (0.0 - f1) * (a2 - a1) / (f2 - f1)
            cx, cy, cz = corners[b]
            index[kk_] = len(vertices)
            vertices.append((p[1] * resolution + cx, -p[0] * resolution + cy, p[2] * resolution + cz))

    triangles, triangle_block = [], []
    for b in range(len(fields)):
        for tri in triangle_edges(rec[b]).tolist():
            ids = [index[key(b, *e)] for e in tri]
            triangles.append((ids[1], ids[0], ids[2]))  # block_mesh's winding flip
            triangle_block.append(b)
    return (np.array(vertices, dtype=np.float64).reshape(-1, 3), np.array(triangles, dtype=np.uint32).reshape(-1, 3),
            np.array(triangle_block, dtype=np.uint32))


def index_manifold_report(triangles, n_vertices):
    """Closedness of an indexed mesh with no tolerance: every directed edge once and its reverse once,
    every vertex referenced; also V - E + F (= V - T/2 when closed)."""
    t = np.asarray(triangles, dtype=np.int64).reshape(-1, 3)
    directed = np.concatenate([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]])
    code = directed[:, 0] * int(n_vertices) + directed[:, 1]
    uniq, counts = np.unique(code, return_counts=True)
    reverse = (code % int(n_vertices)) * int(n_vertices) + code // int(n_vertices)
    paired = np.isin(reverse, uniq)
    return {"repeated_edges": int((counts > 1).sum()), "unpaired_edges": int((~paired).sum()),
            "unreferenced_vertices": int(n_vertices) - len(np.unique(t)),
            "euler": int(n_vertices) - len(uniq) // 2 + len(t)}
