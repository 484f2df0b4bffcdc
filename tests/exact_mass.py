"""TEST INFRASTRUCTURE — true values of the integrals behind the assembly mass properties (DESIGN.md 4.11,
cc_assembly_mass_properties_exact), independent of the hierarchy, the part masks, the pair rule and the accumulator:

- exact integrals of axis-aligned boxes and of their intersections, in fractions.Fraction;
- the accumulator bound B_i of each integral (cc_api.cpp mass_quanta), which the tolerances are multiples of;
- a dense float64 count over every leaf cell of the plan's top block, for curved and rotated parts;
- groups of aligned boxes whose counted region is exactly the analytic one;
- the plumbing the GPU tests share (program buffers, the level plan, limbs -> integrals).

Integrals are in the library's order: one, x, y, z, xx, yy, zz, xy, xz, yz.

Why aligned boxes are exact: with a dyadic resolution s and dyadic corners, every leaf-cell centre and every fp32 cell
coordinate is exact, and a box whose faces lie on leaf-cell boundaries has no leaf-cell centre closer than s/2 to a face.
Each counted cube's integrals are exact per cube (x^2 over a cube of side s centred at b is s^3 (b^2 + s^2/12)), and the
coarse levels decide correctly for exact distance fields, so the counted region of a part is its box and that of a pair
is the boxes' intersection."""
import importlib
import math
from fractions import Fraction

import numpy as np

import oracle
import programs as P

NAMES = ("one", "x", "y", "z", "xx", "yy", "zz", "xy", "xz", "yz")
_SQUARES = ((0, 0), (1, 1), (2, 2), (0, 1), (0, 2), (1, 2))  # the axes of xx, yy, zz, xy, xz, yz


# ---- exact integrals of boxes ----------------------------------------------------------------------------------------

def box_integrals(lo, hi):
    """the ten integrals of the box [lo, hi] (3-tuples of exactly representable numbers) as Fractions; zeros if empty"""
    lo = [Fraction(v) for v in lo]
    hi = [Fraction(v) for v in hi]
    if any(h <= l for l, h in zip(lo, hi)):
        return [Fraction(0)] * 10
    m0 = [h - l for l, h in zip(lo, hi)]                     # int 1 along an axis
    m1 = [(h * h - l * l) / 2 for l, h in zip(lo, hi)]       # int x
    m2 = [(h ** 3 - l ** 3) / 3 for l, h in zip(lo, hi)]     # int x^2
    vol = m0[0] * m0[1] * m0[2]
    first = [m1[k] * m0[(k + 1) % 3] * m0[(k + 2) % 3] for k in range(3)]
    second = []
    for j, k in _SQUARES:
        if j == k:
            second.append(m2[j] * m0[(j + 1) % 3] * m0[(j + 2) % 3])
        else:
            second.append(m1[j] * m1[k] * m0[3 - j - k])
    return [vol] + first + second


def box_intersection(a, b):
    """the intersection of boxes a = (lo, hi) and b (possibly empty: some hi <= lo)"""
    return tuple(max(x, y) for x, y in zip(a[0], b[0])), tuple(min(x, y) for x, y in zip(a[1], b[1]))


def finish_exact(ints):
    """mass_properties.finish in Fractions: (volume, centroid[3], inertia 3x3 about the centroid); None if empty"""
    one, x, y, z, xx, yy, zz, xy, xz, yz = ints
    if one == 0:
        return None
    c = [x / one, y / one, z / one]
    first = (x, y, z)
    s = {}
    for (j, k), v in zip(_SQUARES, (xx, yy, zz, xy, xz, yz)):
        s[j, k] = v - c[j] * first[k] - c[k] * first[j] + c[j] * c[k] * one
    inertia = [[s[1, 1] + s[2, 2], -s[0, 1], -s[0, 2]],
               [-s[0, 1], s[0, 0] + s[2, 2], -s[1, 2]],
               [-s[0, 2], -s[1, 2], s[0, 0] + s[1, 1]]]
    return one, c, inertia


def exact_sets(boxes):
    """Fraction integrals [sets][10] of a group of boxes: the parts, then the pairs {a < b} at pair_index"""
    n = len(boxes)
    rows = [box_integrals(*b) for b in boxes]
    for a in range(n):
        for b in range(a + 1, n):
            rows.append(box_integrals(*box_intersection(boxes[a], boxes[b])))
    return rows


def as_float(rows):
    return np.array([[float(v) for v in row] for row in rows])


# ---- the plan and the accumulator bounds -----------------------------------------------------------------------------

def plan(box_a, box_b, resolution, grid):
    """(box_a, box_b, level plan) as the library's planner gives it (codecad_b200.subdivision.calculate_block_sizes)"""
    from codecad_b200.geometry import Vector
    from codecad_b200.subdivision import calculate_block_sizes
    a, b = Vector(*box_a), Vector(*box_b)
    return a, b, calculate_block_sizes((a, b), 3, resolution, grid, overlap=False)


def bounds(box_a, resolution, block_sizes):
    """B_i of cc_api.cpp mass_quanta, same float64 operations: V, V M_k, V M_j M_k of the plan's top-level block, with
    V its volume and M_k the largest |coordinate| along axis k plus one top-level cell"""
    cell, dims = block_sizes[0]
    s0 = resolution * float(cell)
    ext = [int(d) * s0 for d in dims]
    M, V = [], 1.0
    for k in range(3):
        M.append(max(abs(float(box_a[k])), abs(float(box_a[k]) + ext[k])) + s0)
        V *= ext[k]
    return np.array([V, V * M[0], V * M[1], V * M[2], V * M[0] * M[0], V * M[1] * M[1], V * M[2] * M[2],
                     V * M[0] * M[1], V * M[0] * M[2], V * M[1] * M[2]])


# ---- the library's calls (need the native library) -------------------------------------------------------------------

def buffers(words_list):
    from codecad_b200.cl_util.buffer import ProgramBuffer
    return [ProgramBuffer(np.asarray(w, np.float32)) for w in words_list]


def integrals(limbs, exps):
    mpm = importlib.import_module("codecad_b200.mass_properties")  # (the package exports a function of that name)
    return np.array([mpm.limbs_to_integrals(row, exps) for row in np.atleast_2d(limbs)])


def part_box(parts, margin=0.5):
    """a box around parts of tests/programs.py: each part's centre (where its placement puts its frame's origin) +- a
    radius that bounds the part"""
    lo, hi = [], []
    for p in parts:
        centre = -(P.quat_matrix(p.q).T @ np.asarray(p.t))
        kind = p.profile[0]
        r = float(np.linalg.norm(p.profile[1], axis=1).max()) if kind == "polygon" else \
            float(np.hypot(p.profile[1], p.profile[2])) if kind == "rectangle" else p.profile[1]
        r = float(np.hypot(r, p.h)) + (p.offset or 0.0) + margin
        lo.append(centre - r)
        hi.append(centre + r)
    return tuple(np.min(lo, axis=0).tolist()), tuple(np.max(hi, axis=0).tolist())


def snap_box(box_a, box_b, resolution):
    """box_a rounded down and box_b up to multiples of a dyadic resolution: the leaf cells' fp32 centres are exact"""
    return (tuple(math.floor(v / resolution) * resolution for v in box_a),
            tuple(math.ceil(v / resolution) * resolution for v in box_b))


# ---- the dense float64 reference -------------------------------------------------------------------------------------

def _cell_sums(lo, inside):
    """integer sums over the cells of a boolean grid whose [0, 0, 0] is leaf cell `lo`: n, sum i_k, sum i_j i_k"""
    n = int(inside.sum())
    if n == 0:
        return None
    idx = [np.arange(inside.shape[k], dtype=np.int64) + int(lo[k]) for k in range(3)]
    proj = [inside.sum(axis=tuple(a for a in range(3) if a != k), dtype=np.int64) for k in range(3)]
    first = [int(proj[k] @ idx[k]) for k in range(3)]
    second = []
    for j, k in _SQUARES:
        if j == k:
            second.append(int(proj[j] @ (idx[j] * idx[j])))
        else:
            plane = inside.sum(axis=3 - j - k, dtype=np.int64)   # axes (j, k) in ascending order
            second.append(int(idx[j] @ plane @ idx[k]))
    return n, first, second


def cell_integrals(box_a, resolution, lo, inside):
    """the ten integrals of the union of the leaf cells set in `inside` (cell [0, 0, 0] is leaf cell `lo` of the grid
    at box_a), each cube integrated exactly: the float64 of the exact sum"""
    sums = _cell_sums(lo, inside)
    if sums is None:
        return np.zeros(10)
    n, first, second = sums
    s = Fraction(resolution)
    c = [Fraction(float(v)) + s / 2 for v in box_a]  # centre of cell 0; cell i is at c + i s
    s3 = s ** 3
    out = [s3 * n] + [s3 * (n * c[k] + s * first[k]) for k in range(3)]
    for (j, k), t in zip(_SQUARES, second):
        if j == k:
            out.append(s3 * (n * (c[j] * c[j] + s * s / 12) + 2 * c[j] * s * first[j] + s * s * t))
        else:
            out.append(s3 * (n * c[j] * c[k] + c[j] * s * first[k] + c[k] * s * first[j] + s * s * t))
    return np.array([float(v) for v in out])


class DenseResult:
    """sets: float64 integrals [sets][10] (parts, then pairs at pair_index); marginal: cells whose float64 distance to
    some part was within the margin; disagreements: how many of those the fp32 oracle classified differently"""

    def __init__(self, sets, marginal, disagreements):
        self.sets, self.marginal, self.disagreements = sets, marginal, disagreements


def dense_reference(parts, box_a, resolution, block_sizes, eps=1e-5, slab=16):
    """Every leaf cell of the plan's top block, classified per part at its centre box_a + (i + 1/2) res: inside iff
    programs.eval_part's float64 distance <= 0, except marginal cells (|d| <= eps (1 + M), M the largest |coordinate|
    of the top block), which the fp32 oracle decides at the same point (inside iff its distance <= 0, as the leaf
    level's threshold 0).  With dyadic res and box_a those points are the library's fp32 cell coordinates.  A part is
    evaluated only inside its own bounding box (part_box), and a pair is the cells inside both parts."""
    cell, dims = block_sizes[0]
    n_cells = np.array([int(cell) * int(d) for d in dims])
    a = np.array([float(v) for v in box_a])
    M = float(np.max(np.maximum(np.abs(a), np.abs(a + n_cells * resolution))))
    tol = eps * (1.0 + M)
    grids, marginal, disagree = [], 0, 0
    for part in parts:
        words = P.program(part)
        plo, phi = part_box([part], margin=resolution)
        lo = np.clip(np.floor((np.asarray(plo) - a) / resolution).astype(np.int64), 0, n_cells)
        hi = np.clip(np.ceil((np.asarray(phi) - a) / resolution).astype(np.int64) + 1, 0, n_cells)
        inside = np.zeros(tuple(int(v) for v in np.maximum(hi - lo, 0)), bool)
        ys = a[1] + (np.arange(lo[1], hi[1]) + 0.5) * resolution
        zs = a[2] + (np.arange(lo[2], hi[2]) + 0.5) * resolution
        for x0 in range(int(lo[0]), int(hi[0]), slab):
            xs = a[0] + (np.arange(x0, min(x0 + slab, int(hi[0]))) + 0.5) * resolution
            pts = np.stack(np.meshgrid(xs, ys, zs, indexing="ij"), -1).reshape(-1, 3)
            d = P.eval_part(part, pts)[0]
            ins = d <= 0
            m = np.abs(d) <= tol
            if m.any():
                d32 = oracle.evaluate_points(words, pts[m])[:, 3]
                o = d32 <= 0                                    # (NaN: outside)
                marginal += int(m.sum())
                disagree += int((o != ins[m]).sum())
                ins[m] = o
            inside[x0 - lo[0]:x0 - lo[0] + len(xs)] = ins.reshape(len(xs), len(ys), len(zs))
        grids.append((lo, inside))
    rows = [cell_integrals(a, resolution, lo, g) for lo, g in grids]
    n = len(parts)
    for i in range(n):
        for j in range(i + 1, n):
            (lo_i, g_i), (lo_j, g_j) = grids[i], grids[j]
            lo = np.maximum(lo_i, lo_j)
            hi = np.minimum(lo_i + g_i.shape, lo_j + g_j.shape)
            if np.any(hi <= lo):
                rows.append(np.zeros(10))
                continue
            si = tuple(slice(int(l - o), int(h - o)) for l, h, o in zip(lo, hi, lo_i))
            sj = tuple(slice(int(l - o), int(h - o)) for l, h, o in zip(lo, hi, lo_j))
            rows.append(cell_integrals(a, resolution, lo, g_i[si] & g_j[sj]))
    return DenseResult(np.array(rows), marginal, disagree)


# ---- groups of aligned boxes -----------------------------------------------------------------------------------------
# A group is (parts, boxes, box_a, box_b): tests/programs.py parts, their exact boxes (lo, hi), and a dyadic box around
# them two leaf cells wider.  Sizes are in leaf cells of the resolution `res`, a power of two.

def _group(centres_halves, res, offset=(0.0, 0.0, 0.0)):
    parts, boxes = [], []
    for c, h in centres_halves:
        c = [(ci * res) + o for ci, o in zip(c, offset)]
        h = [hi * res for hi in h]
        parts.append(P.Part.placed(P.Part.box(h[0], h[1], h[2]), c))
        boxes.append((tuple(ci - hi for ci, hi in zip(c, h)), tuple(ci + hi for ci, hi in zip(c, h))))
    box_a = tuple(min(b[0][k] for b in boxes) - 2 * res for k in range(3))
    box_b = tuple(max(b[1][k] for b in boxes) + 2 * res for k in range(3))
    return parts, boxes, box_a, box_b


def _lattice(pitch):
    """32 (centre, half sizes) in leaf cells on a 4 x 4 x 2 lattice `pitch` (even) cells apart around the origin: half
    sizes pitch/2 + delta with delta in {-1, 0, 1, 2} per part and axis, so face neighbours are 2 or 1 cells apart,
    touch, or overlap by 1 to 4 cells, and some edge and corner neighbours overlap in small boxes"""
    out = []
    for i in range(4):
        for j in range(4):
            for k in range(2):
                delta = [(i + 2 * j + 3 * k + 5 * ax + i * j * ax) % 4 - 1 for ax in range(3)]
                centre = ((2 * i - 3) * pitch // 2, (2 * j - 3) * pitch // 2, (2 * k - 1) * pitch // 2)
                out.append((centre, tuple(pitch // 2 + d for d in delta)))
    return out


def lattice32(res, pitch=8):
    return _group(_lattice(pitch), res)


def nested(res, size=24):
    """a large box L (half size `size` cells); a box inside it touching its inner +x face; a box straddling its +y face;
    a box inside the inner box (L, the inner box and it overlap: each of their three pairs counts the whole triple
    region); the inner box again ([A, A])"""
    q = size // 4
    inner = ((size - 2 * q, 0, 0), (2 * q, 2 * q, 2 * q))           # its +x face is L's
    spec = [((0, 0, 0), (size, size, size)),
            inner,
            ((-q, size, q), (q + 1, q, q + 2)),                      # straddles L's +y face
            ((size - 2 * q + 1, 1, -1), (q, q - 1, q + 1)),          # inside the inner box
            inner]
    return _group(spec, res)


def corner8(res, pitch=8, offset=(0.0, 0.0, 0.0)):
    """the 2 x 2 x 2 corner of lattice32: 8 parts, face, edge and corner neighbours"""
    return _group([s for s in _lattice(pitch) if max(s[0][:2]) < 0], res, offset)


FAR = (2048.0, -1920.0, 2176.0)   # a dyadic offset: fp32 cell centres stay exact at 2^11 with res >= 2^-7


def far(res, pitch=8):
    """corner8 moved by FAR: the moments about the origin dwarf the centroidal ones"""
    return corner8(res, pitch, FAR)


# ---- curved and rotated groups (1-Lipschitz: the hierarchy's coarse decisions hold) ----------------------------------

def lipschitz_parts(kind):
    box = P.Part.placed(P.Part.box(1.0, 1.5, 1.2), (0.0, 0.0, 0.0), P.quat((1.0, 2.0, 0.5), 0.3))
    cyl = P.Part.placed(P.Part.cylinder(1.1, 1.0), (1.2, 0.4, 0.3), P.quat((0.2, 1.0, 0.1), 0.7))
    if kind == "two":
        return [box, cyl]
    far_box = P.Part.placed(P.Part.box(0.8, 0.8, 0.8), (-1.6, -0.4, 0.2))  # overlaps the box, not the cylinder
    return [box, cyl, far_box]


# name -> (marginal cells, disagreements) of dense_reference at the default margin
CURVED = {"cloud8": (1638, 0), "lipschitz_two": (142, 0), "lipschitz_three": (151, 0)}


def curved_group(name, res=1 / 32, grid=16):
    """(parts, box_a, box_b, res, grid): rotated boxes and cylinders with offsets (programs.primitive_cloud), or the
    groups of lipschitz_parts; the box snapped to the dyadic res"""
    if name == "cloud8":
        parts = P.primitive_cloud(np.random.default_rng(7), 8, (0.0, 0.0, 0.0), 2.5, 1.5)
    else:
        parts = lipschitz_parts(name.split("_")[1])
    box_a, box_b = snap_box(*part_box(parts), res)
    return parts, box_a, box_b, res, grid
