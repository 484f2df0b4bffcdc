"""A small builder of wire programs in the layouts the reference's node compiler emits, and a float64
restatement of the geometry it builds.

Part (an assembly's component; what dsdf3d_mirror_3d's parts look like):
    initial_transformation_to(q, t)  _store r  <2-D profile>  extrusion r [h]  [offset d]
    transformation_from(q^-1)
A union tree puts a value in the running register: `left  _store k  right  union k [r]`, with k the
depth of the node, so that every stored operand ends where the running operand begins (the post-order
layout analyse_parts cuts into parts).  Forest primitives (cfg_synthetic32) are the same parts with a
rectangle or circle profile: the loader fuses them into one micro-op.

The transform maps a world point p to the part's frame as R(q) p + t; the part's distance is then
R(q)^T-rotated back (its gradient) and, for a unit quaternion, keeps its value.
"""
import math

import numpy as np

from codecad_b200.opcodes import OPCODE, REGISTER_COUNT


def ins(name, reg=0, *params):
    return [float(OPCODE[name] * REGISTER_COUNT + reg)] + [float(p) for p in params]


# ---- quaternions (x, y, z, w) ----

def quat(axis, angle):
    """unit quaternion of a rotation by `angle` about `axis`, rounded to float32 (what the wire carries)"""
    a = np.asarray(axis, np.float64)
    a = a / np.linalg.norm(a)
    s = math.sin(angle / 2)
    return tuple(float(np.float32(v)) for v in (a[0] * s, a[1] * s, a[2] * s, math.cos(angle / 2)))


IDENTITY = (0.0, 0.0, 0.0, 1.0)


def quat_inverse(q):
    return (-q[0], -q[1], -q[2], q[3])


def quat_matrix(q):
    """row-major 3x3 of v -> 2 v (v.p) + 2 w (v x p) + (w^2 - v.v) p, in float64 (oracle/sdf_oracle.c)"""
    x, y, z, w = (float(v) for v in q)
    k = w * w - (x * x + y * y + z * z)
    return np.array([[2 * x * x + k, 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 2 * y * y + k, 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 2 * z * z + k]])


# ---- the geometry: parts and union trees ----

class Part:
    """An extruded 2-D profile: ('polygon', vertices) | ('rectangle', hw, hh) | ('circle', r), half height h,
    optional offset d, placed by the transform p -> R(q) p + t."""

    def __init__(self, profile, h, q=IDENTITY, t=(0.0, 0.0, 0.0), offset=None):
        self.profile = profile
        self.h = float(np.float32(h))
        self.q = tuple(float(np.float32(v)) for v in q)
        self.t = tuple(float(np.float32(v)) for v in t)
        self.offset = None if offset is None else float(np.float32(offset))

    @staticmethod
    def polygon(vertices, h, **kw):
        v = np.asarray(vertices, np.float64).astype(np.float32)
        return Part(("polygon", v), h, **kw)

    @staticmethod
    def box(hw, hh, h, **kw):
        return Part(("rectangle", float(np.float32(hw)), float(np.float32(hh))), h, **kw)

    @staticmethod
    def cylinder(r, h, **kw):
        return Part(("circle", float(np.float32(r))), h, **kw)

    @staticmethod
    def placed(profile_part, centre, q=IDENTITY):
        """the same part with its frame's origin at world point `centre` (the translation carries it)"""
        R = quat_matrix(q)
        t = -(R @ np.asarray(centre, np.float64))
        return Part(profile_part.profile, profile_part.h, q=q, t=t, offset=profile_part.offset)

    def words(self, tmp):
        w = ins("initial_transformation_to", 0, *self.q, *self.t) + ins("_store", tmp)
        kind = self.profile[0]
        if kind == "polygon":
            v = self.profile[1]
            w += ins("polygon2d", 0, len(v), *v.ravel())
        elif kind == "rectangle":
            w += ins("rectangle", 0, self.profile[1], self.profile[2])
        else:
            w += ins("circle", 0, self.profile[1])
        w += ins("extrusion", tmp, self.h)
        if self.offset is not None:
            w += ins("offset", 0, self.offset)
        return w + ins("transformation_from", 0, *quat_inverse(self.q))

    def max_coordinate(self):
        """largest |constant coordinate| of the part: translation and vertices"""
        m = max(abs(v) for v in self.t)
        if self.profile[0] == "polygon":
            m = max(m, float(np.abs(self.profile[1]).max()))
        return m


class Union:
    def __init__(self, left, right, r=-1.0):
        self.left, self.right, self.r = left, right, float(np.float32(r))


def balanced(items, r=-1.0):
    """a balanced tree of unions over `items` (parts or subtrees)"""
    items = list(items)
    if len(items) == 1:
        return items[0]
    mid = len(items) // 2
    return Union(balanced(items[:mid], r), balanced(items[mid:], r), r)


def comb(items, r=-1.0):
    """a right-leaning chain a u (b u (c u ...)): its evaluation stack is as deep as it is long"""
    items = list(items)
    node = items[-1]
    for it in reversed(items[:-1]):
        node = Union(it, node, r)
    return node


def _emit(node, depth, out):
    if isinstance(node, Part):
        out += node.words(depth)
        return
    _emit(node.left, depth, out)
    out += ins("_store", depth)
    _emit(node.right, depth + 1, out)
    out += ins("union", depth, node.r)


def program(tree):
    """wire words of the union tree (or a single part)"""
    out = []
    _emit(tree, 0, out)
    out += ins("_return")
    return np.array(out, np.float32)


def polygon_program(vertices):
    """a 2-D scene: one polygon at the origin of the plane"""
    v = np.asarray(vertices, np.float32)
    return np.array(ins("initial_transformation_to", 0, *IDENTITY, 0, 0, 0) + ins("polygon2d", 0, len(v), *v.ravel())
                    + ins("_return"), np.float32)


def leaves(node):
    if isinstance(node, Part):
        return [node]
    return leaves(node.left) + leaves(node.right)


# ---- float64 restatement ----
# Every function returns (distance, gradient, value margin, gradient margin): a margin is the smallest float64
# gap of a decision the evaluation took (the blend's conditions; which operand of a max / min passes its
# gradient on).  The distance of a sharp tree is continuous in every such decision; a rounded union reads the
# gradients and its own conditions, so their gaps enter its value margin.  A point whose value margin is within
# the rounding of float32 may take the other branch there and is not comparable.

def _perp(a, ga, b, gb):
    """perpendicular intersection (oracle: common.cl:15-31) of two distances with their gradients"""
    both = (a > 0) & (b > 0)
    dist = np.where(both, np.hypot(a, b), np.maximum(a, b))
    safe = np.where(both, dist, 1.0)
    g_both = (ga * (a / safe)[:, None] + gb * (b / safe)[:, None])
    g_max = np.where((a > b)[:, None], ga, gb)
    g = np.where(both[:, None], g_both, g_max)
    # (the max's choice matters only for the gradient, and only where both are <= 0)
    gmargin = np.where((a <= 0) & (b <= 0), np.abs(a - b), np.inf)
    return dist, g, gmargin


def _polygon2d(v, x, y):
    """signed distance to a closed polygon (negative inside, even-odd rule) and its gradient"""
    v = np.asarray(v, np.float64)
    best = np.full(len(x), np.inf)
    gx = np.zeros(len(x))
    gy = np.zeros(len(x))
    inside = np.zeros(len(x), bool)
    for k in range(len(v)):
        px, py = v[k - 1]
        cx, cy = v[k]
        dx, dy = cx - px, cy - py
        qx, qy = x - px, y - py
        t = np.clip((qx * dx + qy * dy) / (dx * dx + dy * dy), 0.0, 1.0)
        ex, ey = qx - t * dx, qy - t * dy
        d2 = ex * ex + ey * ey
        better = d2 < best
        best = np.where(better, d2, best)
        gx = np.where(better, ex, gx)
        gy = np.where(better, ey, gy)
        crosses = (py <= y) != (cy <= y)      # crossings of the ray to +x
        with np.errstate(divide="ignore", invalid="ignore"):
            inside ^= crosses & (x < px + (y - py) * dx / dy)
    d = np.sqrt(best)
    s = np.where(inside, -1.0, 1.0)
    safe = np.where(d > 0, d, 1.0)
    g = np.stack([s * gx / safe, s * gy / safe, np.zeros(len(x))], 1)
    return s * d, g, np.full(len(x), np.inf)


def eval_part(part, p):
    p = np.asarray(p, np.float64)
    R = quat_matrix(part.q)
    loc = p @ R.T + np.asarray(part.t)
    x, y, z = loc[:, 0], loc[:, 1], loc[:, 2]
    kind = part.profile[0]
    zero = np.zeros(len(p))
    if kind == "polygon":
        d2, g2, m2 = _polygon2d(part.profile[1], x, y)
    elif kind == "rectangle":
        ax, ay = np.abs(x) - part.profile[1], np.abs(y) - part.profile[2]
        d2, g2, m2 = _perp(ax, np.stack([np.sign(x), zero, zero], 1), ay, np.stack([zero, np.sign(y), zero], 1))
    else:
        ln = np.hypot(x, y)
        safe = np.where(ln > 0, ln, 1.0)
        d2, g2, m2 = ln - part.profile[1], np.stack([x / safe, y / safe, zero], 1), np.full(len(p), np.inf)
    dz = np.abs(z) - part.h
    d, g, m = _perp(dz, np.stack([zero, zero, np.sign(z)], 1), d2, g2)
    if part.offset is not None:
        d = d - part.offset
    return d, g @ R, np.full(len(p), np.inf), np.minimum(m, m2)


def _rounded_union(r, a, b):
    """oracle/sdf_oracle.c rounded_union: sharp (r < 0) is min"""
    (d1, g1, v1, m1), (d2, g2, v2, m2) = a, b
    vmargin = np.minimum(v1, v2)
    gmargin = np.minimum(np.minimum(m1, m2), np.abs(d1 - d2))   # (which operand's gradient survives)
    if r < 0:
        return np.minimum(d1, d2), np.where((d1 < d2)[:, None], g1, g2), vmargin, gmargin
    c = np.sum(g1 * g2, axis=1)
    x1, x2 = r - d1, r - d2
    blend = (c * x1 < x2) & (c * x2 < x1) & ((x1 > 0) | (x2 > 0))
    num = x1 * x1 + x2 * x2 - 2 * c * x1 * x2
    den = 1 - c * c
    with np.errstate(divide="ignore", invalid="ignore"):
        db = r - np.sqrt(np.maximum(num / den, 0.0))
    # the blend is continuous where its conditions switch it on or off, but not in the gradients it reads,
    # and 1 - c^2 divides; its gradient (zero) differs from min's, which matters to a rounded union above
    vmargin = np.minimum(vmargin, np.where(blend, np.where(den < 0.05, 0.0, np.minimum(m1, m2)), np.inf))
    cond = np.minimum(np.abs(c * x1 - x2), np.abs(c * x2 - x1))
    d = np.where(blend, db, np.minimum(d1, d2))
    g = np.where(blend[:, None], 0.0, np.where((d1 < d2)[:, None], g1, g2))
    return d, g, vmargin, np.minimum(gmargin, cond)


def evaluate(tree, p):
    """(distance, gradient, value margin, gradient margin) of the union tree at world points p, in float64"""
    if isinstance(tree, Part):
        return eval_part(tree, p)
    return _rounded_union(tree.r, evaluate(tree.left, p), evaluate(tree.right, p))


def ulp32(x):
    """spacing of float32 at |x|"""
    x = np.abs(np.asarray(x, np.float32))
    return np.spacing(x).astype(np.float64)


# ---- the scenes of the culling tests ----

def tilted_quad(centre, along, across, length, width):
    """a thin quad of the given length and width around `centre` (2-D), long side along `along`"""
    c = np.asarray(centre, np.float64)
    u = np.asarray(along, np.float64) / np.linalg.norm(along)
    v = np.asarray(across, np.float64) / np.linalg.norm(across)
    L, W = length / 2, width / 2
    return np.array([c - L * u - W * v, c + L * u - W * v, c + L * u + W * v, c - L * u + W * v])


TILT = 0.05          # radians off the grid axes: the medial surfaces between quads cross bricks at every offset


def near_tie_assembly(offset, n=3, gap=1.0, carried_by="vertices", length=40.0, width=0.3, h=5.0):
    """`n` parallel thin extruded quads, `gap` apart (centre to centre), tilted TILT off the x and y axes,
    around world point (offset, offset, 0).  carried_by="vertices": the offset is in the polygon's vertices
    and the transforms are identities; "translation": the vertices are near the origin and the translation of
    initial_transformation_to carries the offset.  The medial surfaces between neighbours are near-ties of
    two parts over their whole length."""
    along = (math.cos(TILT), math.sin(TILT))
    across = (-math.sin(TILT), math.cos(TILT))
    parts = []
    for k in range(n):
        s = (k - (n - 1) / 2) * gap
        local = tilted_quad((s * across[0], s * across[1]), along, across, length, width)
        if carried_by == "vertices":
            parts.append(Part.polygon(local + offset, h))
        else:
            parts.append(Part.placed(Part.polygon(local, h), (offset, offset, 0.0)))
    return balanced(parts)


# the extrusion axis off every grid axis, by the quaternion alone (no translation): no column split
OBLIQUE = quat((1.0, 0.7, 0.2), 0.6)


def oblique_assembly(offset=0.0, n=3, gap=1.0):
    """near_tie_assembly's quads rotated off the grid axes by OBLIQUE: its vertices carry the offset in the
    rotated frame, so the scene sits around R(q)^T (offset, offset, 0) in the world"""
    along = (math.cos(TILT), math.sin(TILT))
    across = (-math.sin(TILT), math.cos(TILT))
    parts = []
    for k in range(n):
        s = (k - (n - 1) / 2) * gap
        local = tilted_quad((s * across[0], s * across[1]), along, across, 40.0, 0.3)
        parts.append(Part.polygon(local + offset, 5.0, q=OBLIQUE))
    return balanced(parts)


def oblique_centre(offset):
    return quat_matrix(OBLIQUE).T @ np.array([offset, offset, 0.0])


def primitive_cloud(rng, n, centre, spread, size, rotate=True):
    """`n` boxes and cylinders (alternating) of about `size` at random places within `spread` of `centre`"""
    parts = []
    for k in range(n):
        c = np.asarray(centre, np.float64) + rng.uniform(-spread, spread, 3)
        q = quat(rng.normal(size=3), rng.uniform(0, math.pi)) if rotate else IDENTITY
        off = float(rng.uniform(0, 0.2 * size))
        if k % 2 == 0:
            proto = Part.box(rng.uniform(0.2, 1) * size, rng.uniform(0.2, 1) * size, rng.uniform(0.2, 1) * size, offset=off)
        else:
            proto = Part.cylinder(rng.uniform(0.2, 1) * size, rng.uniform(0.2, 1) * size, offset=off)
        parts.append(Part.placed(proto, c, q))
    return parts


# ---- polygons for the edge-group skip (cc_ops.cuh: groups of 8 edges, every 4th vertex bounds the search) ----

def test_polygons(rng, scales=(1e-2, 1.0, 1e2, 1e4, 1e6)):
    """(name, vertices) of polygons of 9 to 2000 vertices: long diagonal stars, slivers, combs and circles
    far from the origin, at every scale in `scales`"""
    out = []
    for scale in scales:
        for n in (9, 17, 64, 301, 2000):
            ang = np.sort(rng.uniform(0, 2 * np.pi, n))
            r = scale * 10 ** rng.uniform(-2, 0, n)
            out.append(("star%d@%g" % (n, scale), np.stack([r * np.cos(ang), r * np.sin(ang)], 1)))
        for n in (10, 40, 400):
            x = np.sort(rng.uniform(0, scale, n // 2))
            v = np.concatenate([np.stack([x, rng.uniform(0, 1e-3, len(x)) * scale], 1),
                                np.stack([x[::-1], -rng.uniform(0, 1e-3, len(x)) * scale], 1)])
            c, s = math.cos(0.7), math.sin(0.7)     # a sliver along a diagonal
            out.append(("sliver%d@%g" % (n, scale), v @ np.array([[c, s], [-s, c]])))
        for n in (12, 130):
            v = []
            for i in range(n // 2):
                v += [(i * scale / n, 0.0), ((i + 0.5) * scale / n, scale * rng.uniform(1, 30))]
            out.append(("comb%d@%g" % (n, scale), np.array(v + [(scale, -scale)])))
        ang = np.linspace(0, 2 * np.pi, 97, endpoint=False)
        out.append(("far_circle97@%g" % scale, np.stack([np.cos(ang), np.sin(ang)], 1) * scale * 1e-2 + scale))
    return [(name, np.asarray(v, np.float64).astype(np.float32)) for name, v in out]


def _segment_distance(v, k, p):
    a, b = v[k - 1].astype(np.float64), v[k].astype(np.float64)
    d = b - a
    t = np.clip(((p - a) @ d) / (d @ d), 0.0, 1.0)
    return np.linalg.norm(p - a - t[:, None] * d, axis=1)


def near_tie_points(rng, v, m):
    """float32 points aimed at near-ties of the polygon's distance: about m on the bisector of two edges in
    different 8-edge groups, about m between a vertex the bound samples (every 4th) and one it does not,
    with their float32 neighbours"""
    v = np.asarray(v, np.float32)
    n = len(v)
    pts = []
    if n > 8:
        for _ in range(m // 8):
            i = int(rng.integers(0, n))
            j = int(rng.integers(0, n))
            if i // 8 == j // 8:
                j = (i + 8 * int(rng.integers(1, max(2, n // 8)))) % n
                if i // 8 == j // 8:
                    continue
            mi, mj = (v[i - 1].astype(np.float64) + v[i]) / 2, (v[j - 1].astype(np.float64) + v[j]) / 2
            lo, hi = np.zeros(8), np.ones(8)
            jitter = rng.normal(size=(8, 2)) * 0.05 * np.linalg.norm(mj - mi)
            for _ in range(60):     # bisection of d_i - d_j along the segment mi -> mj (+ a sideways jitter)
                s = (lo + hi) / 2
                p = mi + s[:, None] * (mj - mi) + jitter * (s * (1 - s))[:, None]
                f = _segment_distance(v, i, p) - _segment_distance(v, j, p)
                lo, hi = np.where(f < 0, s, lo), np.where(f < 0, hi, s)
            pts.append(p)
    for _ in range(m // 8):
        i = 4 * int(rng.integers(0, (n + 3) // 4))
        j = (i + int(rng.integers(1, 4))) % n if n > 1 else i
        a, b = v[i].astype(np.float64), v[j].astype(np.float64)
        perp = np.array([-(b - a)[1], (b - a)[0]])
        pts.append((a + b) / 2 + rng.normal(size=8)[:, None] * 3 * perp)
    p = np.concatenate(pts).astype(np.float32)
    p = np.concatenate([p, np.nextafter(p, np.float32(np.inf)), np.nextafter(p, np.float32(-np.inf))])
    return np.concatenate([p, np.zeros((len(p), 1), np.float32)], 1)


def near_edge_points(rng, v, m):
    """float32 points along the edges and near the vertices at small normal offsets, and in the box around"""
    v = np.asarray(v, np.float64)
    lo, hi = v.min(0), v.max(0)
    ext = np.maximum(hi - lo, 1e-3 * max(1.0, float(np.abs(v).max())))
    a = lo + ext * (rng.random((m // 2, 2)) * 1.4 - 0.2)
    i = rng.integers(0, len(v), m - m // 2)
    d = v[i] - v[i - 1]
    nrm = np.stack([-d[:, 1], d[:, 0]], 1) / (np.linalg.norm(d, axis=1, keepdims=True) + 1e-30)
    b = v[i - 1] + d * rng.random(m - m // 2)[:, None] + nrm * (10 ** rng.uniform(-7, 0, m - m // 2) * ext.max())[:, None] \
        * rng.choice([-1, 1], m - m // 2)[:, None]
    p = np.concatenate([a, b]).astype(np.float32)
    return np.concatenate([p, np.zeros((len(p), 1), np.float32)], 1)
