// Program loader: codecad wire format -> device microcode (see cc_microcode.h).
//
// Wire format: /root/reference/codecad/nodes/program.py:39-71 (encoding),
// /root/reference/codecad/nodes/node.py:12-56 (opcode table), interpreter semantics
// /root/reference/codecad/nodes/codegen.py:17-63.  Host-only code; compiled with
// -ffp-contract=off because the per-instruction constants below are part of the
// canonical arithmetic (DESIGN.md "cc-arith") and must not be fused.
#include "cc_internal.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

namespace {

enum WireOp {
    W_RETURN = 0, W_STORE, W_LOAD, W_RECTANGLE, W_CIRCLE, W_REGULAR_POLYGON2D, W_POLYGON2D,
    W_SPHERE, W_HALF_SPACE, W_REVOLUTION_TO, W_TWIST_REVOLUTION_TO,
    W_INITIAL_TRANSFORMATION_TO, W_TRANSFORMATION_TO, W_TRANSFORMATION_FROM, W_MIRROR,
    W_SYMMETRICAL_TO, W_OFFSET, W_SHELL, W_REPETITION, W_CIRCULAR_REPETITION_TO,
    W_CIRCULAR_REPETITION_FROM, W_INVOLUTE_GEAR, W_EXTRUSION, W_REVOLUTION_FROM,
    W_TWIST_REVOLUTION_FROM, W_SYMMETRICAL_FROM, W_UNION, W_INTERSECTION, W_SUBTRACTION,
    W_COUNT
};

// parameter words and arity per wire opcode (node.py:18-52); -1 = polygon2d (1 + 2n)
const int kParams[W_COUNT] = {0, 0, 0, 2, 1, 2, -1, 1, 0, 0, 2, 7, 7, 4, 0, 0,
                              1, 1, 3, 1, 1, 2, 1, 0, 3, 0, 1, 1, 1};
const int kArity[W_COUNT] = {1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 1, 1, 1, 1,
                             1, 1, 1, 1, 2, 1, 2, 2, 2, 2, 2, 2, 2};
const unsigned kRegisterCount = 512;  // EVAL_REGISTER_COUNT, nodes/__init__.py:6

const float kPiF = 3.14159274101257324f;
const float kPi2F = 1.57079637050628662f;

struct WireIns {
    int op;
    unsigned reg;
    const float *p;
    int np;
};

struct Interval {
    int store_idx;  // wire instruction index of the _store
    int last_read;  // wire instruction index of the last read, -1 = dead
    bool point_only;  // every read is the point operand of a *_from / extrusion op
    unsigned slot;
    int n_reads;
};

bool is_point_consumer(int op)
{
    return op == W_EXTRUSION || op == W_REVOLUTION_FROM || op == W_TWIST_REVOLUTION_FROM ||
           op == W_SYMMETRICAL_FROM || op == W_CIRCULAR_REPETITION_FROM;
}

// quaternion (x,y,z,w) -> row-major 3x3 of the map  p -> 2 v (v.p) + 2 w (v x p) + (w^2 - v.v) p
// (shapes/common.cl:1-6) evaluated in double, optionally divided by |q|^2
// (shapes/common.cl:100-110), then rounded to fp32.  Same expression tree as the
// oracle's quat_matrix().
void quat_matrix(const float *q, bool divide_by_scale, float *m, float *scale)
{
    double x = q[0], y = q[1], z = q[2], w = q[3];
    double k = w * w - (x * x + y * y + z * z);
    double d[9];
    d[0] = 2.0 * (x * x) + k;
    d[1] = 2.0 * (x * y - w * z);
    d[2] = 2.0 * (x * z + w * y);
    d[3] = 2.0 * (x * y + w * z);
    d[4] = 2.0 * (y * y) + k;
    d[5] = 2.0 * (y * z - w * x);
    d[6] = 2.0 * (x * z - w * y);
    d[7] = 2.0 * (y * z + w * x);
    d[8] = 2.0 * (z * z) + k;
    double s = (x * x + y * y) + (z * z + w * w);
    for (int i = 0; i < 9; ++i) m[i] = (float)(divide_by_scale ? d[i] / s : d[i]);
    if (scale) *scale = (float)s;
}

// bit k set <=> m[k] != 0 (cc-arith: zero coefficients are omitted from the row sums, cc_ops.cuh)
uint32_t matrix_mask(const float *m)
{
    uint32_t k = 0;
    for (int i = 0; i < 9; ++i)
        if (m[i] != 0.0f) k |= 1u << i;
    return k;
}
float mask_word(uint32_t mask)
{
    float f;
    std::memcpy(&f, &mask, 4);
    return f;
}
bool is_identity_from(const float *m, float scale)
{
    for (int i = 0; i < 9; ++i)
        if (m[i] != ((i % 4 == 0) ? 1.0f : 0.0f)) return false;
    return scale == 1.0f;
}

struct Emitter {
    std::vector<uint32_t> code;
    size_t last_header = (size_t)-1;  // index of the most recent instruction header

    float *emit(uint32_t op, uint32_t src, uint32_t len_words)
    {
        last_header = code.size();
        code.resize(code.size() + len_words, 0u);
        code[last_header] = CC_HDR(op, src, CC_SLOT_NONE, len_words);
        return reinterpret_cast<float *>(&code[last_header + 1]);
    }
    bool can_fold_store() const
    {
        if (last_header == (size_t)-1) return false;
        uint32_t h = code[last_header];
        return CC_HDR_DST(h) == CC_SLOT_NONE && CC_HDR_OP(h) != MOP_RETURN;
    }
    void fold_store(uint32_t dst)
    {
        uint32_t h = code[last_header];
        code[last_header] = CC_HDR(CC_HDR_OP(h), CC_HDR_SRC(h), dst, CC_HDR_LEN(h));
    }
};

}  // namespace


// ---- union forests ------------------------------------------------------------------------------
// Recognises microcode that is ONE tree of (rounded) unions over fused primitives — the shape of a
// scene assembled from many boxes and cylinders, BASELINE config 5 — and tabulates what
// cc_forest.cu needs to cull primitives per tile: for every primitive a bounding ball of its
// distance function, for every union the leaf ranges of its two operands, and the evaluation order
// as a stack program (PUSH / PRIM / COMBINE).
//
// Bounds.  A fused primitive computes  w = scale * (solid(M p + o) - d)  with M = s * rotation,
// solid = the signed distance of a box (half extents a, b, h) or cylinder (radius a, half height h).
// With c = -M^-1 o, rho the circumradius and r_in the inradius of the solid:
//     scale * (smin |p - c| - rho - d)  <=  w  <=  scale * (smax |p - c| - r_in - d),   w >= -scale * (r_in + d)
// (circumscribed / inscribed ball, centre value), where smin, smax bound the singular values of M.
// The computed fp32 value differs from the exact one by a few ulps of the magnitudes involved;
// err_a + err_b * max|p| bounds those magnitudes, and the kernel allows 2^-16 of it (>100 ulps).
namespace {

bool invert3(const double *m, double *inv)
{
    const double c0 = m[4] * m[8] - m[5] * m[7], c1 = m[5] * m[6] - m[3] * m[8], c2 = m[3] * m[7] - m[4] * m[6];
    const double det = m[0] * c0 + m[1] * c1 + m[2] * c2;
    if (!(std::fabs(det) > 1e-30) || !std::isfinite(det)) return false;
    inv[0] = c0 / det; inv[1] = (m[2] * m[7] - m[1] * m[8]) / det; inv[2] = (m[1] * m[5] - m[2] * m[4]) / det;
    inv[3] = c1 / det; inv[4] = (m[0] * m[8] - m[2] * m[6]) / det; inv[5] = (m[2] * m[3] - m[0] * m[5]) / det;
    inv[6] = c2 / det; inv[7] = (m[1] * m[6] - m[0] * m[7]) / det; inv[8] = (m[0] * m[4] - m[1] * m[3]) / det;
    return true;
}

bool prim_bounds(const uint32_t *op_words, bool rect, float *out8, double *err_a, double *err_b)
{
    float q[27];
    std::memcpy(q, op_words + 1, sizeof q);
    double M[9], inv[9];
    for (int i = 0; i < 9; ++i) M[i] = q[i];
    for (int i = 0; i < 27; ++i)
        if (i != 26 && !std::isfinite(q[i])) return false;
    if (!invert3(M, inv)) return false;
    double c[3];
    for (int i = 0; i < 3; ++i) c[i] = -(inv[3 * i] * q[9] + inv[3 * i + 1] * q[10] + inv[3 * i + 2] * q[11]);
    // M^T M = s^2 (I + E): singular values of M lie in s * sqrt(1 -+ |E|_F)
    double g[9], s2 = 0;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) g[3 * i + j] = M[i] * M[j] + M[3 + i] * M[3 + j] + M[6 + i] * M[6 + j];
    s2 = (g[0] + g[4] + g[8]) / 3;
    if (!(s2 > 1e-30)) return false;
    double ef = 0;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            const double e = g[3 * i + j] / s2 - (i == j ? 1.0 : 0.0);
            ef += e * e;
        }
    ef = std::sqrt(ef);
    if (!(ef < 0.25)) return false;  // not a similarity transform: no forest
    const double s = std::sqrt(s2), smin = s * std::sqrt(1 - ef) * (1 - 1e-6), smax = s * std::sqrt(1 + ef) * (1 + 1e-6);
    const double a = q[12], b = q[13], h = q[14], d = q[15], scale = q[25];
    if (!(scale > 0) || !(a >= 0) || !(h >= 0) || (rect && !(b >= 0))) return false;
    const double rho = rect ? std::sqrt(a * a + b * b + h * h) : std::sqrt(a * a + h * h);
    const double rin = rect ? std::min(a, std::min(b, h)) : std::min(a, h);
    const double tiny = 1e-6 * (rho + std::fabs(d));
    out8[0] = (float)c[0]; out8[1] = (float)c[1]; out8[2] = (float)c[2];
    // rounding the centre to fp32 moves it by < 2^-23 |c|; covered by the error budget below
    out8[3] = (float)(scale * smin * (1 - 1e-6));                 // g_lo
    out8[4] = (float)(scale * (rho + d + tiny) * (1 + 1e-6) + 1e-30);   // r_lb   (w >= g_lo |p-c| - r_lb)
    out8[5] = (float)(scale * smax * (1 + 1e-6));                 // g_hi
    out8[6] = (float)(scale * (rin + d - tiny) - 1e-6 * std::fabs(scale * (rin + d)));  // r_ub   (w <= g_hi |p-c| - r_ub)
    out8[7] = (float)std::max(0.0, scale * (rin + d + tiny) * (1 + 1e-6));               // depth  (w >= -depth)
    for (int i = 3; i < 8; ++i)
        if (!std::isfinite(out8[i])) return false;
    // magnitudes that enter the computed value: |M| |p| + |o|, the solid's size, the offset
    const double cn = std::sqrt(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]);
    *err_a = std::max(*err_a, scale * (smax * cn + std::fabs((double)q[9]) + std::fabs((double)q[10]) + std::fabs((double)q[11]) + rho + std::fabs(d)));
    *err_b = std::max(*err_b, scale * smax * 3.0);
    return true;
}

void analyse_forest(const std::vector<uint32_t> &code, cc_forest *f)
{
    *f = cc_forest();
    struct Node { uint32_t lo, hi; };
    struct Union { uint32_t lo, mid, hi, pc, kind; float r; };
    std::vector<Node> nodes;
    std::vector<Union> unions;
    std::vector<uint32_t> leaf_pc, leaf_kind;
    std::vector<int> slot_node(CC_SLOT_NONE + 1, -1);
    int L = -1;
    bool L_stored = true;
    // pass 1: the tree
    std::vector<std::pair<uint32_t, int>> order;  // (pc, union index or -1 - leaf) in microcode order
    for (uint32_t pc = 0;;) {
        if (pc >= code.size()) return;
        const uint32_t hd = code[pc], op = CC_HDR_OP(hd), src = CC_HDR_SRC(hd), dst = CC_HDR_DST(hd);
        if (op == MOP_RETURN) break;
        int made = -1;
        if (op == MOP_PRIM_CIRCLE || op == MOP_PRIM_RECT || op == MOP_PRIM_CIRCLE_M || op == MOP_PRIM_RECT_M) {
            if (L >= 0 && !L_stored) return;  // a value would be lost
            const uint32_t k = (uint32_t)leaf_pc.size();
            leaf_pc.push_back(pc);
            leaf_kind.push_back(op);
            nodes.push_back(Node{k, k + 1});
            made = (int)nodes.size() - 1;
            order.emplace_back(pc, -1 - (int)k);
        } else if (op == MOP_UNION || op == MOP_UNION_R) {
            if (src == CC_SLOT_NONE || slot_node[src] < 0 || L < 0 || L_stored) return;
            const Node A = nodes[(size_t)slot_node[src]], B = nodes[(size_t)L];
            slot_node[src] = -1;
            if (A.hi != B.lo) return;  // operands must be adjacent subtrees, stored one first
            float r = 0.0f;
            std::memcpy(&r, &code[pc + 1], 4);
            if (op == MOP_UNION_R && !(r >= 0.0f && std::isfinite(r))) return;
            unions.push_back(Union{A.lo, A.hi, B.hi, pc, op, op == MOP_UNION_R ? r : 0.0f});
            nodes.push_back(Node{A.lo, B.hi});
            made = (int)nodes.size() - 1;
            order.emplace_back(pc, (int)unions.size() - 1);
        } else {
            return;  // any other micro-op: not a pure union forest
        }
        L = made;
        L_stored = false;
        if (dst != CC_SLOT_NONE) {
            if (slot_node[dst] >= 0) return;  // overwrites a value nobody consumed
            slot_node[dst] = made;
            L_stored = true;
        }
        pc += CC_HDR_LEN(hd);
    }
    const uint32_t n = (uint32_t)leaf_pc.size();
    if (n < CC_FOREST_MIN_LEAVES || n > 60000u || L < 0 || L_stored) return;
    if (nodes[(size_t)L].lo != 0 || nodes[(size_t)L].hi != n) return;
    for (int v : slot_node)
        if (v >= 0) return;
    // pass 2: events in evaluation order; a union's PUSH sits just before the first leaf of its second operand
    std::vector<int> mid_of(n, -1);
    for (size_t u = 0; u < unions.size(); ++u) mid_of[unions[u].mid] = (int)u;
    auto push_event = [&](uint32_t w0, uint32_t w1, uint32_t w2, float r) {
        uint32_t rb;
        std::memcpy(&rb, &r, 4);
        f->events.insert(f->events.end(), {w0, w1, w2, rb});
    };
    uint32_t depth = 0, max_depth = 0;
    for (auto &o : order) {
        if (o.second < 0) {
            const uint32_t k = (uint32_t)(-1 - o.second);
            if (mid_of[k] >= 0) {
                const Union &u = unions[(size_t)mid_of[k]];
                push_event(CC_FOREST_EVENT(CC_FOREST_PUSH, u.kind, u.pc), u.lo | (u.mid << 16), u.hi, u.r);
                max_depth = std::max(max_depth, ++depth);
            }
            push_event(CC_FOREST_EVENT(CC_FOREST_PRIM, leaf_kind[k], leaf_pc[k]), k, 0, 0.0f);
        } else {
            const Union &u = unions[(size_t)o.second];
            push_event(CC_FOREST_EVENT(CC_FOREST_COMBINE, u.kind, u.pc), u.lo | (u.mid << 16), u.hi, u.r);
            --depth;
        }
    }
    if (code.size() >= (1u << 24)) return;
    f->bounds.resize((size_t)n * 8);
    double ea = 0, eb = 0;
    for (uint32_t k = 0; k < n; ++k) {
        const bool rect = leaf_kind[k] == MOP_PRIM_RECT || leaf_kind[k] == MOP_PRIM_RECT_M;
        if (!prim_bounds(&code[leaf_pc[k]], rect, &f->bounds[(size_t)k * 8], &ea, &eb)) {
            *f = cc_forest();
            return;
        }
    }
    float rmax = 0.0f;
    for (const Union &u : unions) rmax = std::max(rmax, u.r);
    f->n_leaves = n;
    f->n_unions = (uint32_t)unions.size();
    f->n_events = (uint32_t)(f->events.size() / 4);
    f->max_depth = std::max(1u, max_depth);
    f->rmax = rmax;
    f->err_a = (float)(ea * 1.01 + rmax);
    f->err_b = (float)(eb * 1.01);
    f->enabled = true;
}

}  // namespace


// ---- parts of an assembly --------------------------------------------------------------------------
// Finds the shape  post-ops( union( union(part, part), part ... ) )  with sharp unions: the result at a
// point is the part with the smallest distance, passed through whole.  A part that is provably farther
// than some other part over a whole brick is never selected there.  The proof needs a Lipschitz bound
// of every part's value, derived op by op:
//   coordinates: transformation M -> largest singular value of M; mirror / |x| / revolution keep it;
//   distances of exact primitives (circle, sphere, rectangle, polygon, half-space): that of the coordinates;
//   extrusion: sqrt(a^2 + b^2) or max(a, b) of a distance in x, y and a slab in z — orthogonal
//   arguments of the same coordinates, so the maximum of the two constants;
//   involute gear: sqrt(1 + g^2) with g the largest angle that scales the radius (gears.cl:24);
//   offset, shell, sharp union / intersection / subtraction: maximum of the operands'; inverse
//   transformation: times its scale.  Anything else (twists, repetitions, regular polygons, rounded
//   combinators) yields no bound and the part is always evaluated.
namespace {

bool sigma_max(const float *m, double *out)
{
    double g[9], s2;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) g[3 * i + j] = (double)m[i] * m[j] + (double)m[3 + i] * m[3 + j] + (double)m[6 + i] * m[6 + j];
    s2 = (g[0] + g[4] + g[8]) / 3;
    if (!(s2 > 1e-30) || !std::isfinite(s2)) return false;
    double ef = 0;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            const double e = g[3 * i + j] / s2 - (i == j ? 1.0 : 0.0);
            ef += e * e;
        }
    *out = std::sqrt(s2) * std::sqrt(1 + std::sqrt(ef)) * (1 + 1e-6);
    return std::isfinite(*out);
}

// ---- columns: which micro-ops can see the grid coordinate along one axis (cc_internal.h cc_columns) ----
// Forward data flow over the straight-line microcode with one bit per component (x, y, z, w) of the
// running value and of every slot: "may differ between two cells of one column along the axis".  The rules below
// follow the op library (cc_ops.cuh) and cc-arith's matrix form, where a zero coefficient is not a
// multiplication by zero but an omitted term — the remaining terms never see that operand:
//   transforms          row r depends on what its non-zero coefficients read
//   2-D primitives      read x, y; write (nx, ny, 0, d)
//   mirror/offset/nop   component-wise; repetition too; circular repetition turns (x, y), passes z
//   everything else     any dependent input makes every output component dependent
static void analyse_columns_along(const std::vector<uint32_t> &code, int axis, cc_columns *out)
{
    *out = cc_columns();
    out->axis = axis;
    enum { X = 1, Y = 2, Z = 4, W = 8, ALL = 15 };
    struct Op { uint32_t pc, op; int in_l, in_s; uint8_t dep; uint32_t cost; };
    std::vector<Op> ops;
    std::vector<uint8_t> split_prim;
    std::vector<int> slot_prod(CC_SLOT_NONE + 1, -1);
    int L = -1, root = -1;
    auto fl = [&](uint32_t pc, int k) { float f; std::memcpy(&f, &code[pc + 1 + (uint32_t)k], 4); return f; };
    for (uint32_t pc = 0;;) {
        if (pc >= code.size()) return;
        const uint32_t hd = code[pc], op = CC_HDR_OP(hd), src = CC_HDR_SRC(hd), dst = CC_HDR_DST(hd);
        if (op == MOP_RETURN) { root = L; break; }
        Op o{pc, op, -1, -1, 0, 4};
        const bool from_point = op == MOP_T_INIT || op == MOP_T_INIT_M || op == MOP_PRIM_CIRCLE || op == MOP_PRIM_RECT ||
                                op == MOP_PRIM_CIRCLE_M || op == MOP_PRIM_RECT_M;
        if (!from_point && op != MOP_LOAD) {
            if (L < 0) return;
            o.in_l = L;
        }
        if (src != CC_SLOT_NONE) {
            if (slot_prod[src] < 0) return;
            o.in_s = slot_prod[src];
        }
        const uint8_t dl = o.in_l >= 0 ? ops[(size_t)o.in_l].dep : 0, ds = o.in_s >= 0 ? ops[(size_t)o.in_s].dep : 0;
        auto rows = [&](uint8_t in, bool carries_w) {  // a 3 x 3 matrix at words 1..9 applied to (x, y, z)
            uint8_t d = 0;
            for (int r = 0; r < 3; ++r)
                for (int k = 0; k < 3; ++k)
                    if (fl(pc, 3 * r + k) != 0.0f && (in & (1 << k))) d |= (uint8_t)(1 << r);
            if (carries_w && (in & W)) d |= W;
            return d;
        };
        switch (op) {
        case MOP_T_INIT: case MOP_T_INIT_M: {  // the grid point: only its coordinate along the axis varies
            // A coefficient of z that is rounding residue (a half turn written as a quaternion leaves
            // cos(pi/2) = 6e-17 behind) is not omitted by cc-arith, so the row does see z — in the last bits of
            // a value near zero, if at all.  Such rows count as invariant here and are CHECKED per column at run
            // time: each row is a monotone function of z (a chain of correctly rounded FMAs), so equal bits at
            // both ends of the column mean equal bits at every cell between them (cc_jit.cpp `invariant`).
            uint8_t d = 0;
            for (int r = 0; r < 3; ++r) {
                const float big = std::max(std::fabs(fl(pc, 3 * r + (axis + 1) % 3)), std::fabs(fl(pc, 3 * r + (axis + 2) % 3)));
                const float mz = std::fabs(fl(pc, 3 * r + axis));
                if (mz != 0.0f && !(mz <= big * 9.313225746154785e-10f)) d |= (uint8_t)(1 << r);  // 2^-30
                else if (mz != 0.0f) out->checked_rows.push_back((uint32_t)ops.size() * 4u + (uint32_t)r);
            }
            o.dep = d;
            o.cost = 18;
            break;
        }
        case MOP_T_TO: case MOP_T_TO_M: o.dep = rows(dl, false); o.cost = 18; break;
        case MOP_T_FROM: case MOP_T_FROM_M: o.dep = rows(dl, true); o.cost = 18; break;
        case MOP_MIRROR: case MOP_SYM_TO: case MOP_OFFSET: case MOP_NOP: o.dep = dl; o.cost = 1; break;
        case MOP_LOAD: o.dep = ds; o.cost = 0; break;
        case MOP_CIRCLE: o.dep = (dl & (X | Y)) ? (X | Y | W) : 0; o.cost = 10; break;
        case MOP_RECTANGLE: o.dep = (dl & (X | Y)) ? (X | Y | W) : 0; o.cost = 17; break;
        case MOP_REGPOLY: o.dep = (dl & (X | Y)) ? (X | Y | W) : 0; o.cost = 120; break;
        case MOP_GEAR: o.dep = (dl & (X | Y)) ? (X | Y | W) : 0; o.cost = 200; break;
        case MOP_POLYGON: o.dep = (dl & (X | Y)) ? (X | Y | W) : 0; o.cost = 12u * (uint32_t)fl(pc, 0) + 30u; break;
        case MOP_SYM_FROM: o.dep = (uint8_t)(dl | ((ds & X) ? X : 0)); o.cost = 2; break;
        // unsafe.cl:1-23: repetition works component by component; the circular one turns (x, y) and passes z (and w) on
        case MOP_REPETITION: o.dep = (uint8_t)(dl & (X | Y | Z)); o.cost = 30; break;
        case MOP_CREP_TO: o.dep = (uint8_t)(((dl & (X | Y)) ? (X | Y) : 0) | (dl & Z)); o.cost = 60; break;
        case MOP_CREP_FROM: o.dep = (uint8_t)((((dl | ds) & (X | Y)) ? (X | Y) : 0) | (dl & (Z | W))); o.cost = 60; break;
        case MOP_PRIM_CIRCLE: case MOP_PRIM_RECT: case MOP_PRIM_CIRCLE_M: case MOP_PRIM_RECT_M: {
            // fused transform -> circle | rectangle -> extrusion -> offset -> inverse transform: as a whole it sees every axis; its
            // 2-D half does not when rows x and y of the matrix have no (or only a residue, checked per column) coefficient
            // along the axis — the extrusion is then along the columns
            o.dep = ALL;
            o.cost = 100;
            bool split = true;
            std::vector<uint32_t> residue;
            for (int r = 0; r < 2; ++r) {
                const float big = std::max(std::fabs(fl(pc, 3 * r + (axis + 1) % 3)), std::fabs(fl(pc, 3 * r + (axis + 2) % 3)));
                const float mz = std::fabs(fl(pc, 3 * r + axis));
                if (mz != 0.0f && !(mz <= big * 9.313225746154785e-10f)) split = false;
                else if (mz != 0.0f) residue.push_back((uint32_t)ops.size() * 4u + (uint32_t)r);
            }
            if (split) {
                split_prim.resize(ops.size() + 1, 0);
                split_prim[ops.size()] = 1;
                out->checked_rows.insert(out->checked_rows.end(), residue.begin(), residue.end());
            }
            break;
        }
        default:
            o.dep = (dl | ds) ? ALL : 0;
            o.cost = (op == MOP_UNION || op == MOP_ISECT || op == MOP_SUB) ? 5 : 30;
            break;
        }
        ops.push_back(o);
        L = (int)ops.size() - 1;
        if (dst != CC_SLOT_NONE) slot_prod[dst] = L;
        pc += CC_HDR_LEN(hd);
    }
    const int n = (int)ops.size();
    if (root < 0 || n < 3) return;
    // what the loop needs (dependent ops, from the result backwards) and what must run ahead of it
    // (invariant ops that feed the loop, and whatever feeds those — possibly dependent ops again, whose
    // invariant components are what is read)
    std::vector<char> in_loop((size_t)n, 0), ahead((size_t)n, 0);
    std::vector<int> todo;
    auto want = [&](int v) {
        if (v < 0) return;
        std::vector<char> &set = ops[(size_t)v].dep ? in_loop : ahead;
        if (!set[(size_t)v]) { set[(size_t)v] = 1; todo.push_back(v); }
    };
    want(root);
    while (!todo.empty()) {
        const int v = todo.back();
        todo.pop_back();
        if (ops[(size_t)v].dep && in_loop[(size_t)v]) { want(ops[(size_t)v].in_l); want(ops[(size_t)v].in_s); }
    }
    for (int v = n - 1; v >= 0; --v) {  // inputs precede their readers: one backward sweep closes `ahead`
        if (!ahead[(size_t)v]) continue;
        for (int p : {ops[(size_t)v].in_l, ops[(size_t)v].in_s})
            if (p >= 0) ahead[(size_t)p] = 1;
    }
    out->phase.assign((size_t)n, 0);
    out->op_cost.resize((size_t)n);
    for (int v = 0; v < n; ++v) out->op_cost[(size_t)v] = ops[(size_t)v].cost;
    out->restore_from.assign((size_t)n, -1);
    out->save_l.assign((size_t)n, 0);
    uint64_t total = 0, hoisted = 0, repeated = 0;
    split_prim.resize((size_t)n, 0);
    out->split_prim.assign((size_t)n, 0);
    for (int v = 0; v < n; ++v) {
        out->phase[(size_t)v] = (uint8_t)((ahead[(size_t)v] ? 1 : 0) | (in_loop[(size_t)v] ? 2 : 0));
        if (split_prim[(size_t)v] && in_loop[(size_t)v] && !ahead[(size_t)v]) {  // its 2-D half joins the column pass
            // (not counted towards the invariant share: a program of boxes and cylinders alone gains too little from
            // moving half a primitive to pay for the column pass; with gears or polygons to hoist it comes for free)
            out->split_prim[(size_t)v] = 1;
            out->phase[(size_t)v] |= 1;
        }
        if (ahead[(size_t)v] || in_loop[(size_t)v]) total += ops[(size_t)v].cost;
        if (ahead[(size_t)v] && !in_loop[(size_t)v]) hoisted += ops[(size_t)v].cost;
        if (ahead[(size_t)v] && in_loop[(size_t)v]) repeated += ops[(size_t)v].cost;
        const int p = ops[(size_t)v].in_l;
        if (in_loop[(size_t)v] && p >= 0 && !in_loop[(size_t)p]) {
            out->restore_from[(size_t)v] = p;
            out->save_l[(size_t)p] = 1;
        }
    }
    if (!in_loop[(size_t)root]) {
        out->root_restore = root;
        out->save_l[(size_t)root] = 1;
    }
    if (getenv("CODECAD_B200_COLUMNS_DEBUG"))
        for (int v = 0; v < n; ++v)
            std::fprintf(stderr, "op %3d  mop %2u  in_l %3d in_s %3d  dep %x  phase %u  save %u restore %d cost %u\n", v, ops[(size_t)v].op,
                         ops[(size_t)v].in_l, ops[(size_t)v].in_s, ops[(size_t)v].dep, out->phase[(size_t)v], out->save_l[(size_t)v],
                         out->restore_from[(size_t)v], ops[(size_t)v].cost);
    (void)repeated;
    out->invariant_share = total ? (float)((double)hoisted / (double)total) : 0.0f;
    out->enabled = out->invariant_share >= 0.25f;
}

// the grid axis along which most of the program is invariant (z, the fastest index of the output, on ties)
void analyse_columns(const std::vector<uint32_t> &code, cc_columns *out)
{
    analyse_columns_along(code, 2, out);
    for (int axis = 1; axis >= 0; --axis) {
        cc_columns c;
        analyse_columns_along(code, axis, &c);
        if (c.invariant_share > out->invariant_share + 0.05f) *out = c;
    }
}

void analyse_parts(const std::vector<uint32_t> &code, cc_parts *out)
{
    *out = cc_parts();
    struct Op { uint32_t pc, op, src, dst; int in_l, in_s; };  // producers of the two inputs (op index), -1 = none
    std::vector<Op> ops;
    std::vector<int> slot_prod(CC_SLOT_NONE + 1, -1);
    int L = -1, root = -1;
    for (uint32_t pc = 0;;) {
        if (pc >= code.size()) return;
        const uint32_t hd = code[pc], op = CC_HDR_OP(hd), src = CC_HDR_SRC(hd), dst = CC_HDR_DST(hd);
        if (op == MOP_RETURN) { root = L; break; }
        Op o{pc, op, src, dst, -1, -1};
        const bool from_point = op == MOP_T_INIT || op == MOP_T_INIT_M || op == MOP_PRIM_CIRCLE || op == MOP_PRIM_RECT ||
                                op == MOP_PRIM_CIRCLE_M || op == MOP_PRIM_RECT_M;
        if (!from_point && op != MOP_LOAD) {
            if (L < 0) return;
            o.in_l = L;
        }
        if (src != CC_SLOT_NONE) {
            if (slot_prod[src] < 0) return;
            o.in_s = slot_prod[src];
        }
        ops.push_back(o);
        L = (int)ops.size() - 1;  // (NOP and LOAD are nodes too: they move a value)
        if (dst != CC_SLOT_NONE) slot_prod[dst] = L;
        pc += CC_HDR_LEN(hd);
    }
    const int n = (int)ops.size();
    if (root < 0 || n < 8) return;
    std::vector<int> uses((size_t)n, 0);
    for (const Op &o : ops) {
        if (o.in_l >= 0) ++uses[(size_t)o.in_l];
        if (o.in_s >= 0) ++uses[(size_t)o.in_s];
    }
    auto fl = [&](uint32_t pc, int k) { float f; std::memcpy(&f, &code[pc + 1 + (uint32_t)k], 4); return f; };
    // the chain above the union tree: ops that map the winner's distance monotonically
    int top = root;
    std::vector<char> in_chain((size_t)n, 0);
    for (;;) {
        const Op &o = ops[(size_t)top];
        const bool t_from = (o.op == MOP_T_FROM || o.op == MOP_T_FROM_M) && fl(o.pc, 9) > 0.0f;
        if (!(t_from || o.op == MOP_OFFSET || o.op == MOP_NOP) || o.in_l < 0 || uses[(size_t)o.in_l] != 1) break;
        in_chain[(size_t)top] = 1;
        top = o.in_l;
    }
    if (ops[(size_t)top].op != MOP_UNION) return;
    // flatten the tree of sharp unions below `top`
    std::vector<int> part_root;
    std::vector<char> is_tree_union((size_t)n, 0);
    struct Item { int node; };
    std::vector<int> stack{top};
    while (!stack.empty()) {
        const int u = stack.back();
        stack.pop_back();
        const Op &o = ops[(size_t)u];
        if (o.op == MOP_UNION && (u == top || uses[(size_t)u] == 1) && o.in_l >= 0 && o.in_s >= 0) {
            is_tree_union[(size_t)u] = 1;
            stack.push_back(o.in_l);
            stack.push_back(o.in_s);
        } else {
            if (uses[(size_t)u] != 1) return;  // a value shared between parts
            part_root.push_back(u);
        }
    }
    std::sort(part_root.begin(), part_root.end());
    const int P = (int)part_root.size();
    if (P < 2 || P > 32) return;
    // every part = the closure of its root, which must be a contiguous run of micro-ops
    std::vector<int> part_of((size_t)n, -1);
    for (int k = 0; k < P; ++k) {
        std::vector<int> todo{part_root[(size_t)k]};
        int lo = part_root[(size_t)k];
        while (!todo.empty()) {
            const int v = todo.back();
            todo.pop_back();
            if (part_of[(size_t)v] == k) continue;
            if (part_of[(size_t)v] >= 0 || is_tree_union[(size_t)v] || in_chain[(size_t)v]) return;  // shared with another part
            part_of[(size_t)v] = k;
            lo = std::min(lo, v);
            if (ops[(size_t)v].in_l >= 0) todo.push_back(ops[(size_t)v].in_l);
            if (ops[(size_t)v].in_s >= 0) todo.push_back(ops[(size_t)v].in_s);
        }
        for (int v = lo; v <= part_root[(size_t)k]; ++v)
            if (part_of[(size_t)v] != k) return;  // foreign op inside the run
    }
    for (int v = 0; v < n; ++v) {
        if (part_of[(size_t)v] < 0 && !is_tree_union[(size_t)v] && !in_chain[(size_t)v]) return;  // dead or stray code
        // nothing but the part itself (and, for its root, the tree) may read a part's values
        const Op &o = ops[(size_t)v];
        for (int in : {o.in_l, o.in_s})
            if (in >= 0 && part_of[(size_t)in] >= 0 && part_of[(size_t)in] != part_of[(size_t)v] &&
                !(is_tree_union[(size_t)v] && in == part_root[(size_t)part_of[(size_t)in]]))
                return;
    }
    // post-order layout: a union's stored operand ends where its running operand begins, and the union
    // follows its running operand at once — then "skip a part's run" leaves the survivor in L
    std::vector<int> first((size_t)n, 0);
    std::vector<uint32_t> below((size_t)n, 0u);
    for (int v = 0; v < n; ++v) {
        if (part_of[(size_t)v] >= 0 && part_root[(size_t)part_of[(size_t)v]] == v) {
            int lo = v;
            while (lo > 0 && part_of[(size_t)lo - 1] == part_of[(size_t)v]) --lo;
            first[(size_t)v] = lo;
            below[(size_t)v] = 1u << part_of[(size_t)v];
        } else if (is_tree_union[(size_t)v]) {
            const int a = ops[(size_t)v].in_s, b = ops[(size_t)v].in_l;  // stored operand, running operand
            if (b != v - 1 || first[(size_t)b] != a + 1) return;
            first[(size_t)v] = first[(size_t)a];
            below[(size_t)v] = below[(size_t)a] | below[(size_t)b];
        }
    }
    if (first[(size_t)top] != 0) return;
    // Lipschitz bounds, op by op
    const double INF = std::numeric_limits<double>::infinity();
    std::vector<double> lip((size_t)n, INF);     // of the node's distance (or of its coordinates)
    std::vector<int> coords_of((size_t)n, -1);   // the coordinate node a 2-D distance was computed from
    double mag_a = 0, mag_b = 0;
    for (int v = 0; v < n; ++v) {
        if (part_of[(size_t)v] < 0) continue;
        const Op &o = ops[(size_t)v];
        const double li = o.in_l >= 0 ? lip[(size_t)o.in_l] : INF, ls = o.in_s >= 0 ? lip[(size_t)o.in_s] : INF;
        double r = INF;
        switch (o.op) {
        case MOP_T_INIT: case MOP_T_INIT_M: case MOP_T_TO: case MOP_T_TO_M: {
            float m[9];
            for (int i = 0; i < 9; ++i) m[i] = fl(o.pc, i);
            double sm;
            if (!sigma_max(m, &sm)) break;
            const bool init = o.op == MOP_T_INIT || o.op == MOP_T_INIT_M;
            r = init ? sm : sm * li;
            mag_a = std::max(mag_a, (double)std::fabs(fl(o.pc, 9)) + std::fabs(fl(o.pc, 10)) + std::fabs(fl(o.pc, 11)));
            if (std::isfinite(r)) mag_b = std::max(mag_b, 3.0 * r);  // (no bound: the part is never culled, its rounding is moot)
            break;
        }
        case MOP_PRIM_CIRCLE: case MOP_PRIM_RECT: case MOP_PRIM_CIRCLE_M: case MOP_PRIM_RECT_M: {
            float m[9];
            for (int i = 0; i < 9; ++i) m[i] = fl(o.pc, i);
            double sm;
            const double scale = fl(o.pc, 25);
            if (!sigma_max(m, &sm) || !(scale > 0)) break;
            r = sm * scale;
            mag_a = std::max(mag_a, scale * ((double)std::fabs(fl(o.pc, 9)) + std::fabs(fl(o.pc, 10)) + std::fabs(fl(o.pc, 11)) +
                                             std::fabs(fl(o.pc, 12)) + std::fabs(fl(o.pc, 13)) + std::fabs(fl(o.pc, 14)) + std::fabs(fl(o.pc, 15))));
            if (std::isfinite(r)) mag_b = std::max(mag_b, 3.0 * r);
            break;
        }
        case MOP_LOAD: r = ls; coords_of[(size_t)v] = o.in_s >= 0 ? coords_of[(size_t)o.in_s] : -1; break;
        case MOP_NOP: r = li; coords_of[(size_t)v] = o.in_l >= 0 ? coords_of[(size_t)o.in_l] : -1; break;
        case MOP_MIRROR: case MOP_SYM_TO: case MOP_REV_TO: r = li; break;
        case MOP_CIRCLE: case MOP_RECTANGLE:  // r (and a zero word) / half width, half height
            r = li;
            coords_of[(size_t)v] = o.in_l;
            mag_a = std::max(mag_a, (double)std::fabs(fl(o.pc, 0)) + std::fabs(fl(o.pc, 1)));
            break;
        case MOP_POLYGON: {
            // the words are the vertex count and the edge table's offset: the magnitudes are the vertices'
            // (every vertex is the start point of one edge)
            const uint32_t nv = (uint32_t)fl(o.pc, 0), off = code[o.pc + 2];
            for (uint32_t k = 0; k < nv; ++k) {
                float px, py;
                std::memcpy(&px, &code[off + CC_POLY_EDGE_WORDS * k], 4);
                std::memcpy(&py, &code[off + CC_POLY_EDGE_WORDS * k + 1], 4);
                mag_a = std::max(mag_a, (double)std::fabs(px) + std::fabs(py));
            }
            r = li;
            coords_of[(size_t)v] = o.in_l;
            break;
        }
        case MOP_SPHERE: case MOP_HALF_SPACE: r = li; mag_a = std::max(mag_a, (double)std::fabs(fl(o.pc, 0))); break;
        case MOP_GEAR: {
            const double tooth = fl(o.pc, 1), half = fl(o.pc, 2);
            const double gmax = std::max(std::fabs(half), std::fabs(tooth - half));
            r = li * std::sqrt(1 + gmax * gmax) * (1 + 1e-5);
            coords_of[(size_t)v] = o.in_l;
            mag_a = std::max(mag_a, 4.0 * M_PI);  // angles up to 4 pi enter the arithmetic
            break;
        }
        case MOP_OFFSET: case MOP_SHELL:
            r = li;
            coords_of[(size_t)v] = o.in_l >= 0 ? coords_of[(size_t)o.in_l] : -1;
            mag_a = std::max(mag_a, (double)std::fabs(fl(o.pc, 0)));
            break;
        case MOP_EXTRUSION:
            // distance in (x, y) of the coordinates in the slot, slab in their z: orthogonal arguments
            r = (o.in_l >= 0 && coords_of[(size_t)o.in_l] == o.in_s) ? std::max(li, ls) : std::sqrt(li * li + ls * ls);
            mag_a = std::max(mag_a, (double)std::fabs(fl(o.pc, 0)));
            break;
        case MOP_REV_FROM: case MOP_SYM_FROM: r = li; break;
        case MOP_T_FROM: case MOP_T_FROM_M: {
            const double scale = fl(o.pc, 9);
            r = scale > 0 ? li * scale * (1 + 1e-6) : INF;
            break;
        }
        case MOP_UNION: case MOP_ISECT: case MOP_SUB: r = std::max(li, ls); break;
        default: break;  // no bound: the part is never culled
        }
        lip[(size_t)v] = r;
    }
    out->n_parts = (uint32_t)P;
    out->part_of_op = part_of;
    out->union_a.assign((size_t)n, 0u);
    out->union_b.assign((size_t)n, 0u);
    for (int v = 0; v < n; ++v)
        if (is_tree_union[(size_t)v]) {
            out->union_a[(size_t)v] = below[(size_t)ops[(size_t)v].in_s];
            out->union_b[(size_t)v] = below[(size_t)ops[(size_t)v].in_l];
        }
    out->lipschitz.resize((size_t)P);
    int bounded = 0;
    for (int k = 0; k < P; ++k) {
        const double l = lip[(size_t)part_root[(size_t)k]];
        out->lipschitz[(size_t)k] = std::isfinite(l) ? (float)(l * (1 + 1e-5)) : std::numeric_limits<float>::infinity();
        bounded += std::isfinite(l) ? 1 : 0;
    }
    if (!std::isfinite(mag_a) || !std::isfinite(mag_b)) return;
    {  // the table the interpreter tier walks (cc_internal.h)
        std::vector<uint32_t> &t = out->table;
        t.assign(2, 0u);
        t[0] = (uint32_t)P;
        for (int k = 0; k < P; ++k) {
            uint32_t bits;
            std::memcpy(&bits, &out->lipschitz[(size_t)k], 4);
            t.push_back(bits);
        }
        auto end_pc = [&](int v) { return ops[(size_t)v].pc + CC_HDR_LEN(code[ops[(size_t)v].pc]); };
        for (int k = 0; k < P; ++k) {
            int lo = part_root[(size_t)k];
            while (lo > 0 && part_of[(size_t)lo - 1] == k) --lo;
            t.push_back(ops[(size_t)lo].pc);
            t.push_back(end_pc(part_root[(size_t)k]));
        }
        uint32_t n_seg = 0;
        for (int v = 0; v < n;) {
            if (is_tree_union[(size_t)v]) {
                t.insert(t.end(), {CC_SEG_UNION, ops[(size_t)v].pc, out->union_a[(size_t)v], out->union_b[(size_t)v]});
                ++v;
            } else {
                const int k = part_of[(size_t)v];
                int w = v;
                while (w + 1 < n && part_of[(size_t)w + 1] == k && !is_tree_union[(size_t)w + 1]) ++w;
                t.insert(t.end(), {k >= 0 ? CC_SEG_PART : CC_SEG_ALWAYS, ops[(size_t)v].pc, end_pc(w), k >= 0 ? (1u << k) : 0u});
                v = w + 1;
            }
            ++n_seg;
        }
        t[1] = n_seg;
    }
    out->magnitude_a = (float)(mag_a + 1.0);
    out->magnitude_b = (float)std::max(mag_b, 3.0);
    out->enabled = bounded >= 1;  // (at least one part can ever be dropped)
}

}  // namespace

int cc_decode_program(const float *words, uint32_t n_words, cc_decoded *out, std::string *err)
{
    // ---- 1. parse + validate ------------------------------------------------------------
    std::vector<WireIns> ins;
    uint32_t pc = 0;
    unsigned max_reg = 0;
    bool any_reg = false;
    for (;;) {
        if (pc >= n_words) {
            *err = "program ends without _return";
            return CC_ERR_INVALID_PROGRAM;
        }
        float wf = words[pc];
        if (!(wf >= 0.0f) || wf >= (float)(W_COUNT * kRegisterCount) || wf != std::floor(wf)) {
            *err = "invalid instruction word at " + std::to_string(pc);
            return CC_ERR_INVALID_PROGRAM;
        }
        unsigned instruction = (unsigned)wf;
        int op = (int)(instruction / kRegisterCount);
        unsigned reg = instruction % kRegisterCount;
        int np = kParams[op];
        if (np < 0) {
            if (pc + 1 >= n_words || !(words[pc + 1] >= 1.0f) || words[pc + 1] > 65536.0f ||
                words[pc + 1] != std::floor(words[pc + 1])) {
                *err = "invalid polygon2d vertex count at " + std::to_string(pc);
                return CC_ERR_INVALID_PROGRAM;
            }
            np = 1 + 2 * (int)words[pc + 1];
        }
        if (pc + 1 + (uint32_t)np > n_words) {
            *err = "truncated parameters at " + std::to_string(pc);
            return CC_ERR_INVALID_PROGRAM;
        }
        ins.push_back(WireIns{op, reg, words + pc + 1, np});
        if (op == W_STORE || op == W_LOAD || kArity[op] == 2) {
            if (reg + 1 > max_reg) max_reg = reg + 1;
            any_reg = true;
        }
        pc += 1 + (uint32_t)np;
        if (op == W_RETURN) break;
    }
    if (ins.size() < 2 || kArity[ins[0].op] != 0) {
        // the first instruction must produce a value from the grid point
        *err = "program must start with initial_transformation_to";
        return CC_ERR_INVALID_PROGRAM;
    }
    (void)any_reg;

    // ---- 2. liveness of the wire registers ------------------------------------------------
    std::vector<Interval> intervals;
    std::vector<int> open(kRegisterCount, -1);       // reg -> interval index
    std::vector<int> read_interval(ins.size(), -1);  // wire idx -> interval it reads
    std::vector<int> store_interval(ins.size(), -1);
    for (size_t i = 0; i < ins.size(); ++i) {
        const WireIns &w = ins[i];
        if (w.op == W_STORE) {
            intervals.push_back(Interval{(int)i, -1, true, CC_SLOT_NONE, 0});
            open[w.reg] = (int)intervals.size() - 1;
            store_interval[i] = open[w.reg];
        } else if (w.op == W_LOAD || kArity[w.op] == 2) {
            int iv = open[w.reg];
            if (iv < 0) {
                *err = "instruction " + std::to_string(i) + " reads register " +
                       std::to_string(w.reg) + " before any _store";
                return CC_ERR_INVALID_PROGRAM;
            }
            intervals[iv].last_read = (int)i;
            intervals[iv].n_reads += 1;
            if (!is_point_consumer(w.op)) intervals[iv].point_only = false;
            read_interval[i] = iv;
        }
    }

    // ---- 2b. fused primitives --------------------------------------------------------------------
    // initial_transformation_to ; _store p ; circle|rectangle ; extrusion p ; [offset] ;
    // [transformation_from]   with p read by that extrusion only  ->  one MOP_PRIM_* micro-op.
    // fuse_len[i] = number of wire instructions consumed by the fused op starting at i.
    std::vector<int> fuse_len(ins.size(), 0);
    for (size_t i = 0; i + 3 < ins.size(); ++i) {
        if (ins[i].op != W_INITIAL_TRANSFORMATION_TO || ins[i + 1].op != W_STORE) continue;
        if (ins[i + 2].op != W_CIRCLE && ins[i + 2].op != W_RECTANGLE) continue;
        if (ins[i + 3].op != W_EXTRUSION) continue;
        const int iv = store_interval[i + 1];
        if (iv < 0 || read_interval[i + 3] != iv || intervals[iv].n_reads != 1) continue;
        size_t j = i + 4;
        if (j < ins.size() && ins[j].op == W_OFFSET) ++j;
        if (j < ins.size() && ins[j].op == W_TRANSFORMATION_FROM) ++j;
        fuse_len[i] = (int)(j - i);
        intervals[iv].last_read = -1;  // the point lives in registers inside the fused op
        i = j - 1;
    }

    uint32_t n_p = 0;  // fused primitives emitted

    // ---- 4. linear-scan slot allocation for everything else ---------------------------------
    uint32_t n_slots = 0;
    {
        std::vector<unsigned> free_slots;
        // intervals are already sorted by store_idx; expire by last_read
        std::vector<int> active;
        for (size_t k = 0; k < intervals.size(); ++k) {
            Interval &iv = intervals[k];
            if (iv.last_read < 0) continue;
            for (size_t a = 0; a < active.size();) {
                if (intervals[active[a]].last_read < iv.store_idx) {
                    free_slots.push_back(intervals[active[a]].slot);
                    active[a] = active.back();
                    active.pop_back();
                } else {
                    ++a;
                }
            }
            if (!free_slots.empty()) {
                // lowest free slot keeps the hot set dense
                size_t best = 0;
                for (size_t f = 1; f < free_slots.size(); ++f)
                    if (free_slots[f] < free_slots[best]) best = f;
                iv.slot = free_slots[best];
                free_slots[best] = free_slots.back();
                free_slots.pop_back();
            } else {
                iv.slot = n_slots++;
            }
            active.push_back((int)k);
        }
    }
    if (n_slots > CC_MAX_SLOTS) {
        *err = "program needs " + std::to_string(n_slots) + " live values";
        return CC_ERR_TOO_LARGE;
    }

    // ---- 5. emit microcode ------------------------------------------------------------------
    Emitter e;
    std::vector<size_t> poly_fixups;              // header index of every MOP_POLYGON
    std::vector<std::vector<float>> poly_tables;  // their edge tables, appended after RETURN
    uint32_t fmin = 0, fmax = 0, n_micro = 0;
    auto cost = [&](uint32_t lo, uint32_t hi) { fmin += lo; fmax += hi; };
    for (size_t i = 0; i < ins.size(); ++i) {
        const WireIns &w = ins[i];
        const float *p = w.p;
        uint32_t src = CC_SLOT_NONE;
        if (read_interval[i] >= 0) src = intervals[read_interval[i]].slot;
        float *q;
        if (fuse_len[i]) {
            const bool rect = ins[i + 2].op == W_RECTANGLE;
            q = e.emit(rect ? MOP_PRIM_RECT : MOP_PRIM_CIRCLE, CC_SLOT_NONE, CC_LEN_PRIM);
            quat_matrix(p, false, q, nullptr);
            q[9] = p[4]; q[10] = p[5]; q[11] = p[6];
            q[12] = ins[i + 2].p[0];
            q[13] = rect ? ins[i + 2].p[1] : 0.0f;
            q[14] = ins[i + 3].p[0];
            cost(42, 42);
            if (rect) cost(2, 17); else cost(7, 7);
            cost(1, 16);
            size_t j = i + 4;
            q[15] = 0.0f;  // no offset: w - 0 == w
            if (j < i + (size_t)fuse_len[i] && ins[j].op == W_OFFSET) {
                q[15] = ins[j].p[0];
                cost(1, 1);
                ++j;
            }
            if (j < i + (size_t)fuse_len[i] && ins[j].op == W_TRANSFORMATION_FROM) {
                quat_matrix(ins[j].p, true, q + 16, &q[25]);
                cost(50, 50);
            } else {  // identity: 1*x + 0*y + 0*z == x, w * 1 == w
                for (int k = 0; k < 9; ++k) q[16 + k] = (k % 4 == 0) ? 1.0f : 0.0f;
                q[25] = 1.0f;
            }
            {
                const uint32_t mt = matrix_mask(q), mfrom = matrix_mask(q + 16);
                q[26] = mask_word(mt | (mfrom << 9));
                if (mt != 0x1FFu || mfrom != 0x1FFu) {  // re-tag as the masked variant
                    uint32_t &hd = e.code[e.last_header];
                    hd = CC_HDR(rect ? MOP_PRIM_RECT_M : MOP_PRIM_CIRCLE_M, CC_HDR_SRC(hd), CC_HDR_DST(hd), CC_HDR_LEN(hd));
                }
            }
            i += (size_t)fuse_len[i] - 1;
            ++n_micro;
            ++n_p;
            continue;
        }
        switch (w.op) {
        case W_RETURN: e.emit(MOP_RETURN, CC_SLOT_NONE, CC_LEN_0); break;
        case W_STORE: {
            const Interval &iv = intervals[store_interval[i]];
            if (iv.last_read < 0) continue;  // dead store
            if (e.can_fold_store()) {
                e.fold_store(iv.slot);
                continue;
            }
            e.emit(MOP_NOP, CC_SLOT_NONE, CC_LEN_0);
            e.fold_store(iv.slot);
            break;
        }
        case W_LOAD: e.emit(MOP_LOAD, src, CC_LEN_0); break;
        case W_RECTANGLE:
            q = e.emit(MOP_RECTANGLE, src, CC_LEN_0);
            q[0] = p[0]; q[1] = p[1];
            cost(2, 17);
            break;
        case W_CIRCLE:
            q = e.emit(MOP_CIRCLE, src, CC_LEN_0);
            q[0] = p[0];
            cost(7, 7);
            break;
        case W_REGULAR_POLYGON2D:
            q = e.emit(MOP_REGPOLY, src, CC_LEN_7);
            q[0] = p[0]; q[1] = p[1];
            q[2] = p[1] * (float)std::sin((double)p[0]);  // simple2d.cl:25
            q[3] = p[1] * (float)std::cos((double)p[0]);  // simple2d.cl:45
            q[4] = 2.0f * p[0];
            cost(25, 40);
            break;
        case W_POLYGON2D: {
            int n = (int)p[0];
            q = e.emit(MOP_POLYGON, src, CC_LEN_0);
            q[0] = (float)n;
            poly_fixups.push_back(e.last_header);  // word 2 <- offset of the edge table
            std::vector<float> &tab = poly_tables.emplace_back((size_t)CC_POLY_TABLE_WORDS(n));
            float *eg = tab.data();
            for (int k = 0; k < n; ++k) {
                int j = (k + n - 1) % n;  // previous vertex, polygons2d.cl:13,17-18
                float px = p[1 + 2 * j], py = p[2 + 2 * j];
                float cx = p[1 + 2 * k], cy = p[2 + 2 * k];
                float dx = cx - px, dy = cy - py;
                eg[0] = px; eg[1] = py; eg[2] = dx; eg[3] = dy;
                eg[4] = 1.0f / std::fmaf(dx, dx, dy * dy);
                eg[5] = cy;
                eg += CC_POLY_EDGE_WORDS;
            }
            for (int g0 = 0; g0 < n; g0 += CC_POLY_GROUP) {  // bounding interval of every edge group
                const int j = (g0 + n - 1) % n;
                float xmin = p[1 + 2 * j], xmax = xmin, ymin = p[2 + 2 * j], ymax = ymin;
                for (int k = g0; k < std::min(n, g0 + CC_POLY_GROUP); ++k) {
                    xmin = std::fmin(xmin, p[1 + 2 * k]); xmax = std::fmax(xmax, p[1 + 2 * k]);
                    ymin = std::fmin(ymin, p[2 + 2 * k]); ymax = std::fmax(ymax, p[2 + 2 * k]);
                }
                eg[0] = xmin; eg[1] = xmax; eg[2] = ymin; eg[3] = ymax;
                eg += CC_POLY_GROUP_WORDS;
            }
            cost(10 + 15u * (uint32_t)n, 10 + 22u * (uint32_t)n);
            break;
        }
        case W_SPHERE:
            q = e.emit(MOP_SPHERE, src, CC_LEN_0);
            q[0] = p[0];
            cost(11, 11);
            break;
        case W_HALF_SPACE: e.emit(MOP_HALF_SPACE, src, CC_LEN_0); break;
        case W_REVOLUTION_TO: e.emit(MOP_REV_TO, src, CC_LEN_0); cost(4, 4); break;
        case W_TWIST_REVOLUTION_TO:
            q = e.emit(MOP_TWIST_TO, src, CC_LEN_0);
            q[0] = p[0]; q[1] = p[1];
            cost(16, 16);
            break;
        case W_INITIAL_TRANSFORMATION_TO:
        case W_TRANSFORMATION_TO:
            q = e.emit(w.op == W_TRANSFORMATION_TO ? MOP_T_TO : MOP_T_INIT, src, CC_LEN_T);
            quat_matrix(p, false, q, nullptr);
            q[9] = p[4]; q[10] = p[5]; q[11] = p[6];
            q[12] = mask_word(matrix_mask(q));
            if (matrix_mask(q) != 0x1FFu) {
                uint32_t &hd = e.code[e.last_header];
                hd = CC_HDR(w.op == W_TRANSFORMATION_TO ? MOP_T_TO_M : MOP_T_INIT_M, CC_HDR_SRC(hd), CC_HDR_DST(hd), CC_HDR_LEN(hd));
            }
            cost(42, 42);
            break;
        case W_TRANSFORMATION_FROM: {
            float mf[9], scale;
            quat_matrix(p, true, mf, &scale);
            cost(50, 50);
            // identity rotation and unit scale (38 % of the planetary scene's matrices): every row is
            // 1 * v, the distance is w * 1 — the value does not change, so no micro-op is emitted
            // (a following _store folds into the instruction that produced the value)
            if (is_identity_from(mf, scale) && e.last_header != (size_t)-1) continue;
            q = e.emit(MOP_T_FROM, src, CC_LEN_T);
            std::memcpy(q, mf, sizeof mf);
            q[9] = scale;
            q[10] = mask_word(matrix_mask(q));
            if (matrix_mask(q) != 0x1FFu) {
                uint32_t &hd = e.code[e.last_header];
                hd = CC_HDR(MOP_T_FROM_M, CC_HDR_SRC(hd), CC_HDR_DST(hd), CC_HDR_LEN(hd));
            }
            break;
        }
        case W_MIRROR: e.emit(MOP_MIRROR, src, CC_LEN_0); break;
        case W_SYMMETRICAL_TO: e.emit(MOP_SYM_TO, src, CC_LEN_0); break;
        case W_OFFSET:
            q = e.emit(MOP_OFFSET, src, CC_LEN_0);
            q[0] = p[0];
            cost(1, 1);
            break;
        case W_SHELL:
            q = e.emit(MOP_SHELL, src, CC_LEN_0);
            q[0] = p[0];
            cost(1, 1);
            break;
        case W_REPETITION:
            q = e.emit(MOP_REPETITION, src, CC_LEN_0);
            q[0] = p[0]; q[1] = p[1]; q[2] = p[2];
            cost(3, 3);
            break;
        case W_CIRCULAR_REPETITION_TO:
        case W_CIRCULAR_REPETITION_FROM:
            q = e.emit(w.op == W_CIRCULAR_REPETITION_TO ? MOP_CREP_TO : MOP_CREP_FROM, src, CC_LEN_0);
            q[0] = p[0]; q[1] = 2.0f * p[0];
            cost(14, 14);
            break;
        case W_INVOLUTE_GEAR: {
            q = e.emit(MOP_GEAR, src, CC_LEN_7);
            float pa = p[1];
            q[0] = (float)std::cos((double)pa);                          // gears.cl:2
            q[1] = kPiF / p[0];                                          // gears.cl:3
            q[2] = (q[1] * 0.5f + (float)std::tan((double)pa)) - pa;     // gears.cl:6
            q[3] = 2.0f * q[1];
            q[4] = q[0] * q[0];
            cost(20, 30);
            break;
        }
        case W_EXTRUSION:
            q = e.emit(MOP_EXTRUSION, src, CC_LEN_0);
            q[0] = p[0];
            cost(1, 16);
            break;
        case W_REVOLUTION_FROM: e.emit(MOP_REV_FROM, src, CC_LEN_0); cost(7, 7); break;
        case W_TWIST_REVOLUTION_FROM: {
            q = e.emit(MOP_TWIST_FROM, src, CC_LEN_7);
            float minorR = p[0], r = p[1], twist = p[2];
            float arg = std::fmin(kPiF, (kPi2F * kPi2F) / std::fabs(twist));
            float lip = (((r - minorR) * 2.0f) * (float)std::sin((double)arg)) / minorR;
            q[0] = minorR; q[1] = r; q[2] = twist;
            q[3] = std::fmin(1.0f, lip);  // simple3d.cl:86-88
            q[4] = 0.05f * r;             // simple3d.cl:70
            cost(15, 40);
            break;
        }
        case W_SYMMETRICAL_FROM: e.emit(MOP_SYM_FROM, src, CC_LEN_0); break;
        case W_UNION:
        case W_INTERSECTION:
        case W_SUBTRACTION: {
            bool rounded = p[0] >= 0.0f;  // common.cl:47
            uint32_t base = w.op == W_UNION ? MOP_UNION : (w.op == W_INTERSECTION ? MOP_ISECT : MOP_SUB);
            q = e.emit(base + (rounded ? 1u : 0u), src, CC_LEN_0);
            q[0] = p[0];
            if (rounded) cost(9, 21);
            break;
        }
        default:
            *err = "internal: unhandled opcode";
            return CC_ERR_INVALID_PROGRAM;
        }
        ++n_micro;
    }

    for (size_t k = 0; k < poly_fixups.size(); ++k) {
        const uint32_t off = (uint32_t)e.code.size();  // multiple of 4: tables stay 16-byte aligned
        e.code[poly_fixups[k] + 2] = off;
        const std::vector<float> &tab = poly_tables[k];
        e.code.resize(off + (tab.size() + 3) / 4 * 4, 0u);
        std::memcpy(&e.code[off], tab.data(), tab.size() * sizeof(float));
    }
    out->microcode.swap(e.code);
    analyse_forest(out->microcode, &out->forest);
    analyse_parts(out->microcode, &out->parts);
    analyse_columns(out->microcode, &out->columns);
    out->info.n_words = pc;
    out->info.n_instructions = (uint32_t)ins.size();
    out->info.n_micro_ops = n_micro;
    out->info.n_micro_words = (uint32_t)out->microcode.size();
    out->info.n_wire_registers = max_reg;
    out->info.n_slots = n_slots;
    out->info.n_fused = n_p;
    out->info.flops_min = fmin;
    out->info.flops_max = fmax;
    out->info.n_forest_leaves = out->forest.enabled ? out->forest.n_leaves : 0;
    out->info.forest_depth = out->forest.enabled ? out->forest.max_depth : 0;
    out->info.n_parts = out->parts.enabled ? out->parts.n_parts : 0;
    out->info.n_parts_bounded = 0;
    if (out->parts.enabled)
        for (float l : out->parts.lipschitz) out->info.n_parts_bounded += std::isfinite(l) ? 1u : 0u;
    out->info.column_invariant_percent = out->columns.enabled ? (uint32_t)(out->columns.invariant_share * 100.0f) : 0u;
    out->info.column_axis = (uint32_t)out->columns.axis;
    return CC_OK;
}
