// SDF op library, device side: one __device__ function per node type of
// /root/reference/codecad/shapes/*.cl, evaluated in the canonical arithmetic of
// cc_math.cuh.  Values follow the reference convention: .xyz = unit direction
// (gradient) or point coordinates, .w = signed distance (negative inside).
//
// Each function handles ONE point; the interpreter calls it in an unrolled loop over the
// thread's points so that independent points interleave in the FP32 pipes.  Parameters
// arrive as warp-uniform values decoded from the microcode.
#ifndef CC_OPS_CUH
#define CC_OPS_CUH

#include "cc_math.cuh"
#include "cc_device_types.h"

// heavy, rarely dominant ops are real functions: inlining them PTS times per kernel variant
// would push the interpreter out of the instruction cache
#ifndef CC_OPT_NOINLINE_HEAVY
#define CC_OPT_NOINLINE_HEAVY 1
#endif
#if CC_OPT_NOINLINE_HEAVY
#define CC_DEV_HEAVY static __device__ __noinline__
#else
#define CC_DEV_HEAVY __device__ __forceinline__
#endif

CC_DEV float4 cc_neg4(float4 a) { return make_float4(-a.x, -a.y, -a.z, -a.w); }
CC_DEV float4 cc_sel4(bool c, float4 a, float4 b)
{
    return make_float4(c ? a.x : b.x, c ? a.y : b.y, c ? a.z : b.z, c ? a.w : b.w);
}

// shapes/simple2d.cl:1-4 = perpendicular_intersection(slab_x, slab_y)  (common.cl:15-43)
CC_DEV float4 cc_rectangle(float hw, float hh, float4 p)
{
    float sx = copysignf(1.0f, p.x), sy = copysignf(1.0f, p.y);
    float ax = fabsf(p.x) - hw, ay = fabsf(p.y) - hh;
    float dist = cc_len2(ax, ay);
    float inv = cc_rcp(dist);
    bool both = ax > 0.0f && ay > 0.0f;
    bool first = ax > ay;
    float4 r;
    r.x = both ? sx * (ax * inv) : (first ? sx : 0.0f);
    r.y = both ? sy * (ay * inv) : (first ? 0.0f : sy);
    r.z = 0.0f;
    r.w = both ? dist : (first ? ax : ay);
    return r;
}

// shapes/simple3d.cl:18-21 = perpendicular_intersection(slab_z(h, coords), input)
CC_DEV float4 cc_extrusion(float h, float4 in, float cz)
{
    float sz = copysignf(1.0f, cz);
    float az = fabsf(cz) - h;
    float dist = cc_len2(az, in.w);
    float inv = cc_rcp(dist);
    float m1 = az * inv, m2 = in.w * inv;
    bool both = az > 0.0f && in.w > 0.0f;
    bool first = az > in.w;
    float4 r;
    r.x = both ? in.x * m2 : (first ? 0.0f : in.x);
    r.y = both ? in.y * m2 : (first ? 0.0f : in.y);
    r.z = both ? cc_fma(sz, m1, in.z * m2) : (first ? sz : in.z);
    r.w = both ? dist : (first ? az : in.w);
    return r;
}

// shapes/simple2d.cl:6-14
CC_DEV float4 cc_circle(float r, float4 p)
{
    float len = cc_len2(p.x, p.y);
    float inv = cc_rcp(len);
    bool zero = len == 0.0f;
    return make_float4(zero ? 1.0f : p.x * inv, zero ? 0.0f : p.y * inv, 0.0f, len - r);
}

// shapes/simple3d.cl:1-12
CC_DEV float4 cc_sphere(float r, float4 p)
{
    float len = cc_len3(p.x, p.y, p.z);
    float inv = cc_rcp(len);
    bool zero = len == 0.0f;
    return make_float4(zero ? 1.0f : p.x * inv, zero ? 0.0f : p.y * inv, zero ? 0.0f : p.z * inv, len - r);
}

// ---- the same ops over all of a thread's points, with one combined special-operand test ----
// L holds G lane vectors (cc_math.cuh: V = float2 packs two points into FFMA2/FMUL2/FADD2).
// Results are identical to the per-point forms above (which remain the slow path and the
// reference for the oracle): in the fast path every sqrt/rcp operand is in the exact range of
// cc_sqrt_fast / cc_rcp_fast, and a length in that range is never zero.
static __device__ __noinline__ float4 cc_rectangle_slow(float hw, float hh, float4 p) { return cc_rectangle(hw, hh, p); }
static __device__ __noinline__ float4 cc_circle_slow(float r, float4 p) { return cc_circle(r, p); }
static __device__ __noinline__ float4 cc_sphere_slow(float r, float4 p) { return cc_sphere(r, p); }
static __device__ __noinline__ float4 cc_extrusion_slow(float h, float4 in, float cz) { return cc_extrusion(h, in, cz); }

// apply a one-point function to every lane of every vector
template <class V, int G, class F>
CC_DEV void cc_each_lane(cc_val<V> (&L)[G], F f)
{
#pragma unroll
    for (int g = 0; g < G; ++g) {
#pragma unroll
        for (int l = 0; l < cc_lane<V>::N; ++l) cc_lane_put(L[g], l, f(cc_lane_get(L[g], l), g, l));
    }
}

template <bool DEFER, class V, int G>
CC_DEV void cc_rectangle_n_(uint32_t &range, float hw, float hh, cc_val<V> (&L)[G])
{
    typedef typename cc_lane<V>::mask M;
    V ax[G], ay[G], s[G];
    bool sp = false;
#pragma unroll
    for (int g = 0; g < G; ++g) {
        ax[g] = vsub(vabs(L[g].x), vbc<V>(hw));
        ay[g] = vsub(vabs(L[g].y), vbc<V>(hh));
        s[g] = vfma(ax[g], ax[g], vmul(ay[g], ay[g]));
        if (DEFER) vrange(range, s[g]);
        else sp |= vspecial(s[g]);
    }
    if (!DEFER && __any_sync(0xffffffffu, sp)) {  // warp-uniform: keeps the interpreter's control flow convergent
        cc_each_lane(L, [&](float4 p, int, int) { return cc_rectangle_slow(hw, hh, p); });
        return;
    }
#pragma unroll
    for (int g = 0; g < G; ++g) {
        const V one = vbc<V>(1.0f), zero = vbc<V>(0.0f);
        const V sx = vcopysign(one, L[g].x), sy = vcopysign(one, L[g].y);
        const V dist = vsqrt_fast(s[g]);
        const V inv = vrcp_fast(dist);
        const M both = mand(vgt(ax[g], zero), vgt(ay[g], zero));
        const M first = vgt(ax[g], ay[g]);
        cc_val<V> r;
        r.x = vsel(both, vmul(sx, vmul(ax[g], inv)), vsel(first, sx, zero));
        r.y = vsel(both, vmul(sy, vmul(ay[g], inv)), vsel(first, zero, sy));
        r.z = zero;
        r.w = vsel(both, dist, vsel(first, ax[g], ay[g]));
        L[g] = r;
    }
}

template <bool DEFER, class V, int G>
CC_DEV void cc_circle_n_(uint32_t &range, float r, cc_val<V> (&L)[G])
{
    V s[G];
    bool sp = false;
#pragma unroll
    for (int g = 0; g < G; ++g) {
        s[g] = vfma(L[g].x, L[g].x, vmul(L[g].y, L[g].y));
        if (DEFER) vrange(range, s[g]);
        else sp |= vspecial(s[g]);
    }
    if (!DEFER && __any_sync(0xffffffffu, sp)) {  // warp-uniform: keeps the interpreter's control flow convergent
        cc_each_lane(L, [&](float4 p, int, int) { return cc_circle_slow(r, p); });
        return;
    }
#pragma unroll
    for (int g = 0; g < G; ++g) {
        const V len = vsqrt_fast(s[g]);
        const V inv = vrcp_fast(len);
        L[g] = cc_val<V>{vmul(L[g].x, inv), vmul(L[g].y, inv), vbc<V>(0.0f), vsub(len, vbc<V>(r))};
    }
}

template <bool DEFER, class V, int G>
CC_DEV void cc_sphere_n_(uint32_t &range, float r, cc_val<V> (&L)[G])
{
    V s[G];
    bool sp = false;
#pragma unroll
    for (int g = 0; g < G; ++g) {
        s[g] = vfma(L[g].x, L[g].x, vfma(L[g].y, L[g].y, vmul(L[g].z, L[g].z)));
        if (DEFER) vrange(range, s[g]);
        else sp |= vspecial(s[g]);
    }
    if (!DEFER && __any_sync(0xffffffffu, sp)) {  // warp-uniform: keeps the interpreter's control flow convergent
        cc_each_lane(L, [&](float4 p, int, int) { return cc_sphere_slow(r, p); });
        return;
    }
#pragma unroll
    for (int g = 0; g < G; ++g) {
        const V len = vsqrt_fast(s[g]);
        const V inv = vrcp_fast(len);
        L[g] = cc_val<V>{vmul(L[g].x, inv), vmul(L[g].y, inv), vmul(L[g].z, inv), vsub(len, vbc<V>(r))};
    }
}

// cz[g] = z coordinate of the point operand
template <bool DEFER, class V, int G>
CC_DEV void cc_extrusion_n_(uint32_t &range, float h, cc_val<V> (&L)[G], const V (&cz)[G])
{
    typedef typename cc_lane<V>::mask M;
    V az[G], s[G];
    bool sp = false;
#pragma unroll
    for (int g = 0; g < G; ++g) {
        az[g] = vsub(vabs(cz[g]), vbc<V>(h));
        s[g] = vfma(az[g], az[g], vmul(L[g].w, L[g].w));
        if (DEFER) vrange(range, s[g]);
        else sp |= vspecial(s[g]);
    }
    if (!DEFER && __any_sync(0xffffffffu, sp)) {  // warp-uniform: keeps the interpreter's control flow convergent
        cc_each_lane(L, [&](float4 p, int g, int l) { return cc_extrusion_slow(h, p, vlane(cz[g], l)); });
        return;
    }
#pragma unroll
    for (int g = 0; g < G; ++g) {
        const V zero = vbc<V>(0.0f);
        const cc_val<V> in = L[g];
        const V sz = vcopysign(vbc<V>(1.0f), cz[g]);
        const V dist = vsqrt_fast(s[g]);
        const V inv = vrcp_fast(dist);
        const V m1 = vmul(az[g], inv), m2 = vmul(in.w, inv);
        const M both = mand(vgt(az[g], zero), vgt(in.w, zero));
        const M first = vgt(az[g], in.w);
        cc_val<V> r;
        r.x = vsel(both, vmul(in.x, m2), vsel(first, zero, in.x));
        r.y = vsel(both, vmul(in.y, m2), vsel(first, zero, in.y));
        r.z = vsel(both, vfma(sz, m1, vmul(in.z, m2)), vsel(first, sz, in.z));
        r.w = vsel(both, dist, vsel(first, az[g], in.w));
        L[g] = r;
    }
}

// the voting forms, and the deferred ones (last argument `range`): the fast path always, its range test folded into
// `range`, which the caller tests once after all its ops (cc_range_flagged); CC_DEFER_CHECKS=0 makes them vote
template <class V, int G> CC_DEV void cc_rectangle_n(float hw, float hh, cc_val<V> (&L)[G])
{
    uint32_t unused = 0;
    cc_rectangle_n_<false>(unused, hw, hh, L);
}
template <class V, int G> CC_DEV void cc_rectangle_n(float hw, float hh, cc_val<V> (&L)[G], uint32_t &range)
{
    cc_rectangle_n_<CC_DEFER_CHECKS != 0>(range, hw, hh, L);
}
template <class V, int G> CC_DEV void cc_circle_n(float r, cc_val<V> (&L)[G])
{
    uint32_t unused = 0;
    cc_circle_n_<false>(unused, r, L);
}
template <class V, int G> CC_DEV void cc_circle_n(float r, cc_val<V> (&L)[G], uint32_t &range)
{
    cc_circle_n_<CC_DEFER_CHECKS != 0>(range, r, L);
}
template <class V, int G> CC_DEV void cc_sphere_n(float r, cc_val<V> (&L)[G])
{
    uint32_t unused = 0;
    cc_sphere_n_<false>(unused, r, L);
}
template <class V, int G> CC_DEV void cc_sphere_n(float r, cc_val<V> (&L)[G], uint32_t &range)
{
    cc_sphere_n_<CC_DEFER_CHECKS != 0>(range, r, L);
}
template <class V, int G> CC_DEV void cc_extrusion_n(float h, cc_val<V> (&L)[G], const V (&cz)[G])
{
    uint32_t unused = 0;
    cc_extrusion_n_<false>(unused, h, L, cz);
}
template <class V, int G> CC_DEV void cc_extrusion_n(float h, cc_val<V> (&L)[G], const V (&cz)[G], uint32_t &range)
{
    cc_extrusion_n_<CC_DEFER_CHECKS != 0>(range, h, L, cz);
}

// The distance-only forms of the column brick kernel's sweep (DESIGN.md 4.10): exactly the arithmetic of the deferred
// cc_sphere_n_ / cc_extrusion_n_ that produces .w and the range test, none of the gradient's.  P: the sphere's point;
// w: the extrusion's profile distance in, its distance out.
template <class V, int G> CC_DEV void cc_sphere_dist(float r, const cc_val<V> (&P)[G], V (&w)[G], uint32_t &range)
{
#pragma unroll
    for (int g = 0; g < G; ++g) {
        const V s = vfma(P[g].x, P[g].x, vfma(P[g].y, P[g].y, vmul(P[g].z, P[g].z)));
        vrange(range, s);
        w[g] = vsub(vsqrt_fast(s), vbc<V>(r));
    }
}
// The sweep's extrusion picks its result with min / max (CC_SWEEP_MINMAX, DESIGN.md 4.10): fminf(az, w) > 0 for
// az > 0 && w > 0, fmaxf(az, w) for az > w ? az : w.  They differ only where an operand is NaN or both are zeros of
// opposite sign; then s is NaN or 0, the range test flags, and the warp throws its values away.  0 keeps the selects.
#ifndef CC_SWEEP_MINMAX
#define CC_SWEEP_MINMAX 1
#endif
template <class V, int G> CC_DEV void cc_extrusion_dist(float h, V (&w)[G], const V (&cz)[G], uint32_t &range)
{
#pragma unroll
    for (int g = 0; g < G; ++g) {
        const V zero = vbc<V>(0.0f), az = vsub(vabs(cz[g]), vbc<V>(h));
        const V s = vfma(az, az, vmul(w[g], w[g]));
        vrange(range, s);
        const V dist = vsqrt_fast(s);
        if (CC_SWEEP_MINMAX)
            w[g] = vsel(vgt(vmin(az, w[g]), zero), dist, vmax(az, w[g]));
        else
            w[g] = vsel(mand(vgt(az, zero), vgt(w[g], zero)), dist, vsel(vgt(az, w[g]), az, w[g]));
    }
}

// shapes/common.cl:45-64
// cc-arith pins down two cases that the formula leaves to rounding noise (both are no-ops in exact
// arithmetic, where |c| <= 1): (1) the blend is taken only if at least one operand is closer than
// r — with both farther away it would need c > 1, which only a dot product of two unit normals
// rounded ABOVE one can deliver; (2) the radicand is clamped at zero, so the blend value is never
// NaN.  With (1) a union of operands that are all farther than r away is exactly the nearest
// operand, which is what lets whole subtrees be skipped without changing a bit (cc_forest.cu).
// Both tests sit in the rare path.
template <class V>
CC_DEV cc_val<V> cc_rounded_union(float r, cc_val<V> o1, cc_val<V> o2)
{
    typedef typename cc_lane<V>::mask M;
    cc_val<V> res = cc_val_sel(vlt(o1.w, o2.w), o1, o2);
    const V c = vfma(o1.x, o2.x, vfma(o1.y, o2.y, vmul(o1.z, o2.z)));
    const V x1 = vsub(vbc<V>(r), o1.w), x2 = vsub(vbc<V>(r), o2.w);
    const M blend = mand(vlt(vmul(c, x1), x2), vlt(vmul(c, x2), x1));
    if (many(blend)) {  // rare: only within r of both surfaces
        const V zero = vbc<V>(0.0f);
        const M near = mor(vgt(x1, zero), vgt(x2, zero));
        const V num = vfma(vneg(vmul(vmul(vbc<V>(2.0f), c), x1)), x2, vfma(x1, x1, vmul(x2, x2)));
        const V den = vfma(vneg(c), c, vbc<V>(1.0f));
        const cc_val<V> b{zero, zero, zero, vsub(vbc<V>(r), vsqrt(vmax(vdiv(num, den), zero)))};
        res = cc_val_sel(mand(blend, near), b, res);
    }
    return res;
}

// ---- transformations: 3x3 (row-major) * v [+ o]   — common.cl:78-110 in matrix form ----
// cc-arith: a row is accumulated innermost-first (z, y, x) and terms whose coefficient is exactly
// zero are OMITTED (a parameter-only simplification, fixed at load time like the quaternion ->
// matrix conversion; multiplying by a zero coefficient would only decide the sign of an exactly
// zero result).  CAD scenes are full of axis-aligned transforms: 44 % of the matrix entries of
// the planetary scene are zero and 38 % of its matrices are the identity.  `mask` bit k tells
// whether m[k] != 0; the loader stores it next to the matrix, the specialised kernels compute it
// from the immediates (and the branches below fold away at compile time).
#define CC_MASK_FULL 0x1FFu
CC_DEV unsigned cc_matrix_mask(const float (&m)[12])
{
    unsigned k = 0;
#pragma unroll
    for (int i = 0; i < 9; ++i) k |= (m[i] != 0.0f) ? (1u << i) : 0u;
    return k;
}
template <class V>
CC_DEV V cc_row_to(unsigned mask3, float m0, float m1, float m2, float o, V x, V y, V z)
{
    V acc = vbc<V>(o);
    if (mask3 & 4u) acc = vfma(vbc<V>(m2), z, acc);
    if (mask3 & 2u) acc = vfma(vbc<V>(m1), y, acc);
    if (mask3 & 1u) acc = vfma(vbc<V>(m0), x, acc);
    return acc;
}
// first (innermost) term: a plain product; a coefficient of exactly +-1 returns the operand itself
// (1 * v == v, -1 * v == -v for every v), which spares the multiply
template <class V>
CC_DEV V cc_first_term(float m, V v)
{
    if (m == 1.0f) return v;
    if (m == -1.0f) return vneg(v);
    return vmul(vbc<V>(m), v);
}
template <class V>
CC_DEV V cc_row_from(unsigned mask3, float m0, float m1, float m2, V x, V y, V z)
{
    switch (mask3 & 7u) {
    case 0u: return vbc<V>(0.0f);
    case 1u: return cc_first_term(m0, x);
    case 2u: return cc_first_term(m1, y);
    case 3u: return vfma(vbc<V>(m0), x, cc_first_term(m1, y));
    case 4u: return cc_first_term(m2, z);
    case 5u: return vfma(vbc<V>(m0), x, cc_first_term(m2, z));
    case 6u: return vfma(vbc<V>(m1), y, cc_first_term(m2, z));
    default: return vfma(vbc<V>(m0), x, vfma(vbc<V>(m1), y, cc_first_term(m2, z)));
    }
}
// full matrix (no zero coefficient): the straight 9-term form
template <class V>
CC_DEV cc_val<V> cc_transform_full(const float (&m)[12], V x, V y, V z)
{
    return cc_val<V>{vfma(vbc<V>(m[0]), x, vfma(vbc<V>(m[1]), y, vfma(vbc<V>(m[2]), z, vbc<V>(m[9])))),
                     vfma(vbc<V>(m[3]), x, vfma(vbc<V>(m[4]), y, vfma(vbc<V>(m[5]), z, vbc<V>(m[10])))),
                     vfma(vbc<V>(m[6]), x, vfma(vbc<V>(m[7]), y, vfma(vbc<V>(m[8]), z, vbc<V>(m[11])))),
                     vbc<V>(0.0f)};
}
// any matrix: `mask` says which coefficients are non-zero (in the specialised kernels it is a
// compile-time constant and the branches fold; the interpreter runs this for "_M" micro-ops only)
template <class V>
CC_DEV cc_val<V> cc_transform(const float (&m)[12], unsigned mask, V x, V y, V z)
{
    if (mask == CC_MASK_FULL) return cc_transform_full(m, x, y, z);
    return cc_val<V>{cc_row_to(mask, m[0], m[1], m[2], m[9], x, y, z), cc_row_to(mask >> 3, m[3], m[4], m[5], m[10], x, y, z),
                     cc_row_to(mask >> 6, m[6], m[7], m[8], m[11], x, y, z), vbc<V>(0.0f)};
}

// common.cl:100-110 (matrix already divided by |q|^2; m[9] = |q|^2)
template <class V>
CC_DEV cc_val<V> cc_transform_from_full(const float (&m)[12], cc_val<V> in)
{
    return cc_val<V>{vfma(vbc<V>(m[0]), in.x, vfma(vbc<V>(m[1]), in.y, vmul(vbc<V>(m[2]), in.z))),
                     vfma(vbc<V>(m[3]), in.x, vfma(vbc<V>(m[4]), in.y, vmul(vbc<V>(m[5]), in.z))),
                     vfma(vbc<V>(m[6]), in.x, vfma(vbc<V>(m[7]), in.y, vmul(vbc<V>(m[8]), in.z))),
                     vmul(in.w, vbc<V>(m[9]))};
}
template <class V>
CC_DEV cc_val<V> cc_transform_from(const float (&m)[12], unsigned mask, cc_val<V> in)
{
    if (mask == CC_MASK_FULL) return cc_transform_from_full(m, in);
    const V w = (m[9] == 1.0f) ? in.w : vmul(in.w, vbc<V>(m[9]));
    return cc_val<V>{cc_row_from(mask, m[0], m[1], m[2], in.x, in.y, in.z),
                     cc_row_from(mask >> 3, m[3], m[4], m[5], in.x, in.y, in.z),
                     cc_row_from(mask >> 6, m[6], m[7], m[8], in.x, in.y, in.z), w};
}

// shapes/simple2d.cl:16-46; k = (piOverN, r, r*sin, r*cos, 2*piOverN)
CC_DEV_HEAVY float4 cc_regular_polygon2d(float k0, float k1, float k2, float k3, float k4, float4 co)
{
    const float k[5] = {k0, k1, k2, k3, k4};
    float piOverN = k[0], r = k[1];
    float len = cc_len2(co.x, co.y);
    float alpha = (cc_atan2(co.y, co.x) + CC_2PI_F) + piOverN;
    int side = (int)floorf(cc_div(alpha, k[4]));
    float t = (float)(side * 2) * piOverN;
    float modAlpha = (alpha - t) - piOverN;
    float s, c;
    cc_sincos(modAlpha, &s, &c);
    if (fabsf(s * len) > k[2]) {
        float ny, nx;
        cc_sincos(cc_fma(cc_sign(s), piOverN, t), &ny, &nx);
        float dx = co.x - nx * r, dy = co.y - ny * r;
        float dist = cc_len2(dx, dy);
        if (dist > 0.0f) {
            float inv = cc_rcp(dist);
            return make_float4(dx * inv, dy * inv, 0.0f, dist);
        }
    }
    float dy, dx;
    cc_sincos(t, &dy, &dx);
    return make_float4(dx, dy, 0.0f, cc_fma(len, c, -k[3]));
}

// shapes/gears.cl:1-42; k = (baseRadius, toothAngle, halfToothBaseAngle, 2*toothAngle, baseRadius^2)
CC_DEV_HEAVY float4 cc_involute_gear(float k0, float k1, float k2, float k3, float k4, float4 co)
{
    const float k[5] = {k0, k1, k2, k3, k4};
    float baseRadius = k[0], toothAngle = k[1], halfTooth = k[2];
    float len = cc_len2(co.x, co.y);
    float alpha = cc_atan2(co.y, co.x);
    float wrapped = cc_fmod_pos(alpha + CC_2PI_F, k[3]);
    float d = fabsf(wrapped - toothAngle);
    float involuteAlpha = halfTooth - d;
    if (len < baseRadius) {
        float inv = cc_rcp(len);
        float nx = co.y * inv, ny = -(co.x * inv);
        if (wrapped > toothAngle) { nx = -nx; ny = -ny; }
        return make_float4(nx, ny, 0.0f, (d - halfTooth) * len);
    }
    float phi = involuteAlpha + cc_acos(cc_div(baseRadius, len));
    float base = alpha - involuteAlpha;
    float normalAngle = (wrapped < toothAngle) ? (CC_PI_F - phi) - base : phi - base;
    float nx, ny;
    cc_sincos(normalAngle, &nx, &ny);
    float distance = cc_fma(-baseRadius, phi, cc_sqrt(cc_fma(len, len, -k[4])));
    return make_float4(nx, ny, 0.0f, distance);
}

// shapes/simple3d.cl:42-51
CC_DEV_HEAVY float4 cc_twist_revolution_to(float r, float twist, float4 co)
{
    float alpha = cc_fmod_pos(cc_atan2(co.z, co.x) + CC_PI_F, CC_2PI_F);
    float beta = cc_div(twist * alpha, CC_2PI_F);
    float ipx = cc_len2(co.x, co.z) - r, ipy = co.y;
    float s, c;
    cc_sincos(-beta, &s, &c);
    return make_float4(cc_fma(c, ipx, -(s * ipy)), cc_fma(s, ipx, c * ipy), 0.0f, 0.0f);
}

// shapes/simple3d.cl:53-97; k = (minorR, r, twist, min(1, lipschitz), padding)
CC_DEV_HEAVY float4 cc_twist_revolution_from(float k0, float k1, float k2, float k3, float k4, float4 inPlane,
                                             float4 co)
{
    const float k[5] = {k0, k1, k2, k3, k4};
    float minorR = k[0], r = k[1], twist = k[2];
    float ad = cc_len2(co.x, co.z);
    float ipx = ad - r, ipy = co.y;
    float icd = cc_len2(ipx, ipy);
    float wd = icd - minorR;
    float bound, dx, dy;
    if (ad == 0.0f) return make_float4(1.0f, 0.0f, 0.0f, r - minorR);
    if (wd > k[4]) {
        float inv = cc_rcp(icd);
        bound = wd; dx = ipx * inv; dy = ipy * inv;
    } else {
        float alpha = cc_fmod_pos(cc_atan2(co.z, co.x) + CC_PI_F, CC_2PI_F);
        float beta = cc_div(twist * alpha, CC_2PI_F);
        float s, c;
        cc_sincos(beta, &s, &c);
        bound = inPlane.w * k[3];
        dx = cc_fma(c, inPlane.x, -(s * inPlane.y));
        dy = cc_fma(s, inPlane.x, c * inPlane.y);
    }
    float mult = cc_div(dx, ad);
    return make_float4(co.x * mult, dy, co.z * mult, bound);
}

// shapes/unsafe.cl:8-15
CC_DEV_HEAVY float4 cc_circular_repetition_to(float piOverN, float twoPiOverN, float4 co)
{
    float len = cc_len2(co.x, co.y);
    float alpha = (cc_atan2(co.y, co.x) + CC_2PI_F) + piOverN;
    int side = (int)floorf(cc_div(alpha, twoPiOverN));
    float modAlpha = (alpha - (float)(side * 2) * piOverN) - piOverN;
    float s, c;
    cc_sincos(modAlpha, &s, &c);
    return make_float4(len * c, len * s, co.z, 0.0f);
}

// shapes/unsafe.cl:17-23
CC_DEV_HEAVY float4 cc_circular_repetition_from(float piOverN, float twoPiOverN, float4 dist, float4 co)
{
    float alpha = (cc_atan2(co.y, co.x) + CC_2PI_F) + piOverN;
    int side = (int)floorf(cc_div(alpha, twoPiOverN));
    float s, c;
    cc_sincos((float)(side * 2) * piOverN, &s, &c);
    return make_float4(cc_fma(c, dist.x, -(s * dist.y)), cc_fma(s, dist.x, c * dist.y), dist.z, dist.w);
}

// shapes/simple3d.cl:28-39
template <class V>
CC_DEV cc_val<V> cc_revolution_from(cc_val<V> flat, cc_val<V> co)
{
    typedef typename cc_lane<V>::mask M;
    const V len = vlen2(co.x, co.z);
    const M zero = veq(len, vbc<V>(0.0f));
    const V mult = vsel(zero, flat.x, vdiv(flat.x, len));
    const V cx = vsel(zero, vbc<V>(1.0f), co.x);
    return cc_val<V>{vmul(cx, mult), flat.y, vmul(co.z, mult), flat.w};
}

// Fused primitive (loader pattern initial_transformation_to -> [store p] -> circle|rectangle ->
// extrusion p -> [offset] -> [transformation_from]); bit-identical to the unfused sequence.
template <bool RECT, bool MASKED, class V, int G>
CC_DEV void cc_prim_n(const float (&m)[12], const float (&mf)[12], unsigned mask, unsigned mask_from, float pa, float pb,
                      float h, float d, const V (&x)[G], const V (&y)[G], const V (&z)[G], cc_val<V> (&L)[G])
{
    V pz[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
        L[g] = MASKED ? cc_transform(m, mask, x[g], y[g], z[g]) : cc_transform_full(m, x[g], y[g], z[g]);
        pz[g] = L[g].z;
    }
    if (RECT) cc_rectangle_n(pa, pb, L);
    else cc_circle_n(pa, L);
    cc_extrusion_n(h, L, pz);
#pragma unroll
    for (int g = 0; g < G; ++g) {
        L[g].w = vsub(L[g].w, vbc<V>(d));
        L[g] = MASKED ? cc_transform_from(mf, mask_from, L[g]) : cc_transform_from_full(mf, L[g]);
    }
}

// shapes/polygons2d.cl:1-74 over a precomputed edge table (px, py, dx, dy, 1/|d|^2, cy) per
// edge; FETCH(i) returns table word i (the interpreter reads it from the microcode, the
// specialised kernels from a __constant__ array).
//
// The edge loop is branch-free and works on lane vectors: per edge the candidate squared distance
// is selected (segment interior / start vertex / none when t > 1) and only two running values are
// kept per point, the smallest squared distance and the index of the edge that produced it (as a
// float: exact below 2^24 edges).  Which kind of feature won and its normal are recomputed once,
// after the loop, from that edge — the same operations on the same operands, hence the same bits
// as the reference's running (normal, isVertex) pair with its strict `<` update.  The crossing
// test reuses the previous edge's end-point comparison (cy of edge i is py of edge i+1).
template <class FETCH>
CC_DEV float4 cc_polygon2d_finish(const FETCH &fetch, float best, float x, float y, float nearest, float outside)
{
    float nnx = 0.0f, nny = 0.0f;
    bool nearest_is_vertex = false;
    if (best >= 0.0f) {
        const uint32_t e = 6u * (uint32_t)best;
        const float px = fetch(e), py = fetch(e + 1), dx = fetch(e + 2), dy = fetch(e + 3), inv = fetch(e + 4);
        const float tqx = x - px, tqy = y - py;
        const float t = cc_fma(dx, tqx, dy * tqy) * inv;
        nnx = -dy; nny = dx;  // segment normal
        if (!(t >= 0.0f)) {
            const float cd = cc_fma(tqx, tqx, tqy * tqy);
            nearest_is_vertex = cd > 1.1920928955078125e-7f;  // too close to the vertex: keep the segment normal
            if (nearest_is_vertex) { nnx = tqx; nny = tqy; }
        }
    }
    const float distance = outside * cc_sqrt(nearest);
    const float inv = nearest_is_vertex ? cc_rcp(distance) : cc_rcp(cc_len2(nnx, nny));
    return make_float4(nnx * inv, nny * inv, 0.0f, distance);
}

// Edge groups.  The table continues with one entry per group of CC_POLY_GROUP consecutive edges:
// the bounding interval of the group's vertices.  A group is skipped when
// (a) no lane can improve on the nearest distance there: the squared distance to the group's
//     bounding box exceeds B, an upper bound of the FINAL nearest value (the squared distance to the
//     nearest vertex: the candidate chain that starts at a vertex only ever gets closer); every
//     candidate of the group then loses the strict `<` whatever the running value is, and
// (b) no lane's y lies inside the group's y range, so no edge of it can flip the crossing parity.
// Both tests carry a 2e-5 relative margin against the rounding of the candidate distances; the
// skipped work could not have changed a bit.  The points of a warp are neighbours (often they share
// x and y exactly: the extrusion axis is the fastest grid axis), so the votes rarely split.
template <class V, class FETCH>
CC_DEV cc_val<V> cc_polygon2d_v(const FETCH &fetch, uint32_t n, cc_val<V> co)
{
    typedef typename cc_lane<V>::mask M;
    const V zero = vbc<V>(0.0f), one = vbc<V>(1.0f);
    V nearest = vbc<V>(__int_as_float(0x7f800000)), best = vbc<V>(-1.0f), outside = one;
    M prev_below = vlt(vbc<V>(n ? fetch(1) : 0.0f), co.y);  // previousPoint.y < coords.y of edge 0
    const uint32_t gt = CC_POLY_EDGE_WORDS * n, ng = (n + CC_POLY_GROUP - 1) / CC_POLY_GROUP;
    V bound = vbc<V>(__int_as_float(0x7f800000));
#ifndef CC_POLY_BOUND_STRIDE
#define CC_POLY_BOUND_STRIDE 4  // every fourth vertex (airfoil mass_properties: 4.15 / 3.78 / 3.69 / 3.74 ms for 1 / 2 / 4 / 8)
#endif
#pragma unroll 4
    for (uint32_t i = 0; i < n; i += CC_POLY_BOUND_STRIDE) {
        const V qx = vsub(co.x, vbc<V>(fetch(6 * i))), qy = vsub(co.y, vbc<V>(fetch(6 * i + 1)));
        bound = vmin(bound, vfma(qx, qx, vmul(qy, qy)));
    }
    bound = vmul(bound, vbc<V>(1.00002f));
    for (uint32_t g = 0; g < ng; ++g) {
        const float xmin = fetch(gt + 4 * g), xmax = fetch(gt + 4 * g + 1), ymin = fetch(gt + 4 * g + 2), ymax = fetch(gt + 4 * g + 3);
        const V ex = vmax(vmax(vsub(vbc<V>(xmin), co.x), vsub(co.x, vbc<V>(xmax))), zero);
        const V ey = vmax(vmax(vsub(vbc<V>(ymin), co.y), vsub(co.y, vbc<V>(ymax))), zero);
        const V lb = vmul(vfma(ex, ex, vmul(ey, ey)), vbc<V>(0.99998f));
        const M above = vgt(co.y, vbc<V>(ymax));                      // every vertex of the group is below the point
        const M may_cross = mand(vgt(co.y, vbc<V>(ymin)), mnot(above));
        const M may_win = mnot(vgt(lb, bound));                       // (NaN coordinates: never skipped)
        const bool need_win = __any_sync(0xffffffffu, many(may_win));
        if (!need_win && !__any_sync(0xffffffffu, many(may_cross))) {
            prev_below = above;  // = (y of the group's last vertex < coords.y)
            continue;
        }
        const uint32_t i1 = min(n, (g + 1) * CC_POLY_GROUP);
        uint32_t e = CC_POLY_EDGE_WORDS * g * CC_POLY_GROUP;
        if (!need_win) {  // only the crossing parity can change here: a thin shape's groups overlap in y
            for (uint32_t i = g * CC_POLY_GROUP; i < i1; ++i, e += 6) {
                const M cur_below = vlt(vbc<V>(fetch(e + 5)), co.y);
                const M straddle = mxor(prev_below, cur_below);
                if (__any_sync(0xffffffffu, many(straddle))) {
                    const float dx = fetch(e + 2), dy = fetch(e + 3);
                    const V tqx = vsub(co.x, vbc<V>(fetch(e))), tqy = vsub(co.y, vbc<V>(fetch(e + 1)));
                    const V side = vmul(vbc<V>(dy), vfma(vbc<V>(-dy), tqx, vmul(vbc<V>(dx), tqy)));
                    outside = vsel(mand(straddle, vgt(side, zero)), vneg(outside), outside);
                }
                prev_below = cur_below;
            }
            continue;
        }
#pragma unroll 2
        for (uint32_t i = g * CC_POLY_GROUP; i < i1; ++i, e += 6) {
            const float px = fetch(e), py = fetch(e + 1), dx = fetch(e + 2), dy = fetch(e + 3), inv = fetch(e + 4),
                        cy = fetch(e + 5);
            const V tqx = vsub(co.x, vbc<V>(px)), tqy = vsub(co.y, vbc<V>(py));
            // polygons2d.cl:24-26: even-odd crossing test
            const M cur_below = vlt(vbc<V>(cy), co.y);
            const M straddle = mxor(prev_below, cur_below);
            // few edges straddle a point's y, and the points of a warp are neighbours: skip the side
            // test when no lane needs it (warp-uniform branch; `outside` is unchanged in that case)
            if (__any_sync(0xffffffffu, many(straddle))) {
                const V side = vmul(vbc<V>(dy), vfma(vbc<V>(-dy), tqx, vmul(vbc<V>(dx), tqy)));
                outside = vsel(mand(straddle, vgt(side, zero)), vneg(outside), outside);
            }
            prev_below = cur_below;
            // :28-52: nearest point of the edge, t > 1 belongs to the next edge's start vertex
            // For t < 0 (or NaN) the candidate is the start vertex, |toQuery|^2.  Clamping t at zero
            // gives exactly that through the segment formula: fma(-0, d, tq) == tq up to the sign of a
            // zero, which the squares erase; fmaxf returns 0 for a NaN t, the branch the reference's
            // `t >= 0` test takes as well.
            const V t = vmul(vfma(vbc<V>(dx), tqx, vmul(vbc<V>(dy), tqy)), vbc<V>(inv));
            const V tc = vmax(t, zero);
            const V tcx = vfma(vneg(tc), vbc<V>(dx), tqx), tcy = vfma(vneg(tc), vbc<V>(dy), tqy);
            const V cd = vfma(tcx, tcx, vmul(tcy, tcy));
            // :55-60
            const M better = mand(mnot(vgt(t, one)), vlt(cd, nearest));
            nearest = vsel(better, cd, nearest);
            best = vsel(better, vbc<V>((float)i), best);
            (void)py;
        }
    }
    cc_val<V> r;
#pragma unroll
    for (int l = 0; l < cc_lane<V>::N; ++l)
        cc_lane_put(r, l, cc_polygon2d_finish(fetch, cc_lane_scalar(best, l), cc_lane_scalar(co.x, l), cc_lane_scalar(co.y, l),
                                              cc_lane_scalar(nearest, l), cc_lane_scalar(outside, l)));
    return r;
}

struct cc_table_fetch {
    const float *t;
    CC_DEV float operator()(uint32_t i) const { return t[i]; }
};


// ---- out-of-line forms for LARGE programs (specialised kernels of more than a few hundred
// micro-ops): one copy of the code, parameters read from a __constant__ table through a uniform
// pointer.  Inlining 500 fused primitives costs NVRTC minutes and produces 880 KB of straight-line
// code; called like this the kernel compiles in seconds and its body stays in the instruction cache.
// t = the micro-op's parameter words 1..27 (cc_kernels.cu cc_prim): m,o | a b h d | m' | scale | masks
template <bool RECT, class V>
__device__ __noinline__ cc_val<V> cc_prim_table(const float *__restrict__ t, V x, V y, V z)
{
    float m[12], mf[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) m[i] = t[i];
#pragma unroll
    for (int i = 0; i < 10; ++i) mf[i] = t[16 + i];
    mf[10] = mf[11] = 0.f;
    const unsigned masks = __float_as_uint(t[26]);
    const V xs[1] = {x}, ys[1] = {y}, zs[1] = {z};
    cc_val<V> L[1];
    cc_prim_n<RECT, true, V, 1>(m, mf, masks & 0x1FFu, (masks >> 9) & 0x1FFu, t[12], t[13], t[14], t[15], xs, ys, zs, L);
    return L[0];
}
template <class V>
__device__ __noinline__ cc_val<V> cc_rounded_union_fn(float r, cc_val<V> a, cc_val<V> b)
{
    return cc_rounded_union(r, a, b);
}

// ---- one entry point per micro-op over lane vectors (shared by the interpreter and the
//      scene-specialised kernels).  Cheap ops are packed; the heavy, rarely dominant ones run
//      their one-point form lane by lane. ----------------------------------------------------
template <class V, class F>
CC_DEV cc_val<V> cc_map1(cc_val<V> a, F f)
{
    cc_val<V> r;
#pragma unroll
    for (int l = 0; l < cc_lane<V>::N; ++l) cc_lane_put(r, l, f(cc_lane_get(a, l)));
    return r;
}
template <class V, class F>
CC_DEV cc_val<V> cc_map2(cc_val<V> a, cc_val<V> b, F f)
{
    cc_val<V> r;
#pragma unroll
    for (int l = 0; l < cc_lane<V>::N; ++l) cc_lane_put(r, l, f(cc_lane_get(a, l), cc_lane_get(b, l)));
    return r;
}

template <class V> CC_DEV cc_val<V> cc_op_half_space(cc_val<V> a)  // simple3d.cl:14-16
{
    return cc_val<V>{vbc<V>(0.0f), vbc<V>(-1.0f), vbc<V>(0.0f), vneg(a.y)};
}
template <class V> CC_DEV cc_val<V> cc_op_rev_to(cc_val<V> a)  // simple3d.cl:23-26
{
    return cc_val<V>{vlen2(a.x, a.z), a.y, vbc<V>(0.0f), vbc<V>(0.0f)};
}
template <class V> CC_DEV cc_val<V> cc_op_shell(float d, cc_val<V> a)  // common.cl:128-131
{
    cc_val<V> s = cc_val_sel(vge(a.w, vbc<V>(0.0f)), a, cc_val_neg(a));
    s.w = vsub(s.w, vbc<V>(d));
    return s;
}
template <class V> CC_DEV cc_val<V> cc_op_repetition(float ox, float oy, float oz, cc_val<V> a)  // unsafe.cl:1-6
{
    return cc_map1(a, [&](float4 p) { return make_float4(cc_remainder(p.x, ox), cc_remainder(p.y, oy), cc_remainder(p.z, oz), 0.0f); });
}
template <class V> CC_DEV cc_val<V> cc_op_sym_from(cc_val<V> a, cc_val<V> point)  // common.cl:120-122
{
    a.x = vsel(vlt(point.x, vbc<V>(0.0f)), vneg(a.x), a.x);
    return a;
}
// CSG with r < 0 (common.cl:60-76): the second operand comes from a slot
template <class V> CC_DEV cc_val<V> cc_op_union(cc_val<V> a, cc_val<V> b) { return cc_val_sel(vlt(a.w, b.w), a, b); }
template <class V> CC_DEV cc_val<V> cc_op_isect(cc_val<V> a, cc_val<V> b)  // -min(-a, -b)
{
    return cc_val_sel(vlt(vneg(a.w), vneg(b.w)), a, b);
}
template <class V> CC_DEV cc_val<V> cc_op_sub(cc_val<V> a, cc_val<V> b)  // -min(-a, b)
{
    return cc_val_sel(vlt(vneg(a.w), b.w), a, cc_val_neg(b));
}
template <class V> CC_DEV cc_val<V> cc_op_isect_r(float r, cc_val<V> a, cc_val<V> b)
{
    return cc_val_neg(cc_rounded_union(r, cc_val_neg(a), cc_val_neg(b)));
}
template <class V> CC_DEV cc_val<V> cc_op_sub_r(float r, cc_val<V> a, cc_val<V> b)
{
    return cc_val_neg(cc_rounded_union(r, cc_val_neg(a), b));
}
// heavy ops, lane by lane
template <class V> CC_DEV cc_val<V> cc_op_regpoly(float k0, float k1, float k2, float k3, float k4, cc_val<V> a)
{
    return cc_map1(a, [&](float4 p) { return cc_regular_polygon2d(k0, k1, k2, k3, k4, p); });
}
CC_DEV cc_val<float> cc_op_gear(float k0, float k1, float k2, float k3, float k4, cc_val<float> a)
{
    return cc_map1(a, [&](float4 p) { return cc_involute_gear(k0, k1, k2, k3, k4, p); });
}
// shapes/gears.cl:1-42 for two points at once: the operation sequence of cc_involute_gear lane by
// lane, arithmetic packed.  Preconditions of the unchecked division / square-root steps (operand
// magnitudes in [2^-40, 2^60], parameters in [2^-30, 2^30]) are tested up front; anything else
// (points on an axis, degenerate parameters) takes the one-point form, whose results are identical.
#ifndef CC_OPT_GEAR_INLINE
#define CC_OPT_GEAR_INLINE 0
#endif
#if CC_OPT_GEAR_INLINE
CC_DEV
#else
static __device__ __noinline__
#endif
cc_val<float2> cc_involute_gear2(float k0, float k1, float k2, float k3, float k4, cc_val<float2> co)
{
    const float baseRadius = k0, toothAngle = k1, halfTooth = k2;
    const uint32_t lo = 0x2b800000u /* 2^-40 */, span = 0x5d800000u /* 2^60 */ - 0x2b800000u;
    const uint32_t plo = 0x30800000u /* 2^-30 */, pspan = 0x4e800000u /* 2^30 */ - 0x30800000u;
    const bool lanes_ok = ((__float_as_uint(co.x.x) & 0x7fffffffu) - lo) <= span &&
                          ((__float_as_uint(co.x.y) & 0x7fffffffu) - lo) <= span &&
                          ((__float_as_uint(co.y.x) & 0x7fffffffu) - lo) <= span &&
                          ((__float_as_uint(co.y.y) & 0x7fffffffu) - lo) <= span;
    const bool params_ok = (__float_as_uint(baseRadius) - plo) <= pspan && (__float_as_uint(k3) - plo) <= pspan;
    if (__builtin_expect(!(lanes_ok && params_ok), 0))
        return cc_map1(co, [&](float4 p) { return cc_involute_gear(k0, k1, k2, k3, k4, p); });
    typedef float2 V;
    const V zero = vbc<V>(0.0f);
    const V len = vsqrt_fast(vfma(co.x, co.x, vmul(co.y, co.y)));
    V mn_, mx_;
    const V alpha = vatan2_fast(co.y, co.x, &mn_, &mx_);  // operands are in range (lanes_ok)
    const V wrapped = vfmod_pos_fast(vadd(alpha, vbc<V>(CC_2PI_F)), k3);
    const V d = vabs(vsub(wrapped, vbc<V>(toothAngle)));
    const V involuteAlpha = vsub(vbc<V>(halfTooth), d);
    const cc_mask2 inner = vlt(len, vbc<V>(baseRadius));
    cc_val<V> res{zero, zero, zero, zero};
    if (many(inner)) {
        const V inv = vrcp_fast(len);
        V nx = vmul(co.y, inv), ny = vneg(vmul(co.x, inv));
        const cc_mask2 flip = vgt(wrapped, vbc<V>(toothAngle));
        nx = vsel(flip, vneg(nx), nx);
        ny = vsel(flip, vneg(ny), ny);
        res = cc_val<V>{nx, ny, zero, vmul(vsub(d, vbc<V>(halfTooth)), len)};
    }
    if (!mall(inner)) {
        // lanes of the inner regime get a harmless length so that they stay on the fast paths
        const V lenO = vsel(inner, vbc<V>(2.0f * baseRadius), len);
        const V q = vdiv_fast(vbc<V>(baseRadius), lenO);
        V t = vfma(vneg(q), q, vbc<V>(1.0f));
        t = vsel(vlt(t, zero), zero, t);
        const V phi = vadd(involuteAlpha, vatan2(vsqrt(t), q));  // cc_acos
        const V base = vsub(alpha, involuteAlpha);
        const V normalAngle = vsel(vlt(wrapped, vbc<V>(toothAngle)), vsub(vsub(vbc<V>(CC_PI_F), phi), base), vsub(phi, base));
        V nx, ny;
        vsincos(normalAngle, &nx, &ny);
        const V distance = vfma(vbc<V>(-baseRadius), phi, vsqrt(vfma(lenO, lenO, vbc<V>(-k4))));
        const cc_val<V> outer{nx, ny, zero, distance};
        res = cc_val_sel(inner, res, outer);
    }
    return res;
}
CC_DEV cc_val<float2> cc_op_gear(float k0, float k1, float k2, float k3, float k4, cc_val<float2> a)
{
    return cc_involute_gear2(k0, k1, k2, k3, k4, a);
}
template <class V> CC_DEV cc_val<V> cc_op_twist_to(float r, float twist, cc_val<V> a)
{
    return cc_map1(a, [&](float4 p) { return cc_twist_revolution_to(r, twist, p); });
}
template <class V>
CC_DEV cc_val<V> cc_op_twist_from(float k0, float k1, float k2, float k3, float k4, cc_val<V> a, cc_val<V> point)
{
    return cc_map2(a, point, [&](float4 p, float4 q) { return cc_twist_revolution_from(k0, k1, k2, k3, k4, p, q); });
}
template <class V> CC_DEV cc_val<V> cc_op_crep_to(float a0, float a1, cc_val<V> a)
{
    return cc_map1(a, [&](float4 p) { return cc_circular_repetition_to(a0, a1, p); });
}
template <class V> CC_DEV cc_val<V> cc_op_crep_from(float a0, float a1, cc_val<V> a, cc_val<V> point)
{
    return cc_map2(a, point, [&](float4 p, float4 q) { return cc_circular_repetition_from(a0, a1, p, q); });
}
// inlined on purpose: `table` is then a known __constant__ array and the loop counter is uniform, so
// the six edge parameters are constant-bank operands of the arithmetic instead of loads
template <class V> CC_DEV cc_val<V> cc_op_polygon_table(const float *table, uint32_t n, cc_val<V> a)
{
    return cc_polygon2d_v<V>(cc_table_fetch{table}, n, a);
}

// ---- shared-memory value slots (interpreter) / value cells (specialised kernels) ----
// Value slots in shared memory: float4 regs[slot][PTS][CC_THREADS].  A packed pair of points
// (V = float2) occupies two consecutive float4 rows: (x0,x1,y0,y1) and (z0,z1,w0,w1).
CC_DEV void cc_slot_store(float4 *base, const cc_val<float> &v) { base[0] = make_float4(v.x, v.y, v.z, v.w); }
CC_DEV void cc_slot_store(float4 *base, const cc_val<float2> &v)
{
    base[0] = make_float4(v.x.x, v.x.y, v.y.x, v.y.y);
    base[CC_THREADS] = make_float4(v.z.x, v.z.y, v.w.x, v.w.y);
}
CC_DEV void cc_slot_load(const float4 *base, cc_val<float> &v)
{
    const float4 f = base[0];
    v = cc_val<float>{f.x, f.y, f.z, f.w};
}
CC_DEV void cc_slot_load(const float4 *base, cc_val<float2> &v)
{
    const float4 a = base[0], b = base[CC_THREADS];
    v = cc_val<float2>{make_float2(a.x, a.y), make_float2(a.z, a.w), make_float2(b.x, b.y), make_float2(b.z, b.w)};
}
// opaque 128-bit shared load: the compiler may not forward the stored registers to it
CC_DEV float4 cc_lds128_opaque(const float4 *p)
{
    float4 r;
    const unsigned a = (unsigned)__cvta_generic_to_shared(p);
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(a));
    return r;
}
CC_DEV void cc_slot_load_opaque(const float4 *base, cc_val<float> &v)
{
    const float4 f = cc_lds128_opaque(base);
    v = cc_val<float>{f.x, f.y, f.z, f.w};
}
CC_DEV void cc_slot_load_opaque(const float4 *base, cc_val<float2> &v)
{
    const float4 a = cc_lds128_opaque(base), b = cc_lds128_opaque(base + CC_THREADS);
    v = cc_val<float2>{make_float2(a.x, a.y), make_float2(a.z, a.w), make_float2(b.x, b.y), make_float2(b.z, b.w)};
}
CC_DEV float2 cc_lds64_opaque(const float2 *p)
{
    float2 r;
    const unsigned a = (unsigned)__cvta_generic_to_shared(p);
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "r"(a));
    return r;
}
CC_DEV void cc_slot_load_x_opaque(const float4 *base, float &x) { x = cc_lds128_opaque(base).x; }
CC_DEV void cc_slot_load_x_opaque(const float4 *base, float2 &x) { x = cc_lds64_opaque(reinterpret_cast<const float2 *>(base)); }
CC_DEV void cc_slot_load_z_opaque(const float4 *base, float &z) { z = cc_lds128_opaque(base).z; }
CC_DEV void cc_slot_load_z_opaque(const float4 *base, float2 &z)
{
    z = cc_lds64_opaque(reinterpret_cast<const float2 *>(base + CC_THREADS));
}
CC_DEV void cc_slot_load_x(const float4 *base, float &x) { x = base[0].x; }
CC_DEV void cc_slot_load_x(const float4 *base, float2 &x) { x = *reinterpret_cast<const float2 *>(base); }
CC_DEV void cc_slot_load_z(const float4 *base, float &z) { z = base[0].z; }
CC_DEV void cc_slot_load_z(const float4 *base, float2 &z) { z = *reinterpret_cast<const float2 *>(base + CC_THREADS); }
// store only the z component (cells whose every reader is an extrusion)
CC_DEV void cc_slot_store_z(float4 *base, float z) { reinterpret_cast<float *>(base)[2] = z; }
CC_DEV void cc_slot_store_z(float4 *base, float2 z) { *reinterpret_cast<float2 *>(base + CC_THREADS) = z; }
// a distance and its leaf id (the column brick kernel's sweep): one float4 row, (w0,w1,id0,id1) for a packed pair
CC_DEV void cc_slot_store_wi(float4 *base, float w, float id) { *reinterpret_cast<float2 *>(base) = make_float2(w, id); }
CC_DEV void cc_slot_store_wi(float4 *base, float2 w, float2 id) { base[0] = make_float4(w.x, w.y, id.x, id.y); }
CC_DEV void cc_slot_load_wi_opaque(const float4 *base, float &w, float &id)
{
    const float2 f = cc_lds64_opaque(reinterpret_cast<const float2 *>(base));
    w = f.x;
    id = f.y;
}
CC_DEV void cc_slot_load_wi_opaque(const float4 *base, float2 &w, float2 &id)
{
    const float4 f = cc_lds128_opaque(base);
    w = make_float2(f.x, f.y);
    id = make_float2(f.z, f.w);
}


#endif
