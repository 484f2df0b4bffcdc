// The microcode interpreter (cc_interpret) and where it reads the microcode from (Prog<MODE>): shared by
// cc_kernels.cu (grid sinks, point lists, renderers) and cc_parts.cu (part culling on the interpreter
// tier).  Every translation unit that includes this file gets its own __constant__ window c_code.
#ifndef CC_INTERP_CUH
#define CC_INTERP_CUH

#include "cc_internal.h"
#include "cc_ops.cuh"

__constant__ uint32_t c_code[CC_CONST_WORDS];

// Where the microcode is read from.  MODE 0: everything from the constant bank.  MODE 1:
// everything from the shared-memory copy.  MODE 2 (hybrid): instruction headers from the
// constant bank — decode and dispatch stay in the uniform datapath — and parameters from the
// shared-memory copy with one broadcast LDS.128 per four words.
template <int MODE>
struct Prog {
    const uint32_t *s;
    CC_DEV uint32_t u(uint32_t i) const { return MODE == 1 ? s[i] : c_code[i]; }
    CC_DEV float f(uint32_t i) const { return __uint_as_float(MODE == 0 ? c_code[i] : s[i]); }
    // 16-byte aligned group of four words
    CC_DEV float4 f4(uint32_t i) const
    {
        if (MODE != 0) return *reinterpret_cast<const float4 *>(s + i);
        // constant bank: vector LDC.64 pairs.  (Measured on B200, profiles/r1_ab_variants.md:
        // four scalar uniform LDCU reads instead are 17 % slower on the planetary scene.)
        return *reinterpret_cast<const float4 *>(c_code + i);
    }
};

// Copies `words` words of microcode (a multiple of four) from global to shared memory with 16-byte cp.async, all threads
// of the CTA, and waits for them.  The caller makes sure no thread still reads what s_code held before.
CC_DEV void cc_stage_code(const uint32_t *code, uint32_t words, uint32_t *s_code)
{
    const uint32_t n4 = words / 4;
    for (uint32_t i = threadIdx.x; i < n4; i += CC_THREADS) {
        uint32_t dsts = (uint32_t)__cvta_generic_to_shared(s_code + 4 * i);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dsts), "l"(code + 4 * i) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
}

template <int MODE>
struct ProgFetch {
    Prog<MODE> P;
    uint32_t base;
    CC_DEV float operator()(uint32_t i) const { return P.f(base + i); }
};
// polygons2d.cl:1-74; the edge table lives after the RETURN instruction, word 2 = its offset
template <class V, int MODE>
CC_DEV_HEAVY cc_val<V> cc_polygon2d(const Prog<MODE> &P, uint32_t pc, cc_val<V> co)
{
    return cc_polygon2d_v<V>(ProgFetch<MODE>{P, P.u(pc + 2)}, (uint32_t)P.f(pc + 1), co);
}

// ---- the interpreter ------------------------------------------------------------------------
// Fused primitive (loader pattern: initial_transformation_to -> [store p] -> circle|rectangle
// -> extrusion p -> [offset] -> [transformation_from]): one dispatch, the transformed point
// never leaves registers.  Bit-identical to the unfused sequence (absent offset = 0, absent
// transformation_from = identity matrix and scale 1).
// words: 1..12 m,o | 13 a | 14 b | 15 h | 16 d | 17..25 m' | 26 scale
template <bool RECT, bool MASKED, class V, int G, int SMEM>
CC_DEV void cc_prim(const Prog<SMEM> &P, uint32_t pc, const V (&x)[G], const V (&y)[G], const V (&z)[G],
                    cc_val<V> (&L)[G])
{
    float m[12], mf[12];
    const float4 a = P.f4(pc), b = P.f4(pc + 4), c = P.f4(pc + 8), d = P.f4(pc + 12), e = P.f4(pc + 16),
                 f = P.f4(pc + 20), g = P.f4(pc + 24);
    m[0] = a.y; m[1] = a.z; m[2] = a.w; m[3] = b.x; m[4] = b.y; m[5] = b.z;
    m[6] = b.w; m[7] = c.x; m[8] = c.y; m[9] = c.z; m[10] = c.w; m[11] = d.x;
    mf[0] = e.y; mf[1] = e.z; mf[2] = e.w; mf[3] = f.x; mf[4] = f.y; mf[5] = f.z;
    mf[6] = f.w; mf[7] = g.x; mf[8] = g.y; mf[9] = g.z; mf[10] = 0.f; mf[11] = 0.f;
    const uint32_t masks = MASKED ? __float_as_uint(g.w) : 0u;
    cc_prim_n<RECT, MASKED, V, G>(m, mf, masks & 0x1FFu, (masks >> 9) & 0x1FFu, d.y, d.z, d.w, e.x, x, y, z, L);
}

// RANGED: run the micro-ops in [pc_begin, pc_end) only, continuing from the running value L that the
// caller passes in (part culling: a part's run, or a single union of the tree).
template <int PTS, int SMEM, bool RANGED = false>
CC_DEV void cc_interpret(const Prog<SMEM> P, float4 *__restrict__ regs, const typename cc_pts<PTS>::V (&gx)[cc_pts<PTS>::G],
                         const typename cc_pts<PTS>::V (&gy)[cc_pts<PTS>::G],
                         const typename cc_pts<PTS>::V (&gz)[cc_pts<PTS>::G],
                         cc_val<typename cc_pts<PTS>::V> (&L)[cc_pts<PTS>::G], uint32_t pc_begin = 0, uint32_t pc_end = 0xffffffffu)
{
    typedef typename cc_pts<PTS>::V V;
    typedef cc_val<V> Val;
    constexpr int G = cc_pts<PTS>::G, NL = cc_lane<V>::N;
    float4 *const myregs = regs + threadIdx.x;
    if (!RANGED) {
#pragma unroll
        for (int g = 0; g < G; ++g) L[g] = Val{vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f)};
    }
#define CC_SLOT_BASE(slot, g) (myregs + ((slot) * PTS + (g) * NL) * CC_THREADS)
#define CC_EACH for (int g = 0; g < G; ++g)
#define CC_LOAD_B(g) Val B; cc_slot_load(CC_SLOT_BASE(src, g), B)
    uint32_t pc = RANGED ? pc_begin : 0u;
    for (;;) {
        if (RANGED && pc >= pc_end) return;
        const uint32_t h = P.u(pc);
        const uint32_t op = CC_HDR_OP(h), src = CC_HDR_SRC(h), dst = CC_HDR_DST(h);
        switch (op) {
        case MOP_RETURN: return;
        case MOP_LOAD:
#pragma unroll
            CC_EACH cc_slot_load(CC_SLOT_BASE(src, g), L[g]);
            pc += CC_LEN_0;
            break;
        case MOP_NOP: pc += CC_LEN_0; break;
        // NB: pc only ever advances by IMMEDIATE amounts (every micro-op has a fixed length; the
        // polygon edge table is out of line), after each op, and the batched ops branch on a warp
        // vote.  That is what lets nvcc prove pc warp-uniform and keep decode + dispatch in the
        // uniform datapath (LDCU/UISETP/BRA.U); deriving the increment from a loaded word or
        // advancing before a per-thread branch silently demotes everything to vector code (-11 %).
        case MOP_PRIM_CIRCLE:
            cc_prim<false, false, V, G, SMEM>(P, pc, gx, gy, gz, L);
            pc += CC_LEN_PRIM;
            break;
        case MOP_PRIM_RECT:
            cc_prim<true, false, V, G, SMEM>(P, pc, gx, gy, gz, L);
            pc += CC_LEN_PRIM;
            break;
        case MOP_PRIM_CIRCLE_M:
            cc_prim<false, true, V, G, SMEM>(P, pc, gx, gy, gz, L);
            pc += CC_LEN_PRIM;
            break;
        case MOP_PRIM_RECT_M:
            cc_prim<true, true, V, G, SMEM>(P, pc, gx, gy, gz, L);
            pc += CC_LEN_PRIM;
            break;
        case MOP_RECTANGLE: {
            const float4 q = P.f4(pc);
            cc_rectangle_n(q.y, q.z, L);
            pc += CC_LEN_0;
            break;
        }
        case MOP_CIRCLE: {
            const float r = P.f(pc + 1);
            cc_circle_n(r, L);
            pc += CC_LEN_0;
            break;
        }
        case MOP_REGPOLY: {
            float k[5];
#pragma unroll
            for (int i = 0; i < 5; ++i) k[i] = P.f(pc + 1 + i);
#pragma unroll
            CC_EACH L[g] = cc_op_regpoly(k[0], k[1], k[2], k[3], k[4], L[g]);
            pc += CC_LEN_7;
            break;
        }
        case MOP_POLYGON: {
#pragma unroll
            CC_EACH L[g] = cc_polygon2d<V, SMEM>(P, pc, L[g]);
            pc += CC_LEN_0;
            break;
        }
        case MOP_SPHERE: {
            const float r = P.f(pc + 1);
            cc_sphere_n(r, L);
            pc += CC_LEN_0;
            break;
        }
        case MOP_HALF_SPACE:
#pragma unroll
            CC_EACH L[g] = cc_op_half_space(L[g]);
            pc += CC_LEN_0;
            break;
        case MOP_REV_TO:
#pragma unroll
            CC_EACH L[g] = cc_op_rev_to(L[g]);
            pc += CC_LEN_0;
            break;
        case MOP_TWIST_TO: {
            const float r = P.f(pc + 1), twist = P.f(pc + 2);
#pragma unroll
            CC_EACH L[g] = cc_op_twist_to(r, twist, L[g]);
            pc += CC_LEN_0;
            break;
        }
        case MOP_T_INIT:
        case MOP_T_TO: {
            float m[12];
            {
                const float4 a = P.f4(pc), b = P.f4(pc + 4), c = P.f4(pc + 8), d = P.f4(pc + 12);
                m[0] = a.y; m[1] = a.z; m[2] = a.w; m[3] = b.x; m[4] = b.y; m[5] = b.z;
                m[6] = b.w; m[7] = c.x; m[8] = c.y; m[9] = c.z; m[10] = c.w; m[11] = d.x;
            }
            if (op == MOP_T_INIT) {
#pragma unroll
                CC_EACH L[g] = cc_transform_full(m, gx[g], gy[g], gz[g]);
            } else {
#pragma unroll
                CC_EACH L[g] = cc_transform_full(m, L[g].x, L[g].y, L[g].z);
            }
            pc += CC_LEN_T;
            break;
        }
        case MOP_T_INIT_M:
        case MOP_T_TO_M: {
            float m[12];
            const float4 a = P.f4(pc), b = P.f4(pc + 4), c = P.f4(pc + 8), d = P.f4(pc + 12);
            m[0] = a.y; m[1] = a.z; m[2] = a.w; m[3] = b.x; m[4] = b.y; m[5] = b.z;
            m[6] = b.w; m[7] = c.x; m[8] = c.y; m[9] = c.z; m[10] = c.w; m[11] = d.x;
            const uint32_t mask = __float_as_uint(d.y);
            if (op == MOP_T_INIT_M) {
#pragma unroll
                CC_EACH L[g] = cc_transform(m, mask, gx[g], gy[g], gz[g]);
            } else {
#pragma unroll
                CC_EACH L[g] = cc_transform(m, mask, L[g].x, L[g].y, L[g].z);
            }
            pc += CC_LEN_T;
            break;
        }
        case MOP_T_FROM: {
            float m[12];
            {
                const float4 a = P.f4(pc), b = P.f4(pc + 4), c = P.f4(pc + 8);
                m[0] = a.y; m[1] = a.z; m[2] = a.w; m[3] = b.x; m[4] = b.y; m[5] = b.z;
                m[6] = b.w; m[7] = c.x; m[8] = c.y; m[9] = c.z; m[10] = 0.f; m[11] = 0.f;
            }
#pragma unroll
            CC_EACH L[g] = cc_transform_from_full(m, L[g]);
            pc += CC_LEN_T;
            break;
        }
        case MOP_T_FROM_M: {
            float m[12];
            const float4 a = P.f4(pc), b = P.f4(pc + 4), c = P.f4(pc + 8);
            m[0] = a.y; m[1] = a.z; m[2] = a.w; m[3] = b.x; m[4] = b.y; m[5] = b.z;
            m[6] = b.w; m[7] = c.x; m[8] = c.y; m[9] = c.z; m[10] = 0.f; m[11] = 0.f;
            const uint32_t mask = __float_as_uint(c.w);
#pragma unroll
            CC_EACH L[g] = cc_transform_from(m, mask, L[g]);
            pc += CC_LEN_T;
            break;
        }
        case MOP_MIRROR:  // common.cl:112-114
#pragma unroll
            CC_EACH L[g].x = vneg(L[g].x);
            pc += CC_LEN_0;
            break;
        case MOP_SYM_TO:  // common.cl:116-118
#pragma unroll
            CC_EACH L[g].x = vabs(L[g].x);
            pc += CC_LEN_0;
            break;
        case MOP_OFFSET: {  // common.cl:124-126
            const float d = P.f(pc + 1);
#pragma unroll
            CC_EACH L[g].w = vsub(L[g].w, vbc<V>(d));
            pc += CC_LEN_0;
            break;
        }
        case MOP_SHELL: {
            const float d = P.f(pc + 1);
#pragma unroll
            CC_EACH L[g] = cc_op_shell(d, L[g]);
            pc += CC_LEN_0;
            break;
        }
        case MOP_REPETITION: {
            const float4 q = P.f4(pc);
#pragma unroll
            CC_EACH L[g] = cc_op_repetition(q.y, q.z, q.w, L[g]);
            pc += CC_LEN_0;
            break;
        }
        case MOP_CREP_TO: {
            const float a = P.f(pc + 1), b = P.f(pc + 2);
#pragma unroll
            CC_EACH L[g] = cc_op_crep_to(a, b, L[g]);
            pc += CC_LEN_0;
            break;
        }
        case MOP_GEAR: {
            float k[5];
#pragma unroll
            for (int i = 0; i < 5; ++i) k[i] = P.f(pc + 1 + i);
#pragma unroll
            CC_EACH L[g] = cc_op_gear(k[0], k[1], k[2], k[3], k[4], L[g]);
            pc += CC_LEN_7;
            break;
        }
        // ---- ops whose second operand is a point held in a slot ----
        case MOP_EXTRUSION: {
            const float hh = P.f(pc + 1);
            V cz[G];
#pragma unroll
            CC_EACH cc_slot_load_z(CC_SLOT_BASE(src, g), cz[g]);
            cc_extrusion_n(hh, L, cz);
            pc += CC_LEN_0;
            break;
        }
        case MOP_REV_FROM:
#pragma unroll
            CC_EACH {
                CC_LOAD_B(g);
                L[g] = cc_revolution_from(L[g], B);
            }
            pc += CC_LEN_0;
            break;
        case MOP_SYM_FROM:
#pragma unroll
            CC_EACH {
                Val B;
                cc_slot_load_x(CC_SLOT_BASE(src, g), B.x);
                L[g] = cc_op_sym_from(L[g], B);
            }
            pc += CC_LEN_0;
            break;
        case MOP_TWIST_FROM: {
            float k[5];
#pragma unroll
            for (int i = 0; i < 5; ++i) k[i] = P.f(pc + 1 + i);
#pragma unroll
            CC_EACH {
                CC_LOAD_B(g);
                L[g] = cc_op_twist_from(k[0], k[1], k[2], k[3], k[4], L[g], B);
            }
            pc += CC_LEN_7;
            break;
        }
        case MOP_CREP_FROM: {
            const float a = P.f(pc + 1), b = P.f(pc + 2);
#pragma unroll
            CC_EACH {
                CC_LOAD_B(g);
                L[g] = cc_op_crep_from(a, b, L[g], B);
            }
            pc += CC_LEN_0;
            break;
        }
        // ---- CSG combinators: second operand is always a slot ----
        case MOP_UNION:
#pragma unroll
            CC_EACH {
                CC_LOAD_B(g);
                L[g] = cc_op_union(L[g], B);
            }
            pc += CC_LEN_0;
            break;
        case MOP_UNION_R: {
            const float r = P.f(pc + 1);
#pragma unroll
            CC_EACH {
                CC_LOAD_B(g);
                L[g] = cc_rounded_union(r, L[g], B);
            }
            pc += CC_LEN_0;
            break;
        }
        case MOP_ISECT:
#pragma unroll
            CC_EACH {
                CC_LOAD_B(g);
                L[g] = cc_op_isect(L[g], B);
            }
            pc += CC_LEN_0;
            break;
        case MOP_ISECT_R: {
            const float r = P.f(pc + 1);
#pragma unroll
            CC_EACH {
                CC_LOAD_B(g);
                L[g] = cc_op_isect_r(r, L[g], B);
            }
            pc += CC_LEN_0;
            break;
        }
        case MOP_SUB:
#pragma unroll
            CC_EACH {
                CC_LOAD_B(g);
                L[g] = cc_op_sub(L[g], B);
            }
            pc += CC_LEN_0;
            break;
        case MOP_SUB_R: {
            const float r = P.f(pc + 1);
#pragma unroll
            CC_EACH {
                CC_LOAD_B(g);
                L[g] = cc_op_sub_r(r, L[g], B);
            }
            pc += CC_LEN_0;
            break;
        }
        default: __builtin_unreachable();  // the loader only emits the micro-ops above
        }
        if (dst != CC_SLOT_NONE) {
#pragma unroll
            CC_EACH cc_slot_store(CC_SLOT_BASE(dst, g), L[g]);
        }
    }
#undef CC_SLOT_BASE
#undef CC_EACH
#undef CC_LOAD_B
}


#endif
