// sm_100a kernels of the codecad SDF hot path.
//
//   cc_eval_kernel<PTS, SMEM_PROG, SINK>   the SDF interpreter (replaces the generated
//       OpenCL `evaluate()`  /root/reference/codecad/nodes/codegen.py:17-63) fused with
//       one of four sinks that replace the reference's __kernel entry points:
//         FLOAT4    grid_eval            grid_eval.cl:23-34
//         PYMCUBES  grid_eval_pymcubes   grid_eval.cl:2-21
//         CLASSIFY  subdivision_step     subdivision.cl:12-30
//         MASS      mass_properties      mass_properties.cl:7-56
//
// Execution model.  Every thread of a warp walks the SAME microcode stream (the program is
// identical for all grid points), so instruction fetch/decode is warp-uniform: header and
// parameters are broadcast reads from shared memory (program staged once per CTA with
// cp.async) or from the constant bank.  Each thread owns PTS grid points that differ
// only in their linear cell index (stride = CTA size, so that every global store of the
// warp is one contiguous 512-byte float4 run); the points' running values (`lastValue` of
// the reference) live in registers and independent points interleave in the FP32 pipes,
// which amortises decode over PTS points and hides the 4-cycle FMA latency.  The
// reference's 512-entry private register array becomes a handful of liveness-renamed
// slots in shared memory, laid out [slot][point][thread] as float4 so that a warp's
// access is a conflict-free 512-byte LDS.128/STS.128; the commonest producer/consumer chain
// (transform -> 2-D primitive -> extrusion -> offset -> inverse rotation) is fused into one
// micro-op by the loader so that its intermediate point never leaves registers.
//
// Compile with -fmad=false (see cc_math.cuh).
#include <cuda_runtime.h>
#include <stdint.h>

#include "cc_internal.h"
#include "cc_ops.cuh"
#include "cc_body.cuh"
#include "cc_render.cuh"

#include "cc_interp.cuh"

template <int PTS, int SMEM>
struct InterpEval {
    typedef typename cc_pts<PTS>::V V;
    Prog<SMEM> P;
    float4 *regs;
    CC_DEV void operator()(const V (&gx)[cc_pts<PTS>::G], const V (&gy)[cc_pts<PTS>::G], const V (&gz)[cc_pts<PTS>::G],
                           cc_val<V> (&L)[cc_pts<PTS>::G]) const
    {
        if (SMEM != 0) {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            __syncthreads();
        }
        cc_interpret<PTS, SMEM>(P, regs, gx, gy, gz, L);
    }
};

template <int PTS, int SMEM, int SINK, bool POINTS = false>
__global__ void __launch_bounds__(CC_THREADS) cc_eval_kernel(const cc_eval_args a)
{
    extern __shared__ float4 smem4[];
    float4 *regs = smem4;  // [n_slots][PTS][CC_THREADS]
    uint32_t *s_code = reinterpret_cast<uint32_t *>(smem4 + (size_t)a.n_slots * PTS * CC_THREADS);
    if (SMEM != 0) {
        // stage the microcode once per CTA: 16-byte cp.async, all threads
        const uint32_t n4 = a.code_words / 4;
        for (uint32_t i = threadIdx.x; i < n4; i += CC_THREADS) {
            uint32_t dsts = (uint32_t)__cvta_generic_to_shared(s_code + 4 * i);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dsts), "l"(a.code + 4 * i) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    InterpEval<PTS, SMEM> eval{Prog<SMEM>{s_code}, regs};
    cc_kernel_body<PTS, SINK, InterpEval<PTS, SMEM>, POINTS>(a, eval);
}

// ---- host-side launch ---------------------------------------------------------------------------

uint32_t cc_tile_points(const cc_launch_cfg &cfg) { return (uint32_t)(CC_THREADS * cfg.pts); }

size_t cc_eval_smem_bytes(const cc_launch_cfg &cfg, uint32_t n_slots, uint32_t code_words)
{
    size_t b = (size_t)n_slots * cfg.pts * CC_THREADS * sizeof(float4);
    if (cfg.prog_space != 1) b += (size_t)code_words * 4;  // shared copy (2 = shared, 3 = hybrid)
    return b;
}

int cc_upload_constant_program(const uint32_t *h_code, uint32_t n_words, void *stream)
{
    return (int)cudaMemcpyToSymbolAsync(c_code, h_code, (size_t)n_words * 4, 0, cudaMemcpyHostToDevice,
                                        (cudaStream_t)stream);
}

template <int PTS, int SMEM, int SINK, bool POINTS = false>
static int launch_one(const cc_eval_args &a, size_t smem, uint32_t grid, cudaStream_t st)
{
    auto k = cc_eval_kernel<PTS, SMEM, SINK, POINTS>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    k<<<grid, CC_THREADS, smem, st>>>(a);
    return (int)cudaGetLastError();
}

template <int SINK>
static int launch_sink(const cc_launch_cfg &cfg, const cc_eval_args &a, size_t smem, uint32_t grid, cudaStream_t st)
{
    // prog_space: 1 = constant bank, 2 = shared copy, 3 = hybrid  ->  Prog MODE 0 / 1 / 2
#define CC_LAUNCH_PTS(P)                                                                \
    (cfg.prog_space == 1 ? launch_one<P, 0, SINK>(a, smem, grid, st)                    \
                         : cfg.prog_space == 2 ? launch_one<P, 1, SINK>(a, smem, grid, st) \
                                               : launch_one<P, 2, SINK>(a, smem, grid, st))
#ifdef CC_EXPERIMENT_PTS  // compile-time experiments: instantiate a single variant
    return launch_one<CC_EXPERIMENT_PTS, CC_EXPERIMENT_MODE, SINK>(a, smem, grid, st);
#else
    switch (cfg.pts) {
    case 1: return CC_LAUNCH_PTS(1);
    case 2: return CC_LAUNCH_PTS(2);
    default: return CC_LAUNCH_PTS(4);
    }
#endif
#undef CC_LAUNCH_PTS
}

int cc_launch_eval(int sink, const cc_launch_cfg &cfg, const cc_eval_args &a, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = cc_eval_smem_bytes(cfg, a.n_slots, a.code_words);
    const uint32_t grid = a.n_blocks * a.tiles_per_block;
    if (grid == 0) return 0;
    if (a.points) {
        // point lists: FLOAT4 sink, 1 or 2 points per thread, constant bank or shared copy
        if (sink != CC_SINK_FLOAT4 || cfg.pts > 2 || cfg.prog_space > 2) return (int)cudaErrorInvalidValue;
        if (cfg.pts == 1)
            return cfg.prog_space == 1 ? launch_one<1, 0, CC_SINK_FLOAT4, true>(a, smem, grid, st)
                                       : launch_one<1, 1, CC_SINK_FLOAT4, true>(a, smem, grid, st);
        return cfg.prog_space == 1 ? launch_one<2, 0, CC_SINK_FLOAT4, true>(a, smem, grid, st)
                                   : launch_one<2, 1, CC_SINK_FLOAT4, true>(a, smem, grid, st);
    }
    switch (sink) {
    case CC_SINK_FLOAT4: return launch_sink<CC_SINK_FLOAT4>(cfg, a, smem, grid, st);
    case CC_SINK_PYMCUBES: return launch_sink<CC_SINK_PYMCUBES>(cfg, a, smem, grid, st);
    case CC_SINK_CLASSIFY: return launch_sink<CC_SINK_CLASSIFY>(cfg, a, smem, grid, st);
    default: return launch_sink<CC_SINK_MASS>(cfg, a, smem, grid, st);
    }
}

// ---- image renderers around evaluate() (SURVEY.md 8(f) rank 4): bodies in cc_render.cuh --------
template <int SMEM>
struct InterpPointEval {
    Prog<SMEM> P;
    float4 *regs;
    CC_DEV void operator()(const float (&gx)[1], const float (&gy)[1], const float (&gz)[1], cc_val<float> (&L)[1]) const
    {
        cc_interpret<1, SMEM>(P, regs, gx, gy, gz, L);
    }
};

template <int SMEM>
CC_DEV const uint32_t *cc_stage_program(const cc_render_args &a, float4 *smem4)
{
    uint32_t *s_code = reinterpret_cast<uint32_t *>(smem4 + (size_t)a.n_slots * CC_THREADS);
    if (SMEM != 0) {
        const uint32_t n4 = a.code_words / 4;
        for (uint32_t i = threadIdx.x; i < n4; i += CC_THREADS) {
            uint32_t dsts = (uint32_t)__cvta_generic_to_shared(s_code + 4 * i);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dsts), "l"(a.code + 4 * i) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
    }
    return s_code;
}

template <int SMEM>
__global__ void __launch_bounds__(CC_THREADS) cc_bitmap_kernel(const cc_render_args a)
{
    extern __shared__ float4 smem4[];
    InterpPointEval<SMEM> eval{Prog<SMEM>{cc_stage_program<SMEM>(a, smem4)}, smem4};
    cc_bitmap_body(a, eval);
}

template <int SMEM>
__global__ void __launch_bounds__(CC_THREADS) cc_ray_caster_kernel(const cc_render_args a)
{
    extern __shared__ float4 smem4[];
    InterpPointEval<SMEM> eval{Prog<SMEM>{cc_stage_program<SMEM>(a, smem4)}, smem4};
    cc_ray_caster_body(a, eval);
}

template <int SMEM>
static int launch_render(bool ray, const cc_render_args &a, size_t smem, cudaStream_t st)
{
    const uint32_t tiles = ((a.w + 7) / 8) * ((a.h + 3) / 4);  // one warp each
    const uint32_t grid = (tiles + CC_THREADS / 32 - 1) / (CC_THREADS / 32);
    if (grid == 0) return 0;
    if (ray) {
        auto k = cc_ray_caster_kernel<SMEM>;
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        k<<<grid, CC_THREADS, smem, st>>>(a);
    } else {
        auto k = cc_bitmap_kernel<SMEM>;
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        k<<<grid, CC_THREADS, smem, st>>>(a);
    }
    return (int)cudaGetLastError();
}

// prog_space 1 = constant bank (program already uploaded by the caller), 2 = shared copy,
// 0 = scene-specialised kernel of `prog`
int cc_launch_render(int ray, int prog_space, const cc_program *prog, const cc_render_launch &r, void *stream, int dev_index)
{
    cc_render_args a;
    a.code = r.code; a.code_words = r.code_words; a.n_slots = r.n_slots;
    a.ox = r.origin[0]; a.oy = r.origin[1]; a.oz = r.origin[2];
    a.fx = r.forward[0]; a.fy = r.forward[1]; a.fz = r.forward[2];
    a.ux = r.up[0]; a.uy = r.up[1]; a.uz = r.up[2];
    a.rx = r.right[0]; a.ry = r.right[1]; a.rz = r.right[2];
    a.pixel_tolerance = r.pixel_tolerance; a.box_radius = r.box_radius;
    a.min_distance = r.min_distance; a.max_distance = r.max_distance; a.floor_z = r.floor_z;
    a.step_size = r.step_size; a.options = r.options; a.w = r.w; a.h = r.h; a.out = r.out;
    a.eval_count = r.eval_count;
    if (prog_space == 0) return cc_jit_launch_render(prog, ray ? CC_SINK_RAY : CC_SINK_BITMAP, a, stream, dev_index);
    cc_launch_cfg cfg{1, prog_space};
    const size_t smem = cc_eval_smem_bytes(cfg, a.n_slots, a.code_words);
    return prog_space == 1 ? launch_render<0>(ray != 0, a, smem, (cudaStream_t)stream)
                           : launch_render<1>(ray != 0, a, smem, (cudaStream_t)stream);
}

// ---- hierarchy helper kernels (float64 host math of the reference, moved on device) ----------

// subdivision.py:55-65: shifted_corner = (int_corner + int_step/2) * resolution + origin,
// rounded to fp32 per block by Vector.as_float4() (util/geometry.py:98-99).
__global__ void cc_make_blocks_subdiv_kernel(const int64_t *__restrict__ corners, uint32_t n, cc_level_geom g,
                                             cc_block_desc *__restrict__ out)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double x = __dadd_rn((double)corners[3 * i + 0], g.half_cell);
    double y = __dadd_rn((double)corners[3 * i + 1], g.half_cell);
    double z = __dadd_rn((double)corners[3 * i + 2], g.dimension == 3 ? g.half_cell : 0.0);
    cc_block_desc b;
    b.cx = (float)__dadd_rn(__dmul_rn(x, g.resolution), g.ox);
    b.cy = (float)__dadd_rn(__dmul_rn(y, g.resolution), g.oy);
    b.cz = (float)__dadd_rn(__dmul_rn(z, g.resolution), g.oz);
    b.pad = 0;
    out[i] = b;
}

// subdivision.py:91-94: child int corner = (i,j,k) * int_step + parent int corner.
// With world > 1 hit h goes to rank h % world (round-robin deal of the first refined level).
__global__ void cc_expand_children_kernel(const int64_t *__restrict__ parents, const uint32_t *__restrict__ hit_block,
                                          const uchar4 *__restrict__ hit_xyz, uint32_t n_hits, int64_t int_step,
                                          uint32_t rank, uint32_t world, int64_t *__restrict__ out)
{
    uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= n_hits || (h % world) != rank) return;
    uint32_t o = h / world;
    uint32_t b = hit_block[h];
    uchar4 c = hit_xyz[h];
    out[3 * o + 0] = parents[3 * b + 0] + (int64_t)c.x * int_step;
    out[3 * o + 1] = parents[3 * b + 1] + (int64_t)c.y * int_step;
    out[3 * o + 2] = parents[3 * b + 2] + (int64_t)c.z * int_step;
}

// mass_properties.py:86: shifted_corner = box_corner + box_step / 2 (float64), then as_float4()
__global__ void cc_mass_make_blocks_kernel(const double *__restrict__ corners, uint32_t n, double half,
                                           cc_block_desc *__restrict__ out)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    cc_block_desc b;
    b.cx = (float)__dadd_rn(corners[3 * i + 0], half);
    b.cy = (float)__dadd_rn(corners[3 * i + 1], half);
    b.cz = (float)__dadd_rn(corners[3 * i + 2], half);
    b.pad = 0;
    out[i] = b;
}

// mass_properties.py:154-157: child corner = Vector(i,j,k) * s + box_corner (float64).  With mask arrays (the assembly's
// hierarchy, cc_assembly.cu) the hit's two part masks go to the child block too.
__global__ void cc_mass_expand_children_kernel(const double *__restrict__ parents,
                                               const uint32_t *__restrict__ hit_block,
                                               const uchar4 *__restrict__ hit_xyz, uint32_t n_hits, double s,
                                               uint32_t rank, uint32_t world, double *__restrict__ out,
                                               const uint2 *__restrict__ hit_masks, uint2 *__restrict__ out_masks)
{
    uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= n_hits || (h % world) != rank) return;
    uint32_t o = h / world;
    uint32_t b = hit_block[h];
    uchar4 c = hit_xyz[h];
    out[3 * o + 0] = __dadd_rn(__dmul_rn((double)c.x, s), parents[3 * b + 0]);
    out[3 * o + 1] = __dadd_rn(__dmul_rn((double)c.y, s), parents[3 * b + 1]);
    out[3 * o + 2] = __dadd_rn(__dmul_rn((double)c.z, s), parents[3 * b + 2]);
    if (hit_masks) out_masks[o] = hit_masks[h];
}

// mass_properties.py:119-148: per block, index sums -> the ten integrals, in float64 with the
// reference's expression order.  The reference then adds the blocks up with a Kahan sum in job
// order; here every block's ten values go into an EXACT accumulator instead, so that the total
// does not depend on the order of the blocks, on how a level is chunked, or on how the hierarchy
// is dealt to GPUs and ranks: value i is truncated to a multiple of 2^q.e[i] (a quantum ~2^-97 of
// a bound on the integral, cc_api.cpp mass_quanta()), the 128-bit integer is cut into four 32-bit
// limbs, limbs are summed as signed 64-bit integers (warp shuffle tree, one atomic per warp and
// limb).  Integer addition is associative, so one GPU, eight GPUs in one process and eight ranks
// with an int64 all-reduce produce the same bits.
__device__ __forceinline__ void cc_to_limbs(double v, int quantum_exp, long long (&limb)[4], unsigned &overflow)
{
    const long long bits = __double_as_longlong(v);
    int ex = (int)((bits >> 52) & 0x7ff);
    unsigned long long m = (unsigned long long)bits & ((1ull << 52) - 1);
    if (ex == 0) ex = 1; else m |= 1ull << 52;  // value = m * 2^(ex - 1075)
    const int sh = (ex - 1075) - quantum_exp;
    unsigned __int128 t = 0;
    if (ex == 0x7ff || sh > 70) {  // inf / nan / beyond the stated bound
        if (m != 0 || ex == 0x7ff) overflow = 1u;
    } else if (sh >= 0) {
        t = (unsigned __int128)m << sh;
    } else if (sh > -64) {
        t = (unsigned __int128)(m >> (-sh));
    }
    const long long sign = bits < 0 ? -1 : 1;
#pragma unroll
    for (int k = 0; k < 4; ++k) limb[k] = sign * (long long)((unsigned long long)(t >> (32 * k)) & 0xffffffffull);
}

// Several sets of sums per block (an assembly's parts and pairs): set blockIdx.y of block b is at
// sums + b * set_stride + 10 * blockIdx.y and goes into accumulator acc + 41 * blockIdx.y.  One set: stride 10.
__global__ void __launch_bounds__(256) cc_mass_integrals_kernel(const double *__restrict__ corners,
                                                                const uint32_t *__restrict__ sums,
                                                                uint32_t n_blocks, double s, cc_mass_quanta qe,
                                                                unsigned long long *__restrict__ acc, uint32_t set_stride)
{
    const uint32_t b = blockIdx.x * 256u + threadIdx.x;
    sums += 10u * blockIdx.y;
    acc += 41u * blockIdx.y;
    const double s2 = __dmul_rn(s, s);
    const double s3 = __dmul_rn(s, s2);
    const double half = __ddiv_rn(s, 2.0);
    const double s2_12 = __ddiv_rn(s2, 12.0);
    double v[10];
#pragma unroll
    for (int i = 0; i < 10; ++i) v[i] = 0.0;
    if (b < n_blocks && sums[(size_t)b * set_stride + 9] != 0) {
        const uint32_t *q = sums + (size_t)b * set_stride;
        const double sxx = q[0], sxy = q[1], sxz = q[2], sx = q[3], syy = q[4], syz = q[5], sy = q[6],
                     szz = q[7], sz = q[8], n = q[9];
        const double bx = __dadd_rn(corners[3 * b + 0], half);
        const double by = __dadd_rn(corners[3 * b + 1], half);
        const double bz = __dadd_rn(corners[3 * b + 2], half);
        const double tx = s * sx, ty = s * sy, tz = s * sz;
        const double txx = s2 * sxx, tyy = s2 * syy, tzz = s2 * szz;
        const double txy = s2 * sxy, txz = s2 * sxz, tyz = s2 * syz;
        v[0] = s3 * n;
        v[1] = s3 * (n * bx + tx);
        v[2] = s3 * (n * by + ty);
        v[3] = s3 * (n * bz + tz);
        v[4] = s3 * (n * (bx * bx + s2_12) + 2.0 * bx * tx + txx);
        v[5] = s3 * (n * (by * by + s2_12) + 2.0 * by * ty + tyy);
        v[6] = s3 * (n * (bz * bz + s2_12) + 2.0 * bz * tz + tzz);
        v[7] = s3 * (n * bx * by + bx * ty + by * tx + txy);
        v[8] = s3 * (n * bx * bz + bx * tz + bz * tx + txz);
        v[9] = s3 * (n * by * bz + by * tz + bz * ty + tyz);
    }
    unsigned overflow = 0;
    const uint32_t lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        long long limb[4];
        cc_to_limbs(v[i], qe.e[i], limb, overflow);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            long long x = limb[k];
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) x += __shfl_down_sync(0xffffffffu, x, d);
            if (lane == 0 && x != 0) atomicAdd(acc + 4 * i + k, (unsigned long long)x);
        }
    }
    if (__any_sync(0xffffffffu, overflow != 0) && lane == 0) atomicAdd(acc + 40, 1ull);
}

int cc_launch_make_blocks_subdiv(const int64_t *d_int_corners, uint32_t n, cc_level_geom g,
                                 cc_block_desc *d_blocks, void *stream)
{
    if (!n) return 0;
    cc_make_blocks_subdiv_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(d_int_corners, n, g, d_blocks);
    return (int)cudaGetLastError();
}

int cc_launch_expand_children(const int64_t *d_parent_corners, const uint32_t *d_hit_block,
                              const uint8_t *d_hit_xyz, uint32_t n_hits, int64_t int_step, uint32_t rank,
                              uint32_t world, int64_t *d_child_corners, void *stream)
{
    if (!n_hits) return 0;
    cc_expand_children_kernel<<<(n_hits + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        d_parent_corners, d_hit_block, reinterpret_cast<const uchar4 *>(d_hit_xyz), n_hits, int_step, rank,
        world, d_child_corners);
    return (int)cudaGetLastError();
}

int cc_launch_mass_make_blocks(const double *d_corners, uint32_t n, double s, cc_block_desc *d_blocks,
                               void *stream)
{
    if (!n) return 0;
    cc_mass_make_blocks_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(d_corners, n, s / 2, d_blocks);
    return (int)cudaGetLastError();
}

int cc_launch_mass_expand_children(const double *d_parent_corners, const uint32_t *d_hit_block,
                                   const uint8_t *d_hit_xyz, uint32_t n_hits, double s, uint32_t rank,
                                   uint32_t world, double *d_child_corners, void *stream,
                                   const uint32_t *d_hit_masks, uint32_t *d_child_masks)
{
    if (!n_hits) return 0;
    cc_mass_expand_children_kernel<<<(n_hits + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        d_parent_corners, d_hit_block, reinterpret_cast<const uchar4 *>(d_hit_xyz), n_hits, s, rank, world,
        d_child_corners, reinterpret_cast<const uint2 *>(d_hit_masks), reinterpret_cast<uint2 *>(d_child_masks));
    return (int)cudaGetLastError();
}

int cc_launch_mass_integrals(const double *d_corners, const uint32_t *d_sums, uint32_t n_blocks, double s,
                             cc_mass_quanta q, unsigned long long *d_limbs, void *stream, uint32_t n_sets)
{
    if (!n_blocks) return 0;
    const dim3 grid((n_blocks + 255) / 256, n_sets);
    cc_mass_integrals_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_corners, d_sums, n_blocks, s, q, d_limbs, 10u * n_sets);
    return (int)cudaGetLastError();
}
