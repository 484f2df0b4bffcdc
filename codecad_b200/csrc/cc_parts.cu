// Part culling on the INTERPRETER tier (DESIGN.md 4.9): what cc_jit.cpp generates as straight-line code
// with `if (mask & bit)` blocks, done by walking the loader's segment table (cc_internal.h cc_parts) —
// so that an assembly is evaluated brick by brick with only the parts that can matter from its very
// first launch, before NVRTC has produced the specialised pair.  Same bricks (8 x 8 x 16 cells), same
// mask rule, same bits.  The microcode is staged in shared memory (this translation unit has no use
// for the __constant__ window).  Compile with -fmad=false.
#include <cuda_runtime.h>
#include <stdint.h>

#include "cc_interp.cuh"
#include "cc_body.cuh"

struct cc_parts_interp_args {
    cc_eval_args a;
    const uint32_t *table;
    uint32_t n_bricks;
};

CC_DEV const uint32_t *ccp_stage(const cc_eval_args &a, float4 *smem4, int pts)
{
    uint32_t *s_code = reinterpret_cast<uint32_t *>(smem4 + (size_t)a.n_slots * pts * CC_THREADS);
    cc_stage_code(a.code, a.code_words, s_code);
    return s_code;
}

// one thread per brick: every part at the brick centre -> the brick's mask (rule: cc_body.cuh cc_part_centers_body)
__global__ void __launch_bounds__(CC_THREADS) cc_parts_centers_kernel(const cc_parts_interp_args A)
{
    extern __shared__ float4 smem4[];
    const cc_eval_args &a = A.a;
    const Prog<1> P{ccp_stage(a, smem4, 1)};
    const uint32_t n_parts = A.table[0];
    const uint32_t *ranges = A.table + 2 + n_parts;
    const uint32_t brick = blockIdx.x * CC_THREADS + threadIdx.x;
    uint32_t x0, y0, z0;
    cc_brick_of(a, min(brick, A.n_bricks - 1u), x0, y0, z0);
    const float gx[1] = {cc_fma(a.step, (float)(x0 + a.x_offset) + 0.5f * (CC_BRICK_X - 1), a.cx)};
    const float gy[1] = {cc_fma(a.step, (float)y0 + 0.5f * (CC_BRICK_Y - 1), a.cy)};
    const float gz[1] = {cc_fma(a.step, (float)z0 + 0.5f * (CC_BRICK_Z - 1), a.cz)};
    const float r = fabsf(a.step) * (0.5f * 1.0001f) *
                    sqrtf((float)((CC_BRICK_X - 1) * (CC_BRICK_X - 1) + (CC_BRICK_Y - 1) * (CC_BRICK_Y - 1) + (CC_BRICK_Z - 1) * (CC_BRICK_Z - 1)));
    float w[32];
    float upper = __int_as_float(0x7f800000);
    for (uint32_t k = 0; k < n_parts; ++k) {  // (uniform: every thread walks the same runs)
        cc_val<float> L[1];
        L[0] = cc_val<float>{0.f, 0.f, 0.f, 0.f};
        cc_interpret<1, 1, true>(P, smem4, gx, gy, gz, L, ranges[2 * k], ranges[2 * k + 1]);
        w[k] = L[0].w;
        upper = fminf(upper, L[0].w + (__uint_as_float(A.table[2 + k]) * r + a.part_slack));
    }
    uint32_t mask = 0;
    for (uint32_t k = 0; k < n_parts; ++k)
        if (!(w[k] - (__uint_as_float(A.table[2 + k]) * r + a.part_slack) > upper)) mask |= 1u << k;
    if (brick < A.n_bricks) a.part_masks[brick] = mask;
}

// one CTA of 128 threads x 2 points per QUARTER brick (two x-planes of 8 x 16 cells): walk the segment table
__global__ void __launch_bounds__(CC_THREADS) cc_parts_eval_kernel(const cc_parts_interp_args A)
{
    typedef float2 V;
    extern __shared__ float4 smem4[];
    const cc_eval_args &a = A.a;
    const Prog<1> P{ccp_stage(a, smem4, 2)};
    const uint32_t brick = blockIdx.x >> 2, quarter = blockIdx.x & 3u;
    const uint32_t mask = a.part_masks[brick];
    uint32_t x0, y0, z0;
    cc_brick_of(a, brick, x0, y0, z0);
    const uint32_t tid = threadIdx.x;
    uint32_t ix[2], iy[2], iz[2];
    float gx[2], gy[2], gz[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const uint32_t c = (uint32_t)j * CC_THREADS + tid;  // 256 cells: z fastest (16), y (8), x (2)
        ix[j] = x0 + 2u * quarter + (c >> 7);
        iy[j] = y0 + ((c >> 4) & 7u);
        iz[j] = z0 + (c & 15u);
        gx[j] = cc_fma(a.step, (float)(ix[j] + a.x_offset), a.cx);
        gy[j] = cc_fma(a.step, (float)iy[j], a.cy);
        gz[j] = cc_fma(a.step, (float)iz[j], a.cz);
    }
    V vx[1] = {make_float2(gx[0], gx[1])}, vy[1] = {make_float2(gy[0], gy[1])}, vz[1] = {make_float2(gz[0], gz[1])};
    cc_val<V> L[1];
    L[0] = cc_val<V>{vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f)};
    const uint32_t n_parts = A.table[0], n_seg = A.table[1];
    const uint32_t *seg = A.table + 2 + 3 * n_parts;
    for (uint32_t s = 0; s < n_seg; ++s, seg += 4) {
        const uint32_t kind = seg[0];
        if (kind == CC_SEG_UNION) {
            if ((mask & seg[2]) && (mask & seg[3])) {
                cc_interpret<2, 1, true>(P, smem4, vx, vy, vz, L, seg[1], seg[1] + CC_LEN_0);
            } else {  // the survivor is already the running value; the union's store still happens
                const uint32_t dst = CC_HDR_DST(P.u(seg[1]));
                if (dst != CC_SLOT_NONE) cc_slot_store(smem4 + tid + (size_t)dst * 2 * CC_THREADS, L[0]);
            }
        } else if (kind == CC_SEG_ALWAYS || (mask & seg[3])) {
            cc_interpret<2, 1, true>(P, smem4, vx, vy, vz, L, seg[1], seg[2]);
        }
    }
    float4 *out = reinterpret_cast<float4 *>(a.out);
#pragma unroll
    for (int j = 0; j < 2; ++j)
        if (ix[j] < a.nx && iy[j] < a.ny && iz[j] < a.nz)
            __stcs(out + ((size_t)ix[j] * a.ny + iy[j]) * a.nz + iz[j], cc_lane_get(L[0], j));  // INDEX3
}

size_t cc_parts_smem_bytes(uint32_t n_slots, uint32_t code_words, int pts)
{
    return (size_t)n_slots * pts * CC_THREADS * sizeof(float4) + (size_t)code_words * 4;
}

// cost of every brick layer (8 x-planes) of a dense grid from its bricks' part masks: sum over the bricks of the layer of
// base + sum of the weights of the parts the brick keeps (load balancing of x-slabs, cc_grid_eval_cost_profile)
__global__ void __launch_bounds__(256) cc_layer_cost_kernel(const uint32_t *__restrict__ masks, uint32_t bricks_per_layer, cc_layer_weights w,
                                                            double *__restrict__ out)
{
    __shared__ double s_sum[256];
    const uint32_t *m = masks + (size_t)blockIdx.x * bricks_per_layer;
    double sum = 0.0;
    for (uint32_t i = threadIdx.x; i < bricks_per_layer; i += 256) {
        uint32_t bits = m[i];
        float c = w.base;
        while (bits) {
            c += w.part[__ffs((int)bits) - 1];
            bits &= bits - 1u;
        }
        sum += (double)c;
    }
    s_sum[threadIdx.x] = sum;
    __syncthreads();
    for (int d = 128; d > 0; d >>= 1) {
        if ((int)threadIdx.x < d) s_sum[threadIdx.x] += s_sum[threadIdx.x + d];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[blockIdx.x] = s_sum[0];
}

int cc_launch_layer_cost(const uint32_t *d_masks, uint32_t n_layers, uint32_t bricks_per_layer, const cc_layer_weights &w, double *d_out,
                         void *stream)
{
    if (n_layers == 0) return 0;
    cc_layer_cost_kernel<<<n_layers, 256, 0, (cudaStream_t)stream>>>(d_masks, bricks_per_layer, w, d_out);
    return (int)cudaGetLastError();
}

int cc_launch_parts_interp(const cc_eval_args &a, const uint32_t *d_table, uint32_t n_bricks, void *stream, bool centers_only)
{
    if (n_bricks == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    cc_parts_interp_args A{a, d_table, n_bricks};
    size_t smem = cc_parts_smem_bytes(a.n_slots, a.code_words, 1);
    cudaError_t e = cudaFuncSetAttribute(cc_parts_centers_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    cc_parts_centers_kernel<<<(n_bricks + CC_THREADS - 1) / CC_THREADS, CC_THREADS, smem, st>>>(A);
    e = cudaGetLastError();
    if (e != cudaSuccess || centers_only) return (int)e;
    smem = cc_parts_smem_bytes(a.n_slots, a.code_words, 2);
    e = cudaFuncSetAttribute(cc_parts_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    cc_parts_eval_kernel<<<n_bricks * 4u, CC_THREADS, smem, st>>>(A);
    return (int)cudaGetLastError();
}
