// Mass properties of every part of an assembly and of every pair's overlap, in one hierarchy pass (DESIGN.md 4.11).
// The level loop is mass_properties' (cc_api.cpp assembly_share); each block also carries two part masks, `eval` (the
// parts undecided at its parent cell) and `inside` (the parts decided inside at an ancestor cell).  A CTA evaluates the
// parts of `eval` one after the other on the interpreter, each with its own microcode staged in shared memory, classifies
// every cell per part with the MASS sink's comparisons, adds the cells newly inside a part to the part's sums and to the
// sums of the pairs they complete, and lists the cells still near some part as child blocks.  Compile with -fmad=false.
#include <cuda_runtime.h>
#include <stdint.h>

#include "cc_interp.cuh"
#include "cc_body.cuh"

// the set of pair {p < q} among n parts: after the n parts, pairs in lexicographic order
CC_DEV uint32_t cc_pair_set(uint32_t n, uint32_t p, uint32_t q) { return n + p * n - p * (p + 1u) / 2u + (q - p - 1u); }

// the warp's ten sums into dst: REDUX across the warp, one atomic per warp and moment (as the MASS sink)
CC_DEV void cc_flush_moments(uint32_t *dst, const uint32_t (&sum)[10])
{
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t w = __reduce_add_sync(0xffffffffu, sum[i]);
        if ((threadIdx.x & 31u) == 0 && w) atomicAdd(dst + i, w);
    }
}

// blocks x linear tiles of CC_THREADS x 2 cells in ticket order, as cc_kernel_body
__global__ void __launch_bounds__(CC_THREADS) cc_assembly_kernel(const cc_assembly_args A)
{
    constexpr int PTS = 2;
    typedef float2 V;
    extern __shared__ float4 smem4[];  // [max_slots][PTS][CC_THREADS] register slots, then one part's microcode
    __shared__ uint32_t s_tile;
    const cc_eval_args &a = A.a;
    uint32_t *s_code = reinterpret_cast<uint32_t *>(smem4 + (size_t)A.max_slots * PTS * CC_THREADS);
    if (threadIdx.x == 0) s_tile = atomicAdd(a.ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile, block = tile / a.tiles_per_block, tile_in_block = tile - block * a.tiles_per_block;
    const cc_block_desc bd = a.blocks[block];
    const uint2 masks = reinterpret_cast<const uint2 *>(A.masks)[block];  // CTA-uniform
    const uint32_t eval = masks.x, inside = masks.y;

    uint32_t ix[PTS], iy[PTS], iz[PTS];
    float gx[PTS], gy[PTS], gz[PTS];
    bool valid[PTS];
#pragma unroll
    for (int j = 0; j < PTS; ++j) cc_tile_cell<PTS>(a, tile_in_block, j, bd.cx, bd.cy, bd.cz, ix[j], iy[j], iz[j], gx[j], gy[j], gz[j], valid[j]);
    const V vx[1] = {cc_pack<V>(gx)}, vy[1] = {cc_pack<V>(gy)}, vz[1] = {cc_pack<V>(gz)};

    // per cell: the parts it is newly inside of, and the parts it is near
    uint32_t now[PTS] = {0u, 0u}, near[PTS] = {0u, 0u};
    for (uint32_t rest = eval; rest; rest &= rest - 1u) {
        const uint32_t k = (uint32_t)__ffs((int)rest) - 1u;
        __syncthreads();  // no warp still reads the previous part's microcode
        cc_stage_code(A.part[k].code, A.part[k].code_words, s_code);
        cc_val<V> L[1];
        cc_interpret<PTS, 1>(Prog<1>{s_code}, smem4, vx, vy, vz, L);
#pragma unroll
        for (int j = 0; j < PTS; ++j) {
            const float v = cc_lane_get(L[0], j).w;
            const bool in = valid[j] && (v <= -a.threshold);       // mass_properties.cl:31
            const bool nr = valid[j] && !in && (v < a.threshold);  // mass_properties.cl:43
            now[j] |= (in ? 1u : 0u) << k;
            near[j] |= (nr ? 1u : 0u) << k;
        }
    }

    const uint32_t n = A.n_parts, n_sets = n + n * (n - 1u) / 2u;
    uint32_t *sums = A.sums + (size_t)block * n_sets * 10u;
    const uint32_t warp_now = __reduce_or_sync(0xffffffffu, now[0] | now[1]);
    for (uint32_t rest = warp_now; rest; rest &= rest - 1u) {
        const uint32_t k = (uint32_t)__ffs((int)rest) - 1u;
        uint32_t sum[10] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
#pragma unroll
        for (int j = 0; j < PTS; ++j)
            if ((now[j] >> k) & 1u) cc_add_moments(sum, ix[j], iy[j], iz[j]);
        cc_flush_moments(sums + 10u * k, sum);
    }
    // Pair {p, q} gets a cell when one of them is newly inside and the other newly inside or inside at an ancestor: the
    // iteration (p, q) takes the cells with p newly inside and q in the cell's inside set, unless q is newly inside too
    // and q < p (that cell belongs to the iteration (q, p)).  Warp-uniform loops; nothing to do without two parts.
    const uint32_t warp_in = warp_now | inside;
    if (warp_now && (warp_in & (warp_in - 1u))) {
        for (uint32_t rp = warp_now; rp; rp &= rp - 1u) {
            const uint32_t p = (uint32_t)__ffs((int)rp) - 1u;
            for (uint32_t rq = warp_in & ~(1u << p); rq; rq &= rq - 1u) {
                const uint32_t q = (uint32_t)__ffs((int)rq) - 1u;
                bool pair[PTS];
#pragma unroll
                for (int j = 0; j < PTS; ++j)
                    pair[j] = ((now[j] >> p) & 1u) && (((now[j] | inside) >> q) & 1u) && (!((now[j] >> q) & 1u) || p < q);
                if (!__any_sync(0xffffffffu, pair[0] || pair[1])) continue;
                uint32_t sum[10] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
#pragma unroll
                for (int j = 0; j < PTS; ++j)
                    if (pair[j]) cc_add_moments(sum, ix[j], iy[j], iz[j]);
                cc_flush_moments(sums + 10u * cc_pair_set(n, min(p, q), max(p, q)), sum);
            }
        }
    }
    // the leaf level runs with threshold 0: no cell can be near (as the MASS sink, cc_kernel_body)
    if (a.threshold == 0.0f) return;
    bool hit[PTS];
    uint32_t pos[PTS];
#pragma unroll
    for (int j = 0; j < PTS; ++j) hit[j] = near[j] != 0u;
    cc_tile_rank<PTS>(a, tile, hit, pos);
#pragma unroll
    for (int j = 0; j < PTS; ++j) {
        if (hit[j]) {
            reinterpret_cast<uchar4 *>(a.list)[pos[j]] = make_uchar4((unsigned char)ix[j], (unsigned char)iy[j], (unsigned char)iz[j], 0);
            a.list_block[pos[j]] = block;
            reinterpret_cast<uint2 *>(A.hit_masks)[pos[j]] = make_uint2(near[j], inside | now[j]);
        }
    }
}

int cc_launch_assembly(const cc_assembly_args &A, size_t smem, void *stream)
{
    const uint32_t grid = A.a.n_blocks * A.a.tiles_per_block;
    if (grid == 0) return 0;
    cudaError_t e = cudaFuncSetAttribute(cc_assembly_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    cc_assembly_kernel<<<grid, CC_THREADS, smem, (cudaStream_t)stream>>>(A);
    return (int)cudaGetLastError();
}
