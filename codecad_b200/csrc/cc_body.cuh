// The part of the evaluation kernels that does not depend on HOW a point is evaluated:
// tile -> cell indices -> grid coordinates, then one of the four sinks (dense float4 store,
// PyMCubes store, ordered classification list, mass-property sums + list).  Shared by the
// microcode interpreter (cc_kernels.cu) and the NVRTC scene-specialised kernels (cc_jit.cpp),
// so that both produce bit-identical coordinates, layouts and list orders.
#ifndef CC_BODY_CUH
#define CC_BODY_CUH

#include "cc_device_types.h"
#include "cc_math.cuh"

#include "cc_scan.cuh"

// EVAL: functor  void operator()(const V (&gx)[G], const V (&gy)[G], const V (&gz)[G], cc_val<V> (&L)[G])
// with V, G = cc_pts<PTS> (cc_math.cuh): for PTS >= 2 the points j = 2g, 2g+1 are the two lanes
// of packed vector g.
// POINTS: the launch evaluates a list of points (a.points) instead of grid coordinates; a
// compile-time switch so that the grid kernels carry nothing for it (a run-time branch cost the
// 64-register specialised kernel 3.5 % more instructions).
// optional hook: a functor with locate(a, tile, block, ix, iy, iz) is told, before it is called, which cells of which
// tile and block the thread evaluates (the tile's part mask; the column kernels look up their columns, cc_col_locate)
template <class EVAL, class... T> CC_DEV void cc_eval_locate_(long, EVAL &, const T &...) {}
template <class EVAL, class... T>
CC_DEV auto cc_eval_locate_(int, EVAL &e, const T &...t) -> decltype(e.locate(t...), void())
{
    e.locate(t...);
}

// Point j of a thread of a linear tile of the block with corner (cx, cy, cz): the cell
// tile_in_block * CC_THREADS * PTS + j * CC_THREADS + tid in INDEX3 order (0 past the block's last cell, where `valid`
// is false; returned) and its fp32 grid coordinates.  Every body over blocks x linear tiles takes its points from here
// (cc_kernel_body, cc_assembly.cu): results that must agree bit for bit across them rest on these lines.
template <int PTS>
CC_DEV uint32_t cc_tile_cell(const cc_eval_args &a, uint32_t tile_in_block, int j, float cx, float cy, float cz, uint32_t &ix,
                             uint32_t &iy, uint32_t &iz, float &gx, float &gy, float &gz, bool &valid)
{
    const uint32_t cells = a.nx * a.ny * a.nz, nyz = a.ny * a.nz;
    uint32_t c = tile_in_block * (CC_THREADS * PTS) + j * CC_THREADS + threadIdx.x;
    valid = c < cells;
    c = valid ? c : 0u;
    ix = c / nyz;
    const uint32_t r = c - ix * nyz;
    iy = r / a.nz;
    iz = r - iy * a.nz;
    // grid_eval.cl:13,31: corner + step * convert_float(id), one FMA per axis
    gx = cc_fma(a.step, (float)(ix + a.x_offset), cx);
    gy = cc_fma(a.step, (float)iy, cy);
    gz = cc_fma(a.step, (float)iz, cz);
    return c;
}

// A cell's ten index products, added to the MASS sink's sums: mass_properties.cl:34-41, order xx,xy,xz,x,yy,yz,y,zz,z,n
CC_DEV void cc_add_moments(uint32_t (&sum)[10], uint32_t x, uint32_t y, uint32_t z)
{
    sum[0] += x * x; sum[1] += x * y; sum[2] += x * z; sum[3] += x;
    sum[4] += y * y; sum[5] += y * z; sum[6] += y; sum[7] += z * z;
    sum[8] += z; sum[9] += 1u;
}

// Ordered compaction of a tile's hits (CTA-wide): the list position of every point j with hit[j], in cell order (j major,
// then warp, then lane) after the hits of all earlier tiles (ticket order, decoupled look-back on a.tile_status); the
// tile of the launch's last ticket writes the final list length to *a.counter.
template <int PTS>
CC_DEV void cc_tile_rank(const cc_eval_args &a, uint32_t tile, const bool (&hit)[PTS], uint32_t (&pos)[PTS])
{
    __shared__ uint32_t s_warp[PTS * (CC_THREADS / 32)];
    __shared__ uint32_t s_base;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t ballot[PTS];
#pragma unroll
    for (int j = 0; j < PTS; ++j) {
        ballot[j] = __ballot_sync(0xffffffffu, hit[j]);
        if (lane == 0) s_warp[j * (CC_THREADS / 32) + warp] = __popc(ballot[j]);
    }
    __syncthreads();
    if (warp == 0) {
        // exclusive scan of the PTS * 4 warp counts (<= 32 entries) with shuffles
        constexpr int NW = PTS * (CC_THREADS / 32);
        static_assert(NW <= 32, "the warp-count scan covers at most 32 entries");
        uint32_t v = (lane < NW) ? s_warp[lane] : 0u;
        uint32_t incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        if (lane < NW) s_warp[lane] = incl - v;
        uint32_t base = cc_lookback(a.tile_status, tile, total, a.counter);
        if (lane == 0) {
            s_base = base;
            if (tile == gridDim.x - 1) *a.counter = base + total;  // final list length
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < PTS; ++j) pos[j] = s_base + s_warp[j * (CC_THREADS / 32) + warp] + __popc(ballot[j] & ((1u << lane) - 1u));
}

template <int PTS, int SINK, class EVAL, bool POINTS = false>
CC_DEV void cc_kernel_body(const cc_eval_args &a, EVAL &eval)
{
    __shared__ uint32_t s_tile;

    const uint32_t tid = threadIdx.x;
    constexpr bool ORDERED = (SINK == CC_SINK_CLASSIFY || SINK == CC_SINK_MASS);
    // tile id: launch order for pure stores; ticket order where tiles wait on predecessors
    uint32_t tile = blockIdx.x;
    if (ORDERED) {
        if (tid == 0) s_tile = atomicAdd(a.ticket, 1u);
        __syncthreads();
        tile = s_tile;
    }
    const uint32_t block = tile / a.tiles_per_block;
    const uint32_t tile_in_block = tile - block * a.tiles_per_block;
    float cx = a.cx, cy = a.cy, cz = a.cz;
    if (a.blocks) {
        const cc_block_desc bd = a.blocks[block];
        cx = bd.cx; cy = bd.cy; cz = bd.cz;
    }
    const uint32_t cells = a.nx * a.ny * a.nz;  // <= 2^31 per launch (host checks)

    typedef typename cc_pts<PTS>::V V;
    constexpr int G = cc_pts<PTS>::G, NL = cc_lane<V>::N;
    float gx[PTS], gy[PTS], gz[PTS];
    uint32_t ix[PTS], iy[PTS], iz[PTS];
    bool valid[PTS];
#pragma unroll
    for (int j = 0; j < PTS; ++j) {
        const uint32_t c = cc_tile_cell<PTS>(a, tile_in_block, j, cx, cy, cz, ix[j], iy[j], iz[j], gx[j], gy[j], gz[j], valid[j]);
        if (POINTS) {
            const float4 p = reinterpret_cast<const float4 *>(a.points)[c];
            gx[j] = p.x; gy[j] = p.y; gz[j] = p.z;
        }
    }

    if (!POINTS) cc_eval_locate_(0, eval, a, tile, block, ix, iy, iz);
    float4 L[PTS];
    {
        V vx[G], vy[G], vz[G];
        cc_val<V> LV[G];
#pragma unroll
        for (int g = 0; g < G; ++g) {
            vx[g] = cc_pack<V>(gx + g * NL);
            vy[g] = cc_pack<V>(gy + g * NL);
            vz[g] = cc_pack<V>(gz + g * NL);
        }
        eval(vx, vy, vz, LV);
#pragma unroll
        for (int j = 0; j < PTS; ++j) L[j] = cc_lane_get(LV[j / NL], j % NL);
    }

    if (SINK == CC_SINK_FLOAT4) {
        float4 *out = reinterpret_cast<float4 *>(a.out) + (size_t)block * cells;
#pragma unroll
        for (int j = 0; j < PTS; ++j) {
            uint32_t c = tile_in_block * (CC_THREADS * PTS) + j * CC_THREADS + tid;
            if (valid[j]) __stcs(out + c, L[j]);  // INDEX3: z + nz*(y + ny*x) == linear cell index
        }
    } else if (SINK == CC_SINK_PYMCUBES) {
        float *out = reinterpret_cast<float *>(a.out) + (size_t)block * cells;
#pragma unroll
        for (int j = 0; j < PTS; ++j) {
            // grid_eval.cl:18: z + (x + (ny - y - 1) * nx) * nz
            size_t idx = (size_t)iz[j] + ((size_t)ix[j] + (size_t)(a.ny - iy[j] - 1) * a.nx) * a.nz;
            if (valid[j]) __stcs(out + idx, L[j].w);
        }
    } else {
        // ---- classification ----
        const uint32_t lane = tid & 31;
        bool hit[PTS];
        uint32_t sum[10];
#pragma unroll
        for (int i = 0; i < 10; ++i) sum[i] = 0;
#pragma unroll
        for (int j = 0; j < PTS; ++j) {
            const float v = L[j].w;
            if (SINK == CC_SINK_CLASSIFY) {
                hit[j] = valid[j] && (v > -a.threshold && v < a.threshold);  // subdivision.cl:25
            } else {
                const bool inside = valid[j] && (v <= -a.threshold);  // mass_properties.cl:31
                hit[j] = valid[j] && !inside && (v < a.threshold);    // mass_properties.cl:43
                if (inside) cc_add_moments(sum, ix[j], iy[j], iz[j]);
            }
        }
        if (SINK == CC_SINK_MASS) {
            // hierarchical reduction: REDUX across the warp, one atomic per warp and moment
            uint32_t *dst = a.sums + (a.blocks ? (size_t)block * 10 : 0);
#pragma unroll
            for (int i = 0; i < 10; ++i) {
                uint32_t w = __reduce_add_sync(0xffffffffu, sum[i]);
                if (lane == 0 && w) atomicAdd(dst + i, w);
            }
        }
        // The leaf level of mass_properties runs with threshold 0 (mass_properties.py:87-90): `inside` is
        // v <= -0 and a hit would need v < 0 on top of !inside — no cell can qualify, the list stays
        // empty, and the tile neither ranks nor waits for its predecessors.  (Warp-uniform: a launch
        // argument.)  The leaf launch is 98 % of a mass_properties call.
        if (SINK == CC_SINK_MASS && a.threshold == 0.0f) return;
        uint32_t pos[PTS];
        cc_tile_rank<PTS>(a, tile, hit, pos);
#pragma unroll
        for (int j = 0; j < PTS; ++j) {
            if (hit[j]) {
                reinterpret_cast<uchar4 *>(a.list)[pos[j]] =
                    make_uchar4((unsigned char)ix[j], (unsigned char)iy[j], (unsigned char)iz[j], 0);
                if (a.list_block) a.list_block[pos[j]] = block;
            }
        }
    }
}

// ---- part culling (DESIGN.md 4.9): the dense float4 grid in bricks of 8 x 8 x 16 cells ------------------
// One CTA of 512 threads x 2 points per brick (z fastest inside the brick: a warp's store is two 256-byte
// runs); bricks in z-fastest order.  EVAL carries the brick's part mask.
CC_DEV void cc_brick_of(const cc_eval_args &a, uint32_t brick, uint32_t &x0, uint32_t &y0, uint32_t &z0)
{
    const uint32_t nbz = (a.nz + CC_BRICK_Z - 1) / CC_BRICK_Z, nby = (a.ny + CC_BRICK_Y - 1) / CC_BRICK_Y;
    const uint32_t bz = brick % nbz, t = brick / nbz;
    z0 = bz * CC_BRICK_Z;
    y0 = (t % nby) * CC_BRICK_Y;
    x0 = (t / nby) * CC_BRICK_X;
}

template <int PTS, class EVAL>
CC_DEV void cc_kernel_body_bricks_at(const cc_eval_args &a, EVAL &eval, uint32_t brick)
{
    static_assert(PTS == 2 && CC_THREADS * PTS == CC_BRICK_X * CC_BRICK_Y * CC_BRICK_Z, "one brick per CTA");
    typedef typename cc_pts<PTS>::V V;
    uint32_t x0, y0, z0;
    cc_brick_of(a, brick, x0, y0, z0);
    const uint32_t tid = threadIdx.x;
    uint32_t ix[PTS], iy[PTS], iz[PTS];
    float gx[PTS], gy[PTS], gz[PTS];
#pragma unroll
    for (int j = 0; j < PTS; ++j) {
        const uint32_t c = (uint32_t)j * CC_THREADS + tid;  // cell of the brick: z fastest, then y, then x
        ix[j] = x0 + (c >> 7);
        iy[j] = y0 + ((c >> 4) & 7u);
        iz[j] = z0 + (c & 15u);
        // grid_eval.cl:13,31: corner + step * convert_float(id), one FMA per axis (same as cc_kernel_body)
        gx[j] = cc_fma(a.step, (float)(ix[j] + a.x_offset), a.cx);
        gy[j] = cc_fma(a.step, (float)iy[j], a.cy);
        gz[j] = cc_fma(a.step, (float)iz[j], a.cz);
    }
    V vx[1], vy[1], vz[1];
    cc_val<V> LV[1];
    vx[0] = cc_pack<V>(gx);
    vy[0] = cc_pack<V>(gy);
    vz[0] = cc_pack<V>(gz);
    eval(vx, vy, vz, LV);
    float4 *out = reinterpret_cast<float4 *>(a.out);
#pragma unroll
    for (int j = 0; j < PTS; ++j)
        if (ix[j] < a.nx && iy[j] < a.ny && iz[j] < a.nz)
            __stcs(out + ((size_t)ix[j] * a.ny + iy[j]) * a.nz + iz[j], cc_lane_get(LV[0], j));  // INDEX3
}

// ---- columns (DESIGN.md 4.10): what cannot see the grid's z is evaluated once per z-column -----------------
// Three kernels around two generated functors.  AHEAD runs, for every (x, y) column of the launch, the
// micro-ops that cannot depend on z and writes the values the rest of the program reads from them into the
// column buffer  float4 columns[nx * ny][CC_COL_VALUES];  LOOP is the rest of the program, run per
// cell by the brick kernel, which reads those values instead of computing them.  A column for which the
// run-time check of AHEAD::invariant() fails (cc_jit.cpp) flags its bricks; they are evaluated by the full
// walk in a third launch.
#ifndef CC_COL_VALUES
#define CC_COL_VALUES 1  // values per column record (the generated source defines it)
#endif
#ifndef CC_COL_AXIS
#define CC_COL_AXIS 2    // the grid axis the columns run along: the program is (mostly) invariant along it
#endif
// columns are numbered over the two other axes (u slow, v fast): z-columns by (x, y), y-columns by (x, z), x-columns by (y, z)
CC_DEV uint32_t cc_col_dim_u(const cc_eval_args &a) { return CC_COL_AXIS == 0 ? a.ny : a.nx; }
CC_DEV uint32_t cc_col_dim_v(const cc_eval_args &a) { return CC_COL_AXIS == 2 ? a.ny : a.nz; }
CC_DEV uint32_t cc_col_len(const cc_eval_args &a) { return CC_COL_AXIS == 0 ? a.nx : CC_COL_AXIS == 1 ? a.ny : a.nz; }
struct cc_col_ref {
    float4 *rec[2];  // the column record of each point of the thread's pair: float4 rec[CC_COL_VALUES]
    bool ok[2];
};
template <class V> CC_DEV void cc_col_store(const cc_col_ref &r, uint32_t k, const cc_val<V> &v)
{
#pragma unroll
    for (int l = 0; l < cc_lane<V>::N; ++l)
        if (r.ok[l]) r.rec[l][k] = cc_lane_get(v, l);
}
template <class V> CC_DEV cc_val<V> cc_col_load(const cc_col_ref &r, uint32_t k)
{
    cc_val<V> v;
#pragma unroll
    for (int l = 0; l < cc_lane<V>::N; ++l) cc_lane_put(v, l, __ldg(r.rec[l] + k));
    return v;
}
// The brick kernel pairs a thread's two cells along the columns' axis (CC_COL_PAIR), so both read one record:
// one load, and the same value in both lanes.  0 keeps the brick order of cc_kernel_body_bricks_at.
#ifndef CC_COL_PAIR
#define CC_COL_PAIR 1
#endif
struct cc_col_one {
    const float4 *rec;  // the column record of both points of the thread's pair
};
template <class V> CC_DEV cc_val<V> cc_col_load(const cc_col_one &r, uint32_t k)
{
    const float4 c = __ldg(r.rec + k);
    cc_val<V> v;
#pragma unroll
    for (int l = 0; l < cc_lane<V>::N; ++l) cc_lane_put(v, l, c);
    return v;
}
#if CC_COL_PAIR
typedef cc_col_one cc_brick_col_ref;
#else
typedef cc_col_ref cc_brick_col_ref;
#endif
CC_DEV bool cc_same_bits(float a, float b) { return __float_as_uint(a) == __float_as_uint(b) && a == a; }
CC_DEV bool cc_same_bits(float2 a, float2 b) { return cc_same_bits(a.x, b.x) && cc_same_bits(a.y, b.y); }

// one thread per pair of columns 2t, 2t + 1
template <int PTS, class AHEAD>
CC_DEV void cc_column_profiles_body(const cc_eval_args &a, AHEAD &ahead)
{
    static_assert(PTS == 2, "two columns per thread");
    typedef typename cc_pts<PTS>::V V;
    const uint32_t dim_v = cc_col_dim_v(a), per_block = cc_col_dim_u(a) * dim_v, ncol = per_block * max(a.n_blocks, 1u),
                   t = blockIdx.x * CC_THREADS + threadIdx.x;
    const uint32_t last = cc_col_len(a) - 1u;
    float gx[PTS], gy[PTS], gz[PTS], gl[PTS];
    uint32_t col[PTS];
#pragma unroll
    for (int j = 0; j < PTS; ++j) {
        const uint32_t c = 2u * t + (uint32_t)j;
        ahead.cr.ok[j] = c < ncol;
        col[j] = min(c, ncol - 1u);  // (every thread evaluates: the ops vote across the warp)
        ahead.cr.rec[j] = reinterpret_cast<float4 *>(a.columns) + (size_t)col[j] * CC_COL_VALUES;
        const uint32_t block = col[j] / per_block, in_block = col[j] - block * per_block;
        const uint32_t u = in_block / dim_v, v = in_block - u * dim_v;
        const uint32_t ix = CC_COL_AXIS == 0 ? 0u : u, iy = CC_COL_AXIS == 0 ? u : CC_COL_AXIS == 1 ? 0u : v, iz = CC_COL_AXIS == 2 ? 0u : v;
        float cx = a.cx, cy = a.cy, cz = a.cz;
        if (a.blocks) {  // the block's own corner, as in cc_kernel_body
            const cc_block_desc bd = a.blocks[block];
            cx = bd.cx; cy = bd.cy; cz = bd.cz;
        }
        gx[j] = cc_fma(a.step, (float)(ix + a.x_offset), cx);
        gy[j] = cc_fma(a.step, (float)iy, cy);
        gz[j] = cc_fma(a.step, (float)iz, cz);
        gl[j] = CC_COL_AXIS == 0 ? cc_fma(a.step, (float)(last + a.x_offset), cx)
                                 : cc_fma(a.step, (float)last, CC_COL_AXIS == 1 ? cy : cz);
    }
    V vx[1], vy[1], vz[1], vl[1];
    vx[0] = cc_pack<V>(gx);
    vy[0] = cc_pack<V>(gy);
    vz[0] = cc_pack<V>(gz);
    vl[0] = cc_pack<V>(gl);
    if (a.column_flags) {
        const unsigned char bad = ahead.invariant(vx, vy, vz, vl) ? 0 : 1;
#pragma unroll
        for (int j = 0; j < PTS; ++j)
            if (ahead.cr.ok[j]) a.column_flags[col[j]] = bad;
    }
    ahead(vx, vy, vz);
}

// the columns of the cells a thread of cc_kernel_body evaluates (blocks x linear tiles); returns whether any column
// of the CTA's tile failed the run-time check (CTA-uniform: every thread calls it)
template <int PTS>
CC_DEV bool cc_col_locate(const cc_eval_args &a, uint32_t block, const uint32_t (&ix)[PTS], const uint32_t (&iy)[PTS],
                          const uint32_t (&iz)[PTS], cc_col_ref &cr)
{
    static_assert(PTS == 2, "two points per thread");
    const uint32_t dim_v = cc_col_dim_v(a), per_block = cc_col_dim_u(a) * dim_v;
    int flagged = 0;
#pragma unroll
    for (int j = 0; j < PTS; ++j) {
        const uint32_t u = CC_COL_AXIS == 0 ? iy[j] : ix[j], v = CC_COL_AXIS == 2 ? iy[j] : iz[j];
        const uint32_t col = block * per_block + u * dim_v + v;
        cr.rec[j] = reinterpret_cast<float4 *>(a.columns) + (size_t)col * CC_COL_VALUES;
        cr.ok[j] = true;
        if (a.column_flags) flagged |= a.column_flags[col];
    }
    return a.column_flags ? __syncthreads_or(flagged) != 0 : false;
}

// The runs of the column brick kernel.  The bricks of one set of columns form a stack along the columns' axis; a stack is
// cut into runs of a.brick_run bricks (the last one shorter).  Run `run` starts at brick `first` (its corner x0, y0, z0),
// holds `n` bricks, and its next brick is `stride` bricks further in the z-fastest brick order.
CC_DEV void cc_brick_run_of(const cc_eval_args &a, uint32_t run, uint32_t &first, uint32_t &n, uint32_t &stride, uint32_t &x0,
                            uint32_t &y0, uint32_t &z0)
{
    const uint32_t nbx = (a.nx + CC_BRICK_X - 1) / CC_BRICK_X, nby = (a.ny + CC_BRICK_Y - 1) / CC_BRICK_Y,
                   nbz = (a.nz + CC_BRICK_Z - 1) / CC_BRICK_Z;
    const uint32_t along = CC_COL_AXIS == 0 ? nbx : CC_COL_AXIS == 1 ? nby : nbz;
    const uint32_t per_stack = (along + a.brick_run - 1) / a.brick_run;
    const uint32_t stack = run / per_stack, start = (run - stack * per_stack) * a.brick_run;
    n = min(a.brick_run, along - start);
    // the stack's two other brick coordinates, numbered in the brick order (z fastest)
    const uint32_t other = CC_COL_AXIS == 2 ? nby : nbz, s1 = stack / other, s0 = stack - s1 * other;
    const uint32_t bx = CC_COL_AXIS == 0 ? start : s1, by = CC_COL_AXIS == 0 ? s1 : CC_COL_AXIS == 1 ? start : s0,
                   bz = CC_COL_AXIS == 2 ? start : s0;
    first = (bx * nby + by) * nbz + bz;
    stride = CC_COL_AXIS == 0 ? nby * nbz : CC_COL_AXIS == 1 ? nbz : 1u;
    x0 = bx * CC_BRICK_X;
    y0 = by * CC_BRICK_Y;
    z0 = bz * CC_BRICK_Z;
}

// The brick kernel of cc_kernel_body_bricks with the thread's columns at hand: the cells of a thread in the brick at
// (x0, y0, z0).  With CC_COL_PAIR the two cells of a thread differ only along the columns' axis (z-columns: z and z + 8, a warp's store is four 128-byte runs; y-columns:
// y and y + 4; x-columns: the brick order's x and x + 4 already), so they share one column record.
template <int PTS>
CC_DEV void cc_brick_col_cells(uint32_t x0, uint32_t y0, uint32_t z0, uint32_t (&ix)[PTS], uint32_t (&iy)[PTS], uint32_t (&iz)[PTS])
{
    const uint32_t tid = threadIdx.x;
#pragma unroll
    for (int j = 0; j < PTS; ++j) {
        const uint32_t c = (uint32_t)j * CC_THREADS + tid;
        ix[j] = x0 + (c >> 7);
        iy[j] = y0 + ((c >> 4) & 7u);
        iz[j] = z0 + (c & 15u);
        if (CC_COL_PAIR && CC_COL_AXIS == 2) {
            ix[j] = x0 + (tid >> 6);
            iy[j] = y0 + ((tid >> 3) & 7u);
            iz[j] = z0 + (tid & 7u) + 8u * (uint32_t)j;
        } else if (CC_COL_PAIR && CC_COL_AXIS == 1) {
            ix[j] = x0 + (tid >> 6);
            iy[j] = y0 + ((tid >> 4) & 3u) + 4u * (uint32_t)j;
            iz[j] = z0 + (tid & 15u);
        }
    }
}

// The lazy gradient of the column brick kernel (DESIGN.md 4.10): its per-cell body carries a distance and the id of the
// leaf it came from through the ops (the sweep), then the winning leaf of each cell is evaluated again in full and taken
// along its one path to the root (the replay, REPLAY::leaf).  0 keeps the eager body; CC_LAZY_CHECK=1 poisons a cell
// whose replayed .w differs in any bit from the sweep's.
#ifndef CC_LAZY_GRADIENT
#define CC_LAZY_GRADIENT 1
#endif
#ifndef CC_LAZY_CHECK
#define CC_LAZY_CHECK 0
#endif
// Both cells of the thread won by one leaf: one packed replay.  Otherwise one packed replay per leaf, each keeping its lane.
template <class REPLAY, class V, int G>
CC_DEV void cc_lazy_replay(const REPLAY &r, const V (&gx)[G], const V (&gy)[G], const V (&gz)[G], const V (&w)[G], const V (&id)[G],
                           cc_val<V> (&L)[G])
{
    static_assert(G * cc_lane<V>::N == 2, "two points per thread");
    constexpr int N = cc_lane<V>::N;
    const int k0 = (int)vlane(id[0], 0), k1 = (int)vlane(id[G - 1], N - 1);
    auto take = [&](const cc_val<V> (&T)[G], int j) {
        float4 t = cc_lane_get(T[j / N], j % N);
        const float sw = vlane(w[j / N], j % N);
        if (CC_LAZY_CHECK && __float_as_uint(t.w) != __float_as_uint(sw)) t.x = t.y = t.z = __uint_as_float(0x7fbadbadu);
        t.w = sw;
        cc_lane_put(L[j / N], j % N, t);
    };
    cc_val<V> T[G];
    r.leaf(k0, gx, gy, gz, T);
    take(T, 0);
    if (k1 != k0) r.leaf(k1, gx, gy, gz, T);
    take(T, 1);
}

// A CTA walks a run of bricks along the columns' axis (cc_brick_run_of).  The bricks of a run read the same columns, so
// the run's position, the thread's column record and the column flags are worked out once per run, and the run's part
// masks come in with one load into shared memory.  Per brick the cells' indices and coordinates are rebuilt from the
// brick's corner (a few integer ops and three FMAs per cell: cheaper than keeping them in registers across the per-cell
// body), then the mask, the per-cell body and the stores; the warps go through the run without waiting for each other.
// EVAL (the generated SceneTile): `loop` is the per-cell body, its part mask and its column reference; with
// EVAL::deferred its ops fold their range tests into `range` instead of voting per op (DESIGN.md 4.10), and a warp in
// which some lane flags evaluates its cells again with EVAL::full, the guarded full walk.
template <int PTS, class EVAL>
CC_DEV void cc_kernel_body_brick_columns(const cc_eval_args &a, EVAL &eval)
{
    static_assert(PTS == 2 && CC_THREADS * PTS == CC_BRICK_X * CC_BRICK_Y * CC_BRICK_Z, "one brick per CTA");
    static_assert(CC_BRICK_RUN_MAX <= CC_THREADS, "one thread loads each mask of a run");
    typedef typename cc_pts<PTS>::V V;
    __shared__ uint32_t s_mask[CC_BRICK_RUN_MAX];
    uint32_t first, n, stride, x0, y0, z0;
    cc_brick_run_of(a, blockIdx.x, first, n, stride, x0, y0, z0);
    const uint32_t tid = threadIdx.x;
    if (tid < n) s_mask[tid] = a.part_masks ? a.part_masks[first + tid * stride] : 0xffffffffu;
    uint32_t col[PTS];
    {
        uint32_t ix[PTS], iy[PTS], iz[PTS];
        cc_brick_col_cells<PTS>(x0, y0, z0, ix, iy, iz);
#pragma unroll
        for (int j = 0; j < PTS; ++j) {
            const uint32_t u = CC_COL_AXIS == 0 ? iy[j] : ix[j], v = CC_COL_AXIS == 2 ? iy[j] : iz[j];
            col[j] = min(u, cc_col_dim_u(a) - 1u) * cc_col_dim_v(a) + min(v, cc_col_dim_v(a) - 1u);  // (cells past the edge read a neighbour's column)
        }
    }
#if CC_COL_PAIR
    eval.loop.cr.rec = reinterpret_cast<const float4 *>(a.columns) + (size_t)col[0] * CC_COL_VALUES;
    const int col_flag = a.column_flags ? (int)a.column_flags[col[0]] : 0;
#else
#pragma unroll
    for (int j = 0; j < PTS; ++j) {
        eval.loop.cr.rec[j] = reinterpret_cast<float4 *>(a.columns) + (size_t)col[j] * CC_COL_VALUES;
        eval.loop.cr.ok[j] = true;
    }
    const int col_flag = a.column_flags ? (int)(a.column_flags[col[0]] | a.column_flags[col[1]]) : 0;
#endif
    // (also the barrier behind the masks' stores)
    if (__syncthreads_or(col_flag)) {
        // a column whose "invariant" micro-ops do see z in some bit: every brick of the run takes the full walk
        if (tid < 32) {
            uint32_t at = 0;
            if (tid == 0) {
                at = atomicAdd(a.brick_count, n);
                if (a.flagged_bricks) atomicAdd(a.flagged_bricks, (unsigned long long)n);
            }
            at = __shfl_sync(0xffffffffu, at, 0);
            for (uint32_t i = tid; i < n; i += 32) a.brick_list[at + i] = first + i * stride;
        }
        return;
    }
    for (uint32_t i = 0; i < n; ++i) {
        uint32_t ix[PTS], iy[PTS], iz[PTS];
        cc_brick_col_cells<PTS>(x0 + (CC_COL_AXIS == 0 ? i * CC_BRICK_X : 0u), y0 + (CC_COL_AXIS == 1 ? i * CC_BRICK_Y : 0u),
                                z0 + (CC_COL_AXIS == 2 ? i * CC_BRICK_Z : 0u), ix, iy, iz);
        float gx[PTS], gy[PTS], gz[PTS];
#pragma unroll
        for (int j = 0; j < PTS; ++j) {
            gx[j] = cc_fma(a.step, (float)(ix[j] + a.x_offset), a.cx);
            gy[j] = cc_fma(a.step, (float)iy[j], a.cy);
            gz[j] = cc_fma(a.step, (float)iz[j], a.cz);
        }
        eval.loop.mask = s_mask[i];
        V vx[1], vy[1], vz[1];
        cc_val<V> LV[1];
        vx[0] = cc_pack<V>(gx);
        vy[0] = cc_pack<V>(gy);
        vz[0] = cc_pack<V>(gz);
        uint32_t range = 0;
        eval(vx, vy, vz, LV, range);
        if (EVAL::deferred && __any_sync(0xffffffffu, cc_range_flagged(range))) {
            // some op of some lane had an operand outside its fast path's range: the warp's values are thrown away
            if ((tid & 31u) == 0 && a.check_fallbacks) atomicAdd(a.check_fallbacks, 1ull);
            eval.full(vx, vy, vz, LV);
        }
        float4 *out = reinterpret_cast<float4 *>(a.out);
#pragma unroll
        for (int j = 0; j < PTS; ++j)
            if (ix[j] < a.nx && iy[j] < a.ny && iz[j] < a.nz)
                __stcs(out + ((size_t)ix[j] * a.ny + iy[j]) * a.nz + iz[j], cc_lane_get(LV[0], j));  // INDEX3
    }
}

template <int PTS, class EVAL>
CC_DEV void cc_kernel_body_bricks(const cc_eval_args &a, EVAL &eval)
{
    cc_kernel_body_bricks_at<PTS>(a, eval, blockIdx.x);
}

// ---- part masks for the linear tiles of cc_kernel_body (the hierarchy sinks, blocks x tiles) -------------
// A tile is CC_THREADS * PTS consecutive cells of a block in INDEX3 order: inside one x-plane a run of whole
// y-rows (or a piece of one row); across x-planes every (y, z).  Its index box, conservative:
CC_DEV void cc_tile_bounds(const cc_eval_args &a, uint32_t tile_in_block, uint32_t tile_cells, float (&lo)[3], float (&hi)[3])
{
    const uint32_t cells = a.nx * a.ny * a.nz, nyz = a.ny * a.nz;
    const uint32_t c0 = min(tile_in_block * tile_cells, cells - 1u), c1 = min(c0 + tile_cells, cells) - 1u;
    const uint32_t x0 = c0 / nyz, x1 = c1 / nyz;
    uint32_t y0 = 0, y1 = a.ny - 1u, z0 = 0, z1 = a.nz - 1u;
    if (x0 == x1) {
        const uint32_t r0 = c0 - x0 * nyz, r1 = c1 - x0 * nyz;
        y0 = r0 / a.nz;
        y1 = r1 / a.nz;
        if (y0 == y1) {
            z0 = r0 - y0 * a.nz;
            z1 = r1 - y1 * a.nz;
        }
    }
    lo[0] = (float)(x0 + a.x_offset); hi[0] = (float)(x1 + a.x_offset);
    lo[1] = (float)y0; hi[1] = (float)y1;
    lo[2] = (float)z0; hi[2] = (float)z1;
}

// Tile-centre pass: thread t evaluates every part at the centres of the index boxes of tiles 2t and 2t + 1 and
// writes their masks (the rule of cc_part_centers_body with the box's own half diagonal).
template <int P, int PTS, class EVAL, class V>
CC_DEV void cc_tile_centers_body(const cc_eval_args &a, EVAL &eval, V *pw, const float *lip)
{
    const uint32_t n_tiles = a.tiles_per_block * a.n_blocks;
    const uint32_t t0 = 2u * (blockIdx.x * CC_THREADS + threadIdx.x);
    float gx[2], gy[2], gz[2], r[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const uint32_t tile = min(t0 + (uint32_t)j, n_tiles - 1u);
        const uint32_t block = tile / a.tiles_per_block, tile_in_block = tile - block * a.tiles_per_block;
        float cx = a.cx, cy = a.cy, cz = a.cz;
        if (a.blocks) {
            const cc_block_desc bd = a.blocks[block];
            cx = bd.cx; cy = bd.cy; cz = bd.cz;
        }
        float lo[3], hi[3];
        cc_tile_bounds(a, tile_in_block, (uint32_t)(CC_THREADS * PTS), lo, hi);
        gx[j] = cc_fma(a.step, 0.5f * (lo[0] + hi[0]), cx);
        gy[j] = cc_fma(a.step, 0.5f * (lo[1] + hi[1]), cy);
        gz[j] = cc_fma(a.step, 0.5f * (lo[2] + hi[2]), cz);
        const float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        r[j] = fabsf(a.step) * (0.5f * 1.0001f) * sqrtf(dx * dx + dy * dy + dz * dz);
    }
    V vx[1], vy[1], vz[1];
    cc_val<V> LV[1];
    vx[0] = cc_pack<V>(gx);
    vy[0] = cc_pack<V>(gy);
    vz[0] = cc_pack<V>(gz);
#pragma unroll
    for (int k = 0; k < P; ++k) pw[k] = vbc<V>(__int_as_float(0x7fc00000));  // NaN: "unknown" keeps a part alive
    eval(vx, vy, vz, LV);
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        if (t0 + (uint32_t)j >= n_tiles) break;
        float upper = __int_as_float(0x7f800000);
#pragma unroll
        for (int k = 0; k < P; ++k) upper = fminf(upper, cc_lane_scalar(pw[k], j) + (lip[k] * r[j] + a.part_slack));
        uint32_t mask = 0;
#pragma unroll
        for (int k = 0; k < P; ++k)
            if (!(cc_lane_scalar(pw[k], j) - (lip[k] * r[j] + a.part_slack) > upper)) mask |= 1u << k;
        a.part_masks[t0 + (uint32_t)j] = mask;
    }
}

// Brick-centre pass.  Thread t evaluates every part at the centres of bricks 2t and 2t + 1 (one packed
// pair; `pw` receives the parts' values) and derives the bricks' masks: with |w_k(p) - w_k(centre)| <=
// lip_k * radius + slack for every point p of the brick, part k can be the nearest somewhere in the brick
// only if  w_k(centre) - lip_k r - slack  <=  min_j (w_j(centre) + lip_j r + slack).  Written with negated
// comparisons so that a NaN keeps a part alive.
template <int P, class EVAL, class V>
CC_DEV void cc_part_centers_body(const cc_eval_args &a, EVAL &eval, V *pw, const float *lip)
{
    const uint32_t nbx = (a.nx + CC_BRICK_X - 1) / CC_BRICK_X, nby = (a.ny + CC_BRICK_Y - 1) / CC_BRICK_Y,
                   nbz = (a.nz + CC_BRICK_Z - 1) / CC_BRICK_Z;
    const uint32_t n_bricks = nbx * nby * nbz;
    const uint32_t b0 = 2u * (blockIdx.x * CC_THREADS + threadIdx.x);
    float gx[2], gy[2], gz[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        uint32_t x0, y0, z0;
        cc_brick_of(a, min(b0 + (uint32_t)j, n_bricks - 1u), x0, y0, z0);
        gx[j] = cc_fma(a.step, (float)(x0 + a.x_offset) + 0.5f * (CC_BRICK_X - 1), a.cx);
        gy[j] = cc_fma(a.step, (float)y0 + 0.5f * (CC_BRICK_Y - 1), a.cy);
        gz[j] = cc_fma(a.step, (float)z0 + 0.5f * (CC_BRICK_Z - 1), a.cz);
    }
    V vx[1], vy[1], vz[1];
    cc_val<V> LV[1];
    vx[0] = cc_pack<V>(gx);
    vy[0] = cc_pack<V>(gy);
    vz[0] = cc_pack<V>(gz);
#pragma unroll
    for (int k = 0; k < P; ++k) pw[k] = vbc<V>(__int_as_float(0x7fc00000));  // NaN: "unknown" keeps a part alive
    eval(vx, vy, vz, LV);
    // half diagonal of the brick's cell centres, with head room for the rounding of the coordinates
    const float r = fabsf(a.step) * (0.5f * 1.0001f) *
                    sqrtf((float)((CC_BRICK_X - 1) * (CC_BRICK_X - 1) + (CC_BRICK_Y - 1) * (CC_BRICK_Y - 1) + (CC_BRICK_Z - 1) * (CC_BRICK_Z - 1)));
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        if (b0 + (uint32_t)j >= n_bricks) break;
        float upper = __int_as_float(0x7f800000);
#pragma unroll
        for (int k = 0; k < P; ++k) upper = fminf(upper, cc_lane_scalar(pw[k], j) + (lip[k] * r + a.part_slack));  // (NaN, inf ignored)
        uint32_t mask = 0;
#pragma unroll
        for (int k = 0; k < P; ++k)
            if (!(cc_lane_scalar(pw[k], j) - (lip[k] * r + a.part_slack) > upper)) mask |= 1u << k;
        a.part_masks[b0 + (uint32_t)j] = mask;
    }
}

#endif
