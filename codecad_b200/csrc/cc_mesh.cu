// Marching cubes over the leaf blocks of a subdivision, on the device.
//
// Replaces, for the mesh-export caller of the hot path (SURVEY.md 8(f) rank 1), the per-block loop of
// /root/reference/codecad/rendering/mesh.py:36-74: one grid_eval_pymcubes launch + one blocking
// 8 MiB device->host copy + a CPU mcubes.marching_cubes() call per block.  Here all blocks of a
// chunk are evaluated by one PYMCUBES-sink launch into HBM, classified and triangulated by two
// kernels, and only the triangles come back.
//
// mcubes (PyMCubes 0.0.6, requirements.txt:11) is a third-party package that is not in the
// reference tree; its published algorithm (P. Bourke's polygonise conventions: corner/edge
// numbering, "inside" = value <= isovalue, vertices by linear interpolation in double precision)
// is restated here and in oracle/mc_oracle.py; the case table is generated (tools/make_mc_tables.py).
// Output order is deterministic: blocks in the given order, cells in (i, j, k) order with k
// fastest — mcubes' loop order — and the triangles of a cell in table order.
#include <cuda_runtime.h>
#include <stdint.h>

#include "cc_internal.h"
#include "cc_mc_table.h"

__constant__ unsigned char c_mc_count[256];
__constant__ unsigned char c_mc_tri[256][16];
__constant__ unsigned char c_mc_edge_corner[12][2];

__device__ __forceinline__ uint32_t cc_mc_edge_corner_d(uint32_t e, int which) { return c_mc_edge_corner[e][which]; }
// corner m -> offset along axis 0 (i), 1 (j), 2 (k): v0=(0,0,0) v1=(1,0,0) v2=(1,1,0) v3=(0,1,0), v4..v7 = +k
__device__ __forceinline__ uint32_t cc_mc_corner_d(uint32_t m, int axis)
{
    const uint32_t q = m & 3u;
    return axis == 0 ? (uint32_t)(q == 1u || q == 2u) : axis == 1 ? (uint32_t)(q >= 2u) : (m >> 2);
}

#define CC_MESH_THREADS 256

__device__ __forceinline__ uint32_t cc_mesh_case(const cc_mesh_args &a, const float *f, uint32_t i, uint32_t j, uint32_t k,
                                                 float (&v)[8])
{
    // corners v0..v7 = (i,j,k) + (0,0,0),(1,0,0),(1,1,0),(0,1,0),(0,0,1),(1,0,1),(1,1,1),(0,1,1)
    const size_t s0 = (size_t)a.d1 * a.d2, s1 = a.d2;
    const float *p = f + (size_t)i * s0 + (size_t)j * s1 + k;
    v[0] = p[0]; v[1] = p[s0]; v[2] = p[s0 + s1]; v[3] = p[s1];
    v[4] = p[1]; v[5] = p[s0 + 1]; v[6] = p[s0 + s1 + 1]; v[7] = p[s1 + 1];
    uint32_t c = 0;
#pragma unroll
    for (int m = 0; m < 8; ++m) c |= (v[m] <= 0.0f) ? (1u << m) : 0u;  // mcubes: v[m] <= isovalue, isovalue = 0
    return c;
}

// ---- indexed export: which block owns a sample or an edge (DESIGN.md 4.4) --------------------------
// Array index (i, j, k) of a block with int corner (X, Y, Z) is the lattice point (X + j, Y + n-1-i, Z + k),
// so neighbours are found in array axes: the block shifted by d (d_a in {-1, 0, 1}) holds our sample s as
// s - d*(n-1) when every component of that is inside [0, n-1].
#define CC_KEY_BITS 21
#define CC_KEY_MASK ((1ull << CC_KEY_BITS) - 1)

__device__ __forceinline__ int cc_find_block(const cc_mesh_args &a, uint64_t key)
{
    uint32_t lo = 0, hi = a.n_all;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (a.sorted_key[mid] < key) lo = mid + 1; else hi = mid;
    }
    return (lo < a.n_all && a.sorted_key[lo] == key) ? (int)a.sorted_block[lo] : -1;
}

struct cc_holder {
    uint32_t block;
    int d[3];
};

// The first block in input order that holds sample s of block b, or (edge_axis >= 0) both ends of the
// edge from s along edge_axis: such a block is not shifted along the edge.
__device__ cc_holder cc_first_holder(const cc_mesh_args &a, uint32_t b, const uint32_t (&s)[3], int edge_axis)
{
    const uint32_t m[3] = {a.d0 - 1, a.d1 - 1, a.d2 - 1};
    int lo[3], hi[3];
    bool face = false;
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
        lo[ax] = (ax != edge_axis && s[ax] == 0) ? -1 : 0;
        hi[ax] = (ax != edge_axis && s[ax] == m[ax]) ? 1 : 0;
        face |= lo[ax] != hi[ax];
    }
    cc_holder h{b, {0, 0, 0}};
    if (!face || a.n_all == 1) return h;
    const uint64_t key = a.block_key[b];
    const int64_t q[3] = {(int64_t)((key >> (2 * CC_KEY_BITS)) & CC_KEY_MASK), (int64_t)((key >> CC_KEY_BITS) & CC_KEY_MASK),
                          (int64_t)(key & CC_KEY_MASK)};
    for (int d0 = lo[0]; d0 <= hi[0]; ++d0)
        for (int d1 = lo[1]; d1 <= hi[1]; ++d1)
            for (int d2 = lo[2]; d2 <= hi[2]; ++d2) {
                if (!d0 && !d1 && !d2) continue;
                const int64_t n0 = q[0] + d0, n1 = q[1] + d1, n2 = q[2] + d2;
                if (n0 < 0 || n1 < 0 || n2 < 0 || n0 > (int64_t)CC_KEY_MASK || n1 > (int64_t)CC_KEY_MASK || n2 > (int64_t)CC_KEY_MASK)
                    continue;
                const int nb = cc_find_block(a, ((uint64_t)n0 << (2 * CC_KEY_BITS)) | ((uint64_t)n1 << CC_KEY_BITS) | (uint64_t)n2);
                if (nb >= 0 && (uint32_t)nb < h.block) h = cc_holder{(uint32_t)nb, {d0, d1, d2}};
            }
    return h;
}

// Face f = 2*axis + side (side 1: s[axis] == n-1) of a block is archived as [u][v], u and v the other two
// axes in increasing order.
__device__ __forceinline__ void cc_face_axes(uint32_t axis, uint32_t &ua, uint32_t &va)
{
    ua = axis == 0 ? 1u : 0u;
    va = axis == 2 ? 1u : 2u;
}

__device__ __forceinline__ size_t cc_face_slot(const cc_mesh_args &a, uint32_t block, uint32_t axis, uint32_t side, const uint32_t (&s)[3])
{
    uint32_t ua, va;
    cc_face_axes(axis, ua, va);
    return (((size_t)block * 6 + 2 * axis + side) * a.nf + s[ua]) * a.nf + s[va];
}

// Sample s of block b as the holder h sees it, and a face of h on which it lies (an axis h is shifted along).
__device__ __forceinline__ size_t cc_holder_slot(const cc_mesh_args &a, const cc_holder &h, const uint32_t (&s)[3], uint32_t &axis)
{
    const uint32_t m[3] = {a.d0 - 1, a.d1 - 1, a.d2 - 1};
    uint32_t t[3];
    axis = 0;
#pragma unroll
    for (int ax = 2; ax >= 0; --ax) {
        t[ax] = (uint32_t)((int64_t)s[ax] - (int64_t)h.d[ax] * m[ax]);
        if (h.d[ax]) axis = ax;
    }
    return cc_face_slot(a, h.block, axis, h.d[axis] < 0 ? 1u : 0u, t);
}

// Global index of the vertex on the edge from sample s along `axis` of chunk block `block`.
__device__ __forceinline__ uint32_t cc_vertex_index(const cc_mesh_args &a, uint32_t block, const uint32_t (&s)[3], int axis)
{
    const uint32_t b = a.first_block + block;
    const cc_holder h = cc_first_holder(a, b, s, axis);
    if (h.block == b) {
        const size_t t = ((size_t)block * a.d0 + s[0]) * a.d1 * a.d2 + (size_t)s[1] * a.d2 + s[2];
        return a.vert_base + a.vbase[t] + __popc(a.vmask[t] & ((1u << axis) - 1u));
    }
    // the edge lies on the face cc_holder_slot picks: h is not shifted along the edge's axis
    uint32_t face_axis, ua, va;
    const size_t slot = cc_holder_slot(a, h, s, face_axis);
    cc_face_axes(face_axis, ua, va);
    return a.face_vertex[2 * slot + ((uint32_t)axis == ua ? 0u : 1u)];
}

// Two passes share this kernel.  COUNT writes every tile's number of triangles to tile_offsets[tile];
// cc_mesh_scan_kernel turns them into exclusive offsets (+ the total in *counter); EMIT reads its base
// from there.  (The first version ordered the tiles with a ticket and a decoupled look-back inside the
// emit pass: with 896 k tiles of which 95 % are empty, every CTA sat ~7 us at the barrier behind its
// look-back warp — 11.6 ms for csg_example at 512^3, stall_barrier 30 per issue; profiles/r1_mesh.md.)
// INDEXED: the emit pass of cc_mesh_blocks_indexed, which writes three vertex indices per triangle.
template <bool EMIT, bool INDEXED = false>
__global__ void __launch_bounds__(CC_MESH_THREADS) cc_mesh_kernel(const cc_mesh_args a)
{
    __shared__ uint32_t s_warp[CC_MESH_THREADS / 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // COUNT runs over every tile; EMIT only over the tiles that hold triangles (95 % do not), whose
    // ids the scan compacted into tile_list in increasing order
    const uint32_t tile = EMIT ? a.tile_list[blockIdx.x] : blockIdx.x;
    const uint32_t block = tile / a.tiles_per_block;
    const uint32_t tile_in_block = tile - block * a.tiles_per_block;
    const uint32_t c0 = a.d0 - 1, c1 = a.d1 - 1, c2 = a.d2 - 1;
    const uint32_t cells = c0 * c1 * c2;
    const uint32_t cell = tile_in_block * CC_MESH_THREADS + tid;
    const bool valid = cell < cells;
    uint32_t i = 0, j = 0, k = 0, cs = 0, n = 0;
    float v[8];
    const float *f = a.field + (size_t)block * a.d0 * a.d1 * a.d2;
    if (valid) {
        i = cell / (c1 * c2);
        const uint32_t r = cell - i * (c1 * c2);
        j = r / c2;
        k = r - j * c2;
        cs = cc_mesh_case(a, f, i, j, k, v);
        n = c_mc_count[cs];
    }
    // triangles of this tile: warp scan + scan of the warp totals
    uint32_t incl = n;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = (lane < CC_MESH_THREADS / 32) ? s_warp[lane] : 0u;
        uint32_t wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, wi, d);
            if (lane >= d) wi += t;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, wi, 31);
        if (lane < CC_MESH_THREADS / 32) s_warp[lane] = wi - w;
        if (!EMIT && lane == 0) a.tile_offsets[tile] = total;
    }
    if (!EMIT) return;
    // Emission is spread over the CTA: triangle t of the tile goes to thread t mod 256, whichever
    // cell it belongs to (a serial loop per cell left the few surface threads of a warp working
    // alone on up to five triangles each, and wrote 72-byte pieces far apart).  The owning cell is
    // found by binary search in the tile's inclusive prefix sums; its corner values come from
    // shared memory.  Same arithmetic per triangle, same output order.
    __shared__ uint32_t s_incl[CC_MESH_THREADS];
    __shared__ unsigned char s_case[CC_MESH_THREADS];
    __shared__ float s_v[CC_MESH_THREADS][9];  // padded: 8 corner values per cell
    __syncthreads();
    s_incl[tid] = s_warp[warp] + incl;
    s_case[tid] = (unsigned char)cs;
    if (n) {
#pragma unroll
        for (int m = 0; m < 8; ++m) s_v[tid][m] = v[m];
    }
    __syncthreads();
    const uint32_t tile_total = s_incl[CC_MESH_THREADS - 1];
    const uint32_t tile_base = a.tile_offsets[tile];
    const double cx = a.corner[3 * (size_t)block + 0], cy = a.corner[3 * (size_t)block + 1], cz = a.corner[3 * (size_t)block + 2];
    for (uint32_t t = tid; t < tile_total; t += CC_MESH_THREADS) {
        // owner = first thread whose inclusive sum exceeds t
        uint32_t lo = 0, hi = CC_MESH_THREADS - 1;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (s_incl[mid] > t) hi = mid; else lo = mid + 1;
        }
        const uint32_t owner = lo, ocs = s_case[owner];
        const uint32_t tri = t - (s_incl[owner] - c_mc_count[ocs]);  // index among the owner's triangles
        const uint32_t ocell = tile_in_block * CC_MESH_THREADS + owner;
        const uint32_t oi = ocell / (c1 * c2), orem = ocell - oi * (c1 * c2), oj = orem / c2, ok = orem - oj * c2;
        const uint32_t pos = tile_base + t;
        a.tri_block[pos] = a.first_block + block;
        if (INDEXED) {
            uint32_t idx[3];
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const uint32_t e = c_mc_tri[ocs][3 * tri + q];
                const uint32_t ca = cc_mc_edge_corner_d(e, 0), cb = cc_mc_edge_corner_d(e, 1);
                const uint32_t s[3] = {oi + cc_mc_corner_d(ca, 0), oj + cc_mc_corner_d(ca, 1), ok + cc_mc_corner_d(ca, 2)};
                const int axis = cc_mc_corner_d(ca, 0) != cc_mc_corner_d(cb, 0) ? 0 : cc_mc_corner_d(ca, 1) != cc_mc_corner_d(cb, 1) ? 1 : 2;
                idx[q] = cc_vertex_index(a, block, s, axis);
            }
            uint32_t *dst = a.triangles + (size_t)pos * 3;  // winding flip as below
            dst[0] = idx[1];
            dst[1] = idx[0];
            dst[2] = idx[2];
            continue;
        }
        const double base_idx[3] = {(double)oi, (double)oj, (double)ok};
        const float *ov = s_v[owner];
        double out[3][3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            const uint32_t e = c_mc_tri[ocs][3 * tri + q];
            const uint32_t ca = cc_mc_edge_corner_d(e, 0), cb = cc_mc_edge_corner_d(e, 1);
            double p[3];
#pragma unroll
            for (int ax = 0; ax < 3; ++ax) {
                // mc_add_vertex: c1 + (isovalue - f1) * (c2 - c1) / (f2 - f1) along the edge's axis, in double
                const double a1 = __dadd_rn(base_idx[ax], (double)cc_mc_corner_d(ca, ax));
                const double a2 = __dadd_rn(base_idx[ax], (double)cc_mc_corner_d(cb, ax));
                double val = a1;
                if (a1 != a2) {
                    const double f1 = (double)ov[ca], f2 = (double)ov[cb];
                    val = __dadd_rn(a1, __ddiv_rn(__dmul_rn(__dsub_rn(0.0, f1), __dsub_rn(a2, a1)), __dsub_rn(f2, f1)));
                }
                p[ax] = val;
            }
            // rendering/mesh.py:68-71: swap columns 0 and 1, negate column 1, scale, translate (float64)
            out[q][0] = __dadd_rn(__dmul_rn(p[1], a.resolution), cx);
            out[q][1] = __dadd_rn(__dmul_rn(-p[0], a.resolution), cy);
            out[q][2] = __dadd_rn(__dmul_rn(p[2], a.resolution), cz);
        }
        // rendering/mesh.py:72: triangles[:, [0, 1]] = triangles[:, [1, 0]]
        double *dst = a.vertices + (size_t)pos * 9;
#pragma unroll
        for (int ax = 0; ax < 3; ++ax) {
            dst[0 + ax] = out[1][ax];
            dst[3 + ax] = out[0][ax];
            dst[6 + ax] = out[2][ax];
        }
    }
}

// mc_add_vertex (see cc_mesh_kernel) for the edge from sample s along `axis`, field values f1 at s and
// f2 at its other end, then the post-transform of rendering/mesh.py:68-71 with the block's corner.
__device__ __forceinline__ void cc_edge_vertex(const cc_mesh_args &a, uint32_t block, const uint32_t (&s)[3], int axis, float f1,
                                               float f2, double *dst)
{
    double p[3];
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
        const double a1 = (double)s[ax];
        double val = a1;
        if (ax == axis) {
            const double a2 = __dadd_rn(a1, 1.0);
            val = __dadd_rn(a1, __ddiv_rn(__dmul_rn(__dsub_rn(0.0, (double)f1), __dsub_rn(a2, a1)), __dsub_rn((double)f2, (double)f1)));
        }
        p[ax] = val;
    }
    const double *c = a.corner + 3 * (size_t)block;
    dst[0] = __dadd_rn(__dmul_rn(p[1], a.resolution), c[0]);
    dst[1] = __dadd_rn(__dmul_rn(-p[0], a.resolution), c[1]);
    dst[2] = __dadd_rn(__dmul_rn(p[2], a.resolution), c[2]);
}

__device__ __forceinline__ void cc_sample_of(const cc_mesh_args &a, size_t t, uint32_t &block, uint32_t (&s)[3])
{
    const size_t per = (size_t)a.d0 * a.d1 * a.d2;
    block = (uint32_t)(t / per);
    const uint32_t r = (uint32_t)(t - (size_t)block * per);
    s[0] = r / (a.d1 * a.d2);
    const uint32_t r2 = r - s[0] * (a.d1 * a.d2);
    s[1] = r2 / a.d2;
    s[2] = r2 - s[1] * a.d2;
}

// One thread per (chunk block, face, u, v); samples on a block's edges and corners are visited by
// each face they lie on and get the same value every time.  ARCHIVE copies the chunk's face samples
// into face_field; otherwise every face sample the block does not own takes its owner's value from
// the owner's archive.  An owner's own values are never written, so the two can run in place.
template <bool ARCHIVE>
__global__ void __launch_bounds__(CC_MESH_THREADS) cc_mesh_faces_kernel(const cc_mesh_args a)
{
    const size_t t = (size_t)blockIdx.x * CC_MESH_THREADS + threadIdx.x;
    const size_t per_face = (size_t)a.nf * a.nf;
    if (t >= (size_t)a.n_blocks * 6 * per_face) return;
    const uint32_t block = (uint32_t)(t / (6 * per_face));
    const uint32_t f = (uint32_t)(t / per_face % 6), axis = f >> 1;
    const uint32_t uv = (uint32_t)(t % per_face), u = uv / a.nf, v = uv - u * a.nf;
    const uint32_t dims[3] = {a.d0, a.d1, a.d2};
    uint32_t ua, va;
    cc_face_axes(axis, ua, va);
    if (u >= dims[ua] || v >= dims[va]) return;
    uint32_t s[3];
    s[axis] = (f & 1) ? dims[axis] - 1 : 0;
    s[ua] = u;
    s[va] = v;
    float *field = const_cast<float *>(a.field) + (size_t)block * a.d0 * a.d1 * a.d2 + ((size_t)s[0] * a.d1 + s[1]) * a.d2 + s[2];
    const uint32_t b = a.first_block + block;
    if (ARCHIVE) {
        a.face_field[cc_face_slot(a, b, axis, f & 1, s)] = *field;
        return;
    }
    const cc_holder h = cc_first_holder(a, b, s, -1);
    if (h.block == b) return;
    uint32_t face_axis;
    *field = a.face_field[cc_holder_slot(a, h, s, face_axis)];
}

// One thread per chunk sample: which edges along +i, +j, +k are crossed (both ends inside the block)
// and owned by this block; vbase gets their number (scanned afterwards), vmask the edges.
__global__ void __launch_bounds__(CC_MESH_THREADS) cc_mesh_vertex_count_kernel(const cc_mesh_args a)
{
    const size_t t = (size_t)blockIdx.x * CC_MESH_THREADS + threadIdx.x;
    if (t >= (size_t)a.n_blocks * a.d0 * a.d1 * a.d2) return;
    uint32_t block, s[3];
    cc_sample_of(a, t, block, s);
    const uint32_t dims[3] = {a.d0, a.d1, a.d2};
    const size_t stride[3] = {(size_t)a.d1 * a.d2, a.d2, 1};
    const bool in0 = a.field[t] <= 0.0f;
    uint32_t mask = 0;
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
        if (s[ax] + 1 >= dims[ax] || (a.field[t + stride[ax]] <= 0.0f) == in0) continue;
        if (cc_first_holder(a, a.first_block + block, s, ax).block == a.first_block + block) mask |= 1u << ax;
    }
    a.vmask[t] = (uint8_t)mask;
    a.vbase[t] = __popc(mask);
}

// One thread per chunk sample: the positions of its owned vertices, and their indices in the block's
// face archive for the edges that lie on a face (later blocks that hold them look them up there).
__global__ void __launch_bounds__(CC_MESH_THREADS) cc_mesh_vertex_emit_kernel(const cc_mesh_args a)
{
    const size_t t = (size_t)blockIdx.x * CC_MESH_THREADS + threadIdx.x;
    if (t >= (size_t)a.n_blocks * a.d0 * a.d1 * a.d2) return;
    const uint32_t mask = a.vmask[t];
    if (!mask) return;
    uint32_t block, s[3];
    cc_sample_of(a, t, block, s);
    const uint32_t dims[3] = {a.d0, a.d1, a.d2};
    const size_t stride[3] = {(size_t)a.d1 * a.d2, a.d2, 1};
    uint32_t local = a.vbase[t];
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
        if (!(mask & (1u << ax))) continue;
        cc_edge_vertex(a, block, s, ax, a.field[t], a.field[t + stride[ax]], a.vert_out + 3 * (size_t)local);
        const uint32_t index = a.vert_base + local;
#pragma unroll
        for (int fa = 0; fa < 3; ++fa) {
            if (fa == ax || (s[fa] != 0 && s[fa] != dims[fa] - 1)) continue;
            uint32_t ua, va;
            cc_face_axes(fa, ua, va);
            a.face_vertex[2 * cc_face_slot(a, a.first_block + block, fa, s[fa] != 0, s) + ((uint32_t)ax == ua ? 0u : 1u)] = index;
        }
        ++local;
    }
}

// In-place exclusive scan of the n tile counts (n ~ 10^6) and compaction of the ids of the non-empty
// tiles, three small launches:
//   cc_scan_local_kernel  4096 elements per CTA: exclusive scans of (count, count != 0) inside the CTA,
//                         CTA totals -> part[cta], part_f[cta]
//   cc_scan_parts_kernel  one CTA: exclusive scans of part[] and part_f[], grand totals -> counter[0..1]
//   cc_scan_add_kernel    adds part[cta] to the CTA's offsets and writes the non-empty tile ids
#define CC_SCAN_PER_CTA 4096u
__device__ __forceinline__ uint32_t cc_block_exclusive(uint32_t mine, uint32_t *s_warp, uint32_t *total)
{
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t up = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += up;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = s_warp[lane];
        uint32_t wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t up = __shfl_up_sync(0xffffffffu, wi, d);
            if (lane >= d) wi += up;
        }
        s_warp[lane] = wi - w;
        if (lane == 31) s_warp[32] = wi;
    }
    __syncthreads();
    const uint32_t excl = s_warp[warp] + (incl - mine);
    *total = s_warp[32];
    __syncthreads();  // s_warp is reused by the next call
    return excl;
}

__global__ void __launch_bounds__(1024) cc_scan_local_kernel(uint32_t *__restrict__ v, uint32_t n, uint32_t *__restrict__ part,
                                                             uint32_t *__restrict__ flag_off, uint32_t *__restrict__ part_f)
{
    __shared__ uint32_t s_warp[33];
    const uint32_t t = threadIdx.x;
    const uint32_t i0 = blockIdx.x * CC_SCAN_PER_CTA + 4u * t;
    uint32_t x[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) x[k] = (i0 + k < n) ? v[i0 + k] : 0u;
    uint32_t total, total_f;
    uint32_t run = cc_block_exclusive(x[0] + x[1] + x[2] + x[3], s_warp, &total);
    uint32_t run_f = cc_block_exclusive((x[0] != 0) + (x[1] != 0) + (x[2] != 0) + (x[3] != 0), s_warp, &total_f);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (i0 + k < n) {
            v[i0 + k] = run;
            flag_off[i0 + k] = run_f | (x[k] ? 0x80000000u : 0u);  // top bit: this tile holds triangles
        }
        run += x[k];
        run_f += x[k] != 0;
    }
    if (t == 0) {
        part[blockIdx.x] = total;
        part_f[blockIdx.x] = total_f;
    }
}

// exclusive scan of v[0..n) by one CTA (chunk per thread); returns the total through *out
__device__ __forceinline__ void cc_scan_single_cta(uint32_t *__restrict__ v, uint32_t n, uint32_t *s_part, uint32_t *out)
{
    const uint32_t t = threadIdx.x;
    const uint32_t per = (n + 1023u) / 1024u;
    const uint32_t lo = min(n, t * per), hi = min(n, lo + per);
    uint32_t sum = 0;
    for (uint32_t i = lo; i < hi; ++i) sum += v[i];
    s_part[t] = sum;
    __syncthreads();
    for (uint32_t d = 1; d < 1024u; d <<= 1) {  // Hillis-Steele inclusive scan of the 1024 partial sums
        const uint32_t add = t >= d ? s_part[t - d] : 0u;
        __syncthreads();
        s_part[t] += add;
        __syncthreads();
    }
    uint32_t run = s_part[t] - sum;
    for (uint32_t i = lo; i < hi; ++i) {
        const uint32_t c = v[i];
        v[i] = run;
        run += c;
    }
    if (t == 1023u) *out = s_part[1023];
    __syncthreads();
}

__global__ void __launch_bounds__(1024) cc_scan_parts_kernel(uint32_t *__restrict__ part, uint32_t *__restrict__ part_f, uint32_t n,
                                                             uint32_t *__restrict__ counter)
{
    __shared__ uint32_t s_part[1024];
    cc_scan_single_cta(part, n, s_part, counter);        // counter[0] = triangles
    cc_scan_single_cta(part_f, n, s_part, counter + 1);  // counter[1] = non-empty tiles
}

__global__ void __launch_bounds__(1024) cc_scan_add_kernel(uint32_t *__restrict__ v, uint32_t n, const uint32_t *__restrict__ part,
                                                           const uint32_t *__restrict__ flag_off,
                                                           const uint32_t *__restrict__ part_f, uint32_t *__restrict__ tile_list)
{
    const uint32_t base = part[blockIdx.x], base_f = part_f[blockIdx.x];
    const uint32_t i0 = blockIdx.x * CC_SCAN_PER_CTA + 4u * threadIdx.x;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (i0 + k < n) {
            v[i0 + k] += base;
            const uint32_t f = flag_off[i0 + k];
            if (f & 0x80000000u) tile_list[base_f + (f & 0x7FFFFFFFu)] = i0 + k;
        }
}

// ---- host side ------------------------------------------------------------------------------------

int cc_mesh_upload_tables(void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemcpyToSymbolAsync(c_mc_count, cc_mc_count, sizeof(cc_mc_count), 0, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess)
        e = cudaMemcpyToSymbolAsync(c_mc_tri, cc_mc_tri, sizeof(cc_mc_tri), 0, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess)
        e = cudaMemcpyToSymbolAsync(c_mc_edge_corner, cc_mc_edge_corner, sizeof(cc_mc_edge_corner), 0,
                                    cudaMemcpyHostToDevice, st);
    return (int)e;
}

uint32_t cc_mesh_tiles_per_block(uint32_t d0, uint32_t d1, uint32_t d2)
{
    const uint64_t cells = (uint64_t)(d0 - 1) * (d1 - 1) * (d2 - 1);
    return (uint32_t)((cells + CC_MESH_THREADS - 1) / CC_MESH_THREADS);
}

size_t cc_mesh_scratch_words(uint32_t tiles)
{
    const size_t ctas = (tiles + CC_SCAN_PER_CTA - 1) / CC_SCAN_PER_CTA;
    return 3 * (size_t)tiles + 2 * ctas;  // offsets, flag offsets, tile list; two sets of CTA partials
}

size_t cc_mesh_scan_scratch_words(uint32_t n)
{
    const size_t ctas = (n + CC_SCAN_PER_CTA - 1) / CC_SCAN_PER_CTA;
    return (size_t)n + 2 * ctas;  // flag offsets; two sets of CTA partials
}

int cc_launch_mesh_scan(uint32_t *v, uint32_t n, uint32_t *scratch, uint32_t *list, uint32_t *counter, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) return 0;
    const uint32_t ctas = (n + CC_SCAN_PER_CTA - 1) / CC_SCAN_PER_CTA;
    uint32_t *part = scratch, *flag_off = part + ctas, *part_f = flag_off + n;
    cc_scan_local_kernel<<<ctas, 1024, 0, st>>>(v, n, part, flag_off, part_f);
    cc_scan_parts_kernel<<<1, 1024, 0, st>>>(part, part_f, ctas, counter);
    cc_scan_add_kernel<<<ctas, 1024, 0, st>>>(v, n, part, flag_off, part_f, list);
    return (int)cudaGetLastError();
}

// count pass: all tiles, then the scan (counter[0] = triangles, counter[1] = non-empty tiles).
// emit pass: `emit_tiles` CTAs, one per non-empty tile.
int cc_launch_mesh(const cc_mesh_args &a, bool emit, uint32_t emit_tiles, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    const uint32_t grid = a.n_blocks * a.tiles_per_block;
    if (grid == 0) return 0;
    if (emit) {
        if (emit_tiles) cc_mesh_kernel<true><<<emit_tiles, CC_MESH_THREADS, 0, st>>>(a);
    } else {
        cc_mesh_kernel<false><<<grid, CC_MESH_THREADS, 0, st>>>(a);
        return cc_launch_mesh_scan(a.tile_offsets, grid, a.tile_offsets + grid, a.tile_list, a.counter, stream);
    }
    return (int)cudaGetLastError();
}

static uint32_t cc_ctas(size_t threads) { return (uint32_t)((threads + CC_MESH_THREADS - 1) / CC_MESH_THREADS); }

int cc_launch_mesh_reconcile(const cc_mesh_args &a, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    const size_t faces = (size_t)a.n_blocks * 6 * a.nf * a.nf, samples = (size_t)a.n_blocks * a.d0 * a.d1 * a.d2;
    if (samples == 0) return 0;
    cc_mesh_faces_kernel<true><<<cc_ctas(faces), CC_MESH_THREADS, 0, st>>>(a);
    cc_mesh_faces_kernel<false><<<cc_ctas(faces), CC_MESH_THREADS, 0, st>>>(a);
    cc_mesh_vertex_count_kernel<<<cc_ctas(samples), CC_MESH_THREADS, 0, st>>>(a);
    return (int)cudaGetLastError();
}

int cc_launch_mesh_indexed_emit(const cc_mesh_args &a, uint32_t emit_tiles, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    const size_t samples = (size_t)a.n_blocks * a.d0 * a.d1 * a.d2;
    if (samples == 0) return 0;
    cc_mesh_vertex_emit_kernel<<<cc_ctas(samples), CC_MESH_THREADS, 0, st>>>(a);
    if (emit_tiles) cc_mesh_kernel<true, true><<<emit_tiles, CC_MESH_THREADS, 0, st>>>(a);
    return (int)cudaGetLastError();
}
