// Plain-old-data types shared by host code, the precompiled kernels and the NVRTC-compiled
// scene-specialised kernels (no standard headers: this file is also fed to NVRTC).
#ifndef CC_DEVICE_TYPES_H
#define CC_DEVICE_TYPES_H

#ifdef __CUDACC_RTC__
typedef unsigned char uint8_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
typedef unsigned long size_t;
#else
#include <stddef.h>
#include <stdint.h>
#endif

#ifndef CC_THREADS
#define CC_THREADS 128  // CTA size of the precompiled kernels; specialised kernels may override it
#endif

// polygon2d edge table (microcode, after RETURN; __constant__ array in the specialised kernels):
// n edges of (px, py, dx, dy, 1/|d|^2, cy), then
#define CC_POLY_EDGE_WORDS 6
// after the n edges: one entry per group of CC_POLY_GROUP consecutive edges, (xmin, xmax, ymin, ymax of
// the group's vertices) — lets the edge loop skip whole groups exactly
#define CC_POLY_GROUP 8
#define CC_POLY_GROUP_WORDS 4
#define CC_POLY_TABLE_WORDS(n) (CC_POLY_EDGE_WORDS * (n) + CC_POLY_GROUP_WORDS * (((n) + CC_POLY_GROUP - 1) / CC_POLY_GROUP))


enum cc_sink_kind {
    CC_SINK_FLOAT4 = 0, CC_SINK_PYMCUBES, CC_SINK_CLASSIFY, CC_SINK_MASS,
    CC_SINK_RAY, CC_SINK_BITMAP,  // image renderers (cc_render.cuh), one point per thread
    CC_SINK_POINTS,               // FLOAT4 sink fed from a point list (cc_evaluate_points)
    CC_SINK_PARTS,                // FLOAT4 sink over 8 x 8 x 16 bricks with per-brick part masks (cc_jit.cpp, DESIGN.md 4.9)
    CC_SINK_COLUMNS,              // FLOAT4 sink over bricks with the column-invariant micro-ops evaluated once per column (DESIGN.md 4.10)
    // the hierarchy sinks (blocks x linear tiles) with a part mask per tile and / or the column split: one unit each
    CC_SINK_TILES_PYMCUBES, CC_SINK_TILES_CLASSIFY, CC_SINK_TILES_MASS,
    CC_N_SINKS
};

struct cc_block_desc {  // one block of a subdivision level (device resident)
    float cx, cy, cz;   // fp32 corner of the first sample (cell centre), reference rounding
    uint32_t pad;
};

struct cc_eval_args {
    const uint32_t *code;
    uint32_t code_words;
    uint32_t n_slots;
    // geometry: single grid (blocks == nullptr) or a list of equally sized blocks
    float cx, cy, cz, step;
    uint32_t nx, ny, nz, x_offset;
    uint32_t n_blocks;
    uint32_t tiles_per_block;
    const cc_block_desc *blocks;
    // sinks
    void *out;            // float4* / float*            (FLOAT4, PYMCUBES)
    float threshold;      // CLASSIFY, MASS
    uint32_t *counter;    // running length of `list`   (CLASSIFY, MASS)
    uint8_t *list;        // uchar4 (x,y,z,0) per hit
    uint32_t *list_block; // optional: block index of every hit (hierarchy fast path)
    uint32_t *sums;       // MASS: 10 uint32 per block (stride 10), or one set when blocks == nullptr
    // decoupled look-back scratch (ordered compaction)
    uint32_t *ticket;
    unsigned long long *tile_status;
    // optional: evaluate at these points (x, y, z, unused) instead of grid coordinates; cell c of
    // the launch reads points[c] (used with nx = number of points, ny = nz = 1)
    const float *points;  // 16-byte aligned quadruples
    // part culling (CC_SINK_PARTS): one mask per brick, bit k = part k can matter there
    uint32_t *part_masks;
    float part_slack;     // bound on |computed - exact| of a part's value over the launch
    float coord_max;      // launches over blocks: largest |coordinate| any block of the launch can reach (0: unknown, no masks)
    // columns (CC_SINK_COLUMNS, cc_body.cuh): per-column values of the z-invariant micro-ops, columns that
    // failed the run-time check (null: the program has nothing to check), the bricks those send to the full walk
    float *columns;
    unsigned char *column_flags;
    uint32_t *brick_list, *brick_count;
    // warps of the column brick kernel whose deferred range check failed and that took the full walk (cc_body.cuh)
    unsigned long long *check_fallbacks;
    // bricks of the column brick kernel that a flagged column sent to the full walk (cc_body.cuh)
    unsigned long long *flagged_bricks;
    // bricks per CTA of the column brick kernel: a run along the columns' axis, 1 .. CC_BRICK_RUN_MAX (cc_body.cuh)
    uint32_t brick_run;
};

// bricks of the part-culling kernels: a CTA of 512 threads x 2 points
#define CC_BRICK_X 8
#define CC_BRICK_Y 8
#define CC_BRICK_Z 16
// the longest run of bricks one CTA of the column brick kernel walks, and the run it walks unless asked otherwise
// (CODECAD_B200_BRICK_RUN)
#define CC_BRICK_RUN_MAX 64
#define CC_BRICK_RUN_DEFAULT 8

// arguments of the image renderers (rendering/ray_caster.cl:147-156, rendering/bitmap.cl:1-3)
struct cc_render_args {
    const uint32_t *code;
    uint32_t code_words, n_slots;
    float ox, oy, oz;        // origin
    float fx, fy, fz;        // forward * focal length   (ray caster)
    float ux, uy, uz;        // up
    float rx, ry, rz;        // right
    float pixel_tolerance, box_radius, min_distance, max_distance, floor_z;
    float step_size;         // bitmap
    uint32_t options;        // 1 = false colour, 2 = zebra
    uint32_t w, h;
    uint8_t *out;            // [w][h][3], INDEX2: y fastest (cl_util/indexing.h:3)
    unsigned long long *eval_count;  // optional: total evaluate() calls of valid lanes
};

#endif
