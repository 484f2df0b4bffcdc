// Internal declarations shared by the translation units of libcodecad_b200.
#ifndef CC_INTERNAL_H
#define CC_INTERNAL_H

#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/codecad_b200.h"
#include "cc_device_types.h"
#include "cc_microcode.h"

// A program that is one tree of unions over fused primitives ("union forest"): what the loader
// proves about it (cc_program.cpp analyse_forest) so that cc_forest.cu may skip, per tile of the
// grid, every primitive that provably cannot influence a single bit of the tile's results.
struct cc_forest {
    bool enabled = false;
    uint32_t n_leaves = 0, n_unions = 0, n_events = 0, max_depth = 0;
    float rmax = 0.0f;             // largest blend radius of its rounded unions (0: sharp unions only)
    float err_a = 0.0f, err_b = 0.0f;  // |computed - exact| of a primitive's distance <= 2^-16 (err_a + err_b * max|p|)
    std::vector<float> bounds;     // [n_leaves][8]: centre x,y,z, g_lo, r_lb, g_hi, r_ub, depth  (cc_forest.cu)
    std::vector<uint32_t> events;  // [n_events][4]: PUSH / PRIM / COMBINE in evaluation order
};
#define CC_FOREST_PUSH 0u
#define CC_FOREST_PRIM 1u
#define CC_FOREST_COMBINE 2u
#define CC_FOREST_EVENT(type, kind, pc) ((uint32_t)(type) | ((uint32_t)(kind) << 2) | ((uint32_t)(pc) << 8))
#define CC_FOREST_MIN_LEAVES 8u

// A program whose value is a tree of sharp unions over self-contained sub-programs ("parts": the
// components of an assembly), possibly under a chain of distance-monotone ops.  A part whose value
// over a brick provably exceeds another part's cannot be selected there, so its code is skipped
// (cc_program.cpp analyse_parts, cc_jit.cpp, DESIGN.md 4.9).
struct cc_parts {
    bool enabled = false;
    uint32_t n_parts = 0;                 // <= 32
    std::vector<int> part_of_op;          // micro-op index -> part, -1 = outside every part
    std::vector<uint32_t> union_a, union_b;  // micro-op index of a union of the tree -> bit masks of the parts below its two operands (0 elsewhere)
    std::vector<float> lipschitz;         // per part: |w(p) - w(q)| <= lipschitz |p - q|   (inf: never culled)
    float magnitude_a = 0.0f, magnitude_b = 0.0f;  // rounding budget: 2^-13 (a + b max|p|)
    // The same structure for the interpreter tier (cc_parts.cu), device table:
    //   [0] n_parts  [1] n_segments  [2 .. 2+P) Lipschitz constants (float bits)  then P x (pc begin, pc end)
    //   then n_segments x 4 words: (kind, a, b, c)
    //     kind 0: micro-ops [a, b) always        kind 1: micro-ops [a, b) if mask & c (a part's run)
    //     kind 2: the union at pc a if (mask & b) && (mask & c), else kind 3's effect with its dst slot
    std::vector<uint32_t> table;
};
#define CC_SEG_ALWAYS 0u
#define CC_SEG_PART 1u
#define CC_SEG_UNION 2u

// Columns (DESIGN.md 4.10).  On a dense grid the axes of the grid are the axes of the program's point; a 2-D profile
// under an extrusion — transform, polygon, gear, their unions — sees two of them only, so its value is the same for
// every cell of a column along the third.  The loader tracks, op by op and component by component, what can depend
// on the grid coordinate along `axis`, and splits the micro-ops into those that run once per column ("ahead": the
// column pass) and those that run per cell ("loop": the brick / tile kernels) — cc_program.cpp analyse_columns,
// cc_jit.cpp.
struct cc_columns {
    bool enabled = false;
    int axis = 2;                      // the grid axis of the columns: 0 = x, 1 = y, 2 = z
    std::vector<uint8_t> phase;        // per micro-op: bit 0 = runs in the column pass, bit 1 = runs per cell
    std::vector<int> restore_from;     // per micro-op of the per-cell body: the op (of the column pass only) whose result is its running value, else -1
    std::vector<uint8_t> save_l;       // per micro-op: its result is carried into the per-cell body as a running value
    std::vector<uint8_t> split_prim;   // per micro-op: a fused extruded circle / rectangle whose 2-D half (transform rows x, y + the profile)
                                       // cannot see the axis: that half runs in the column pass, extrusion and the rest per cell
    int root_restore = -1;             // the program's result itself is column-invariant: op index, else -1
    std::vector<uint32_t> checked_rows;  // (micro-op index * 4 + row) of T_INIT rows whose coefficient along the axis is rounding residue: verified per column
    float invariant_share = 0.0f;      // estimated share of the arithmetic that leaves the per-cell body
    std::vector<uint32_t> op_cost;     // per micro-op: the rough cost the estimate uses (instructions per point pair)
};

struct cc_decoded {
    std::vector<uint32_t> microcode;
    cc_program_info info;
    cc_forest forest;
    cc_parts parts;
    cc_columns columns;
};

// cc_program.cpp
int cc_decode_program(const float *words, uint32_t n_words, cc_decoded *out, std::string *err);

struct cc_jit_cfg {
    int pts = 2;         // points per thread
    int threads = 512;   // CTA size
    int min_blocks = 2;  // __launch_bounds__ min CTAs per SM (register cap)
    int smem_min_len = 12;   // values live for at least this many micro-ops go to shared-memory cells
    int smem_max_cells = 6;  // budget of cells (0 = keep everything in registers)
    int segment_ops = 96;    // programs longer than ~1.5x this are cut into functions of this many micro-ops
};
struct cc_jit_job;
// what the column kernels of a program need from the host (filled by the code generator; default for a unit without them)
struct cc_columns_meta {
    uint32_t n_values = 0;  // carried values: the column buffer holds 4 * n_values floats per column
    bool checks = false;    // some transform row is verified per column: flags, brick list and the full-walk kernel exist
    int axis = 2;           // the grid axis of the columns
    bool columns = false;   // the unit has the column split (a tile unit of a program with parts only has not)
};

#define CC_AUX_CENTERS 0
#define CC_AUX_COLUMNS 1
#define CC_AUX_FULL 2

// columns of an nx x ny x nz grid along `axis`: the cells of the plane across it
inline uint64_t columns_along(int axis, uint32_t nx, uint32_t ny, uint32_t nz)
{
    return axis == 2 ? (uint64_t)nx * ny : axis == 1 ? (uint64_t)nx * nz : (uint64_t)ny * nz;
}

// bricks of the launch along `axis`
inline uint32_t bricks_along(int axis, const cc_eval_args &a)
{
    return axis == 0 ? (a.nx + CC_BRICK_X - 1) / CC_BRICK_X : axis == 1 ? (a.ny + CC_BRICK_Y - 1) / CC_BRICK_Y : (a.nz + CC_BRICK_Z - 1) / CC_BRICK_Z;
}
// CTAs of the column brick kernel: every stack of bricks along the columns' axis in runs of a.brick_run (cc_brick_run_of)
inline uint64_t brick_runs(int axis, const cc_eval_args &a)
{
    const uint64_t stacks = (uint64_t)bricks_along(0, a) * bricks_along(1, a) * bricks_along(2, a) / bricks_along(axis, a);
    return stacks * ((bricks_along(axis, a) + a.brick_run - 1) / a.brick_run);
}

#define CC_MAX_DEVICES 16  // devices one process can drive (cc_init_devices)

struct cc_program {
    cc_decoded dec;
    uint32_t *d_code[CC_MAX_DEVICES] = {};  // device copies of the microcode, one per initialised device (made on first use)
    void *d_forest[CC_MAX_DEVICES] = {};    // device copies of the forest tables (bounds, then events)
    uint32_t *d_parts[CC_MAX_DEVICES] = {};  // device copies of cc_parts::table
    uint64_t id = 0;             // identifies what is currently loaded in a device's __constant__ window
    // scene-specialised kernels (cc_jit.cpp), one library per sink; null until compiled
    void *jit_library[CC_N_SINKS] = {};
    void *jit_kernel[CC_N_SINKS] = {};
    // companion kernels of the same library (CC_SINK_PARTS, CC_SINK_COLUMNS, CC_SINK_TILES_*), null where a slot does not
    // apply: [CC_AUX_CENTERS] brick / tile centres (part masks), [CC_AUX_COLUMNS] column pass, [CC_AUX_FULL] full walk of the
    // flagged bricks
    void *jit_aux[CC_N_SINKS][3] = {};
    cc_columns_meta jit_meta[CC_N_SINKS];  // column buffer layout of each unit (columns false: no column split)
    cc_jit_cfg jit_cfg[CC_N_SINKS];
    size_t jit_smem[CC_N_SINKS] = {};  // dynamic shared memory of each specialised kernel
    bool jit_attr_done[CC_N_SINKS][CC_MAX_DEVICES] = {};  // MaxDynamicSharedMemorySize is a per-device attribute
    cc_jit_job *jit_job[CC_N_SINKS] = {};  // background compiles in flight
    bool jit_failed[CC_N_SINKS] = {};
    size_t jit_cubin_bytes = 0;
    double jit_seconds = 0;  // background compile time spent so far
    bool use_jit = true;     // per-program switch (cc_program_use_specialized)
};

// cc_jit.cpp
cc_jit_cfg cc_jit_default_cfg(const cc_decoded &dec, int pts);
bool cc_jit_is_segmented(const cc_decoded &dec);
int cc_jit_source(const cc_decoded &dec, int pts, unsigned sink_mask, std::string *src, std::string *err);
int cc_jit_nvrtc(const std::string &src, std::vector<char> *cubin, std::string *err);
int cc_jit_compile(cc_program *prog, int pts, unsigned sink_mask, double *seconds, std::string *err);
void cc_jit_start(cc_program *prog, int sink);
int cc_jit_poll(cc_program *prog, int sink, bool wait, std::string *err);
void cc_jit_release(cc_program *prog);
// dev_index = index of the library context (device) the launch goes to
int cc_jit_launch(const cc_program *prog, int sink, const cc_eval_args &a, void *stream, int dev_index);
// the brick and tile units (CC_SINK_PARTS, CC_SINK_COLUMNS, CC_SINK_TILES_*) over `n_units` bricks or tiles, one CTA each
// (CC_SINK_COLUMNS: one CTA per run of a.brick_run bricks, brick_runs):
// [centres ->] [column pass ->] main kernel [-> full walk of the flagged bricks].  A companion runs where the unit has it and
// the caller prepared its buffer (a.part_masks, a.columns, a.column_flags); `centers_only` stops after the centres.
int cc_jit_launch_units(const cc_program *prog, int sink, const cc_eval_args &a, uint64_t n_units, int sm_count, void *stream,
                        int dev_index, int *n_launches, bool centers_only = false);
int cc_jit_launch_render(const cc_program *prog, int sink, const cc_render_args &a, void *stream, int dev_index);
cc_jit_cfg cc_jit_render_cfg(const cc_decoded &dec);
#define CC_SINK_MASK_ALL ((1u << CC_N_SINKS) - 1u)
#define CC_RENDER_THREADS 128  // CTA size of the specialised image renderers

// ---- kernel launch layer (cc_kernels.cu) ------------------------------------------------

#include "cc_device_types.h"

struct cc_launch_cfg {
    int pts;         // points per thread: 1, 2, 4
    int prog_space;  // 1 = __constant__, 2 = shared
};

// launches on `stream`; returns cudaError_t as int
int cc_launch_eval(int sink, const cc_launch_cfg &cfg, const cc_eval_args &args, void *stream);
int cc_upload_constant_program(const uint32_t *h_code, uint32_t n_words, void *stream);
uint32_t cc_tile_points(const cc_launch_cfg &cfg);
size_t cc_eval_smem_bytes(const cc_launch_cfg &cfg, uint32_t n_slots, uint32_t code_words);

// image renderers around evaluate() (rendering/ray_caster.cl, rendering/bitmap.cl)
struct cc_render_launch {
    const uint32_t *code;
    uint32_t code_words, n_slots;
    float origin[3], forward[3], up[3], right[3];
    float pixel_tolerance, box_radius, min_distance, max_distance, floor_z, step_size;
    uint32_t options, w, h;
    uint8_t *out;
    unsigned long long *eval_count;
};
// prog_space 1 = constant bank, 2 = shared copy (interpreter kernels); 0 = the specialised kernel of `prog`
struct cc_program;
int cc_launch_render(int ray, int prog_space, const cc_program *prog, const cc_render_launch &r, void *stream, int dev_index);

// union-forest kernel (cc_forest.cu): dense float4 grids with per-tile culling
struct cc_forest_launch {
    const float *bounds;     // device, [n_leaves][8]
    const uint32_t *events;  // device, [n_events][4]
    uint32_t n_leaves, n_events, max_depth;
    float rmax, slack;
};
size_t cc_forest_smem_bytes(const cc_forest &f);          // of the (rare) second launch, the larger one
uint32_t cc_forest_overflow_words(const cc_eval_args &a);  // scratch the launch needs: deferred super-tiles
int cc_launch_forest(const cc_eval_args &a, const cc_forest_launch &f, uint32_t *d_overflow, int sm_count, void *stream);

// part culling on the interpreter tier (cc_parts.cu): brick-centre pass + one CTA per quarter brick
size_t cc_parts_smem_bytes(uint32_t n_slots, uint32_t code_words, int pts);
int cc_launch_parts_interp(const cc_eval_args &a, const uint32_t *d_table, uint32_t n_bricks, void *stream, bool centers_only = false);
struct cc_layer_weights {
    float base;      // per brick
    float part[32];  // per part a brick keeps
};
int cc_launch_layer_cost(const uint32_t *d_masks, uint32_t n_layers, uint32_t bricks_per_layer, const cc_layer_weights &w, double *d_out,
                         void *stream);

// hierarchy helper kernels
struct cc_level_geom {
    double ox, oy, oz;      // origin
    double resolution;
    double half_cell;       // int_step / 2 (leaf units) added to the int corner; 0 on flat axes
    int dimension;
};
// subdivision: corner = fp32((int_corner + int_step/2) * resolution + origin)   subdivision.py:55-65
int cc_launch_make_blocks_subdiv(const int64_t *d_int_corners, uint32_t n, cc_level_geom g,
                                 cc_block_desc *d_blocks, void *stream);
// children int corners from hits: child = parent + (x,y,z) * int_step         subdivision.py:91-94
int cc_launch_expand_children(const int64_t *d_parent_corners, const uint32_t *d_hit_block,
                              const uint8_t *d_hit_xyz, uint32_t n_hits, int64_t int_step,
                              uint32_t rank, uint32_t world, int64_t *d_child_corners, void *stream);
// mass properties: float64 corner chain + per-block integrals
int cc_launch_mass_make_blocks(const double *d_corners, uint32_t n, double s, cc_block_desc *d_blocks,
                               void *stream);
// d_hit_masks / d_child_masks (assemblies): the (eval, inside) part masks of every hit, copied to its child block
int cc_launch_mass_expand_children(const double *d_parent_corners, const uint32_t *d_hit_block,
                                   const uint8_t *d_hit_xyz, uint32_t n_hits, double s,
                                   uint32_t rank, uint32_t world, double *d_child_corners, void *stream,
                                   const uint32_t *d_hit_masks = nullptr, uint32_t *d_child_masks = nullptr);
// per-block integrals (mass_properties.py:139-148, float64) added to an exact fixed-point accumulator:
// d_limbs[10][4] signed 64-bit sums of the 32-bit limbs of trunc(value / 2^quantum_exp[i]); d_limbs[40]
// counts values outside the accumulator's range (must stay 0)
struct cc_mass_quanta { int e[10]; };
// n_sets sets of ten sums per block (stride 10 * n_sets), each into its own accumulator of 41 limbs
int cc_launch_mass_integrals(const double *d_corners, const uint32_t *d_sums, uint32_t n_blocks, double s,
                             cc_mass_quanta q, unsigned long long *d_limbs /* [n_sets][41] */, void *stream,
                             uint32_t n_sets = 1);

// ---- mass properties of an assembly's parts and pairs in one hierarchy pass (cc_assembly.cu, DESIGN.md 4.11) --------
#define CC_ASSEMBLY_MAX_PARTS 32
struct cc_assembly_part {
    const uint32_t *code;  // the part program's microcode on the launch's device
    uint32_t code_words, n_slots;
};
struct cc_assembly_args {
    cc_eval_args a;         // blocks x linear tiles of CC_THREADS x 2 cells; threshold, hit list, ticket and look-back
    cc_assembly_part part[CC_ASSEMBLY_MAX_PARTS];
    uint32_t n_parts;
    uint32_t max_slots;     // the dynamic shared memory (cc_parts_smem_bytes, 2 points) holds max_slots register slots, then one microcode
    const uint32_t *masks;  // per block: (eval, inside) part masks
    uint32_t *hit_masks;    // per hit: the child block's (eval, inside)
    uint32_t *sums;         // per block: n_parts + n_parts (n_parts - 1) / 2 sets of ten sums
};
int cc_launch_assembly(const cc_assembly_args &A, size_t smem, void *stream);

// ---- 2-D outline extraction (cc_polygon.cu, rendering/polygon2d.cl) -----------------------------
#ifdef __CUDACC__
#include <vector_types.h>
#else
struct float4;
struct float2;
#endif
struct cc_polygon_args {
    float corner_x, corner_y, step;  // boxCorner, boxStep (single block)
    const float *block_corners;      // optional: [n_blocks][2] fp32 corners (batched form)
    uint32_t cx, cy;                 // the OpenCL global size: cells per axis = samples - 1
    uint32_t n_blocks;
    const float4 *corners;           // [n_blocks][cx+1][cy+1]
    float2 *vertices;                // [n_blocks][cx][cy][2]
    uint32_t *links;                 // same shape
    uint32_t *starts;                // [n_blocks][max_starts]
    uint32_t *start_counter;         // [n_blocks], zeroed by the caller
    uint32_t max_starts;             // <= 1024
};
int cc_launch_process_polygon(const cc_polygon_args &a, void *stream);
int cc_launch_slice_repack(const void *d_field, uint32_t w, uint32_t h, float *d_out, void *stream);

// ---- marching cubes over leaf blocks (cc_mesh.cu) ---------------------------------------------
struct cc_mesh_args {
    const float *field;    // [n_blocks][d0*d1*d2], the array mcubes would receive: index (i*d1 + j)*d2 + k
    uint32_t d0, d1, d2;   // its numpy shape (the reference passes max_box_size, rendering/mesh.py:20)
    uint32_t n_blocks;
    uint32_t tiles_per_block;
    const double *corner;  // [n_blocks][3] box_corner (float64)
    double resolution;     // box_resolution (float64)
    uint32_t *counter;     // [2]: total triangles, non-empty tiles (written by the scan after the count pass)
    double *vertices;      // [n_triangles][3 vertices][3]  (emit pass)
    uint32_t *tri_block;   // [n_triangles] block of every triangle (emit pass)
    uint32_t first_block;  // added to the block index written to tri_block
    uint32_t *tile_offsets; // cc_mesh_scratch_words(tiles) words: triangle counts (count pass) -> exclusive offsets; scan scratch
    uint32_t *tile_list;    // ids of the tiles that hold triangles, increasing (inside the same scratch)

    // ---- indexed export only (cc_mesh_blocks_indexed); blocks are cubic when there are several ----
    // Block table of the whole call: block coordinates (int corner / (n-1)) in array axes (i = -y,
    // j = x, k = z), shifted to be non-negative, packed 21 bits each (i highest).
    const uint64_t *block_key;   // [n_all] key of every block, input order
    const uint64_t *sorted_key;  // [n_all] the same keys, increasing
    const uint32_t *sorted_block; // [n_all] block index of sorted_key[r]
    uint32_t n_all;              // blocks in the call
    uint32_t nf;                 // face archive row length: max(d0, d1, d2)
    float *face_field;           // [n_all][6 faces][nf][nf] each block's face samples as evaluated
    uint32_t *face_vertex;       // [n_all][6][nf][nf][2] global index of the owned vertex on each in-face edge
    uint32_t *vbase;             // [n_blocks * samples] owned crossed edges per sample -> exclusive vertex offsets in the chunk
    uint8_t *vmask;              // [n_blocks * samples] bit a: the edge along array axis a from this sample is owned and crossed
    uint32_t vert_base;          // vertices of the earlier chunks
    double *vert_out;            // [chunk vertices][3] (emit pass)
    uint32_t *triangles;         // [n_triangles][3] vertex indices (emit pass)
};

int cc_mesh_upload_tables(void *stream);
uint32_t cc_mesh_tiles_per_block(uint32_t d0, uint32_t d1, uint32_t d2);
int cc_launch_mesh(const cc_mesh_args &a, bool emit, uint32_t emit_tiles, void *stream);
size_t cc_mesh_scratch_words(uint32_t tiles);
// In-place exclusive scan of v[0..n) with the ids of the non-zero elements in `list`; scratch holds
// cc_mesh_scan_scratch_words(n) words.  counter[0] = sum, counter[1] = non-zero elements.
size_t cc_mesh_scan_scratch_words(uint32_t n);
int cc_launch_mesh_scan(uint32_t *v, uint32_t n, uint32_t *scratch, uint32_t *list, uint32_t *counter, void *stream);
// Indexed export, per chunk (after the PYMCUBES evaluation into a.field):
//   reconcile: archive the chunk's face samples, then replace every sample a block does not own with
//              its owner's value; then count the owned crossed edges per sample into vbase / vmask.
//   emit: vertex positions and face vertex indices, then (the tiles listed by the count pass) the
//         triangles as vertex indices.
int cc_launch_mesh_reconcile(const cc_mesh_args &a, void *stream);
int cc_launch_mesh_indexed_emit(const cc_mesh_args &a, uint32_t emit_tiles, void *stream);

#endif
