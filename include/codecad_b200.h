/* libcodecad_b200 — C ABI of the B200-native codecad SDF hot path.
 *
 * This library replaces the reference's OpenCL layer (codecad/cl_util + the .cl
 * kernels).  Every entry point is what a foreign-function binding of the reference
 * would bind in place of a pyopencl call; the reference interface each one replaces is
 * cited as /root/reference-relative file:line.  The Python ctypes binding lives in
 * codecad_b200/_lib.py; INTEGRATION.md shows the reference-side shim.
 *
 * Conventions: plain pointers and sizes only.  Every function returning `int` returns
 * 0 on success and a negative cc_status on failure; cc_last_error() then returns a
 * thread-local message.  One process drives one GPU (cc_init; one rank per GPU under
 * torchrun) or several (cc_init_devices); per device the library owns one compute stream and
 * one copy stream.  Host pointers are caller-owned; device pointers and handles are
 * library-owned until the matching *_free / *_destroy.  There is NO CPU fallback: with
 * no usable CUDA device cc_init() fails and every other call fails after it.
 */
#ifndef CODECAD_B200_H
#define CODECAD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum cc_status {
    CC_OK = 0,
    CC_ERR_CUDA = -1,          /* a CUDA runtime call failed (message has the detail)   */
    CC_ERR_NOT_INITIALIZED = -2,
    CC_ERR_INVALID_PROGRAM = -3, /* malformed word stream (bad opcode / truncated)      */
    CC_ERR_INVALID_ARGUMENT = -4,
    CC_ERR_TOO_LARGE = -5,     /* program or register demand exceeds device limits      */
    CC_ERR_OPEN_OUTLINE = -6   /* polygon(): an outline leaves the subdivided region (the
                                  reference's final assertion, rendering/polygon2d.py:172-173) */
} cc_status;

typedef struct cc_program cc_program; /* decoded node program resident on the device */
typedef struct cc_event cc_event;     /* completion marker on a library stream        */

/* output layouts of cc_grid_eval */
#define CC_LAYOUT_INDEX3_FLOAT4 0 /* grid_eval.cl:23-34  out[z + nz*(y + ny*x)] = (grad.xyz, dist) */
#define CC_LAYOUT_PYMCUBES_FLOAT 1 /* grid_eval.cl:2-21   out[z + (x + (ny-1-y)*nx)*nz] = dist      */

/* ---- context: replaces OpenCLManager.__init__  cl_util/opencl_manager.py:87-98 ------- */
int cc_init(int device);            /* idempotent for the same device */
/* Several GPUs driven by ONE process (the reference's user is a single Python script with one
 * context and one queue, cl_util/opencl_manager.py:89-98; SURVEY.md 8(b) asks for exactly this
 * entry point).  devices[0] is the primary device: buffers, events and every per-launch kernel
 * call live there, as after cc_init(devices[0]).  The calls that shard — cc_grid_eval_to_host
 * (x-slabs), cc_subdivide and cc_mass_properties (blocks of the hierarchy) — then use all n
 * devices, one worker thread, compute stream and copy stream per device, programs replicated on
 * first use, and return exactly what one device returns.  May be called after cc_init(devices[0]). */
int cc_init_devices(const int *devices, int n);
int cc_active_devices(void);        /* devices initialised in this process (0 before cc_init)  */
void cc_shutdown(void);
int cc_device_count(void);          /* 0 when no CUDA device/driver is usable */
const char *cc_last_error(void);
typedef struct cc_device_info {
    int device, sm_count, sm_clock_khz, l2_bytes;
    size_t total_mem;
    char name[64];
} cc_device_info;
/* PCI address ("0000:17:00.0") of CUDA device `device`, without creating a context on it: lets
 * the host side place its page-locked buffers on the NUMA node next to the GPU. */
int cc_device_pci_bus_id(int device, char *out, int capacity);
int cc_get_device_info(cc_device_info *out);
int cc_synchronize(void);
/* counters since cc_init / the last reset: kernels launched by this library and grid
 * points evaluated (the reference's dead `kernel_invocations` / `function_evaluations`
 * mass_properties.py:66-67,110-111). */
int cc_get_counters(uint64_t *kernel_launches, uint64_t *points_evaluated);
void cc_reset_counters(void);
/* warps of the column brick kernel (DESIGN.md 4.10) since cc_init / the last reset whose deferred
 * range check failed, so that they evaluated their cells again with the guarded full walk; waits
 * for the work queued so far. */
int cc_get_check_fallbacks(uint64_t *warps);
/* bricks of the column brick kernel since cc_init / the last reset that a column failing its run-time
 * check sent to the full walk (DESIGN.md 4.10); waits for the work queued so far. */
int cc_get_flagged_bricks(uint64_t *bricks);
/* tuning knobs, mainly for bench.py / profiling: points per thread (1,2,4; 0 = auto),
 * and where the microcode is fetched from (0 = auto, 1 = __constant__, 2 = shared). */
int cc_set_tuning(int points_per_thread, int program_space);

/* ---- programs: replaces make_program_buffer  nodes/program.py:79-84 ------------------- */
/* Copies and validates `n_words` float32 words (opcode table nodes/node.py:12-56,
 * encoding nodes/program.py:39-71), decodes them to device microcode, renames the
 * 512 wire registers to a dense slot set, uploads. */
int cc_program_create(const float *words, uint32_t n_words, cc_program **out);
void cc_program_destroy(cc_program *prog);
typedef struct cc_program_info {
    uint32_t n_words;        /* wire words consumed (up to and including _return)   */
    uint32_t n_instructions; /* wire instructions                                    */
    uint32_t n_micro_ops;    /* decoded instructions (stores folded)                 */
    uint32_t n_micro_words;  /* decoded length in 32-bit words                       */
    uint32_t n_wire_registers; /* highest wire register used + 1                     */
    uint32_t n_slots;        /* shared-memory value slots after liveness renaming    */
    uint32_t n_fused;        /* fused primitive micro-ops (MOP_PRIM_*)               */
    uint32_t flops_min;      /* static algorithmic flop/point, SURVEY.md 8(a3) rules */
    uint32_t flops_max;
    uint32_t n_forest_leaves; /* primitives of a union forest (cc_set_forest_mode), 0 = not one */
    uint32_t forest_depth;    /* its evaluation stack depth                                    */
    uint32_t n_parts;         /* parts of an assembly (cc_set_parts_mode), 0 = none            */
    uint32_t n_parts_bounded; /* of them: with a Lipschitz bound, i.e. cullable                */
    uint32_t column_invariant_percent; /* estimated share of the arithmetic that does not depend on the grid's z
                                          (2-D profiles under extrusions); evaluated once per z-column of a dense
                                          grid when >= 25 (cc_set_columns_mode), 0 = nothing to gain          */
    uint32_t column_axis;     /* the grid axis those columns run along: 0 = x, 1 = y, 2 = z                */
} cc_program_info;
int cc_program_get_info(const cc_program *prog, cc_program_info *out);
/* copies the decoded microcode (for tests / disassembly); returns the microcode length */
int cc_program_get_microcode(const cc_program *prog, uint32_t *out, uint32_t capacity);
/* Host-only decode (no device, no cc_init needed): validates `words`, fills `info` and
 * copies up to `capacity` microcode words to `out` (may be NULL).  Returns the microcode
 * length in words, or a negative cc_status.  Lets the loader be tested without a GPU. */
int cc_program_decode(const float *words, uint32_t n_words, cc_program_info *info,
                      uint32_t *out, uint32_t capacity);

/* ---- scene-specialised kernels (optional accelerator; SURVEY.md 8(f) rank 2) -------------
 * cc_program_specialize() turns the program's microcode into straight-line CUDA C++ that calls
 * the same op library, compiles it with NVRTC for sm_100a (-fmad=false) and loads it; afterwards
 * every kernel launched for this program uses the specialised code (bit-identical results, no
 * instruction fetch/dispatch).  Costs seconds of compile time, so it is opt-in; without NVRTC it
 * fails and the interpreter stays in use.  points_per_thread: 1, 2 or 4 (0 = default 2);
 * sink_mask: which kernels to build, bit k = sink k (1 float4 grid, 2 PyMCubes grid,
 * 4 subdivision_step, 8 mass_properties; 0 = all four) — each costs its own compile time,
 * sinks left out keep using the interpreter.
 * The reference can emit a straight-line C evaluator too: nodes/codegen.py:137-204. */
int cc_program_specialize(cc_program *prog, int points_per_thread, unsigned sink_mask,
                          double *compile_seconds);
int cc_program_use_specialized(cc_program *prog, int enable); /* returns 1 if specialised code is active */
/* Tiered execution (default): every program starts on the interpreter kernels while its
 * specialised kernel for the sink in use compiles on a background thread (cached in memory and in
 * $CODECAD_B200_CACHE or ~/.cache/codecad_b200); launches switch over when it is ready.  Results
 * are bit-identical in both tiers.  mode: 0 = interpreter only, 1 = background (default),
 * 2 = compile at first use and wait.  Environment: CODECAD_B200_JIT.  Programs with more than
 * CODECAD_B200_JIT_MAX_OPS (4096) micro-ops are only specialised on request; programs of more than a
 * few hundred micro-ops are compiled as segments that call shared, table-driven op functions.  Returns the old mode. */
int cc_set_jit_mode(int mode);
/* Union forests.  A program that is one tree of (rounded) unions over fused boxes / cylinders
 * (SURVEY.md 8(d) config C5: 500 rounded boxes) is recognised at load time; its dense float4 grids
 * (cc_grid_eval, cc_grid_eval_to_host) are then evaluated tile by tile, skipping in each tile the
 * primitives that provably cannot change a bit of its results (csrc/cc_forest.cu; the reference
 * walks the whole program for every point, nodes/codegen.py:17-63).  Bit-identical to the full
 * evaluation; needs no compilation and has no size limit short of 60 000 primitives.  mode 1 = on
 * (default; environment CODECAD_B200_FOREST), 0 = always evaluate everything.  Returns the old mode.
 * cc_program_get_forest_info: returns 1 and fills {primitives, unions, stack depth, events} if the
 * program is a union forest, else 0. */
int cc_set_forest_mode(int mode);
/* Parts.  A program whose value is a tree of sharp unions over self-contained sub-programs — the
 * components of an assembly, SURVEY.md 8(d) config C4 — gets, next to its specialised kernels, a pair
 * that evaluates dense float4 grids brick by brick and skips in every brick the parts that provably
 * cannot be the nearest there (Lipschitz bound of every part from the brick centre; csrc/cc_body.cuh).
 * Bit-identical to the full evaluation.  The interpreter kernels apply the same masks (a program is culled from its
 * first launch, not from the arrival of its specialised kernels), and the hierarchy kernels — subdivision,
 * mass_properties, the PyMCubes-layout fields of the mesh export — get a mask per tile of 1024 consecutive cells the
 * same way.  mode 1 = on (default; CODECAD_B200_PARTS), 0 = off. */
int cc_set_parts_mode(int mode);
/* Columns.  On a dense grid the grid's z axis is the z axis of the program's point, and a 2-D profile
 * under an extrusion (transform, polygon2d, involute gear, their CSG: shapes/simple2d.cl, polygons2d.cl,
 * gears.cl before simple3d.cl extrusion) reads x and y only: its value is the same in every cell of a
 * z-column.  The loader proves, micro-op by micro-op and component by component, what cannot depend on
 * the grid's z — or x, or y: the axis with the largest invariant share is taken — (cc_program_info.
 * column_invariant_percent, column_axis); the column kernels evaluate that once per column and only the
 * rest per cell.  Same arithmetic on the same operands: bit-identical.  Combines with
 * the parts' masks.  mode 1 = on (default; CODECAD_B200_COLUMNS), 0 = off.  Returns the old mode. */
int cc_set_columns_mode(int mode);
/* Load balance of x-slabs (SURVEY.md 8(e): "over-decompose"): with part culling the planes of a grid are no longer
 * equal work — the rim of an assembly's box is emptier than its middle.  Fills layer_cost[i], i < ceil(nx / 8), with an
 * estimate of the work in the i-th layer of eight x-planes: per brick a constant plus the micro-ops of the parts its
 * mask keeps (the brick-centre pass of cc_set_parts_mode; a program without parts reports equal layers).  Callers
 * cut the prefix sums into as many slabs as they have GPUs (codecad_b200.grid_eval.balanced_slabs).  Results of
 * grid_eval do not depend on where the slabs are cut. */
int cc_grid_eval_cost_profile(const cc_program *prog, const float corner[3], float step, uint32_t nx, uint32_t ny,
                              uint32_t nz, uint32_t x_offset, double *layer_cost, uint32_t n_layers);
int cc_program_get_forest_info(const cc_program *prog, uint32_t out[4]);
/* Blocks until the specialised kernels of the sinks in `sink_mask` (0 = all) are compiled and
 * loaded, starting their compilation if necessary; returns how many are ready.  compile_seconds
 * receives the background compile time spent on this program so far. */
int cc_program_specialize_wait(cc_program *prog, unsigned sink_mask, double *compile_seconds);
/* Host-only (no device): generate the source for `words` (returns its length, copies up to
 * `capacity` bytes incl. NUL), and optionally run NVRTC on it (compile != 0; returns the cubin
 * size through *cubin_bytes).  For tests and inspection. */
int cc_specialize_source(const float *words, uint32_t n_words, int points_per_thread,
                         unsigned sink_mask, char *out, uint32_t capacity, int compile,
                         uint64_t *cubin_bytes);

/* ---- buffers and events: replaces cl_util.Buffer  cl_util/cl_buffer.py:9-131 ---------- */
int cc_buffer_alloc(size_t bytes, void **dptr);
int cc_buffer_free(void *dptr);
int cc_host_alloc(size_t bytes, void **hptr); /* pinned; ALLOC_HOST_PTR cl_buffer.py:36-40 */
int cc_host_free(void *hptr);
int cc_memcpy_h2d_async(void *dptr, const void *hptr, size_t bytes, cc_event **ev);
int cc_memcpy_d2h_async(void *hptr, const void *dptr, size_t bytes, cc_event **ev);
int cc_memset_async(void *dptr, int value, size_t bytes, cc_event **ev);
int cc_event_record(cc_event **ev);     /* on the compute stream */
int cc_event_wait(cc_event *ev);        /* pyopencl.Event.wait()  */
int cc_event_elapsed_ms(cc_event *start, cc_event *end, float *ms); /* Event.profile */
void cc_event_destroy(cc_event *ev);

/* ---- kernels with the reference's per-launch semantics (the `opencl_manager.k.*`
 *      proxy, cl_util/opencl_manager.py:73-84).  `ev` may be NULL. ---------------------- */

/* grid_eval / grid_eval_pymcubes  grid_eval.cl:2-34.
 * point(x,y,z) = corner + step * (x + x_offset, y, z); d_out holds nx*ny*nz elements of
 * the layout's type.  x_offset lets a rank evaluate a slab of a larger grid with
 * bit-identical coordinates. */
int cc_grid_eval(const cc_program *prog, const float corner[3], float step,
                 uint32_t nx, uint32_t ny, uint32_t nz, uint32_t x_offset, int layout,
                 void *d_out, cc_event **ev);

/* evaluate() at arbitrary points: d_points = n x (x, y, z, unused) float4 on the device, d_out = n
 * float4 (gradient, distance).  This is what the reference's other kernels do around evaluate()
 * (tests/test_dsdf.cl:7-72 estimate_direction / actual_distance_to_surface, rendering/ray_caster.cl,
 * rendering/bitmap.cl): the call lets such callers live on the host side of the boundary. */
int cc_evaluate_points(const cc_program *prog, const float *d_points, uint64_t n, void *d_out, cc_event **ev);

/* ---- image renderers around evaluate() (SURVEY.md 8(f) rank 4) --------------------------------
 * ray_caster  rendering/ray_caster.cl:147-256, launched by rendering/ray_caster.py:55-71 with global
 * size (width, height): sphere tracing with over-relaxation, soft shadow ray, 4-tap ambient
 * occlusion and floor shadow.  Arguments are the kernel's own (forward is already scaled by the
 * focal length, ray_caster.py:39-43); render_options: 1 = false colour, 2 = zebra
 * (ray_caster.py:13-15).  d_out = width*height*3 bytes in the reference's INDEX2 order
 * ((y + height*x)*3, cl_util/indexing.h:3), i.e. the numpy array [width][height][3] that
 * ray_caster.py:89 transposes.  eval_count (may be NULL; makes the call blocking) receives the
 * number of evaluate() calls the rays made. */
int cc_ray_caster(const cc_program *prog, const float origin[3], const float forward[3], const float up[3],
                  const float right[3], float pixel_tolerance, float box_radius, float min_distance,
                  float max_distance, float floor_z, uint32_t render_options, uint32_t width, uint32_t height,
                  uint8_t *d_out, uint64_t *eval_count, cc_event **ev);

/* bitmap  rendering/bitmap.cl:1-18 (global size (width, height), rendering/bitmap.py:27-29):
 * pixel (x, y) shows the sign of the distance at origin + step_size * (x, height - y - 1, 0). */
int cc_bitmap(const cc_program *prog, const float origin[3], float step_size, uint32_t width, uint32_t height,
              uint8_t *d_out, cc_event **ev);

/* Same, result delivered to HOST memory: slabs of the grid are evaluated into a device
 * ring and copied out on the copy stream while the next slab computes.  Blocking.
 * Replaces kernel + Buffer.read()  (rendering/mesh.py:53-61). */
int cc_grid_eval_to_host(const cc_program *prog, const float corner[3], float step,
                         uint32_t nx, uint32_t ny, uint32_t nz, uint32_t x_offset, int layout,
                         void *h_out);

/* subdivision_step  subdivision.cl:12-30: cells with -thr < dist < thr are appended to
 * d_list as uchar4 (x,y,z,0) starting at *d_counter, which is advanced.  Unlike the
 * reference's atomic_inc the order is deterministic: INDEX3 order (x slowest). */
int cc_subdivision_step(const cc_program *prog, const float corner[3], float step, float threshold,
                        uint32_t nx, uint32_t ny, uint32_t nz,
                        uint32_t *d_counter, uint8_t *d_list, cc_event **ev);

/* mass_properties  mass_properties.cl:7-56: dist <= -thr adds the 10 index products
 * (order xx,xy,xz,x,yy,yz,y,zz,z,n) to d_sums; -thr < dist < thr appends to d_list. */
int cc_mass_properties_step(const cc_program *prog, const float corner[3], float step, float threshold,
                            uint32_t nx, uint32_t ny, uint32_t nz, uint32_t *d_sums,
                            uint32_t *d_counter, uint8_t *d_list, cc_event **ev);

/* ---- whole-hierarchy fast paths (device-resident work lists, one launch per level) ---- */
typedef struct cc_level {
    int64_t cell_size;   /* in leaf units (subdivision.calculate_block_sizes [i][0]) */
    uint32_t nx, ny, nz; /* grid dims of a block at this level ([i][1])              */
} cc_level;

/* subdivision()  subdivision.py:169-253 for n_levels >= 2.  origin = expanded bbox.a,
 * float64 like the reference's host math.  Returns the int corners (resolution units)
 * of the leaf blocks owned by `rank` of `world`: the hits of the level that feeds the last
 * classified level are dealt round-robin, the (tiny) levels above it are evaluated by everyone.
 * With several devices (cc_init_devices) the rank's share is dealt on over them and merged back
 * into the order one device produces.  *out_corners is a malloc'ed int64[n][3] released with
 * cc_free.  cc_sort_leaf_corners puts a union of per-rank lists into that same order (level by
 * level: parent block order, then INDEX3 cell order), so that results can be compared as arrays. */
int cc_subdivide(const cc_program *prog, const double origin[3], double resolution,
                 const cc_level *levels, uint32_t n_levels, int dimension,
                 uint32_t rank, uint32_t world, int64_t **out_corners, uint64_t *out_count);
int cc_sort_leaf_corners(int64_t *corners, uint64_t n, const cc_level *levels, uint32_t n_levels);

/* mass_properties()  mass_properties.py:30-177: the ten integrals (one,x,y,z,xx,yy,zz,xy,xz,yz)
 * over the part of the hierarchy owned by `rank` of `world` (all of it for world = 1), shared out
 * over the devices of cc_init_devices; finish with mass_properties.py:179-229.
 * stats[0..3] = launches, evaluated cells, blocks, levels.
 *
 * Exactness.  Each block's ten float64 values (mass_properties.py:139-148, the reference's
 * expression order) are added in an exact fixed-point accumulator instead of the reference's
 * Kahan sum in job order (util/math.py:4-21), so the result does not depend on the order of the
 * blocks nor on how they are dealt to devices and ranks: 1, 2, 4 and 8 GPUs return the same bits.
 * cc_mass_properties_exact returns the accumulator itself: limbs[10][4] = signed sums of the
 * 32-bit limbs of trunc(value / 2^exponents[i]); ranks add their limbs (an int64 all-reduce, NCCL
 * or gloo) and convert once with cc_mass_limbs_to_integrals.  exponents depend on the arguments
 * only.  stats[4..7] = blocks of the dealt level owned, devices used, cells evaluated by the
 * busiest and by the least busy device. */
int cc_mass_properties(const cc_program *prog, const double box_a[3], double resolution,
                       const cc_level *levels, uint32_t n_levels,
                       uint32_t rank, uint32_t world, double integrals[10], uint64_t stats[4]);
int cc_mass_properties_exact(const cc_program *prog, const double box_a[3], double resolution,
                             const cc_level *levels, uint32_t n_levels, uint32_t rank, uint32_t world,
                             int64_t limbs[40], int32_t exponents[10], uint64_t stats[8]);
int cc_mass_limbs_to_integrals(const int64_t limbs[40], const int32_t exponents[10], double integrals[10]);

/* Mass properties of an assembly: every part, and the overlap of every pair of parts, in one
 * hierarchy pass (DESIGN.md 4.11).  parts[0..n_parts) (1 <= n_parts <= 32) are ordinary programs,
 * already placed; box_a, resolution and levels are those of cc_mass_properties_exact.
 *
 * The hierarchy is mass_properties' (same blocks, float64 corner chain, fp32 cell coordinates and
 * thresholds; leaf threshold 0).  Every block carries `eval`, the parts undecided at its parent
 * cell (the root: all), and `inside`, the parts decided inside at an ancestor cell (the root:
 * none).  In a cell only the parts of `eval` are evaluated; part k is inside if D_k <= -thr, near
 * if not inside and D_k < thr, outside otherwise (NaN included).  With N the parts newly inside and
 * U the parts near:
 *   - the cell's ten index products go into part k's sums for every k in N;
 *   - ... and into pair {a, b}'s sums for every a in N, b in N u inside, a != b (once per pair);
 *   - U nonempty: the cell becomes a child block with eval = U, inside = inside u N.
 * So set k is bit for bit cc_mass_properties_exact(parts[k], ...) (part k is evaluated in exactly
 * the blocks of its own hierarchy), and pair {a, b} is the intersection of the two parts' counted
 * regions: [A, A] gives pair = A.  For 1-Lipschitz fields vol(A u B) = vol A + vol B - vol AB.
 *
 * limbs[sets][40] with sets = n_parts + n_parts (n_parts - 1) / 2: the parts, then pair {a < b}
 * at n_parts + a n_parts - a (a + 1) / 2 + (b - a - 1); each set is an accumulator of
 * cc_mass_properties_exact (same exponents, same sharding over ranks and devices).  stats as
 * there.  CC_ERR_INVALID_ARGUMENT: no parts, more than 32, a null part, bad rank / world, an
 * accumulator out of range; CC_ERR_TOO_LARGE: the parts' slots and microcode exceed a CTA's shared
 * memory. */
int cc_assembly_mass_properties_exact(const cc_program *const *parts, uint32_t n_parts, const double box_a[3],
                                      double resolution, const cc_level *levels, uint32_t n_levels,
                                      uint32_t rank, uint32_t world, int64_t *limbs /* sets x 40 */,
                                      int32_t exponents[10], uint64_t stats[8]);

/* matplotlib_slice  rendering/matplotlib_slice.cl:1-20 (global size (width, height),
 * rendering/matplotlib_slice.py:44-52): d_out[(x + y*width)*3 + 0..2] = distance, gradient x,
 * gradient y at corner + step * (x, y, 0) — the numpy array [height][width][3] the viewer plots. */
int cc_matplotlib_slice(const cc_program *prog, const float corner[3], float step, uint32_t width, uint32_t height,
                        float *d_out, cc_event **ev);

/* ---- 2-D outlines (SURVEY.md 8(f) rank 4): rendering/polygon2d.cl + the device half of
 * rendering/polygon2d.py:36-173.
 * process_polygon  polygon2d.cl:82-175 with global size (cells_x, cells_y, 2): d_corners is the
 * float4 grid [cells_x+1][cells_y+1] grid_eval wrote (INDEX2), d_vertices float2 and d_links uint32
 * per triangle in INDEX3 order t + 2*(y + cells_y*x), d_starts the encoded starts of open chains and
 * *d_start_counter (zeroed by the caller, polygon2d.py:100) their number.  Unlike the reference's
 * atomic_inc order the starts come out ordered by cell index.  max_starts (<= 1024) is the capacity
 * of d_starts (cells_x + cells_y in the reference, polygon2d.py:63-69). */
int cc_process_polygon(const float box_corner[2], float box_step, uint32_t cells_x, uint32_t cells_y,
                       const void *d_corners, void *d_vertices, uint32_t *d_links, uint32_t *d_starts,
                       uint32_t max_starts, uint32_t *d_start_counter, cc_event **ev);

/* The per-box loop of polygon2d.py:80-117 for n_blocks equally sized boxes in two launches:
 * grid_eval of every box (gx*gy samples at fp32(corners[b]) + step*(x, y), corners float64 [n][3])
 * and process_polygon of every box; results land in caller-owned HOST arrays
 * h_vertices [n][2*(gx-1)*(gy-1)][2] float, h_links [n][2*(gx-1)*(gy-1)], h_starts [n][gx+gy-2],
 * h_start_counts [n].  Vertices of triangles the outline does not cross are zero.  Blocking. */
int cc_polygon_blocks(const cc_program *prog, const double *corners, double resolution, uint32_t gx, uint32_t gy,
                      uint32_t n_blocks, float *h_vertices, uint32_t *h_links, uint32_t *h_starts,
                      uint32_t *h_start_counts);

/* Host half of polygon() (no device work, usable without cc_init): follows the links that
 * process_polygon wrote for n_blocks boxes (arrays as returned by cc_polygon_blocks; `links` is
 * overwritten with visit marks) into closed outlines — rendering/polygon2d.py:15-31 and :119-170.
 * Chains closed inside a box come out in increasing order of their first triangle; chains that cross
 * box borders are joined through the (box corner, side + row) keys of polygon2d.py:131,141-144, with
 * int_corners [n][3] and int_step = int_resolution * (box_size - 1).  Results: malloc'ed
 * out_vertices float[total][2] and out_offsets uint64[chains + 1] (release with cc_free).
 * CC_ERR_OPEN_OUTLINE if a chain never closes. */
int cc_polygon_assemble(const float *vertices, uint32_t *links, const uint32_t *starts,
                        const uint32_t *start_counts, const int64_t *int_corners, int64_t int_step,
                        uint32_t cells, uint32_t max_starts, uint32_t n_blocks, float **out_vertices,
                        uint64_t **out_offsets, uint64_t *out_chains);

/* ---- mesh export (SURVEY.md 8(f) rank 1): replaces the per-block loop of rendering/mesh.py:36-74
 * (grid_eval_pymcubes launch + blocking device->host copy + mcubes.marching_cubes on the CPU).
 * For each of the n_blocks equally sized leaf blocks (nx,ny,nz samples, float64 corners[n][3] =
 * box_corner, rounded to fp32 per block like Vector.as_float4()): evaluate the distance field in
 * the PyMCubes layout on the device, run marching cubes at isovalue 0 (PyMCubes 0.0.6 conventions,
 * vertices interpolated in float64) and apply the reference's post-transform (mesh.py:68-72: swap
 * x/y, negate y, scale by `resolution`, translate by the corner, flip the winding).  Returns a
 * triangle soup in world coordinates: malloc'ed vertices[n_triangles][3][3] (float64) and the block
 * index of every triangle, blocks in input order, cells in (i,j,k) order; release with cc_free. */
int cc_mesh_blocks(const cc_program *prog, const double *corners, double resolution,
                   uint32_t nx, uint32_t ny, uint32_t nz, uint32_t n_blocks,
                   double **out_vertices, uint32_t **out_triangle_block, uint64_t *out_triangles);

/* Welded mesh of the same blocks: every vertex once, triangles as vertex indices, watertight by
 * construction.  int_corners[n][3] are the blocks' int corners (resolution units, LeafBlocks.int_corners).
 * Neighbouring blocks share their face samples; each block evaluates them from its own fp32 corner,
 * so the copies can differ in their last bits.  Here every shared sample takes the value of the
 * first block in input order that holds it (array index (i,j,k) of a block is the lattice point
 * (X + j, Y + ny-1-i, Z + k)), and marching cubes runs on these fields with the triangle order,
 * winding and triangle_block of cc_mesh_blocks.  One vertex per crossed lattice edge, placed as
 * cc_mesh_blocks places it in the edge's owner (the first block holding both ends); vertices are
 * ordered by owner block, then lower end in (i,j,k) order, then edge axis.  Results, page-locked,
 * released with cc_free: vertices[n_vertices][3] (float64), triangles[n_triangles][3] (uint32) and
 * triangle_block[n_triangles].  Where no shared sample differs, vertices[triangles] is
 * cc_mesh_blocks' soup bit for bit.  CC_ERR_INVALID_ARGUMENT for several blocks that are not cubic,
 * int corners that are not all congruent modulo n-1, repeated int corners, or blocks spread over
 * 2^21 or more block widths along an axis. */
int cc_mesh_blocks_indexed(const cc_program *prog, const double *corners, const int64_t *int_corners,
                           double resolution, uint32_t nx, uint32_t ny, uint32_t nz, uint32_t n_blocks,
                           double **out_vertices, uint64_t *out_n_vertices, uint32_t **out_triangles,
                           uint32_t **out_triangle_block, uint64_t *out_n_triangles);

void cc_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* CODECAD_B200_H */
