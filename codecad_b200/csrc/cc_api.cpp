// C ABI of libcodecad_b200 (see include/codecad_b200.h): context, programs, buffers,
// events, the four reference-semantics kernels and the device-resident hierarchy drivers.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <thread>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "cc_internal.h"

struct cc_event {
    cudaEvent_t ev;
};

namespace {

thread_local std::string g_err;

struct Context {
    bool ready = false;
    int device = -1;
    cudaDeviceProp prop;
    cudaStream_t compute = nullptr, copy = nullptr, copy2 = nullptr;
    uint64_t launches = 0, points = 0;
    int pts = 0, prog_space = 0;  // tuning overrides, 0 = auto
    int jit_mode = 1;             // 0 never, 1 background (default), 2 compile at first use and wait
    int forest_mode = 1;          // 1: dense grids of union-forest programs use the culling kernel (cc_forest.cu)
    int parts_mode = 1;           // 1: dense grids of assemblies skip, per brick, the parts that cannot be nearest
    int columns_mode = 1;         // 1: dense grids evaluate what cannot see z once per z-column (DESIGN.md 4.10)
    void *d_columns = nullptr;    // column buffer of the column kernels (values, flags, brick list)
    size_t columns_cap = 0;
    uint32_t *d_part_masks = nullptr;
    size_t part_masks_cap = 0;
    uint32_t jit_max_ops = 4096;  // programs longer than this are not specialised automatically
    uint64_t constant_program = 0;  // id of the program in this device's __constant__ window
    int index = 0;                  // position in g_ctx
    bool mesh_tables = false;       // marching-cubes tables uploaded to this device
    // look-back scratch
    uint32_t *d_forest_scratch = nullptr;  // deferred super-tiles of the union-forest kernel
    size_t forest_scratch_words = 0;
    uint32_t *d_ticket = nullptr;
    unsigned long long *d_status = nullptr;
    size_t status_cap = 0;
    // pinned bounce word for counters
    uint32_t *h_word = nullptr;
    // device ring + events of cc_grid_eval_to_host, kept between calls
    static const int kRing = 4;
    void *ring[kRing] = {nullptr, nullptr, nullptr, nullptr};
    size_t ring_bytes = 0;
    cudaEvent_t ring_computed[kRing] = {}, ring_copied[kRing] = {};
};
// One context per device the process drives (cc_init: one; cc_init_devices: several).  Every
// function body below works on "the current context" `g`: contexts[0] on the caller's thread, and
// contexts[i] on the worker thread that serves device i while a call is fanned out over the
// devices (for_each_device).
Context g_ctx[CC_MAX_DEVICES];
int g_n_ctx = 0;
thread_local Context *tl_ctx = &g_ctx[0];
thread_local int tl_device = -1;  // device this thread last made current through the library
#define g (*tl_ctx)
std::mutex g_mu, g_jit_mu;
std::atomic<uint64_t> g_next_program_id{1};

int fail(int code, const std::string &msg)
{
    g_err = msg;
    return code;
}

int cuda_fail(cudaError_t e, const char *what)
{
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return CC_ERR_CUDA;
}

#define CU(call)                                        \
    do {                                                \
        cudaError_t e_ = (call);                        \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call); \
    } while (0)

// (the CUDA current device is per thread: a caller's thread other than the one that ran cc_init
// would otherwise talk to device 0)
#define NEED_INIT()                                                             \
    do {                                                                        \
        if (!g.ready) return fail(CC_ERR_NOT_INITIALIZED, "cc_init() has not succeeded"); \
        if (tl_device != g.device) {                                            \
            CU(cudaSetDevice(g.device));                                        \
            tl_device = g.device;                                               \
        }                                                                       \
    } while (0)

int make_event(cc_event **ev, cudaStream_t st)
{
    if (!ev) return CC_OK;
    cc_event *e = new cc_event;
    cudaError_t r = cudaEventCreate(&e->ev);
    if (r == cudaSuccess) r = cudaEventRecord(e->ev, st);
    if (r != cudaSuccess) {
        delete e;
        return cuda_fail(r, "cudaEventRecord");
    }
    *ev = e;
    return CC_OK;
}

int ensure_status(size_t tiles)
{
    if (!g.d_ticket) CU(cudaMalloc(&g.d_ticket, 4));
    if (tiles > g.status_cap) {
        if (g.d_status) CU(cudaFree(g.d_status));
        size_t cap = std::max<size_t>(tiles, 1 << 16);
        CU(cudaMalloc(&g.d_status, cap * sizeof(unsigned long long)));
        g.status_cap = cap;
    }
    return CC_OK;
}

// pick points-per-thread / program space for a program
int choose_cfg(const cc_program *prog, uint64_t total_points, cc_launch_cfg *cfg)
{
    const uint32_t words = prog->dec.info.n_micro_words;
    const uint32_t slots = prog->dec.info.n_slots;
    const size_t smem_max = g.prop.sharedMemPerBlockOptin;
    // microcode in the constant bank (uniform loads, parameters stay in uniform registers)
    // whenever it fits the 63 KB window; larger programs are staged in shared memory
    // 1 = constant bank, 2 = shared copy, 3 = hybrid (headers constant, parameters shared)
    int space = g.prog_space;
    if (space == 0) space = 1;  // hybrid (3) measured slower on B200: 2.2 vs 2.7 Gpts/s on planetary
    if (space != 2 && words > CC_CONST_WORDS) space = 2;
    // two points per thread measured best on B200 (profiles/r1_ab_variants.md): four halve the
    // resident warps without enough extra ILP to pay for it
    int pts = g.pts ? g.pts : 2;
    if (pts != 1 && pts != 2 && pts != 4) pts = 2;
    // small launches: fewer points per thread keeps more SMs busy
    if (!g.pts) {
        while (pts > 1 && total_points < (uint64_t)g.prop.multiProcessorCount * 128u * pts * 2u) pts >>= 1;
    }
    for (;;) {
        cfg->pts = pts;
        cfg->prog_space = space;
        size_t need = cc_eval_smem_bytes(*cfg, slots, words);
        // want at least two CTAs per SM when possible
        if (need * 2 <= (size_t)g.prop.sharedMemPerMultiprocessor - 2048 || pts == 1) {
            if (need > smem_max) {
                if (space != 1 && words <= CC_CONST_WORDS) {
                    space = 1;
                    continue;
                }
                return fail(CC_ERR_TOO_LARGE, "program needs " + std::to_string(need) +
                                                  " bytes of shared memory per CTA (limit " +
                                                  std::to_string(smem_max) + ")");
            }
            return CC_OK;
        }
        pts >>= 1;
    }
}

int prepare_program(const cc_program *prog, const cc_launch_cfg &cfg)
{
    if (cfg.prog_space != 2 && g.constant_program != prog->id) {
        int e = cc_upload_constant_program(prog->dec.microcode.data(), prog->dec.info.n_micro_words, g.compute);
        if (e) return cuda_fail((cudaError_t)e, "cudaMemcpyToSymbolAsync");
        g.constant_program = prog->id;
    }
    return CC_OK;
}

// Page-locked result buffers handed to the caller (cc_mesh_blocks) and returned through cc_free.
// A device-to-host copy into fresh pageable memory runs at 3 GB/s (staging + page faults: 110 ms
// for the 328 MB of a 4.3 M-triangle mesh); into pinned memory it runs at PCIe speed (7 ms), but
// cudaHostAlloc itself costs ~0.3 ms/MB, so released buffers are kept (up to kRetain bytes) and
// reused by the next call of similar size.
struct PinnedPool {
    static constexpr size_t kRetain = 2ull << 30;
    std::mutex mu;
    std::multimap<size_t, void *> idle;
    std::unordered_map<void *, size_t> live;
    size_t retained = 0;

    void *get(size_t bytes)
    {
        const size_t granule = 1u << 20;
        const size_t want = (std::max<size_t>(bytes, 1) + granule - 1) / granule * granule;
        {
            std::lock_guard<std::mutex> lk(mu);
            auto it = idle.lower_bound(want);
            if (it != idle.end() && it->first <= want + want / 2) {
                void *p = it->second;
                retained -= it->first;
                live[p] = it->first;
                idle.erase(it);
                return p;
            }
        }
        void *p = nullptr;
        if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            trim(0);  // give idle blocks back and retry once
            if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                return nullptr;
            }
        }
        std::lock_guard<std::mutex> lk(mu);
        live[p] = want;
        return p;
    }
    // true if p was one of ours
    bool put(void *p)
    {
        size_t sz;
        {
            std::lock_guard<std::mutex> lk(mu);
            auto it = live.find(p);
            if (it == live.end()) return false;
            sz = it->second;
            live.erase(it);
            if (retained + sz <= kRetain) {
                idle.emplace(sz, p);
                retained += sz;
                return true;
            }
        }
        cudaFreeHost(p);
        return true;
    }
    void trim(size_t keep)
    {
        std::lock_guard<std::mutex> lk(mu);
        while (retained > keep && !idle.empty()) {
            auto it = std::prev(idle.end());
            cudaFreeHost(it->second);
            retained -= it->first;
            idle.erase(it);
        }
    }
};
PinnedPool g_pinned;

// the program's microcode on the current device (replicated on first use)
int program_on_device(const cc_program *prog, const uint32_t **out)
{
    cc_program *p = const_cast<cc_program *>(prog);
    uint32_t *&d = p->d_code[g.index];
    if (!d) {
        const size_t bytes = p->dec.microcode.size() * 4;
        cudaError_t e = cudaMalloc(&d, bytes);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d, p->dec.microcode.data(), bytes, cudaMemcpyHostToDevice, g.compute);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g.compute);
        if (e != cudaSuccess) {
            if (d) cudaFree(d);
            d = nullptr;
            return cuda_fail(e, "program upload");
        }
    }
    *out = d;
    return CC_OK;
}

int fill_common(cc_eval_args *a, const cc_program *prog)
{
    std::memset(a, 0, sizeof(*a));
    int rc = program_on_device(prog, &a->code);
    if (rc) return rc;
    a->code_words = prog->dec.info.n_micro_words;
    a->n_slots = prog->dec.info.n_slots;
    return CC_OK;
}
#define FILL_COMMON(a, prog)                 \
    do {                                     \
        int rc_ = fill_common(&(a), (prog)); \
        if (rc_) return rc_;                 \
    } while (0)

int check_dims(uint32_t nx, uint32_t ny, uint32_t nz)
{
    if (nx == 0 || ny == 0 || nz == 0) return fail(CC_ERR_INVALID_ARGUMENT, "empty grid");
    uint64_t cells = (uint64_t)nx * ny * nz;
    if (cells > (1ull << 31)) return fail(CC_ERR_INVALID_ARGUMENT, "more than 2^31 cells in one launch");
    return CC_OK;
}

// Tiered execution: a program starts on the interpreter; its scene-specialised kernel for `sink`
// is compiled on a background thread (NVRTC, cached in memory and on disk) and takes over as soon
// as it is ready.  Both tiers produce identical bits (same op library, same -fmad=false contract).
bool jit_ready(cc_program *p, int sink)
{
    std::lock_guard<std::mutex> lk(g_jit_mu);  // device threads of a fanned-out call share the program
    if (!p->use_jit) return false;
    if (p->jit_kernel[sink]) return true;
    if (g.jit_mode == 0 || p->jit_failed[sink]) return false;
    if (p->dec.info.n_micro_ops > g.jit_max_ops) return false;
    cc_jit_start(p, sink);
    std::string err;
    int r = cc_jit_poll(p, sink, g.jit_mode == 2, &err);
    if (r < 0)
        std::fprintf(stderr, "libcodecad_b200: kernel specialisation failed, staying on the interpreter: %s\n",
                     err.c_str());
    return r == 1;
}

// tables of a union-forest program on the current device (replicated on first use)
int forest_on_device(const cc_program *prog, cc_forest_launch *out)
{
    cc_program *p = const_cast<cc_program *>(prog);
    const cc_forest &f = p->dec.forest;
    void *&d = p->d_forest[g.index];
    const size_t nb = f.bounds.size() * 4, ne = f.events.size() * 4;
    if (!d) {
        cudaError_t e = cudaMalloc(&d, nb + ne);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d, f.bounds.data(), nb, cudaMemcpyHostToDevice, g.compute);
        if (e == cudaSuccess) e = cudaMemcpyAsync((char *)d + nb, f.events.data(), ne, cudaMemcpyHostToDevice, g.compute);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g.compute);
        if (e != cudaSuccess) {
            if (d) cudaFree(d);
            d = nullptr;
            return cuda_fail(e, "forest table upload");
        }
    }
    out->bounds = (const float *)d;
    out->events = (const uint32_t *)((char *)d + nb);
    out->n_leaves = f.n_leaves;
    out->n_events = f.n_events;
    out->max_depth = f.max_depth;
    out->rmax = f.rmax;
    return CC_OK;
}

bool forest_applies(int sink_kind, const cc_program *prog, const cc_eval_args &a)
{
    if (!g.forest_mode || sink_kind != CC_SINK_FLOAT4 || a.points || a.blocks) return false;
    const cc_forest &f = prog->dec.forest;
    return f.enabled && cc_forest_smem_bytes(f) <= (size_t)g.prop.sharedMemPerBlockOptin && f.n_events <= 8192 &&
           f.n_leaves <= 8192;
}

int launch_forest(const cc_program *prog, cc_eval_args &a, uint64_t points)
{
    cc_forest_launch f;
    int rc = forest_on_device(prog, &f);
    if (rc) return rc;
    // error budget of the primitives' bounds: 2^-16 of the magnitudes that enter their arithmetic
    const double ext[3] = {std::fabs((double)a.step) * (double)(a.nx + a.x_offset), std::fabs((double)a.step) * a.ny,
                           std::fabs((double)a.step) * a.nz};
    // (forest_applies admits no launch over blocks: the grid's own corner bounds the coordinates)
    const double pmax = std::max(std::fabs((double)a.cx) + ext[0], std::max(std::fabs((double)a.cy) + ext[1], std::fabs((double)a.cz) + ext[2]));
    f.slack = (float)(((double)prog->dec.forest.err_a + (double)prog->dec.forest.err_b * pmax) / 65536.0);
    if (!std::isfinite(f.slack)) return fail(CC_ERR_INVALID_ARGUMENT, "grid coordinates out of range");
    const size_t ow = cc_forest_overflow_words(a);
    if (ow > g.forest_scratch_words) {
        if (g.d_forest_scratch) CU(cudaFree(g.d_forest_scratch));
        g.d_forest_scratch = nullptr;
        g.forest_scratch_words = 0;
        CU(cudaMalloc(&g.d_forest_scratch, ow * 4));
        g.forest_scratch_words = ow;
    }
    int e = cc_launch_forest(a, f, g.d_forest_scratch, g.prop.multiProcessorCount, g.compute);
    if (e) return cuda_fail((cudaError_t)e, "cc_forest_kernel launch");
    g.launches += 1;
    g.points += points;
    return CC_OK;
}

// Dense float4 grid of an assembly through the part-culling kernels (DESIGN.md 4.9); the caller checked
// that the specialised kernels of CC_SINK_PARTS are loaded.
// cc_parts::table on the current device (replicated on first use)
int parts_on_device(const cc_program *prog, const uint32_t **out)
{
    cc_program *p = const_cast<cc_program *>(prog);
    uint32_t *&d = p->d_parts[g.index];
    if (!d) {
        const size_t bytes = p->dec.parts.table.size() * 4;
        cudaError_t e = cudaMalloc(&d, bytes);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d, p->dec.parts.table.data(), bytes, cudaMemcpyHostToDevice, g.compute);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g.compute);
        if (e != cudaSuccess) {
            if (d) cudaFree(d);
            d = nullptr;
            return cuda_fail(e, "part table upload");
        }
    }
    *out = d;
    return CC_OK;
}

// the brick masks' buffer and the rounding budget of the parts' values
int prepare_part_masks(const cc_program *prog, cc_eval_args &a, uint64_t nb)
{
    if (nb > g.part_masks_cap) {
        if (g.d_part_masks) CU(cudaFree(g.d_part_masks));
        g.d_part_masks = nullptr;
        g.part_masks_cap = 0;
        CU(cudaMalloc(&g.d_part_masks, (size_t)nb * 4));
        g.part_masks_cap = (size_t)nb;
    }
    // rounding budget of a part's value: 2^-13 of the magnitudes that enter its arithmetic (a part is at
    // most a few hundred fp32 operations deep: ~1e-5 relative; this allows 1.2e-4)
    const double ext[3] = {std::fabs((double)a.step) * (double)(a.nx + a.x_offset), std::fabs((double)a.step) * a.ny,
                           std::fabs((double)a.step) * a.nz};
    // (launches over blocks: a.cx/cy/cz are zero and the corners are in the block descriptors; the caller's
    // bound on every block's coordinates stands in for them)
    const double pmax = a.blocks ? (double)a.coord_max + std::max(ext[0], std::max(ext[1], ext[2]))
                                 : std::max(std::fabs((double)a.cx) + ext[0], std::max(std::fabs((double)a.cy) + ext[1], std::fabs((double)a.cz) + ext[2]));
    a.part_slack = (float)(((double)prog->dec.parts.magnitude_a + (double)prog->dec.parts.magnitude_b * pmax) / 8192.0);
    if (!std::isfinite(a.part_slack)) return fail(CC_ERR_INVALID_ARGUMENT, "grid coordinates out of range");
    a.part_masks = g.d_part_masks;
    return CC_OK;
}

// `specialised`: the NVRTC pair is loaded; otherwise the interpreter-tier pair of cc_parts.cu
int launch_parts(const cc_program *prog, cc_eval_args &a, uint64_t points, bool specialised)
{
    const uint64_t nb = (uint64_t)((a.nx + CC_BRICK_X - 1) / CC_BRICK_X) * ((a.ny + CC_BRICK_Y - 1) / CC_BRICK_Y) *
                        ((a.nz + CC_BRICK_Z - 1) / CC_BRICK_Z);
    if (nb >= (1ull << 31)) return fail(CC_ERR_INVALID_ARGUMENT, "too many bricks in one launch");
    int prc = prepare_part_masks(prog, a, nb);
    if (prc) return prc;
    int e;
    if (specialised) {
        e = cc_jit_launch_parts(prog, a, (uint32_t)nb, g.compute, g.index);
    } else {
        const uint32_t *table = nullptr;
        int rc = parts_on_device(prog, &table);
        if (rc) return rc;
        e = cc_launch_parts_interp(a, table, (uint32_t)nb, g.compute);
    }
    if (e) return cuda_fail((cudaError_t)e, "part-culling kernel launch");
    g.launches += 2;
    g.points += points;
    return CC_OK;
}

// Dense float4 grid through the column kernel (DESIGN.md 4.10): one warp per 8 x 8 x 16 brick, what does not
// depend on z evaluated once per column; with the parts' masks when the scene is an assembly.
int launch_columns(const cc_program *prog, cc_eval_args &a, uint64_t points, bool with_parts)
{
    const uint64_t nb = (uint64_t)((a.nx + CC_BRICK_X - 1) / CC_BRICK_X) * ((a.ny + CC_BRICK_Y - 1) / CC_BRICK_Y) *
                        ((a.nz + CC_BRICK_Z - 1) / CC_BRICK_Z);
    if (nb >= (1ull << 31)) return fail(CC_ERR_INVALID_ARGUMENT, "too many bricks in one launch");
    const cc_columns_meta &meta = prog->jit_columns;
    const int axis = meta.axis;
    const uint64_t ncol = axis == 2 ? (uint64_t)a.nx * a.ny : axis == 1 ? (uint64_t)a.nx * a.nz : (uint64_t)a.ny * a.nz;
    // column buffer (+ flags, brick list, counter behind it when some transform row is checked per column)
    const size_t values = (size_t)ncol * 4 * std::max(1u, meta.n_values) * sizeof(float);
    const size_t flags_at = (values + 255) & ~(size_t)255, list_at = (flags_at + ncol + 255) & ~(size_t)255;
    const size_t bytes = meta.checks ? list_at + ((size_t)nb + 1) * 4 : values;
    if (bytes > g.columns_cap) {
        if (g.d_columns) CU(cudaFree(g.d_columns));
        g.d_columns = nullptr;
        g.columns_cap = 0;
        CU(cudaMalloc(&g.d_columns, bytes));
        g.columns_cap = bytes;
    }
    a.columns = reinterpret_cast<float *>(g.d_columns);
    a.column_flags = nullptr;
    a.brick_list = a.brick_count = nullptr;
    if (meta.checks) {
        a.column_flags = reinterpret_cast<unsigned char *>(g.d_columns) + flags_at;
        a.brick_count = reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(g.d_columns) + list_at);
        a.brick_list = a.brick_count + 1;
        CU(cudaMemsetAsync(a.brick_count, 0, 4, g.compute));
    }
    a.part_masks = nullptr;
    if (with_parts) {
        int rc = prepare_part_masks(prog, a, nb);
        if (rc) return rc;
    }
    int n_launches = 0;
    int e = cc_jit_launch_columns(prog, a, (uint32_t)nb, g.prop.multiProcessorCount, g.compute, g.index, &n_launches);
    if (e) return cuda_fail((cudaError_t)e, "column kernel launch");
    g.launches += (uint64_t)n_launches;
    g.points += points;
    return CC_OK;
}

// The hierarchy sinks (ordered hit lists, mass sums, PyMCubes fields of blocks) through the brick units' tile
// kernels: with `columns` the column pass covers the columns of every block of the launch and the tile kernel
// runs the per-cell body; with `masks` a tile-centre pass writes a part mask per tile first.
int tile_sink_of(int sink_kind)
{
    return sink_kind == CC_SINK_PYMCUBES ? CC_SINK_TILES_PYMCUBES : sink_kind == CC_SINK_CLASSIFY ? CC_SINK_TILES_CLASSIFY : CC_SINK_TILES_MASS;
}

int launch_tiles(int sink_kind, const cc_program *prog, cc_eval_args &a, uint64_t points, bool columns, bool masks)
{
    const int sink = tile_sink_of(sink_kind);
    const cc_columns_meta &meta = prog->jit_tiles[sink - CC_SINK_TILES_PYMCUBES];
    const uint32_t tile = (uint32_t)(prog->jit_cfg[sink].threads * prog->jit_cfg[sink].pts);
    const uint64_t cells = (uint64_t)a.nx * a.ny * a.nz;
    a.tiles_per_block = (uint32_t)((cells + tile - 1) / tile);
    const uint64_t tiles = (uint64_t)a.tiles_per_block * a.n_blocks;
    if (tiles >= (1ull << 31)) return fail(CC_ERR_INVALID_ARGUMENT, "too many tiles in one launch");
    if (sink_kind == CC_SINK_CLASSIFY || sink_kind == CC_SINK_MASS) {
        int rc = ensure_status((size_t)tiles);
        if (rc) return rc;
        CU(cudaMemsetAsync(g.d_ticket, 0, 4, g.compute));
        CU(cudaMemsetAsync(g.d_status, 0, (size_t)tiles * sizeof(unsigned long long), g.compute));
        a.ticket = g.d_ticket;
        a.tile_status = g.d_status;
    }
    a.columns = nullptr;
    a.column_flags = nullptr;
    if (columns) {
        const int axis = meta.axis;
        const uint64_t ncol = (uint64_t)a.n_blocks * (axis == 2 ? (uint64_t)a.nx * a.ny : axis == 1 ? (uint64_t)a.nx * a.nz : (uint64_t)a.ny * a.nz);
        const size_t values = (size_t)ncol * 4 * std::max(1u, meta.n_values) * sizeof(float);
        const size_t flags_at = (values + 255) & ~(size_t)255;
        const size_t bytes = meta.checks ? flags_at + ncol : values;
        if (bytes > g.columns_cap) {
            if (g.d_columns) CU(cudaFree(g.d_columns));
            g.d_columns = nullptr;
            g.columns_cap = 0;
            CU(cudaMalloc(&g.d_columns, bytes));
            g.columns_cap = bytes;
        }
        a.columns = reinterpret_cast<float *>(g.d_columns);
        a.column_flags = meta.checks ? reinterpret_cast<unsigned char *>(g.d_columns) + flags_at : nullptr;
    }
    a.part_masks = nullptr;
    if (masks) {
        int rc = prepare_part_masks(prog, a, tiles);
        if (rc) return rc;
    }
    int n_launches = 0;
    int e = cc_jit_launch_tiles(prog, sink, a, g.compute, g.index, &n_launches);
    if (e) return cuda_fail((cudaError_t)e, "tile kernel launch");
    g.launches += (uint64_t)n_launches;
    g.points += points;
    return CC_OK;
}

uint64_t axis_len(const cc_program *prog, const cc_eval_args &a)
{
    const int axis = prog->dec.columns.axis;
    return std::max(1u, axis == 0 ? a.nx : axis == 1 ? a.ny : a.nz);
}

bool columns_apply(int sink_kind, const cc_program *prog, const cc_eval_args &a)
{
    const int axis = prog->dec.columns.axis;
    return g.columns_mode && sink_kind == CC_SINK_FLOAT4 && !a.points && !a.blocks && prog->dec.columns.enabled && !cc_jit_is_segmented(prog->dec) &&
           (axis == 0 ? a.nx : axis == 1 ? a.ny : a.nz) >= 8 && (uint64_t)a.nx * a.ny * a.nz >= 4096;
}

bool parts_apply(int sink_kind, const cc_program *prog, const cc_eval_args &a)
{
    return g.parts_mode && sink_kind == CC_SINK_FLOAT4 && !a.points && !a.blocks && prog->dec.parts.enabled &&
           (uint64_t)a.nx * a.ny * a.nz >= 4096;
}

int launch(int sink_kind, const cc_program *prog, cc_eval_args &a, uint64_t points)
{
    if (forest_applies(sink_kind, prog, a)) return launch_forest(prog, a, points);
    if (columns_apply(sink_kind, prog, a)) {
        cc_program *p = const_cast<cc_program *>(prog);
        const bool with_parts = parts_apply(sink_kind, prog, a);
        // (the specialised column kernels or nothing: until they are loaded the other paths serve the launch)
        if (jit_ready(p, CC_SINK_COLUMNS) && (uint64_t)a.nx * a.ny * a.nz / (axis_len(prog, a)) * 16 * std::max(1u, p->jit_columns.n_values) <= (8ull << 30))
            return launch_columns(prog, a, points, with_parts);
    }
    if ((sink_kind == CC_SINK_CLASSIFY || sink_kind == CC_SINK_MASS || (sink_kind == CC_SINK_PYMCUBES && a.blocks)) && !a.points &&
        !cc_jit_is_segmented(prog->dec) && (uint64_t)a.nx * a.ny * a.nz >= 512) {
        // blocks x linear tiles: the per-cell body of the column split and / or a part mask per tile (one unit per sink)
        cc_program *p = const_cast<cc_program *>(prog);
        const bool masks = g.parts_mode && prog->dec.parts.enabled && (!a.blocks || a.coord_max > 0.0f);
        const bool cols = g.columns_mode && prog->dec.columns.enabled && axis_len(prog, a) >= 8;
        if ((masks || cols) && jit_ready(p, tile_sink_of(sink_kind))) {
            const cc_columns_meta &meta = p->jit_tiles[tile_sink_of(sink_kind) - CC_SINK_TILES_PYMCUBES];
            const bool fits = (uint64_t)a.n_blocks * a.nx * a.ny * a.nz / axis_len(prog, a) * 16 * std::max(1u, meta.n_values) <= (8ull << 30);
            // (the unit's per-cell body reads the column buffer whenever the program has a split: no columns, no unit)
            if (!meta.columns || (cols && fits)) return launch_tiles(sink_kind, prog, a, points, meta.columns, masks);
        }
    }
    if (parts_apply(sink_kind, prog, a)) {
        if (!cc_jit_is_segmented(prog->dec) && jit_ready(const_cast<cc_program *>(prog), CC_SINK_PARTS)) return launch_parts(prog, a, points, true);
        // interpreter tier: the same culling by walking the segment table (needs the microcode in shared memory)
        if (!prog->dec.parts.table.empty() && prog->dec.parts.n_parts <= 32 &&
            cc_parts_smem_bytes(prog->dec.info.n_slots, prog->dec.info.n_micro_words, 2) * 2 <= (size_t)g.prop.sharedMemPerMultiprocessor)
            return launch_parts(prog, a, points, false);
    }
    // which specialised kernel serves the launch: point lists have their own (cc_jit_points)
    const int sink = a.points ? (int)CC_SINK_POINTS : sink_kind;
    if (jit_ready(const_cast<cc_program *>(prog), sink)) {
        // scene-specialised kernel: slots are registers, parameters immediates
        const uint32_t tile = (uint32_t)(prog->jit_cfg[sink].threads * prog->jit_cfg[sink].pts);
        const uint64_t cells = (uint64_t)a.nx * a.ny * a.nz;
        a.tiles_per_block = (uint32_t)((cells + tile - 1) / tile);
        const uint64_t tiles = (uint64_t)a.tiles_per_block * a.n_blocks;
        if (tiles >= (1ull << 31)) return fail(CC_ERR_INVALID_ARGUMENT, "too many tiles in one launch");
        if (sink == CC_SINK_CLASSIFY || sink == CC_SINK_MASS) {
            int rc = ensure_status((size_t)tiles);
            if (rc) return rc;
            CU(cudaMemsetAsync(g.d_ticket, 0, 4, g.compute));
            CU(cudaMemsetAsync(g.d_status, 0, (size_t)tiles * sizeof(unsigned long long), g.compute));
            a.ticket = g.d_ticket;
            a.tile_status = g.d_status;
        }
        int e = cc_jit_launch(prog, sink, a, g.compute, g.index);
        if (e) return cuda_fail((cudaError_t)e, "specialised kernel launch");
        g.launches += 1;
        g.points += points;
        return CC_OK;
    }
    cc_launch_cfg cfg;
    int rc = choose_cfg(prog, points, &cfg);
    if (rc) return rc;
    if (a.points) {  // the point-list kernels exist for 1 / 2 points per thread, constant or shared program
        if (cfg.pts > 2) cfg.pts = 2;
        if (cfg.prog_space == 3) cfg.prog_space = 1;
    }
    rc = prepare_program(prog, cfg);
    if (rc) return rc;
    const uint32_t tile = cc_tile_points(cfg);
    const uint64_t cells = (uint64_t)a.nx * a.ny * a.nz;
    a.tiles_per_block = (uint32_t)((cells + tile - 1) / tile);
    const uint64_t tiles = (uint64_t)a.tiles_per_block * a.n_blocks;
    if (tiles >= (1ull << 31)) return fail(CC_ERR_INVALID_ARGUMENT, "too many tiles in one launch");
    if (sink == CC_SINK_CLASSIFY || sink == CC_SINK_MASS) {
        rc = ensure_status((size_t)tiles);
        if (rc) return rc;
        CU(cudaMemsetAsync(g.d_ticket, 0, 4, g.compute));
        CU(cudaMemsetAsync(g.d_status, 0, (size_t)tiles * sizeof(unsigned long long), g.compute));
        a.ticket = g.d_ticket;
        a.tile_status = g.d_status;
    }
    int e = cc_launch_eval(sink_kind, cfg, a, g.compute);
    if (e) return cuda_fail((cudaError_t)e, "cc_eval_kernel launch");
    g.launches += 1;
    g.points += points;
    return CC_OK;
}


int init_context(Context &c, int device, int index)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(CC_ERR_CUDA, "no CUDA device available; libcodecad_b200 has no CPU fallback");
    }
    if (device < 0 || device >= n) return fail(CC_ERR_INVALID_ARGUMENT, "no such device");
    CU(cudaSetDevice(device));
    tl_device = device;
    CU(cudaGetDeviceProperties(&c.prop, device));
    if (c.prop.major < 10)
        return fail(CC_ERR_CUDA, std::string("device ") + c.prop.name + " is not sm_100 (built for sm_100a only)");
    CU(cudaStreamCreateWithFlags(&c.compute, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c.copy, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c.copy2, cudaStreamNonBlocking));
    CU(cudaMallocHost(&c.h_word, 64));
    {
        // keep freed work-list memory in the pool instead of returning it to the driver at every sync
        cudaMemPool_t pool = nullptr;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        } else {
            cudaGetLastError();
        }
    }
    c.device = device;
    c.index = index;
    const char *p = getenv("CODECAD_B200_PTS");
    if (p) c.pts = atoi(p);
    p = getenv("CODECAD_B200_PROG_SPACE");
    if (p) c.prog_space = atoi(p);
    p = getenv("CODECAD_B200_JIT");
    if (p) c.jit_mode = std::max(0, std::min(2, atoi(p)));
    p = getenv("CODECAD_B200_JIT_MAX_OPS");
    if (p) c.jit_max_ops = (uint32_t)atoi(p);
    p = getenv("CODECAD_B200_FOREST");
    if (p) c.forest_mode = atoi(p) != 0;
    p = getenv("CODECAD_B200_PARTS");
    if (p) c.parts_mode = atoi(p) != 0;
    p = getenv("CODECAD_B200_COLUMNS");
    if (p) c.columns_mode = atoi(p) != 0;
    c.ready = true;
    return CC_OK;
}

// ---- one worker thread per additional device ----------------------------------------------------
// A call that shards (cc_mass_properties, cc_subdivide, cc_grid_eval_to_host) runs its single-device
// body once per device: device 0 on the caller's thread, device i on worker i, whose current
// context is g_ctx[i].  Workers are created on first use and live until cc_shutdown.
struct Worker {
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::function<void()> task;
    bool has_task = false, stop = false;
};
Worker *g_workers[CC_MAX_DEVICES] = {};

void worker_main(Worker *w, int index)
{
    tl_ctx = &g_ctx[index];
    cudaSetDevice(g_ctx[index].device);
    tl_device = g_ctx[index].device;
    for (;;) {
        std::function<void()> task;
        {
            std::unique_lock<std::mutex> lk(w->mu);
            w->cv.wait(lk, [&] { return w->has_task || w->stop; });
            if (w->stop) return;
            task.swap(w->task);
            w->has_task = false;
        }
        task();
    }
}

void stop_workers()
{
    for (int i = 0; i < CC_MAX_DEVICES; ++i) {
        Worker *w = g_workers[i];
        if (!w) continue;
        {
            std::lock_guard<std::mutex> lk(w->mu);
            w->stop = true;
        }
        w->cv.notify_all();
        if (w->th.joinable()) w->th.join();
        delete w;
        g_workers[i] = nullptr;
    }
}

// fn(device index) -> status, once per initialised device, concurrently; returns the first failure
template <class F>
int for_each_device(F fn)
{
    const int n = g_n_ctx;
    if (n <= 1 || tl_ctx != &g_ctx[0]) return fn(g.index);
    std::vector<int> rc((size_t)n, CC_OK);
    std::vector<std::string> errs((size_t)n);
    std::mutex done_mu;
    std::condition_variable done_cv;
    int pending = n - 1;
    for (int i = 1; i < n; ++i) {
        if (!g_workers[i]) {
            g_workers[i] = new Worker;
            g_workers[i]->th = std::thread(worker_main, g_workers[i], i);
        }
        Worker *w = g_workers[i];
        {
            std::lock_guard<std::mutex> lk(w->mu);
            w->task = [&, i] {
                rc[(size_t)i] = fn(i);
                if (rc[(size_t)i]) errs[(size_t)i] = g_err;
                std::lock_guard<std::mutex> dl(done_mu);
                if (--pending == 0) done_cv.notify_one();
            };
            w->has_task = true;
        }
        w->cv.notify_one();
    }
    rc[0] = fn(0);
    {
        std::unique_lock<std::mutex> lk(done_mu);
        done_cv.wait(lk, [&] { return pending == 0; });
    }
    for (int i = 0; i < n; ++i)
        if (rc[(size_t)i]) {
            if (i) g_err = "device " + std::to_string(g_ctx[i].device) + ": " + errs[(size_t)i];
            return rc[(size_t)i];
        }
    return CC_OK;
}

}  // namespace

extern "C" {

const char *cc_last_error(void) { return g_err.c_str(); }

int cc_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int cc_init(int device)
{
    std::lock_guard<std::mutex> lk(g_mu);
    Context &c = g_ctx[0];
    if (c.ready) {
        if (c.device == device) return CC_OK;
        return fail(CC_ERR_INVALID_ARGUMENT, "already initialised on another device");
    }
    int rc = init_context(c, device, 0);
    if (rc) return rc;
    g_n_ctx = 1;
    tl_ctx = &g_ctx[0];
    return CC_OK;
}

int cc_init_devices(const int *devices, int n)
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (!devices || n < 1 || n > CC_MAX_DEVICES) return fail(CC_ERR_INVALID_ARGUMENT, "1.." + std::to_string(CC_MAX_DEVICES) + " devices");
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < i; ++j)
            if (devices[i] == devices[j]) return fail(CC_ERR_INVALID_ARGUMENT, "a device is listed twice");
    if (g_ctx[0].ready && g_ctx[0].device != devices[0])
        return fail(CC_ERR_INVALID_ARGUMENT, "already initialised with another first device");
    if (g_n_ctx > n) return fail(CC_ERR_INVALID_ARGUMENT, "already initialised with more devices");
    for (int i = 0; i < n; ++i) {
        Context &c = g_ctx[i];
        if (c.ready) {
            if (c.device != devices[i]) return fail(CC_ERR_INVALID_ARGUMENT, "already initialised with other devices");
            continue;
        }
        int rc = init_context(c, devices[i], i);
        if (rc) return rc;
        g_n_ctx = std::max(g_n_ctx, i + 1);
    }
    // the caller's thread keeps driving the first device
    tl_ctx = &g_ctx[0];
    CU(cudaSetDevice(g_ctx[0].device));
    tl_device = g_ctx[0].device;
    return CC_OK;
}

int cc_active_devices(void) { return g_n_ctx; }

void cc_shutdown(void)
{
    std::lock_guard<std::mutex> lk(g_mu);
    stop_workers();
    g_pinned.trim(0);
    for (int k = 0; k < g_n_ctx; ++k) {
        Context &c = g_ctx[k];
        if (!c.ready) continue;
        cudaSetDevice(c.device);
        cudaDeviceSynchronize();
        if (c.d_ticket) cudaFree(c.d_ticket);
        if (c.d_status) cudaFree(c.d_status);
        if (c.d_forest_scratch) cudaFree(c.d_forest_scratch);
        if (c.d_part_masks) cudaFree(c.d_part_masks);
        if (c.d_columns) cudaFree(c.d_columns);
        if (c.h_word) cudaFreeHost(c.h_word);
        for (int i = 0; i < Context::kRing; ++i) {
            if (c.ring[i]) cudaFree(c.ring[i]);
            if (c.ring_computed[i]) cudaEventDestroy(c.ring_computed[i]);
            if (c.ring_copied[i]) cudaEventDestroy(c.ring_copied[i]);
        }
        cudaStreamDestroy(c.compute);
        cudaStreamDestroy(c.copy);
        cudaStreamDestroy(c.copy2);
        c = Context();
    }
    g_n_ctx = 0;
    tl_ctx = &g_ctx[0];
    tl_device = -1;
}

int cc_device_pci_bus_id(int device, char *out, int capacity)
{
    if (!out || capacity < 13) return fail(CC_ERR_INVALID_ARGUMENT, "buffer too small for a PCI bus id");
    cudaError_t e = cudaDeviceGetPCIBusId(out, capacity, device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceGetPCIBusId");
    return CC_OK;
}

int cc_get_device_info(cc_device_info *out)
{
    NEED_INIT();
    std::memset(out, 0, sizeof(*out));
    out->device = g.device;
    out->sm_count = g.prop.multiProcessorCount;
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, g.device);
    out->sm_clock_khz = khz;
    out->l2_bytes = g.prop.l2CacheSize;
    out->total_mem = g.prop.totalGlobalMem;
    std::strncpy(out->name, g.prop.name, sizeof(out->name) - 1);
    return CC_OK;
}

int cc_synchronize(void)
{
    NEED_INIT();
    CU(cudaStreamSynchronize(g.compute));
    CU(cudaStreamSynchronize(g.copy));
    CU(cudaStreamSynchronize(g.copy2));
    return CC_OK;
}

int cc_get_counters(uint64_t *kernel_launches, uint64_t *points_evaluated)
{
    uint64_t l = 0, p = 0;
    for (int i = 0; i < std::max(g_n_ctx, 1); ++i) {
        l += g_ctx[i].launches;
        p += g_ctx[i].points;
    }
    if (kernel_launches) *kernel_launches = l;
    if (points_evaluated) *points_evaluated = p;
    return CC_OK;
}

void cc_reset_counters(void)
{
    for (int i = 0; i < CC_MAX_DEVICES; ++i) g_ctx[i].launches = g_ctx[i].points = 0;
}

int cc_set_tuning(int points_per_thread, int program_space)
{
    if (points_per_thread != 0 && points_per_thread != 1 && points_per_thread != 2 && points_per_thread != 4)
        return fail(CC_ERR_INVALID_ARGUMENT, "points_per_thread must be 0, 1, 2 or 4");
    if (program_space < 0 || program_space > 3) return fail(CC_ERR_INVALID_ARGUMENT, "program_space must be 0..3");
    for (int i = 0; i < CC_MAX_DEVICES; ++i) {
        g_ctx[i].pts = points_per_thread;
        g_ctx[i].prog_space = program_space;
    }
    return CC_OK;
}

// ---- programs -------------------------------------------------------------------------------------

int cc_program_create(const float *words, uint32_t n_words, cc_program **out)
{
    NEED_INIT();
    if (!words || !out) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    cc_program *p = new cc_program();
    std::string err;
    int rc = cc_decode_program(words, n_words, &p->dec, &err);
    if (rc != CC_OK) {
        delete p;
        return fail(rc, err);
    }
    const uint32_t *d = nullptr;
    rc = program_on_device(p, &d);  // the caller's device now; other devices on first use
    if (rc != CC_OK) {
        delete p;
        return rc;
    }
    p->id = g_next_program_id++;
    *out = p;
    return CC_OK;
}

void cc_program_destroy(cc_program *prog)
{
    if (!prog) return;
    if (g.ready) {
        for (int i = 0; i < g_n_ctx; ++i) {
            Context &c = g_ctx[i];
            if (!c.ready) continue;
            cudaSetDevice(c.device);
            cudaStreamSynchronize(c.compute);
            if (prog->d_code[i]) cudaFree(prog->d_code[i]);
            if (prog->d_forest[i]) cudaFree(prog->d_forest[i]);
            if (prog->d_parts[i]) cudaFree(prog->d_parts[i]);
            if (c.constant_program == prog->id) c.constant_program = 0;
        }
        cudaSetDevice(g.device);
        tl_device = g.device;
        cc_jit_release(prog);
    }
    delete prog;
}

int cc_program_get_info(const cc_program *prog, cc_program_info *out)
{
    if (!prog || !out) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    *out = prog->dec.info;
    return CC_OK;
}

int cc_program_get_microcode(const cc_program *prog, uint32_t *out, uint32_t capacity)
{
    if (!prog) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    uint32_t n = (uint32_t)prog->dec.microcode.size();
    if (out) std::memcpy(out, prog->dec.microcode.data(), (size_t)std::min(n, capacity) * 4);
    return (int)n;
}

int cc_program_decode(const float *words, uint32_t n_words, cc_program_info *info, uint32_t *out,
                      uint32_t capacity)
{
    if (!words) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    cc_decoded dec;
    std::string err;
    int rc = cc_decode_program(words, n_words, &dec, &err);
    if (rc != CC_OK) return fail(rc, err);
    if (info) *info = dec.info;
    uint32_t n = (uint32_t)dec.microcode.size();
    if (out) std::memcpy(out, dec.microcode.data(), (size_t)std::min(n, capacity) * 4);
    return (int)n;
}

int cc_program_specialize(cc_program *prog, int points_per_thread, unsigned sink_mask, double *compile_seconds)
{
    NEED_INIT();
    if (!prog) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaStreamSynchronize(g.compute));
    std::string err;
    int rc = cc_jit_compile(prog, points_per_thread, sink_mask, compile_seconds, &err);
    if (rc) return fail(rc, err);
    return CC_OK;
}

int cc_program_use_specialized(cc_program *prog, int enable)
{
    if (!prog) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    prog->use_jit = enable != 0;
    bool any = false;
    for (int k = 0; k < CC_N_SINKS; ++k) any = any || prog->jit_kernel[k] != nullptr;
    return (prog->use_jit && any) ? 1 : 0;
}

int cc_set_jit_mode(int mode)
{
    const int old = g.jit_mode;
    if (mode < 0 || mode > 2) return fail(CC_ERR_INVALID_ARGUMENT, "jit mode must be 0, 1 or 2");
    for (int i = 0; i < CC_MAX_DEVICES; ++i) g_ctx[i].jit_mode = mode;
    return old;
}

int cc_set_forest_mode(int mode)
{
    const int old = g.forest_mode;
    if (mode != 0 && mode != 1) return fail(CC_ERR_INVALID_ARGUMENT, "forest mode must be 0 or 1");
    for (int i = 0; i < CC_MAX_DEVICES; ++i) g_ctx[i].forest_mode = mode;
    return old;
}

int cc_grid_eval_cost_profile(const cc_program *prog, const float corner[3], float step, uint32_t nx, uint32_t ny, uint32_t nz,
                              uint32_t x_offset, double *layer_cost, uint32_t n_layers)
{
    NEED_INIT();
    if (!prog || !corner || !layer_cost) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    int rc = check_dims(nx, ny, nz);
    if (rc) return rc;
    const uint32_t nbx = (nx + CC_BRICK_X - 1) / CC_BRICK_X, nby = (ny + CC_BRICK_Y - 1) / CC_BRICK_Y, nbz = (nz + CC_BRICK_Z - 1) / CC_BRICK_Z;
    if (n_layers != nbx) return fail(CC_ERR_INVALID_ARGUMENT, "one cost per layer of 8 x-planes: n_layers must be ceil(nx / 8)");
    const cc_parts &parts = prog->dec.parts;
    const uint64_t per_layer = (uint64_t)nby * nbz, nb = per_layer * nbx;
    if (!g.parts_mode || !parts.enabled || parts.table.empty() || nb >= (1ull << 31)) {
        for (uint32_t i = 0; i < n_layers; ++i) layer_cost[i] = (double)per_layer;  // nothing known: every layer the same
        return CC_OK;
    }
    cc_eval_args a;
    FILL_COMMON(a, prog);
    a.cx = corner[0]; a.cy = corner[1]; a.cz = corner[2]; a.step = step;
    a.nx = nx; a.ny = ny; a.nz = nz; a.x_offset = x_offset; a.n_blocks = 1;
    if ((rc = prepare_part_masks(prog, a, nb))) return rc;
    int e;
    cc_program *p = const_cast<cc_program *>(prog);
    if (!cc_jit_is_segmented(prog->dec) && jit_ready(p, CC_SINK_PARTS)) {
        e = cc_jit_launch_parts(prog, a, (uint32_t)nb, g.compute, g.index, true);
    } else {
        const uint32_t *table = nullptr;
        if ((rc = parts_on_device(prog, &table))) return rc;
        e = cc_launch_parts_interp(a, table, (uint32_t)nb, g.compute, true);
    }
    if (e) return cuda_fail((cudaError_t)e, "brick-centre kernel launch");
    // weights: a brick costs its set-up and stores plus the micro-ops of the parts it keeps
    cc_layer_weights w;
    w.base = 60.0f;
    for (int k = 0; k < 32; ++k) w.part[k] = 0.0f;
    const cc_columns &cols = prog->dec.columns;
    const bool split = g.columns_mode && cols.enabled && !cc_jit_is_segmented(prog->dec);  // (the dense path then runs the per-cell body only)
    for (size_t v = 0; v < parts.part_of_op.size(); ++v) {
        const int part = parts.part_of_op[v];
        if (part < 0 || part >= 32) continue;
        if (split && v < cols.phase.size() && !(cols.phase[v] & 2)) continue;
        w.part[part] += v < cols.op_cost.size() ? (float)cols.op_cost[v] : 10.0f;
    }
    double *d_cost = nullptr;
    CU(cudaMallocAsync((void **)&d_cost, (size_t)n_layers * sizeof(double), g.compute));
    e = cc_launch_layer_cost(a.part_masks, n_layers, (uint32_t)per_layer, w, d_cost, g.compute);
    cudaError_t ce = e ? (cudaError_t)e : cudaMemcpyAsync(layer_cost, d_cost, (size_t)n_layers * sizeof(double), cudaMemcpyDeviceToHost, g.compute);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(g.compute);
    cudaFreeAsync(d_cost, g.compute);
    if (ce != cudaSuccess) return cuda_fail(ce, "layer cost kernel");
    g.launches += 2;
    return CC_OK;
}

int cc_set_columns_mode(int mode)
{
    const int old = g.columns_mode;
    if (mode != 0 && mode != 1) return fail(CC_ERR_INVALID_ARGUMENT, "columns mode must be 0 or 1");
    for (int i = 0; i < CC_MAX_DEVICES; ++i) g_ctx[i].columns_mode = mode;
    return old;
}

int cc_set_parts_mode(int mode)
{
    const int old = g.parts_mode;
    if (mode != 0 && mode != 1) return fail(CC_ERR_INVALID_ARGUMENT, "parts mode must be 0 or 1");
    for (int i = 0; i < CC_MAX_DEVICES; ++i) g_ctx[i].parts_mode = mode;
    return old;
}

int cc_program_get_forest_info(const cc_program *prog, uint32_t out[4])
{
    if (!prog || !out) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    const cc_forest &f = prog->dec.forest;
    out[0] = f.enabled ? f.n_leaves : 0;
    out[1] = f.enabled ? f.n_unions : 0;
    out[2] = f.enabled ? f.max_depth : 0;
    out[3] = f.enabled ? f.n_events : 0;
    return f.enabled ? 1 : 0;
}

int cc_program_specialize_wait(cc_program *prog, unsigned sink_mask, double *compile_seconds)
{
    NEED_INIT();
    if (!prog) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    if ((sink_mask & CC_SINK_MASK_ALL) == 0) sink_mask = 15u;
    // dense float4 grids of an assembly run on the part-culling kernels: "ready" includes them
    const bool small = !cc_jit_is_segmented(prog->dec);
    const bool parts = small && prog->dec.parts.enabled && g.parts_mode, cols = small && prog->dec.columns.enabled && g.columns_mode;
    if ((sink_mask & (1u << CC_SINK_FLOAT4)) && parts) sink_mask |= 1u << CC_SINK_PARTS;
    if ((sink_mask & (1u << CC_SINK_FLOAT4)) && cols) sink_mask |= 1u << CC_SINK_COLUMNS;
    for (int k : {(int)CC_SINK_PYMCUBES, (int)CC_SINK_CLASSIFY, (int)CC_SINK_MASS})
        if ((sink_mask & (1u << k)) && (parts || cols)) sink_mask |= 1u << tile_sink_of(k);
    int ready = 0;
    for (int k = 0; k < CC_N_SINKS; ++k) {
        if (!(sink_mask & (1u << k))) continue;
        cc_jit_start(prog, k);
        std::string err;
        int r = cc_jit_poll(prog, k, true, &err);
        if (r < 0) return fail(r, err);
        ready += r;
    }
    if (compile_seconds) *compile_seconds = prog->jit_seconds;
    return ready;
}

int cc_specialize_source(const float *words, uint32_t n_words, int points_per_thread, unsigned sink_mask,
                         char *out, uint32_t capacity, int compile, uint64_t *cubin_bytes)
{
    if (!words) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    cc_decoded dec;
    std::string err, src;
    int rc = cc_decode_program(words, n_words, &dec, &err);
    if (rc == CC_OK) rc = cc_jit_source(dec, points_per_thread, sink_mask, &src, &err);
    if (rc != CC_OK) return fail(rc, err);
    if (out && capacity) {
        size_t n = std::min<size_t>(src.size(), capacity - 1);
        std::memcpy(out, src.data(), n);
        out[n] = 0;
    }
    if (compile) {
        std::vector<char> cubin;
        rc = cc_jit_nvrtc(src, &cubin, &err);
        if (rc != CC_OK) return fail(rc, err);
        if (cubin_bytes) *cubin_bytes = cubin.size();
    }
    return (int)src.size();
}

// ---- buffers / events ---------------------------------------------------------------------------------

// Stream-ordered allocations from the device's default pool on the compute stream (every kernel
// and copy that touches a caller's buffer is issued on that stream; cc_init keeps the pool warm):
// a cl_util.Buffer costs microseconds instead of a cudaMalloc + a device-wide cudaFree.
int cc_buffer_alloc(size_t bytes, void **dptr)
{
    NEED_INIT();
    if (!dptr) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaMallocAsync(dptr, bytes ? bytes : 1, g.compute));
    return CC_OK;
}

int cc_buffer_free(void *dptr)
{
    NEED_INIT();
    if (!dptr) return CC_OK;
    CU(cudaStreamSynchronize(g.copy));  // the slab pipeline may still be reading from it
    CU(cudaStreamSynchronize(g.copy2));
    CU(cudaFreeAsync(dptr, g.compute));
    return CC_OK;
}

int cc_host_alloc(size_t bytes, void **hptr)
{
    NEED_INIT();
    if (!hptr) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    *hptr = g_pinned.get(bytes);  // pooled: page-locking costs ~0.3 ms per MB
    if (!*hptr) return fail(CC_ERR_CUDA, "cudaHostAlloc failed for " + std::to_string(bytes) + " bytes");
    return CC_OK;
}

int cc_host_free(void *hptr)
{
    NEED_INIT();
    if (!hptr) return CC_OK;
    // an asynchronous copy into the block may still be in flight
    CU(cudaStreamSynchronize(g.compute));
    CU(cudaStreamSynchronize(g.copy));
    if (!g_pinned.put(hptr)) CU(cudaFreeHost(hptr));
    return CC_OK;
}

int cc_memcpy_h2d_async(void *dptr, const void *hptr, size_t bytes, cc_event **ev)
{
    NEED_INIT();
    CU(cudaMemcpyAsync(dptr, hptr, bytes, cudaMemcpyHostToDevice, g.compute));
    return make_event(ev, g.compute);
}

int cc_memcpy_d2h_async(void *hptr, const void *dptr, size_t bytes, cc_event **ev)
{
    NEED_INIT();
    CU(cudaMemcpyAsync(hptr, dptr, bytes, cudaMemcpyDeviceToHost, g.compute));
    return make_event(ev, g.compute);
}

int cc_memset_async(void *dptr, int value, size_t bytes, cc_event **ev)
{
    NEED_INIT();
    CU(cudaMemsetAsync(dptr, value, bytes, g.compute));
    return make_event(ev, g.compute);
}

int cc_event_record(cc_event **ev)
{
    NEED_INIT();
    if (!ev) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    return make_event(ev, g.compute);
}

int cc_event_wait(cc_event *ev)
{
    NEED_INIT();
    if (!ev) return CC_OK;
    CU(cudaEventSynchronize(ev->ev));
    return CC_OK;
}

int cc_event_elapsed_ms(cc_event *start, cc_event *end, float *ms)
{
    NEED_INIT();
    if (!start || !end || !ms) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaEventElapsedTime(ms, start->ev, end->ev));
    return CC_OK;
}

void cc_event_destroy(cc_event *ev)
{
    if (!ev) return;
    cudaEventDestroy(ev->ev);
    delete ev;
}

void cc_free(void *p)
{
    if (p && !g_pinned.put(p)) free(p);
}

// ---- reference-semantics kernels ---------------------------------------------------------------------

int cc_grid_eval(const cc_program *prog, const float corner[3], float step, uint32_t nx, uint32_t ny,
                 uint32_t nz, uint32_t x_offset, int layout, void *d_out, cc_event **ev)
{
    NEED_INIT();
    if (!prog || !corner || !d_out) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    if (layout != CC_LAYOUT_INDEX3_FLOAT4 && layout != CC_LAYOUT_PYMCUBES_FLOAT)
        return fail(CC_ERR_INVALID_ARGUMENT, "unknown layout");
    if (nx == 0 || ny == 0 || nz == 0) return fail(CC_ERR_INVALID_ARGUMENT, "empty grid");
    const uint64_t plane = (uint64_t)ny * nz;
    if (plane > (1ull << 31)) return fail(CC_ERR_INVALID_ARGUMENT, "y*z plane too large");
    // split along x so that every launch has <= 2^30 cells (the PyMCubes layout is not
    // x-separable, so it must fit one launch)
    uint32_t max_x = (uint32_t)std::max<uint64_t>(1, (1ull << 30) / plane);
    if (layout == CC_LAYOUT_PYMCUBES_FLOAT && nx > max_x)
        return fail(CC_ERR_INVALID_ARGUMENT, "PyMCubes-layout grid too large for one launch");
    const size_t elem = layout == CC_LAYOUT_INDEX3_FLOAT4 ? 16 : 4;
    for (uint32_t x0 = 0; x0 < nx; x0 += max_x) {
        uint32_t cnt = std::min(max_x, nx - x0);
        cc_eval_args a;
        FILL_COMMON(a, prog);
        a.cx = corner[0]; a.cy = corner[1]; a.cz = corner[2]; a.step = step;
        a.nx = cnt; a.ny = ny; a.nz = nz; a.x_offset = x_offset + x0;
        a.n_blocks = 1;
        a.out = (char *)d_out + (size_t)x0 * plane * elem;
        int rc = launch(layout == CC_LAYOUT_INDEX3_FLOAT4 ? CC_SINK_FLOAT4 : CC_SINK_PYMCUBES, prog, a,
                        (uint64_t)cnt * plane);
        if (rc) return rc;
    }
    return make_event(ev, g.compute);
}

int cc_evaluate_points(const cc_program *prog, const float *d_points, uint64_t n, void *d_out, cc_event **ev)
{
    NEED_INIT();
    if (!prog || !d_points || !d_out) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    const uint64_t chunk = 1ull << 30;
    for (uint64_t i0 = 0; i0 < n; i0 += chunk) {
        const uint32_t cnt = (uint32_t)std::min<uint64_t>(chunk, n - i0);
        cc_eval_args a;
        FILL_COMMON(a, prog);
        a.nx = cnt; a.ny = 1; a.nz = 1; a.n_blocks = 1;
        a.points = d_points + 4 * i0;
        a.out = (char *)d_out + i0 * 16;
        int rc = launch(CC_SINK_FLOAT4, prog, a, cnt);
        if (rc) return rc;
    }
    return make_event(ev, g.compute);
}

// Dense float4 grid into host memory on the current device: slabs of ~64 MiB are computed on the
// compute stream into a device ring (kept between calls) and copied out on the copy stream; a ring
// entry is re-used only after its copy has finished.
static int grid_to_host_share(const cc_program *prog, const float corner[3], float step, uint32_t nx, uint32_t ny,
                              uint32_t nz, uint32_t x_offset, void *h_out)
{
    if (nx == 0) return CC_OK;
    const uint64_t plane = (uint64_t)ny * nz;
    const size_t elem = 16;
    const int layout = CC_LAYOUT_INDEX3_FLOAT4;
    const int RING = Context::kRing;
    // Slab size.  Measured with the culling kernels (21 ms of compute per 1024^3 grid) against 57.0 GB/s for bare
    // copies on the same box: 16 MiB slabs 50.5 GB/s, 32 MiB 51.7, 64 MiB 56.8, 128 MiB 56.9, 256 MiB 56.7
    // (tools/e2e_probe.py).  The brick kernels evaluate 8 x-planes at a time, so a slab is a multiple of 8 planes
    // where that keeps it under 512 MiB: a one-plane slab would have them compute eight planes to keep one.
    static const uint64_t slab_mib = [] {
        const char *t = getenv("CODECAD_B200_SLAB_MIB");
        const long v = t ? atol(t) : 0;
        return (uint64_t)(v > 0 ? v : 64);
    }();
    uint32_t slab_x = (uint32_t)std::max<uint64_t>(1, (slab_mib << 20) / (plane * elem));
    if ((uint64_t)((slab_x + 7u) & ~7u) * plane * elem <= (512ull << 20)) slab_x = (slab_x + 7u) & ~7u;
    slab_x = std::min(slab_x, nx);
    const size_t slab_bytes = (size_t)slab_x * plane * elem;
    if (slab_bytes > g.ring_bytes) {
        for (int i = 0; i < RING; ++i) {
            if (g.ring[i]) CU(cudaFree(g.ring[i]));
            g.ring[i] = nullptr;
        }
        g.ring_bytes = 0;
        for (int i = 0; i < RING; ++i) CU(cudaMalloc(&g.ring[i], slab_bytes));
        g.ring_bytes = slab_bytes;
    }
    if (!g.ring_computed[0])
        for (int i = 0; i < RING; ++i) {
            CU(cudaEventCreateWithFlags(&g.ring_computed[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&g.ring_copied[i], cudaEventDisableTiming));
        }
    int rc = CC_OK;
    int slot = 0;
    for (uint32_t x0 = 0; x0 < nx && rc == CC_OK; x0 += slab_x, slot = (slot + 1) % RING) {
        uint32_t cnt = std::min(slab_x, nx - x0);
        if (x0 >= (uint32_t)RING * slab_x) CU(cudaStreamWaitEvent(g.compute, g.ring_copied[slot], 0));
        rc = cc_grid_eval(prog, corner, step, cnt, ny, nz, x_offset + x0, layout, g.ring[slot], nullptr);
        if (rc) break;
        CU(cudaEventRecord(g.ring_computed[slot], g.compute));
        // two copy streams take the slabs in turn, so that the next transfer is already queued on the
        // copy engine when one ends
        cudaStream_t cs = (slot & 1) ? g.copy2 : g.copy;
        CU(cudaStreamWaitEvent(cs, g.ring_computed[slot], 0));
        CU(cudaMemcpyAsync((char *)h_out + (size_t)x0 * plane * elem, g.ring[slot], (size_t)cnt * plane * elem,
                           cudaMemcpyDeviceToHost, cs));
        CU(cudaEventRecord(g.ring_copied[slot], cs));
    }
    cudaStreamSynchronize(g.compute);
    cudaError_t e = cudaStreamSynchronize(g.copy);
    cudaError_t e2 = cudaStreamSynchronize(g.copy2);
    if (e == cudaSuccess) e = e2;
    if (rc == CC_OK && e != cudaSuccess) rc = cuda_fail(e, "grid_eval_to_host");
    return rc;
}

int cc_grid_eval_to_host(const cc_program *prog, const float corner[3], float step, uint32_t nx, uint32_t ny,
                         uint32_t nz, uint32_t x_offset, int layout, void *h_out)
{
    NEED_INIT();
    if (!prog || !corner || !h_out) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    if (nx == 0 || ny == 0 || nz == 0) return fail(CC_ERR_INVALID_ARGUMENT, "empty grid");
    if (layout != CC_LAYOUT_INDEX3_FLOAT4 && layout != CC_LAYOUT_PYMCUBES_FLOAT)
        return fail(CC_ERR_INVALID_ARGUMENT, "unknown layout");
    const uint64_t plane = (uint64_t)ny * nz;
    if (layout == CC_LAYOUT_PYMCUBES_FLOAT) {
        // y-flipped layout [ny][nx][nz] is not x-separable: evaluate whole (pooled device memory),
        // then copy in pieces so that the first bytes cross PCIe while the driver maps the rest
        const size_t bytes = (size_t)nx * plane * 4;
        void *d = nullptr;
        CU(cudaMallocAsync(&d, bytes, g.compute));
        int rc = cc_grid_eval(prog, corner, step, nx, ny, nz, x_offset, layout, d, nullptr);
        if (rc == CC_OK) {
            const size_t piece = 64ull << 20;
            cudaError_t e = cudaSuccess;
            for (size_t o = 0; o < bytes && e == cudaSuccess; o += piece)
                e = cudaMemcpyAsync((char *)h_out + o, (char *)d + o, std::min(piece, bytes - o), cudaMemcpyDeviceToHost,
                                    g.compute);
            if (e == cudaSuccess) e = cudaStreamSynchronize(g.compute);
            if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemcpyAsync D2H");
        }
        cudaFreeAsync(d, g.compute);
        return rc;
    }
    // x-slabs over the initialised devices (the INDEX3 layout is contiguous in x), each with its
    // own compute/copy pipeline; coordinates stay corner + step * global index
    const uint32_t nd = (uint32_t)std::max(1, g_n_ctx);
    if (nd == 1 || nx < nd) return grid_to_host_share(prog, corner, step, nx, ny, nz, x_offset, h_out);
    return for_each_device([&](int i) {
        const uint32_t base = nx / nd, rem = nx % nd;
        const uint32_t x0 = (uint32_t)i * base + std::min<uint32_t>((uint32_t)i, rem);
        const uint32_t cnt = base + ((uint32_t)i < rem ? 1u : 0u);
        return grid_to_host_share(prog, corner, step, cnt, ny, nz, x_offset + x0, (char *)h_out + (size_t)x0 * plane * 16);
    });
}

int cc_subdivision_step(const cc_program *prog, const float corner[3], float step, float threshold,
                        uint32_t nx, uint32_t ny, uint32_t nz, uint32_t *d_counter, uint8_t *d_list,
                        cc_event **ev)
{
    NEED_INIT();
    if (!prog || !corner || !d_counter || !d_list) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    int rc = check_dims(nx, ny, nz);
    if (rc) return rc;
    if (nx > 256 || ny > 256 || nz > 256)
        return fail(CC_ERR_INVALID_ARGUMENT, "grid dimension > 256 overflows the uchar4 index list");
    cc_eval_args a;
    FILL_COMMON(a, prog);
    a.cx = corner[0]; a.cy = corner[1]; a.cz = corner[2]; a.step = step;
    a.nx = nx; a.ny = ny; a.nz = nz; a.n_blocks = 1;
    a.threshold = threshold; a.counter = d_counter; a.list = d_list;
    rc = launch(CC_SINK_CLASSIFY, prog, a, (uint64_t)nx * ny * nz);
    if (rc) return rc;
    return make_event(ev, g.compute);
}

int cc_mass_properties_step(const cc_program *prog, const float corner[3], float step, float threshold,
                            uint32_t nx, uint32_t ny, uint32_t nz, uint32_t *d_sums, uint32_t *d_counter,
                            uint8_t *d_list, cc_event **ev)
{
    NEED_INIT();
    if (!prog || !corner || !d_sums || !d_counter || !d_list) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    int rc = check_dims(nx, ny, nz);
    if (rc) return rc;
    if (nx > 256 || ny > 256 || nz > 256)
        return fail(CC_ERR_INVALID_ARGUMENT, "grid dimension > 256 overflows the uchar4 index list");
    cc_eval_args a;
    FILL_COMMON(a, prog);
    a.cx = corner[0]; a.cy = corner[1]; a.cz = corner[2]; a.step = step;
    a.nx = nx; a.ny = ny; a.nz = nz; a.n_blocks = 1;
    a.threshold = threshold; a.counter = d_counter; a.list = d_list; a.sums = d_sums;
    rc = launch(CC_SINK_MASS, prog, a, (uint64_t)nx * ny * nz);
    if (rc) return rc;
    return make_event(ev, g.compute);
}

}  // extern "C"

// ---- hierarchy fast paths --------------------------------------------------------------------------------

namespace {

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    // stream-ordered allocations from the device's default pool (kept warm: cc_init raises the
    // release threshold), all on the compute stream like every user of these buffers
    ~DevBuf() { if (p) cudaFreeAsync(p, g.compute); }
    int reserve(size_t bytes)
    {
        if (bytes <= cap) return CC_OK;
        if (p) cudaFreeAsync(p, g.compute);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMallocAsync(&p, bytes, g.compute);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMallocAsync (hierarchy work list)");
        cap = bytes;
        return CC_OK;
    }
    template <class T> T *as() { return static_cast<T *>(p); }
};

int read_counter(uint32_t *d_counter, uint32_t *out)
{
    CU(cudaMemcpyAsync(g.h_word, d_counter, 4, cudaMemcpyDeviceToHost, g.compute));
    CU(cudaStreamSynchronize(g.compute));
    *out = *g.h_word;
    return CC_OK;
}

// Blocks of one level are processed in chunks so that hit lists stay bounded:
// a chunk evaluates at most `kChunkCells` cells and can emit at most that many hits.
const uint64_t kChunkCells = 1ull << 27;

// Which level's hits are dealt to the shares (ranks x devices): the one that feeds the most
// expensive level, so that the unit of distribution is as fine as it gets.  Levels up to and
// including it are evaluated by every share (they are a few thousand cells), everything below is
// evaluated by the share that owns the block.  Hit h of a launch goes to share h % n_shares.
//   subdivision: levels 0 .. n-2 are classified, n-2 is the big one -> deal the hits of n-3
//   mass properties: the leaf level n-1 is the big one           -> deal the hits of n-2
uint32_t deal_level_subdiv(uint32_t n_levels) { return n_levels >= 3 ? n_levels - 3 : 0; }
uint32_t deal_level_mass(uint32_t n_levels) { return n_levels >= 2 ? n_levels - 2 : 0; }

int check_levels(const cc_level *levels, uint32_t n_levels)
{
    for (uint32_t l = 0; l < n_levels; ++l)
        if (levels[l].nx > 256 || levels[l].ny > 256 || levels[l].nz > 256 || !levels[l].nx || !levels[l].ny ||
            !levels[l].nz || levels[l].cell_size < 1)
            return fail(CC_ERR_INVALID_ARGUMENT, "level grid dimensions must be in 1..256");
    return CC_OK;
}

// subdivision() on the current device for share `rank` of `world`: appends the int corners of the
// share's leaf blocks to *out (host), in the order the levels produce them
int subdivide_share(const cc_program *prog, const double origin[3], double resolution, const cc_level *levels,
                    uint32_t n_levels, int dimension, uint32_t rank, uint32_t world, std::vector<int64_t> *out,
                    uint64_t *dealt_blocks)
{
    DevBuf corners_a, corners_b, blocks, hit_xyz, hit_block, counter;
    int rc;
    if ((rc = counter.reserve(4))) return rc;
    // level 0: one block at int corner (0,0,0)
    std::vector<int64_t> cur_host(3, 0);
    uint64_t n_cur = 1;
    if ((rc = corners_a.reserve(3 * sizeof(int64_t)))) return rc;
    CU(cudaMemcpyAsync(corners_a.p, cur_host.data(), 3 * sizeof(int64_t), cudaMemcpyHostToDevice, g.compute));
    DevBuf *cur = &corners_a, *nxt = &corners_b;
    const uint32_t deal = deal_level_subdiv(n_levels);
    if (dealt_blocks) *dealt_blocks = 0;
    // every block of every level lies inside the root block: the bound on coordinates the tile masks' rounding budget needs
    float coord_max = 0.0f;
    for (int i = 0; i < 3; ++i) {
        const double n0 = i == 0 ? levels[0].nx : i == 1 ? levels[0].ny : levels[0].nz;
        const double far = origin[i] + (n0 + 1.0) * (double)levels[0].cell_size * resolution;
        coord_max = std::max(coord_max, (float)std::max(std::fabs(origin[i]), std::fabs(far)));
    }

    for (uint32_t l = 0; l + 1 < n_levels; ++l) {
        const cc_level &L = levels[l];
        const uint64_t cells = (uint64_t)L.nx * L.ny * L.nz;
        const uint64_t chunk_blocks = std::max<uint64_t>(1, kChunkCells / cells);
        const double box_step = (double)L.cell_size * resolution;
        const float thr = (float)(box_step * std::sqrt((double)dimension) / 2);  // subdivision.py:67
        cc_level_geom geo{origin[0], origin[1], origin[2], resolution, (double)L.cell_size / 2, dimension};
        // children of this level, gathered chunk by chunk
        uint64_t n_next = 0;
        size_t next_cap = 0;
        const uint32_t w = (l == deal) ? world : 1u, r = (l == deal) ? rank : 0u;
        for (uint64_t b0 = 0; b0 < n_cur; b0 += chunk_blocks) {
            const uint32_t nb = (uint32_t)std::min<uint64_t>(chunk_blocks, n_cur - b0);
            if ((rc = blocks.reserve((size_t)nb * sizeof(cc_block_desc)))) return rc;
            if ((rc = hit_xyz.reserve((size_t)nb * cells * 4))) return rc;
            if ((rc = hit_block.reserve((size_t)nb * cells * 4))) return rc;
            int e = cc_launch_make_blocks_subdiv(cur->as<int64_t>() + 3 * b0, nb, geo, blocks.as<cc_block_desc>(), g.compute);
            if (e) return cuda_fail((cudaError_t)e, "make_blocks");
            CU(cudaMemsetAsync(counter.p, 0, 4, g.compute));
            cc_eval_args a;
            FILL_COMMON(a, prog);
            a.step = (float)box_step;
            a.nx = L.nx; a.ny = L.ny; a.nz = L.nz; a.n_blocks = nb;
            a.blocks = blocks.as<cc_block_desc>();
            a.coord_max = coord_max;
            a.threshold = thr;
            a.counter = counter.as<uint32_t>();
            a.list = hit_xyz.as<uint8_t>();
            a.list_block = hit_block.as<uint32_t>();
            if ((rc = launch(CC_SINK_CLASSIFY, prog, a, (uint64_t)nb * cells))) return rc;
            uint32_t hits = 0;
            if ((rc = read_counter(counter.as<uint32_t>(), &hits))) return rc;
            const uint64_t mine = (hits > r) ? ((uint64_t)hits - r + w - 1) / w : 0;
            if (mine) {
                size_t need = (size_t)(n_next + mine) * 3 * sizeof(int64_t);
                if (need > next_cap) {
                    // grow, preserving what earlier chunks produced
                    DevBuf bigger;
                    size_t cap = std::max(need, next_cap * 2);
                    if ((rc = bigger.reserve(cap))) return rc;
                    if (n_next) CU(cudaMemcpyAsync(bigger.p, nxt->p, (size_t)n_next * 3 * sizeof(int64_t),
                                                   cudaMemcpyDeviceToDevice, g.compute));
                    CU(cudaStreamSynchronize(g.compute));
                    std::swap(nxt->p, bigger.p);
                    std::swap(nxt->cap, bigger.cap);
                    next_cap = cap;
                }
                e = cc_launch_expand_children(cur->as<int64_t>() + 3 * b0, hit_block.as<uint32_t>(),
                                              hit_xyz.as<uint8_t>(), hits, L.cell_size, r, w,
                                              nxt->as<int64_t>() + 3 * n_next, g.compute);
                if (e) return cuda_fail((cudaError_t)e, "expand_children");
                g.launches += 1;
                n_next += mine;
            }
            g.launches += 1;  // make_blocks
        }
        std::swap(cur, nxt);
        n_cur = n_next;
        if (l == deal && dealt_blocks) *dealt_blocks = n_cur;
        if (n_cur == 0) break;
    }
    // `cur` now holds the int corners of the share's leaf blocks
    if (n_cur) {
        const size_t at = out->size();
        out->resize(at + (size_t)n_cur * 3);
        CU(cudaMemcpyAsync(out->data() + at, cur->p, (size_t)n_cur * 3 * sizeof(int64_t), cudaMemcpyDeviceToHost, g.compute));
        CU(cudaStreamSynchronize(g.compute));
    }
    return CC_OK;
}

// The order in which one GPU lists the leaf blocks: level by level the hits come out by parent
// block and, inside a block, in INDEX3 cell order (x slowest) — i.e. lexicographic in the per-level
// cell coordinates (x0,y0,z0, x1,y1,z1, ...), which can be read off a leaf corner because
// cell_size[l-1] is a multiple of cell_size[l] that exceeds any offset inside the level.
void hierarchy_order(int64_t *corners, uint64_t n, const cc_level *levels, uint32_t n_levels)
{
    const uint32_t nd = n_levels - 1;  // classified levels
    std::vector<uint32_t> key((size_t)n * nd * 3);
    for (uint64_t i = 0; i < n; ++i)
        for (int ax = 0; ax < 3; ++ax) {
            int64_t rest = corners[3 * i + ax];
            for (uint32_t l = 0; l < nd; ++l) {
                const int64_t cs = levels[l].cell_size;
                key[((size_t)i * nd + l) * 3 + ax] = (uint32_t)(rest / cs);
                rest %= cs;
            }
        }
    std::vector<uint64_t> order((size_t)n);
    for (uint64_t i = 0; i < n; ++i) order[(size_t)i] = i;
    const size_t kl = (size_t)nd * 3;
    std::sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) {
        return std::lexicographical_compare(key.begin() + (ptrdiff_t)(a * kl), key.begin() + (ptrdiff_t)((a + 1) * kl),
                                            key.begin() + (ptrdiff_t)(b * kl), key.begin() + (ptrdiff_t)((b + 1) * kl));
    });
    std::vector<int64_t> sorted((size_t)n * 3);
    for (uint64_t i = 0; i < n; ++i)
        for (int ax = 0; ax < 3; ++ax) sorted[3 * (size_t)i + ax] = corners[3 * order[(size_t)i] + ax];
    std::memcpy(corners, sorted.data(), sorted.size() * sizeof(int64_t));
}

// Exponents of the accumulator quanta of the ten integrals (one,x,y,z,xx,yy,zz,xy,xz,yz): the
// hierarchy lives inside the top-level block, so |integral| and every block's contribution are
// bounded by V, V*M_k, V*M_j*M_k with V its volume and M_k the largest |coordinate| along axis k.
// Depends on the arguments only, hence identical on every device and rank.
cc_mass_quanta mass_quanta(const double box_a[3], double resolution, const cc_level &top)
{
    const double s0 = resolution * (double)top.cell_size;
    const double ext[3] = {top.nx * s0, top.ny * s0, top.nz * s0};
    double M[3], V = 1.0;
    for (int k = 0; k < 3; ++k) {
        M[k] = std::max(std::fabs(box_a[k]), std::fabs(box_a[k] + ext[k])) + s0;
        V *= ext[k];
    }
    const double bound[10] = {V, V * M[0], V * M[1], V * M[2], V * M[0] * M[0], V * M[1] * M[1], V * M[2] * M[2],
                              V * M[0] * M[1], V * M[0] * M[2], V * M[1] * M[2]};
    cc_mass_quanta q;
    for (int i = 0; i < 10; ++i) {
        int e = 0;
        std::frexp(bound[i], &e);  // bound < 2^e
        q.e[i] = e + 3 - 100;      // 8x head room; a value is < 2^100 quanta
    }
    return q;
}

// mass_properties() on the current device for share `rank` of `world`: limb sums of the share's
// contribution (limbs[10][4] + overflow count), stats = launches, cells, blocks, blocks of the dealt level
int mass_share(const cc_program *prog, const double box_a[3], double resolution, const cc_level *levels,
               uint32_t n_levels, uint32_t rank, uint32_t world, const cc_mass_quanta &quanta, int64_t limbs[41],
               uint64_t stats[4])
{
    DevBuf corners_a, corners_b, blocks, hit_xyz, hit_block, counter, sums, acc;
    int rc;
    if ((rc = counter.reserve(4))) return rc;
    if ((rc = acc.reserve(41 * sizeof(unsigned long long)))) return rc;
    CU(cudaMemsetAsync(acc.p, 0, 41 * sizeof(unsigned long long), g.compute));
    double root[3] = {box_a[0], box_a[1], box_a[2]};
    if ((rc = corners_a.reserve(3 * sizeof(double)))) return rc;
    CU(cudaMemcpyAsync(corners_a.p, root, sizeof(root), cudaMemcpyHostToDevice, g.compute));
    CU(cudaStreamSynchronize(g.compute));
    DevBuf *cur = &corners_a, *nxt = &corners_b;
    uint64_t n_cur = 1, n_launch = 0, n_cells = 0, n_blocks_total = 0, n_dealt = 0;
    const uint32_t deal = deal_level_mass(n_levels);
    float coord_max = 0.0f;  // (as in subdivide_share)
    for (int i = 0; i < 3; ++i) {
        const double n0 = i == 0 ? levels[0].nx : i == 1 ? levels[0].ny : levels[0].nz;
        const double far = box_a[i] + (n0 + 1.0) * (double)levels[0].cell_size * resolution;
        coord_max = std::max(coord_max, (float)std::max(std::fabs(box_a[i]), std::fabs(far)));
    }

    for (uint32_t l = 0; l < n_levels && n_cur; ++l) {
        const cc_level &L = levels[l];
        const bool leaf = (l + 1 == n_levels);
        const uint64_t cells = (uint64_t)L.nx * L.ny * L.nz;
        const uint64_t chunk_blocks = std::max<uint64_t>(1, kChunkCells / cells);
        const double s = resolution * (double)L.cell_size;                       // mass_properties.py:51-53
        const float thr = leaf ? 0.0f : (float)(s * std::sqrt(3.0) / 2);         // :87-90
        const uint32_t w = (l == deal) ? world : 1u, r = (l == deal) ? rank : 0u;
        uint64_t n_next = 0;
        size_t next_cap = 0;
        for (uint64_t b0 = 0; b0 < n_cur; b0 += chunk_blocks) {
            const uint32_t nb = (uint32_t)std::min<uint64_t>(chunk_blocks, n_cur - b0);
            if ((rc = blocks.reserve((size_t)nb * sizeof(cc_block_desc)))) return rc;
            if ((rc = sums.reserve((size_t)nb * 10 * 4))) return rc;
            if (!leaf) {
                if ((rc = hit_xyz.reserve((size_t)nb * cells * 4))) return rc;
                if ((rc = hit_block.reserve((size_t)nb * cells * 4))) return rc;
            } else {
                if ((rc = hit_xyz.reserve(16))) return rc;
                if ((rc = hit_block.reserve(16))) return rc;
            }
            int e = cc_launch_mass_make_blocks(cur->as<double>() + 3 * b0, nb, s, blocks.as<cc_block_desc>(), g.compute);
            if (e) return cuda_fail((cudaError_t)e, "mass make_blocks");
            CU(cudaMemsetAsync(counter.p, 0, 4, g.compute));
            CU(cudaMemsetAsync(sums.p, 0, (size_t)nb * 10 * 4, g.compute));
            cc_eval_args a;
            FILL_COMMON(a, prog);
            a.step = (float)s;
            a.nx = L.nx; a.ny = L.ny; a.nz = L.nz; a.n_blocks = nb;
            a.blocks = blocks.as<cc_block_desc>();
            a.coord_max = coord_max;
            a.threshold = thr;
            a.counter = counter.as<uint32_t>();
            a.list = hit_xyz.as<uint8_t>();
            a.list_block = hit_block.as<uint32_t>();
            a.sums = sums.as<uint32_t>();
            if ((rc = launch(CC_SINK_MASS, prog, a, (uint64_t)nb * cells))) return rc;
            n_launch += 1;
            n_cells += (uint64_t)nb * cells;
            n_blocks_total += nb;
            // levels up to the dealt one are evaluated by every share; share 0 alone counts their
            // inside cells
            if (l > deal || rank == 0 || world == 1) {
                e = cc_launch_mass_integrals(cur->as<double>() + 3 * b0, sums.as<uint32_t>(), nb, s, quanta,
                                             acc.as<unsigned long long>(), g.compute);
                if (e) return cuda_fail((cudaError_t)e, "mass integrals");
            }
            g.launches += 2;  // make_blocks, integrals
            if (leaf) continue;
            uint32_t hits = 0;
            if ((rc = read_counter(counter.as<uint32_t>(), &hits))) return rc;
            const uint64_t mine = (hits > r) ? ((uint64_t)hits - r + w - 1) / w : 0;
            if (mine) {
                size_t need = (size_t)(n_next + mine) * 3 * sizeof(double);
                if (need > next_cap) {
                    DevBuf bigger;
                    size_t cap = std::max(need, next_cap * 2);
                    if ((rc = bigger.reserve(cap))) return rc;
                    if (n_next) CU(cudaMemcpyAsync(bigger.p, nxt->p, (size_t)n_next * 3 * sizeof(double),
                                                   cudaMemcpyDeviceToDevice, g.compute));
                    CU(cudaStreamSynchronize(g.compute));
                    std::swap(nxt->p, bigger.p);
                    std::swap(nxt->cap, bigger.cap);
                    next_cap = cap;
                }
                e = cc_launch_mass_expand_children(cur->as<double>() + 3 * b0, hit_block.as<uint32_t>(),
                                                   hit_xyz.as<uint8_t>(), hits, s, r, w,
                                                   nxt->as<double>() + 3 * n_next, g.compute);
                if (e) return cuda_fail((cudaError_t)e, "mass expand_children");
                g.launches += 1;
                n_next += mine;
            }
        }
        std::swap(cur, nxt);
        n_cur = n_next;
        if (l == deal) n_dealt = n_cur;
    }
    unsigned long long h_acc[41];
    CU(cudaMemcpyAsync(h_acc, acc.p, sizeof(h_acc), cudaMemcpyDeviceToHost, g.compute));
    CU(cudaStreamSynchronize(g.compute));
    for (int i = 0; i < 41; ++i) limbs[i] = (int64_t)h_acc[i];
    stats[0] = n_launch;
    stats[1] = n_cells;
    stats[2] = n_blocks_total;
    stats[3] = n_dealt;
    return CC_OK;
}

}  // namespace

extern "C" {

int cc_sort_leaf_corners(int64_t *corners, uint64_t n, const cc_level *levels, uint32_t n_levels)
{
    if ((!corners && n) || !levels || n_levels < 2) return fail(CC_ERR_INVALID_ARGUMENT, "bad argument");
    int rc = check_levels(levels, n_levels);
    if (rc) return rc;
    if (n > 1) hierarchy_order(corners, n, levels, n_levels);
    return CC_OK;
}

int cc_subdivide(const cc_program *prog, const double origin[3], double resolution, const cc_level *levels,
                 uint32_t n_levels, int dimension, uint32_t rank, uint32_t world, int64_t **out_corners,
                 uint64_t *out_count)
{
    NEED_INIT();
    if (!prog || !origin || !levels || !out_corners || !out_count)
        return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    if (n_levels < 2) return fail(CC_ERR_INVALID_ARGUMENT, "cc_subdivide needs at least two levels");
    if (dimension != 2 && dimension != 3) return fail(CC_ERR_INVALID_ARGUMENT, "dimension must be 2 or 3");
    if (world == 0 || rank >= world) return fail(CC_ERR_INVALID_ARGUMENT, "bad rank/world");
    int rc = check_levels(levels, n_levels);
    if (rc) return rc;
    *out_count = 0;
    *out_corners = nullptr;
    // every initialised device takes a share of this rank's share
    const uint32_t nd = (uint32_t)std::max(1, g_n_ctx);
    std::vector<std::vector<int64_t>> part(nd);
    rc = for_each_device([&](int i) {
        return subdivide_share(prog, origin, resolution, levels, n_levels, dimension, rank * nd + (uint32_t)i, world * nd,
                               &part[(size_t)i], nullptr);
    });
    if (rc) return rc;
    size_t total = 0;
    for (auto &v : part) total += v.size();
    if (!total) return CC_OK;
    int64_t *h = (int64_t *)malloc(total * sizeof(int64_t));
    if (!h) return fail(CC_ERR_INVALID_ARGUMENT, "out of host memory");
    size_t at = 0;
    for (auto &v : part) {
        if (!v.empty()) std::memcpy(h + at, v.data(), v.size() * sizeof(int64_t));
        at += v.size();
    }
    if (nd > 1) hierarchy_order(h, total / 3, levels, n_levels);  // the order one GPU produces
    *out_corners = h;
    *out_count = total / 3;
    return CC_OK;
}

int cc_mass_properties_exact(const cc_program *prog, const double box_a[3], double resolution, const cc_level *levels,
                             uint32_t n_levels, uint32_t rank, uint32_t world, int64_t limbs[40], int32_t exponents[10],
                             uint64_t stats[8])
{
    NEED_INIT();
    if (!prog || !box_a || !levels || !limbs || !exponents) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    if (n_levels < 1) return fail(CC_ERR_INVALID_ARGUMENT, "no levels");
    if (world == 0 || rank >= world) return fail(CC_ERR_INVALID_ARGUMENT, "bad rank/world");
    int rc = check_levels(levels, n_levels);
    if (rc) return rc;
    if (!(resolution > 0)) return fail(CC_ERR_INVALID_ARGUMENT, "resolution must be positive");
    const cc_mass_quanta quanta = mass_quanta(box_a, resolution, levels[0]);
    const uint32_t nd = (uint32_t)std::max(1, g_n_ctx);
    std::vector<int64_t> part((size_t)nd * 41, 0);
    std::vector<uint64_t> st((size_t)nd * 4, 0);
    rc = for_each_device([&](int i) {
        return mass_share(prog, box_a, resolution, levels, n_levels, rank * nd + (uint32_t)i, world * nd, quanta,
                          part.data() + (size_t)i * 41, st.data() + (size_t)i * 4);
    });
    if (rc) return rc;
    for (int k = 0; k < 40; ++k) limbs[k] = 0;
    int64_t overflow = 0;
    uint64_t s4[4] = {0, 0, 0, 0}, max_cells = 0, min_cells = UINT64_MAX;
    for (uint32_t i = 0; i < nd; ++i) {
        for (int k = 0; k < 40; ++k) limbs[k] += part[(size_t)i * 41 + k];
        overflow += part[(size_t)i * 41 + 40];
        for (int k = 0; k < 4; ++k) s4[k] += st[(size_t)i * 4 + k];
        max_cells = std::max(max_cells, st[(size_t)i * 4 + 1]);
        min_cells = std::min(min_cells, st[(size_t)i * 4 + 1]);
    }
    if (overflow) return fail(CC_ERR_INVALID_ARGUMENT, "mass integrals left the range of the exact accumulator");
    for (int i = 0; i < 10; ++i) exponents[i] = quanta.e[i];
    if (stats) {
        stats[0] = s4[0]; stats[1] = s4[1]; stats[2] = s4[2]; stats[3] = n_levels;
        stats[4] = s4[3];      // blocks of the dealt level owned by this call's devices
        stats[5] = nd;         // devices used
        stats[6] = max_cells;  // cells evaluated by the busiest / the least busy device
        stats[7] = min_cells;
    }
    return CC_OK;
}

int cc_mass_limbs_to_integrals(const int64_t limbs[40], const int32_t exponents[10], double integrals[10])
{
    if (!limbs || !exponents || !integrals) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    for (int i = 0; i < 10; ++i) {
        __int128 t = 0;
        for (int k = 3; k >= 0; --k) t = t * ((__int128)1 << 32) + (__int128)limbs[4 * i + k];
        // (double)__int128 rounds to nearest even; ldexp is exact here
        integrals[i] = std::ldexp((double)t, exponents[i]);
    }
    return CC_OK;
}

int cc_mass_properties(const cc_program *prog, const double box_a[3], double resolution, const cc_level *levels,
                       uint32_t n_levels, uint32_t rank, uint32_t world, double integrals[10], uint64_t stats[4])
{
    if (!integrals) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    int64_t limbs[40];
    int32_t ex[10];
    uint64_t st[8];
    int rc = cc_mass_properties_exact(prog, box_a, resolution, levels, n_levels, rank, world, limbs, ex, st);
    if (rc) return rc;
    if (stats)
        for (int k = 0; k < 4; ++k) stats[k] = st[k];
    return cc_mass_limbs_to_integrals(limbs, ex, integrals);
}

}  // extern "C"

// ---- mesh export: marching cubes over leaf blocks --------------------------------------------------------

namespace {
int launch_render(bool ray, const cc_program *prog, cc_render_launch &r, uint64_t *eval_count)
{
    if (r.w == 0 || r.h == 0) return fail(CC_ERR_INVALID_ARGUMENT, "empty image");
    if ((uint64_t)r.w * r.h > (1ull << 31)) return fail(CC_ERR_INVALID_ARGUMENT, "more than 2^31 pixels");
    const int sink = ray ? CC_SINK_RAY : CC_SINK_BITMAP;
    const bool specialised = jit_ready(const_cast<cc_program *>(prog), sink);
    cc_launch_cfg cfg{1, prog->dec.info.n_micro_words <= CC_CONST_WORDS && g.prog_space != 2 ? 1 : 2};
    if (!specialised) {
        const size_t need = cc_eval_smem_bytes(cfg, prog->dec.info.n_slots, prog->dec.info.n_micro_words);
        if (need > (size_t)g.prop.sharedMemPerBlockOptin)
            return fail(CC_ERR_TOO_LARGE, "program needs " + std::to_string(need) + " bytes of shared memory per CTA");
        int rc = prepare_program(prog, cfg);
        if (rc) return rc;
    }
    {
        int rc = program_on_device(prog, &r.code);
        if (rc) return rc;
    }
    r.code_words = prog->dec.info.n_micro_words;
    r.n_slots = prog->dec.info.n_slots;
    DevBuf count;  // released on every path
    if (eval_count) {
        int rc = count.reserve(8);
        if (rc) return rc;
        CU(cudaMemsetAsync(count.p, 0, 8, g.compute));
    }
    r.eval_count = count.as<unsigned long long>();
    int e = cc_launch_render(ray ? 1 : 0, specialised ? 0 : cfg.prog_space, specialised ? prog : nullptr, r, g.compute, g.index);
    if (e) return cuda_fail((cudaError_t)e, "render kernel launch");
    g.launches += 1;
    g.points += (uint64_t)r.w * r.h;
    if (eval_count) {
        unsigned long long h = 0;
        CU(cudaMemcpyAsync(&h, count.p, 8, cudaMemcpyDeviceToHost, g.compute));
        CU(cudaStreamSynchronize(g.compute));
        *eval_count = h;
    }
    return CC_OK;
}
}  // namespace

// ---- host half of polygon(): follow the links of process_polygon into closed outlines -------------
// (rendering/polygon2d.py:15-31 _collect_polygon / _step_from_overflow_spec, :119-170).  No device
// work: usable without cc_init.
namespace {
constexpr uint32_t kLinkOverflowMask = 0xFFF00000u;  // flags (bits 29-31) + row / column (bits 20-28)
constexpr uint32_t kLinkIndexMask = 0x000FFFFFu;

struct PieceKey {
    int64_t x, y;
    uint32_t spec;
    bool operator==(const PieceKey &o) const { return x == o.x && y == o.y && spec == o.spec; }
};
struct PieceKeyHash {
    size_t operator()(const PieceKey &k) const
    {
        uint64_t h = (uint64_t)k.x * 0x9E3779B97F4A7C15ull;
        h ^= ((uint64_t)k.y + 0x7F4A7C15ull + (h << 6) + (h >> 2));
        h ^= ((uint64_t)k.spec * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2));
        return (size_t)h;
    }
};
struct Piece {
    std::vector<float> v;  // x0, y0, x1, y1, ...
    PieceKey begin, end;
};
// Outline pieces that cross box borders, joinable at either end.
struct OpenChains {
    std::unordered_map<PieceKey, Piece *, PieceKeyHash> by_begin, by_end;
    std::vector<std::unique_ptr<Piece>> store;
    // returns the piece if this addition closed it
    Piece *add(std::vector<float> &&chain, const PieceKey &begin, const PieceKey &end)
    {
        Piece *piece;
        auto it = by_end.find(begin);
        if (it == by_end.end()) {
            store.emplace_back(new Piece{std::move(chain), begin, end});
            piece = store.back().get();
            by_begin[begin] = piece;
        } else {  // continues a chain that ended on this box's border
            piece = it->second;
            by_end.erase(it);
            piece->v.insert(piece->v.end(), chain.begin(), chain.end());
            piece->end = end;
        }
        auto jt = by_begin.find(end);
        if (jt == by_begin.end()) {
            by_end[end] = piece;
            return nullptr;
        }
        Piece *next = jt->second;
        by_begin.erase(jt);
        if (next == piece) return piece;
        piece->v.insert(piece->v.end(), next->v.begin(), next->v.end());
        piece->end = next->end;
        std::vector<float>().swap(next->v);
        by_end[piece->end] = piece;
        return nullptr;
    }
};

// appends the vertices from `index` on; visited links are overwritten with the mask; returns the
// flags of the terminating link, or 0xFFFFFFFF on a link that points outside the box's arrays
uint32_t follow_links(uint32_t *links, const float *vertices, uint32_t cells, uint32_t index, std::vector<float> *chain)
{
    while (!(index & kLinkOverflowMask)) {
        if (index >= cells) return 0xFFFFFFFFu;
        chain->push_back(vertices[2 * (size_t)index]);
        chain->push_back(vertices[2 * (size_t)index + 1]);
        const uint32_t next = links[index];
        links[index] = kLinkOverflowMask;
        index = next;
    }
    return index & kLinkOverflowMask;
}
}  // namespace

extern "C" int cc_polygon_assemble(const float *vertices, uint32_t *links, const uint32_t *starts,
                                   const uint32_t *start_counts, const int64_t *int_corners, int64_t int_step,
                                   uint32_t cells, uint32_t max_starts, uint32_t n_blocks, float **out_vertices,
                                   uint64_t **out_offsets, uint64_t *out_chains)
{
    if (!vertices || !links || !starts || !start_counts || !int_corners || !out_vertices || !out_offsets || !out_chains)
        return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    *out_vertices = nullptr;
    *out_offsets = nullptr;
    *out_chains = 0;
    std::vector<float> all;            // vertices of the finished outlines, in the order they close
    std::vector<uint64_t> offsets{0};  // in vertices
    OpenChains open;
    for (uint32_t b = 0; b < n_blocks; ++b) {
        uint32_t *bl = links + (size_t)b * cells;
        const float *bv = vertices + 2 * (size_t)b * cells;
        const int64_t cx = int_corners[3 * (size_t)b], cy = int_corners[3 * (size_t)b + 1];
        const uint32_t ns = start_counts[b];
        if (ns > max_starts) return fail(CC_ERR_INVALID_ARGUMENT, "more open chains than the start list holds");
        for (uint32_t k = 0; k < ns; ++k) {  // chains that enter through the box border (polygon2d.py:121-163)
            const uint32_t start = starts[(size_t)b * max_starts + k];
            std::vector<float> chain;
            const uint32_t spec = follow_links(bl, bv, cells, start & kLinkIndexMask, &chain);
            if (spec == 0xFFFFFFFFu) return fail(CC_ERR_INVALID_ARGUMENT, "corrupt link");
            const int64_t d = (spec & 0x20000000u) ? -1 : 1;  // polygon2d.py:26-31
            const bool along_y = (spec & 0x40000000u) != 0;
            const PieceKey begin{cx, cy, start & kLinkOverflowMask};
            const PieceKey end{cx + (along_y ? 0 : d * int_step), cy + (along_y ? d * int_step : 0), spec};
            if (Piece *closed = open.add(std::move(chain), begin, end)) {
                all.insert(all.end(), closed->v.begin(), closed->v.end());
                offsets.push_back(all.size() / 2);
                std::vector<float>().swap(closed->v);
            }
        }
        for (uint32_t i = 0; i < cells; ++i) {  // what is left are chains closed inside the box (:165-170)
            if (bl[i] & kLinkOverflowMask) continue;
            const size_t before = all.size();
            const uint32_t spec = follow_links(bl, bv, cells, i, &all);
            if (spec == 0xFFFFFFFFu) return fail(CC_ERR_INVALID_ARGUMENT, "corrupt link");
            (void)before;
            offsets.push_back(all.size() / 2);
        }
    }
    if (!open.by_begin.empty() || !open.by_end.empty())
        return fail(CC_ERR_OPEN_OUTLINE, "an outline left the subdivided region");
    const size_t n_chains = offsets.size() - 1;
    float *v = (float *)malloc(std::max<size_t>(all.size(), 1) * sizeof(float));
    uint64_t *o = (uint64_t *)malloc(offsets.size() * sizeof(uint64_t));
    if (!v || !o) {
        free(v);
        free(o);
        return fail(CC_ERR_INVALID_ARGUMENT, "out of host memory");
    }
    if (!all.empty()) std::memcpy(v, all.data(), all.size() * sizeof(float));
    std::memcpy(o, offsets.data(), offsets.size() * sizeof(uint64_t));
    *out_vertices = v;
    *out_offsets = o;
    *out_chains = n_chains;
    return CC_OK;
}

extern "C" {

int cc_ray_caster(const cc_program *prog, const float origin[3], const float forward[3], const float up[3],
                  const float right[3], float pixel_tolerance, float box_radius, float min_distance,
                  float max_distance, float floor_z, uint32_t render_options, uint32_t width, uint32_t height,
                  uint8_t *d_out, uint64_t *eval_count, cc_event **ev)
{
    NEED_INIT();
    if (!prog || !origin || !forward || !up || !right || !d_out) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    if (render_options & ~3u) return fail(CC_ERR_INVALID_ARGUMENT, "unknown render option");
    cc_render_launch r;
    std::memset(&r, 0, sizeof(r));
    for (int i = 0; i < 3; ++i) {
        r.origin[i] = origin[i]; r.forward[i] = forward[i]; r.up[i] = up[i]; r.right[i] = right[i];
    }
    r.pixel_tolerance = pixel_tolerance; r.box_radius = box_radius; r.min_distance = min_distance;
    r.max_distance = max_distance; r.floor_z = floor_z; r.options = render_options;
    r.w = width; r.h = height; r.out = d_out;
    int rc = launch_render(true, prog, r, eval_count);
    if (rc) return rc;
    return make_event(ev, g.compute);
}

int cc_bitmap(const cc_program *prog, const float origin[3], float step_size, uint32_t width, uint32_t height,
              uint8_t *d_out, cc_event **ev)
{
    NEED_INIT();
    if (!prog || !origin || !d_out) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    cc_render_launch r;
    std::memset(&r, 0, sizeof(r));
    for (int i = 0; i < 3; ++i) r.origin[i] = origin[i];
    r.step_size = step_size; r.w = width; r.h = height; r.out = d_out;
    int rc = launch_render(false, prog, r, nullptr);
    if (rc) return rc;
    return make_event(ev, g.compute);
}

int cc_matplotlib_slice(const cc_program *prog, const float corner[3], float step, uint32_t width, uint32_t height,
                        float *d_out, cc_event **ev)
{
    NEED_INIT();
    if (!prog || !corner || !d_out) return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    int rc = check_dims(width, height, 1);
    if (rc) return rc;
    DevBuf field;
    if ((rc = field.reserve((size_t)width * height * 16))) return rc;
    cc_eval_args a;
    FILL_COMMON(a, prog);
    a.cx = corner[0]; a.cy = corner[1]; a.cz = corner[2]; a.step = step;
    a.nx = width; a.ny = height; a.nz = 1; a.n_blocks = 1;
    a.out = field.p;
    if ((rc = launch(CC_SINK_FLOAT4, prog, a, (uint64_t)width * height))) return rc;
    int e = cc_launch_slice_repack(field.p, width, height, d_out, g.compute);
    if (e) return cuda_fail((cudaError_t)e, "slice repack launch");
    g.launches += 1;
    return make_event(ev, g.compute);
}

int cc_process_polygon(const float box_corner[2], float box_step, uint32_t cells_x, uint32_t cells_y,
                       const void *d_corners, void *d_vertices, uint32_t *d_links, uint32_t *d_starts,
                       uint32_t max_starts, uint32_t *d_start_counter, cc_event **ev)
{
    NEED_INIT();
    if (!box_corner || !d_corners || !d_vertices || !d_links || !d_starts || !d_start_counter)
        return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    if (cells_x == 0 || cells_y == 0) return fail(CC_ERR_INVALID_ARGUMENT, "empty grid");
    if (cells_x >= 512 || cells_y >= 512)
        return fail(CC_ERR_INVALID_ARGUMENT, "grid of 512 or more cells overflows the link encoding");  // polygon2d.py:46
    if (max_starts == 0 || max_starts > 1024) return fail(CC_ERR_INVALID_ARGUMENT, "max_starts must be 1..1024");
    cc_polygon_args a;
    std::memset(&a, 0, sizeof(a));
    a.corner_x = box_corner[0]; a.corner_y = box_corner[1]; a.step = box_step;
    a.cx = cells_x; a.cy = cells_y; a.n_blocks = 1;
    a.corners = (const float4 *)d_corners;
    a.vertices = (float2 *)d_vertices;
    a.links = d_links; a.starts = d_starts; a.start_counter = d_start_counter; a.max_starts = max_starts;
    int e = cc_launch_process_polygon(a, g.compute);
    if (e) return cuda_fail((cudaError_t)e, "process_polygon launch");
    g.launches += 2;
    return make_event(ev, g.compute);
}

int cc_polygon_blocks(const cc_program *prog, const double *corners, double resolution, uint32_t gx, uint32_t gy,
                      uint32_t n_blocks, float *h_vertices, uint32_t *h_links, uint32_t *h_starts,
                      uint32_t *h_start_counts)
{
    NEED_INIT();
    if (!prog || !corners || !h_vertices || !h_links || !h_starts || !h_start_counts)
        return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    if (gx < 2 || gy < 2) return fail(CC_ERR_INVALID_ARGUMENT, "outline extraction needs at least 2 samples per axis");
    if (gx > 512 || gy > 512)
        return fail(CC_ERR_INVALID_ARGUMENT, "grid of more than 512 samples overflows the link encoding");
    if (n_blocks == 0) return CC_OK;
    const uint32_t cx = gx - 1, cy = gy - 1, max_starts = cx + cy;  // polygon2d.py:63-69
    const uint64_t samples = (uint64_t)gx * gy, cells = 2ull * cx * cy;
    const uint32_t chunk = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(n_blocks, (1ull << 26) / samples));
    DevBuf field, descs, d_corner2, vertices, links, starts, counts;
    int rc;
    if ((rc = field.reserve((size_t)chunk * samples * 16))) return rc;
    if ((rc = descs.reserve((size_t)chunk * sizeof(cc_block_desc)))) return rc;
    if ((rc = d_corner2.reserve((size_t)chunk * 8))) return rc;
    if ((rc = vertices.reserve((size_t)chunk * cells * 8))) return rc;
    if ((rc = links.reserve((size_t)chunk * cells * 4))) return rc;
    if ((rc = starts.reserve((size_t)chunk * max_starts * 4))) return rc;
    if ((rc = counts.reserve((size_t)chunk * 4))) return rc;
    std::vector<cc_block_desc> h_desc(chunk);
    std::vector<float> h_c2(2 * (size_t)chunk);
    const float step = (float)resolution;  // numpy.float32(box_resolution), polygon2d.py:96,107
    for (uint32_t b0 = 0; b0 < n_blocks; b0 += chunk) {
        const uint32_t nb = std::min(chunk, n_blocks - b0);
        for (uint32_t b = 0; b < nb; ++b) {  // as_float4() / as_float2(): float64 -> float32 per block
            const double *c = corners + 3 * (size_t)(b0 + b);
            h_desc[b] = cc_block_desc{(float)c[0], (float)c[1], (float)c[2], 0u};
            h_c2[2 * b] = (float)c[0];
            h_c2[2 * b + 1] = (float)c[1];
        }
        CU(cudaMemcpyAsync(descs.p, h_desc.data(), (size_t)nb * sizeof(cc_block_desc), cudaMemcpyHostToDevice, g.compute));
        CU(cudaMemcpyAsync(d_corner2.p, h_c2.data(), (size_t)nb * 8, cudaMemcpyHostToDevice, g.compute));
        cc_eval_args a;
        FILL_COMMON(a, prog);
        a.step = step;
        a.nx = gx; a.ny = gy; a.nz = 1; a.n_blocks = nb;
        a.blocks = descs.as<cc_block_desc>();
        a.out = field.p;
        if ((rc = launch(CC_SINK_FLOAT4, prog, a, (uint64_t)nb * samples))) return rc;
        CU(cudaMemsetAsync(vertices.p, 0, (size_t)nb * cells * 8, g.compute));
        CU(cudaMemsetAsync(starts.p, 0, (size_t)nb * max_starts * 4, g.compute));
        CU(cudaMemsetAsync(counts.p, 0, (size_t)nb * 4, g.compute));
        cc_polygon_args pa;
        std::memset(&pa, 0, sizeof(pa));
        pa.step = step;
        pa.block_corners = d_corner2.as<float>();
        pa.cx = cx; pa.cy = cy; pa.n_blocks = nb;
        pa.corners = (const float4 *)field.p;
        pa.vertices = (float2 *)vertices.p;
        pa.links = links.as<uint32_t>();
        pa.starts = starts.as<uint32_t>();
        pa.start_counter = counts.as<uint32_t>();
        pa.max_starts = max_starts;
        int e = cc_launch_process_polygon(pa, g.compute);
        if (e) return cuda_fail((cudaError_t)e, "process_polygon launch");
        g.launches += 2;
        CU(cudaMemcpyAsync(h_vertices + (size_t)b0 * cells * 2, vertices.p, (size_t)nb * cells * 8, cudaMemcpyDeviceToHost, g.compute));
        CU(cudaMemcpyAsync(h_links + (size_t)b0 * cells, links.p, (size_t)nb * cells * 4, cudaMemcpyDeviceToHost, g.compute));
        CU(cudaMemcpyAsync(h_starts + (size_t)b0 * max_starts, starts.p, (size_t)nb * max_starts * 4, cudaMemcpyDeviceToHost, g.compute));
        CU(cudaMemcpyAsync(h_start_counts + b0, counts.p, (size_t)nb * 4, cudaMemcpyDeviceToHost, g.compute));
        CU(cudaStreamSynchronize(g.compute));  // h_desc / h_c2 are reused by the next chunk
    }
    return CC_OK;
}

int cc_mesh_blocks(const cc_program *prog, const double *corners, double resolution, uint32_t nx, uint32_t ny,
                   uint32_t nz, uint32_t n_blocks, double **out_vertices, uint32_t **out_triangle_block,
                   uint64_t *out_triangles)
{
    NEED_INIT();
    if (!prog || !corners || !out_vertices || !out_triangle_block || !out_triangles)
        return fail(CC_ERR_INVALID_ARGUMENT, "null argument");
    if (nx < 2 || ny < 2 || nz < 2) return fail(CC_ERR_INVALID_ARGUMENT, "marching cubes needs at least 2 samples per axis");
    const uint64_t cells = (uint64_t)nx * ny * nz;
    if (cells > (1ull << 30)) return fail(CC_ERR_INVALID_ARGUMENT, "block too large");
    *out_vertices = nullptr;
    *out_triangle_block = nullptr;
    *out_triangles = 0;
    if (n_blocks == 0) return CC_OK;
    if (!g.mesh_tables) {  // __constant__ tables are per device (and gone after cc_shutdown)
        int e = cc_mesh_upload_tables(g.compute);
        if (e) return cuda_fail((cudaError_t)e, "marching-cubes tables");
        g.mesh_tables = true;
    }
    // Phase A per chunk of blocks: evaluate the field, count triangles per tile, scan.  Phase B per
    // chunk: emit the triangles.  When every chunk's field fits the budget at once (the usual
    // case), all of phase A runs first, the page-locked result is sized from the totals, and each
    // chunk's triangles start crossing PCIe on the copy stream as soon as its emit pass is done,
    // while the next chunk emits.  Larger meshes keep one field buffer, run A + B chunk by chunk
    // and copy at the end.
    struct Chunk {
        uint32_t b0 = 0, nb = 0, n_tri = 0, n_tiles = 0;
        DevBuf field, descs, corner, scratch, vertices, tri_block;
        cc_mesh_args m;
    };
    // (both sizes can be overridden for tests: CODECAD_B200_MESH_FIELD_BUDGET / _MESH_CHUNK_BYTES)
    uint64_t field_budget = 4ull << 30;
    if (const char *t = getenv("CODECAD_B200_MESH_FIELD_BUDGET")) field_budget = strtoull(t, nullptr, 10);
    const bool resident = (uint64_t)n_blocks * cells * 4 <= field_budget;
    // blocks per chunk: ~256 MiB of field when the copies are pipelined (several chunks to overlap),
    // ~1 GiB otherwise
    uint64_t chunk_bytes = resident ? (1ull << 28) : (1ull << 30);
    if (const char *t = getenv("CODECAD_B200_MESH_CHUNK_BYTES")) chunk_bytes = std::max<uint64_t>(1, strtoull(t, nullptr, 10));
    const uint32_t chunk = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(n_blocks, chunk_bytes / (cells * 4)));
    std::vector<std::unique_ptr<Chunk>> chunks;
    DevBuf counter, shared_field;
    int rc;
    if ((rc = counter.reserve(8))) return rc;
    if (!resident && (rc = shared_field.reserve((size_t)chunk * cells * 4))) return rc;
    std::vector<cc_block_desc> h_desc(chunk);
    const float step = (float)resolution;  // numpy.float32(box_resolution), rendering/mesh.py:58
    float mesh_coord_max = 0.0f;  // largest |corner coordinate| seen so far (the tile masks' rounding budget adds the block's extent)

    auto phase_a = [&](Chunk &c) -> int {
        int rc2;
        const uint32_t nb = c.nb;
        if (resident && (rc2 = c.field.reserve((size_t)nb * cells * 4))) return rc2;
        if ((rc2 = c.descs.reserve((size_t)nb * sizeof(cc_block_desc)))) return rc2;
        if ((rc2 = c.corner.reserve((size_t)nb * 3 * sizeof(double)))) return rc2;
        for (uint32_t b = 0; b < nb; ++b) {  // Vector.as_float4(): float64 -> float32 per block
            const double *p = corners + 3 * (size_t)(c.b0 + b);
            h_desc[b] = cc_block_desc{(float)p[0], (float)p[1], (float)p[2], 0u};
            mesh_coord_max = std::max(mesh_coord_max, (float)std::max(std::fabs(p[0]), std::max(std::fabs(p[1]), std::fabs(p[2]))));
        }
        CU(cudaMemcpyAsync(c.descs.p, h_desc.data(), (size_t)nb * sizeof(cc_block_desc), cudaMemcpyHostToDevice, g.compute));
        CU(cudaMemcpyAsync(c.corner.p, corners + 3 * (size_t)c.b0, (size_t)nb * 3 * sizeof(double), cudaMemcpyHostToDevice,
                           g.compute));
        void *field = resident ? c.field.p : shared_field.p;
        cc_eval_args a;
        FILL_COMMON(a, prog);
        a.step = step;
        a.nx = nx; a.ny = ny; a.nz = nz; a.n_blocks = nb;
        a.blocks = c.descs.as<cc_block_desc>();
        a.coord_max = mesh_coord_max;
        a.out = field;
        if ((rc2 = launch(CC_SINK_PYMCUBES, prog, a, (uint64_t)nb * cells))) return rc2;

        cc_mesh_args &m = c.m;
        std::memset(&m, 0, sizeof(m));
        m.field = (const float *)field;
        m.d0 = nx; m.d1 = ny; m.d2 = nz;  // numpy.empty(max_box_size): the array shape mcubes sees
        m.n_blocks = nb;
        m.tiles_per_block = cc_mesh_tiles_per_block(nx, ny, nz);
        m.corner = c.corner.as<double>();
        m.resolution = resolution;
        m.counter = counter.as<uint32_t>();
        m.first_block = c.b0;
        const uint64_t tiles = (uint64_t)m.tiles_per_block * nb;
        if (tiles >= (1ull << 31)) return fail(CC_ERR_INVALID_ARGUMENT, "too many tiles in one launch");
        const size_t words = cc_mesh_scratch_words((uint32_t)tiles);
        if ((rc2 = c.scratch.reserve(words * 4))) return rc2;
        m.tile_offsets = c.scratch.as<uint32_t>();
        m.tile_list = m.tile_offsets + (words - tiles);
        int e = cc_launch_mesh(m, false, 0, g.compute);  // count per tile + scan + list of non-empty tiles
        if (e) return cuda_fail((cudaError_t)e, "marching cubes (count)");
        g.launches += 4;
        uint32_t h2[2] = {0, 0};
        CU(cudaMemcpyAsync(h2, counter.p, 8, cudaMemcpyDeviceToHost, g.compute));
        CU(cudaStreamSynchronize(g.compute));  // also: h_desc is reused by the next chunk
        c.n_tri = h2[0];
        c.n_tiles = h2[1];
        return CC_OK;
    };
    auto phase_b = [&](Chunk &c) -> int {
        if (c.n_tri == 0) return CC_OK;
        int rc2;
        if ((rc2 = c.vertices.reserve((size_t)c.n_tri * 9 * sizeof(double)))) return rc2;
        if ((rc2 = c.tri_block.reserve((size_t)c.n_tri * 4))) return rc2;
        c.m.vertices = c.vertices.as<double>();
        c.m.tri_block = c.tri_block.as<uint32_t>();
        int e = cc_launch_mesh(c.m, true, c.n_tiles, g.compute);
        if (e) return cuda_fail((cudaError_t)e, "marching cubes (emit)");
        g.launches += 1;
        return CC_OK;
    };

    for (uint32_t b0 = 0; b0 < n_blocks; b0 += chunk) {
        chunks.emplace_back(new Chunk);
        Chunk &c = *chunks.back();
        c.b0 = b0;
        c.nb = std::min(chunk, n_blocks - b0);
        if ((rc = phase_a(c))) return rc;
        if (!resident && (rc = phase_b(c))) return rc;  // the shared field is overwritten by the next chunk
    }
    size_t n = 0;
    for (auto &c : chunks) n += c->n_tri;
    *out_triangles = n;
    if (n == 0) return CC_OK;
    double *v = (double *)g_pinned.get(n * 9 * sizeof(double));  // page-locked: the copy runs at PCIe speed
    uint32_t *b = (uint32_t *)g_pinned.get(n * sizeof(uint32_t));
    if (!v || !b) {
        cc_free(v);
        cc_free(b);
        return fail(CC_ERR_INVALID_ARGUMENT, "out of host memory");
    }
    size_t at = 0;
    cudaError_t ce = cudaSuccess;
    rc = CC_OK;
    cudaEvent_t emitted = nullptr;
    if (resident) ce = cudaEventCreateWithFlags(&emitted, cudaEventDisableTiming);
    for (auto &cp : chunks) {
        Chunk &c = *cp;
        if (c.n_tri == 0) continue;
        cudaStream_t copy_on = g.compute;
        if (resident && ce == cudaSuccess) {
            if ((rc = phase_b(c))) break;
            ce = cudaEventRecord(emitted, g.compute);
            if (ce == cudaSuccess) ce = cudaStreamWaitEvent(g.copy, emitted, 0);
            copy_on = g.copy;  // this chunk's triangles cross PCIe while the next chunk emits
        }
        if (ce == cudaSuccess)
            ce = cudaMemcpyAsync(v + at * 9, c.vertices.p, (size_t)c.n_tri * 9 * sizeof(double), cudaMemcpyDeviceToHost, copy_on);
        if (ce == cudaSuccess)
            ce = cudaMemcpyAsync(b + at, c.tri_block.p, (size_t)c.n_tri * 4, cudaMemcpyDeviceToHost, copy_on);
        at += c.n_tri;
    }
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(g.compute);
    cudaError_t ce2 = cudaStreamSynchronize(g.copy);  // before the chunks' device buffers are released
    if (ce == cudaSuccess) ce = ce2;
    if (emitted) cudaEventDestroy(emitted);
    if (rc != CC_OK || ce != cudaSuccess) {
        cc_free(v);
        cc_free(b);
        return rc != CC_OK ? rc : cuda_fail(ce, "triangles D2H");
    }
    *out_vertices = v;
    *out_triangle_block = b;
    return CC_OK;
}

}  // extern "C"
