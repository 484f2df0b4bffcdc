// Scene-specialised kernels: the decoded microcode of one program is turned into straight-line
// CUDA C++ (every parameter an immediate, every value slot a register), compiled at run time
// with NVRTC for sm_100a and loaded through the runtime's library API.
//
// This is SURVEY.md §8(f) rank 2 ("scene-specialised kernels via NVRTC"; the reference
// itself can print a straight-line C evaluator: nodes/codegen.py:137-204).  The generated
// code calls the very same op library (cc_ops.cuh / cc_math.cuh) and the same kernel body
// (cc_body.cuh: coordinates, sinks, ordered compaction) as the interpreter, compiled with the
// same -fmad=false contract, so results are bit-identical; what disappears is instruction
// fetch, decode, dispatch, parameter loads and the shared-memory value slots.
//
// NVRTC is loaded with dlopen: without it cc_program_specialize() reports an error and the
// interpreter kernels remain the (only) path.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <mutex>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "cc_internal.h"

namespace {

// ---- NVRTC through dlopen ------------------------------------------------------------------------
typedef struct _nvrtcProgram *nvrtcProgram;
struct Nvrtc {
    void *handle = nullptr;
    int (*CreateProgram)(nvrtcProgram *, const char *, const char *, int, const char *const *, const char *const *);
    int (*CompileProgram)(nvrtcProgram, int, const char *const *);
    int (*GetProgramLogSize)(nvrtcProgram, size_t *);
    int (*GetProgramLog)(nvrtcProgram, char *);
    int (*GetCUBINSize)(nvrtcProgram, size_t *);
    int (*GetCUBIN)(nvrtcProgram, char *);
    int (*DestroyProgram)(nvrtcProgram *);
    const char *(*GetErrorString)(int);
    int (*Version)(int *, int *);
};

// Leaked on purpose (like the caches below): a background compile thread may still be running when
// the process exits, and must not find these destroyed by static destruction.
std::mutex &g_nvrtc_mu = *new std::mutex;

bool load_nvrtc(Nvrtc *n, std::string *err)
{
    static Nvrtc cached;
    if (cached.handle) {
        *n = cached;
        return true;
    }
    // Candidates: $CODECAD_B200_NVRTC, the CUDA toolkit's copy, whatever the loader finds by name.
    // A process that imported PyTorch resolves "libnvrtc.so.12" to torch's bundled (older) NVRTC,
    // whose code generator does not fold negations into the packed FFMA2 operands (+10 % executed
    // instructions on the planetary scene), so the newest version among the candidates wins.
    std::vector<std::string> names;
    if (const char *e = getenv("CODECAD_B200_NVRTC")) names.push_back(e);
    if (const char *e = getenv("CUDA_HOME")) names.push_back(std::string(e) + "/lib64/libnvrtc.so.12");
    names.push_back("/usr/local/cuda/lib64/libnvrtc.so.12");
    names.push_back("/usr/local/cuda/lib64/libnvrtc.so");
    names.push_back("libnvrtc.so.12");
    names.push_back("libnvrtc.so");
    void *h = nullptr;
    int best = -1;
    for (const std::string &nm : names) {
        void *cand = dlopen(nm.c_str(), RTLD_NOW | RTLD_LOCAL);
        if (!cand) continue;
        int major = 0, minor = 0;
        int (*ver)(int *, int *) = (int (*)(int *, int *))dlsym(cand, "nvrtcVersion");
        if (ver) ver(&major, &minor);
        if (major * 100 + minor > best) {
            best = major * 100 + minor;
            h = cand;
        }
    }
    if (!h) {
        *err = "NVRTC (libnvrtc.so.12) not found: scene-specialised kernels unavailable";
        return false;
    }
    Nvrtc r;
    r.handle = h;
#define SYM(field, name)                                                  \
    *(void **)(&r.field) = dlsym(h, name);                                \
    if (!r.field) {                                                       \
        *err = std::string("NVRTC symbol missing: ") + name;              \
        return false;                                                     \
    }
    SYM(CreateProgram, "nvrtcCreateProgram")
    SYM(CompileProgram, "nvrtcCompileProgram")
    SYM(GetProgramLogSize, "nvrtcGetProgramLogSize")
    SYM(GetProgramLog, "nvrtcGetProgramLog")
    SYM(GetCUBINSize, "nvrtcGetCUBINSize")
    SYM(GetCUBIN, "nvrtcGetCUBIN")
    SYM(DestroyProgram, "nvrtcDestroyProgram")
    SYM(GetErrorString, "nvrtcGetErrorString")
    SYM(Version, "nvrtcVersion")
#undef SYM
    cached = r;
    *n = r;
    return true;
}

std::string source_dir()
{
    Dl_info info;
    if (dladdr((void *)&source_dir, &info) && info.dli_fname) {
        std::string p(info.dli_fname);
        size_t k = p.rfind('/');
        return (k == std::string::npos ? std::string(".") : p.substr(0, k)) + "/csrc/";
    }
    return "csrc/";
}

bool read_file(const std::string &path, std::string *out)
{
    std::ifstream f(path.c_str(), std::ios::binary);
    if (!f) return false;
    std::stringstream ss;
    ss << f.rdbuf();
    *out = ss.str();
    return true;
}

// ---- code generation ---------------------------------------------------------------------------------

struct Gen {
    const std::vector<uint32_t> &code;
    std::ostringstream body, consts, params;
    int n_tables = 0;
    size_t n_params = 0;  // words in the __constant__ parameter table of the out-of-line ops
    int n_cells = 0;

    explicit Gen(const std::vector<uint32_t> &c) : code(c) {}

    std::string F(uint32_t idx) const  // exact fp32 literal of microcode word idx
    {
        char buf[48];
        std::snprintf(buf, sizeof buf, "__uint_as_float(0x%08xu)", code[idx]);
        return buf;
    }
    std::string args(uint32_t pc, int first, int count) const
    {
        std::string s;
        for (int i = 0; i < count; ++i) s += (i ? ", " : "") + F(pc + first + i);
        return s;
    }
    float value(uint32_t idx) const
    {
        float f;
        std::memcpy(&f, &code[idx], 4);
        return f;
    }
    // One matrix row written out term by term with cc-arith's rules (cc_ops.cuh cc_row_to /
    // cc_row_from): innermost-first (z, y, x), zero coefficients omitted.  Emitting the folded form
    // here instead of calling the masked templates keeps NVRTC's work small (compile time).
    std::string row_to(uint32_t m, uint32_t o, const std::string &x, const std::string &y, const std::string &z) const
    {
        std::string acc = "vbc<V>(" + F(o) + ")";
        const std::string v[3] = {x, y, z};
        for (int k = 2; k >= 0; --k)
            if (value(m + k) != 0.0f) acc = "vfma(vbc<V>(" + F(m + k) + "), " + v[k] + ", " + acc + ")";
        return acc;
    }
    std::string row_from(uint32_t m, const std::string &x, const std::string &y, const std::string &z) const
    {
        std::string acc;
        const std::string v[3] = {x, y, z};
        for (int k = 2; k >= 0; --k) {
            if (value(m + k) == 0.0f) continue;
            if (acc.empty()) acc = "cc_first_term(" + F(m + k) + ", " + v[k] + ")";
            else acc = "vfma(vbc<V>(" + F(m + k) + "), " + v[k] + ", " + acc + ")";
        }
        return acc.empty() ? std::string("vbc<V>(0.0f)") : acc;
    }
    // statements computing `dst` (a Val) = matrix(m..m+8) * (x, y, z) + o(m+9..m+11)
    std::string transform_to(uint32_t m, const std::string &x, const std::string &y, const std::string &z) const
    {
        return "Val{" + row_to(m, m + 9, x, y, z) + ", " + row_to(m + 3, m + 10, x, y, z) + ", " +
               row_to(m + 6, m + 11, x, y, z) + ", vbc<V>(0.0f)}";
    }
    // from-matrix at m..m+8, scale at m+9, applied to the Val named `in`
    std::string transform_from(uint32_t m, const std::string &in) const
    {
        const std::string x = in + ".x", y = in + ".y", z = in + ".z";
        const std::string w = value(m + 9) == 1.0f ? in + ".w" : "vmul(" + in + ".w, vbc<V>(" + F(m + 9) + "))";
        return "Val{" + row_from(m, x, y, z) + ", " + row_from(m + 3, x, y, z) + ", " + row_from(m + 6, x, y, z) + ", " + w + "}";
    }
    std::string C(uint32_t idx) const  // constant-expression literal (for __constant__ initialisers)
    {
        float f;
        std::memcpy(&f, &code[idx], 4);
        if (f != f) return "__builtin_nanf(\"\")";
        if (f - f != 0.0f) return f > 0 ? "__builtin_huge_valf()" : "-__builtin_huge_valf()";
        char buf[48];
        std::snprintf(buf, sizeof buf, "%af", (double)f);  // C++17 hexadecimal floating literal: exact
        return buf;
    }
};

// experiments: CODECAD_B200_JIT_DEFINES="A=1,B=0" -> "#define A 1\n#define B 0\n" ahead of the headers
std::string extra_defines()
{
    std::string out;
    const char *e = getenv("CODECAD_B200_JIT_DEFINES");
    if (!e) return out;
    std::stringstream ss(e);
    std::string item;
    while (std::getline(ss, item, ',')) {
        size_t k = item.find('=');
        if (k == std::string::npos) out += "#define " + item + " 1\n";
        else out += "#define " + item.substr(0, k) + " " + item.substr(k + 1) + "\n";
    }
    return out;
}

int generate(const cc_decoded &dec, const cc_jit_cfg &cfg, unsigned sink_mask, std::string *src, size_t *smem_bytes,
             std::string *err, cc_columns_meta *columns_meta = nullptr)
{
    const int pts = cfg.pts;
    // debugging aids: stop after N micro-ops (bisecting a mismatch), force scalar lanes
    const char *stop_env = getenv("CODECAD_B200_JIT_STOP");
    const int stop_after = stop_env ? atoi(stop_env) : -1;
    const bool no_pack = getenv("CODECAD_B200_JIT_NOPACK") != nullptr;
    int n_emitted = 0;
    Gen g(dec.microcode);
    const std::vector<uint32_t> &c = dec.microcode;
    std::ostringstream &o = g.body;
    // part culling (DESIGN.md 4.9): the run of micro-ops of part k is wrapped in `if (mask & (1 << k))`,
    // a union of the tree is taken only if both operands keep a part; generated for CC_SINK_PARTS only
    // columns (DESIGN.md 4.10): the micro-ops that cannot see the grid's z (cc_program.cpp analyse_columns) become
    // one functor that runs once per (x, y) column and leaves its results in the column buffer, the rest another
    // that runs per cell and reads them there; a third is the full walk (brick centres, flagged bricks).
    const cc_columns &cols = dec.columns;
    const cc_parts &parts = dec.parts;
    // tile units (hierarchy sinks): the column split if the program has one, the part masks if it has parts
    const int tile_kind = (sink_mask & (1u << CC_SINK_TILES_PYMCUBES)) ? (int)CC_SINK_PYMCUBES
                        : (sink_mask & (1u << CC_SINK_TILES_CLASSIFY)) ? (int)CC_SINK_CLASSIFY
                        : (sink_mask & (1u << CC_SINK_TILES_MASS)) ? (int)CC_SINK_MASS : -1;
    const bool tiles = tile_kind >= 0;
    if (tiles && !cols.enabled && !parts.enabled) {
        *err = "tile units need a program with parts or column-invariant micro-ops";
        return CC_ERR_INVALID_ARGUMENT;
    }
    const bool columns_mode = (sink_mask & (1u << CC_SINK_COLUMNS)) != 0 || (tiles && cols.enabled);
    const bool parts_mode = (sink_mask & (1u << CC_SINK_PARTS)) != 0 || ((columns_mode || tiles) && parts.enabled);
    if (columns_mode && (!cols.enabled || pts != 2 || cfg.threads * pts != CC_BRICK_X * CC_BRICK_Y * CC_BRICK_Z)) {
        *err = "column kernels need a program with column-invariant micro-ops and 512 threads x 2 points";
        return CC_ERR_INVALID_ARGUMENT;
    }
    if (parts_mode && !columns_mode && (!parts.enabled || pts != 2 || cfg.threads * pts != CC_BRICK_X * CC_BRICK_Y * CC_BRICK_Z)) {
        *err = "part culling needs a program with parts and 512 threads x 2 points";
        return CC_ERR_INVALID_ARGUMENT;
    }
    // the columns unit's per-cell body defers its ops' range checks to one vote per warp (DESIGN.md 4.10) when every
    // micro-op in it is pure arithmetic: no address and no loop bound depends on a value, so an op fed an operand out of
    // its fast path's range yields inf or NaN that the fallback throws away, and cannot fault or loop
    const bool column_unit = columns_mode && !tiles;
    bool defer_checks = column_unit;
    auto deferrable = [](uint32_t op) {
        switch (op) {
        case MOP_RETURN: case MOP_NOP: case MOP_LOAD:
        case MOP_T_INIT: case MOP_T_TO: case MOP_T_FROM: case MOP_T_INIT_M: case MOP_T_TO_M: case MOP_T_FROM_M:
        case MOP_RECTANGLE: case MOP_CIRCLE: case MOP_SPHERE:
        case MOP_PRIM_CIRCLE: case MOP_PRIM_RECT: case MOP_PRIM_CIRCLE_M: case MOP_PRIM_RECT_M:
        case MOP_EXTRUSION: case MOP_OFFSET: case MOP_SHELL: case MOP_MIRROR: case MOP_SYM_TO: case MOP_SYM_FROM:
        case MOP_UNION: case MOP_ISECT: case MOP_SUB:
            return true;
        default:
            return false;
        }
    };
    std::ostringstream hoisted;  // parts mode: value variables are declared ahead of the conditional blocks
    std::ostringstream ahead, in_loop, full;  // columns mode: the three bodies
    int full_open = -1, loop_open = -1;       // the part whose `if` is open in each body
    uint32_t n_carried = 0;                   // values in the column buffer
    std::vector<int> carried_interval, carried_l;  // interval / micro-op -> its place there, -1 = none
    auto col_phase = [&](int op) { return columns_mode && (size_t)op < cols.phase.size() ? cols.phase[(size_t)op] : (uint8_t)3; };

    // ---- value intervals: one per slot definition, from the storing micro-op to its last reader.
    // Each interval becomes its own variable (the microcode is straight-line, so this is SSA).
    // Long-lived intervals are kept in shared memory cells instead of registers: two points per
    // thread need 8 registers per live value, and what does not fit the register cap would be
    // spilled to local memory, i.e. through L1/L2 to DRAM.
    struct Interval {
        int def, last_read, cell;
        bool z_only;  // every reader is an extrusion (needs the point's z only)
        bool carried; // columns mode: defined ahead of the z loop only, read inside it (lives through the loop: a register)
    };
    std::vector<Interval> iv;
    std::vector<int> op_def, op_use;  // per micro-op: interval defined / interval read (-1 = none)
    {
        std::vector<int> cur(CC_SLOT_NONE + 1, -1);
        uint32_t q = 0;
        for (int i = 0;; ++i) {
            if (q >= c.size()) {
                *err = "internal: microcode without RETURN";
                return CC_ERR_INVALID_PROGRAM;
            }
            const uint32_t h = c[q], op = CC_HDR_OP(h), src_slot = CC_HDR_SRC(h), dst = CC_HDR_DST(h);
            int use = -1;
            if (src_slot != CC_SLOT_NONE && op != MOP_RETURN) {
                use = cur[src_slot];
                if (use < 0) {
                    *err = "internal: micro-op reads an undefined slot";
                    return CC_ERR_INVALID_PROGRAM;
                }
                iv[use].last_read = i;
                if (op != MOP_EXTRUSION) iv[use].z_only = false;
                if ((col_phase(i) & 2) && !(col_phase(iv[use].def) & 2)) iv[use].carried = true;
            }
            op_use.push_back(use);
            int def = -1;
            if (dst != CC_SLOT_NONE && op != MOP_RETURN) {
                def = (int)iv.size();
                iv.push_back(Interval{i, i, -1, true, false});
                cur[dst] = def;
            }
            op_def.push_back(def);
            if (op == MOP_RETURN) break;
            q += CC_HDR_LEN(h);
        }
    }
    int n_cells = 0;
    {
        // cells: longest intervals first, interval-graph colouring within the budget
        const int min_len = cfg.smem_min_len, max_cells = cfg.smem_max_cells;
        std::vector<int> order;
        for (int k = 0; k < (int)iv.size(); ++k)
            if (max_cells > 0 && iv[k].last_read - iv[k].def >= min_len && !iv[k].carried) order.push_back(k);
        std::sort(order.begin(), order.end(), [&](int a, int b) {
            return iv[a].last_read - iv[a].def > iv[b].last_read - iv[b].def;
        });
        std::vector<std::vector<int>> cell_members;
        for (int k : order) {
            int chosen = -1;
            for (int cidx = 0; cidx < (int)cell_members.size() && chosen < 0; ++cidx) {
                bool clash = false;
                for (int m : cell_members[cidx])
                    if (!(iv[m].last_read <= iv[k].def || iv[k].last_read <= iv[m].def)) clash = true;
                if (!clash) chosen = cidx;
            }
            if (chosen < 0 && (int)cell_members.size() < max_cells) {
                cell_members.emplace_back();
                chosen = (int)cell_members.size() - 1;
            }
            if (chosen >= 0) {
                cell_members[chosen].push_back(k);
                iv[k].cell = chosen;
            }
        }
        n_cells = (int)cell_members.size();
    }
    // experiment: keep the grid coordinates (live through the whole kernel) in one more cell
    const bool coord_smem = getenv("CODECAD_B200_JIT_COORD_SMEM") != nullptr;
    const int coord_cell = n_cells;
    if (coord_smem) ++n_cells;
    const std::string coord_load = !coord_smem ? std::string() :
        "          V px[G], py[G], pz[G]; CC_EACH { Val P_; cc_slot_load_opaque(CC_CELL(" + std::to_string(coord_cell) +
        ", g), P_); px[g] = P_.x; py[g] = P_.y; pz[g] = P_.z; }\n";
    g.n_cells = n_cells;

    // ---- segments: long programs are cut into __noinline__ functions of seg_ops micro-ops each.
    // One 1000-op function (the 500-box scene) takes NVRTC/ptxas 5 minutes; compile time grows
    // faster than linearly with the function size.  Values that cross a segment boundary travel
    // through a State struct (local memory, L1-resident; a few round trips per hundred micro-ops).
    const int n_ops_total = (int)op_def.size();
    int seg_ops = cfg.segment_ops;
    if (seg_ops <= 0 || n_ops_total <= seg_ops + seg_ops / 2) seg_ops = n_ops_total + 1;
    const bool segmented = seg_ops <= n_ops_total;
    if (segmented && (parts_mode || columns_mode)) {
        *err = "part culling and column kernels are not generated for segmented programs";
        return CC_ERR_INVALID_ARGUMENT;
    }
    auto seg_of = [&](int op) { return op / seg_ops; };
    const int n_segs = segmented ? seg_of(n_ops_total - 1) + 1 : 1;
    std::vector<char> crosses(iv.size(), 0);  // register interval read in a later segment than its definition
    if (segmented)
        for (size_t k = 0; k < iv.size(); ++k)
            crosses[k] = iv[k].cell < 0 && iv[k].last_read != iv[k].def && seg_of(iv[k].def) != seg_of(iv[k].last_read);
    const bool out_of_line = segmented && pts <= 2;  // (the table-driven forms take one lane vector)
    std::vector<std::string> seg_text((size_t)n_segs);
    std::vector<std::vector<int>> seg_copy_in((size_t)n_segs);
    if (segmented)
        for (int i = 0; i < n_ops_total; ++i) {
            const int u = op_use[i];
            if (u >= 0 && crosses[u] && seg_of(i) != seg_of(iv[u].def)) {
                std::vector<int> &lst = seg_copy_in[(size_t)seg_of(i)];
                if (std::find(lst.begin(), lst.end(), u) == lst.end()) lst.push_back(u);
            }
        }

    // the lazy gradient of the columns unit's per-cell body (DESIGN.md 4.10).  The sweep runs the body's ops with a
    // distance and a leaf id per cell in place of each distance value (points stay whole), and the replay has one case
    // per leaf: the leaf's value rebuilt from the cell's coordinates and its column record, then the ops that change
    // a gradient on the leaf's one path to the root.  `lazy` stays true while every per-cell op has such a form and
    // every leaf reaches the root along exactly one path.
    bool lazy = column_unit && !coord_smem;
    std::ostringstream sweep, sweep_hoisted;
    int sweep_open = -1;
    std::vector<char> dist_after, dist_iv(iv.size(), 0);  // per micro-op / interval: a distance (else a point)
    struct Path {
        int leaf;
        std::vector<int> chain;  // op index of a transformation_from, ~op index of a subtrahend's negation
    };
    typedef std::vector<Path> Paths;
    Paths l_paths;                   // the leaves the sweep's running distance may hold
    std::vector<Paths> iv_paths(iv.size());
    std::string l_recipe;            // statements that rebuild the running point into L ("" = unknown)
    std::vector<std::string> iv_recipe(iv.size()), op_core((size_t)n_ops_total + 1), leaf_text;
    bool l_dist = false;
    auto new_leaf = [&](const std::string &text) {
        leaf_text.push_back(text);
        return (int)leaf_text.size() - 1;
    };
    auto set_id = [](int leaf) { return "CC_EACH Li[g] = vbc<V>(" + std::to_string(leaf) + ".0f);\n"; };

    uint32_t pc = 0;
    for (int op_index = 0;; ++op_index) {
        if (pc >= c.size()) {
            *err = "internal: microcode without RETURN";
            return CC_ERR_INVALID_PROGRAM;
        }
        if (segmented && op_index > 0 && op_index % seg_ops == 0) {  // cut: what was emitted so far is one segment
            seg_text[(size_t)seg_of(op_index - 1)] = o.str();
            o.str(std::string());
        }
        const uint32_t h = c[pc], op = CC_HDR_OP(h), src_slot = CC_HDR_SRC(h), dst = CC_HDR_DST(h);
        if (columns_mode) o.str(std::string());  // one micro-op at a time: its text goes to one body or both
        std::string split_fused, split_a, split_b, split_sweep;  // a fused primitive cut in two (cc_columns::split_prim)
        o << "        // pc " << pc << "\n";
        const int my_part = (parts_mode && op != MOP_RETURN && (size_t)op_index < parts.part_of_op.size()) ? parts.part_of_op[(size_t)op_index] : -1;
        const bool tree_union = parts_mode && op == MOP_UNION && (size_t)op_index < parts.union_a.size() &&
                                parts.union_a[(size_t)op_index] != 0;
        if (!columns_mode && my_part >= 0 && (op_index == 0 || parts.part_of_op[(size_t)op_index - 1] != my_part))
            o << "        if (mask & " << (1u << my_part) << "u) {  // part " << my_part << "\n";
        const std::string tree_union_open = !tree_union ? std::string() :
            "        if ((mask & " + std::to_string(parts.union_a[(size_t)op_index]) + "u) && (mask & " +
            std::to_string(parts.union_b[(size_t)op_index]) + "u)) {  // both operands keep a part; otherwise the survivor is already in L\n";
        if (!columns_mode) o << tree_union_open;
        std::string B = "?";
        if (op_use[op_index] >= 0) {
            const int u = op_use[op_index];
            const std::string name = "I" + std::to_string(u);
            if (iv[u].cell < 0) {
                B = name + "[g]";
            } else {  // operand lives in a shared-memory cell: fetch what this op needs
                B = "B" + std::to_string(op_index) + "[g]";
                o << "        Val B" << op_index << "[G]; CC_EACH "
                  << (op == MOP_EXTRUSION ? "cc_slot_load_z_opaque(CC_CELL(" : op == MOP_SYM_FROM ? "cc_slot_load_x_opaque(CC_CELL(" : "cc_slot_load_opaque(CC_CELL(")
                  << iv[u].cell << ", g), " << B << (op == MOP_EXTRUSION ? ".z" : op == MOP_SYM_FROM ? ".x" : "") << ");\n";
            }
        }
        if (columns_mode) o << tree_union_open;  // (after the operand fetch: the other branch needs it too)
        const size_t core_at = lazy ? o.str().size() : 0;
        switch (op) {
        case MOP_RETURN: break;
        case MOP_NOP: break;
        case MOP_LOAD: o << "        CC_EACH L[g] = " << B << ";\n"; break;
        case MOP_PRIM_CIRCLE:
        case MOP_PRIM_RECT:
        case MOP_PRIM_CIRCLE_M:
        case MOP_PRIM_RECT_M: {
            // words: 1..12 m,o | 13 a | 14 b | 15 h | 16 d | 17..25 m' | 26 scale  (cc_prim_n, unrolled)
            const bool rect = (op == MOP_PRIM_RECT || op == MOP_PRIM_RECT_M);
            const std::string X = coord_smem ? "px[g]" : "gx[g]", Y = coord_smem ? "py[g]" : "gy[g]",
                              Z = coord_smem ? "pz[g]" : "gz[g]";
            if (out_of_line) {  // large program: call the shared copy with this op's row of the parameter table
                const size_t off = g.n_params;
                for (int i = 1; i <= 27; ++i) g.params << (g.n_params++ ? ", " : "") << g.C(pc + i);
                o << "        {\n" << coord_load << "          CC_EACH L[g] = cc_prim_table<" << (rect ? "true" : "false")
                  << ", V>(cc_par + " << off << ", " << X << ", " << Y << ", " << Z << ");\n        }\n";
                break;
            }
            {
                const std::string to = g.transform_to(pc + 1, X, Y, Z);
                const std::string profile = rect ? "          cc_rectangle_n(" + g.args(pc, 13, 2) + ", L);\n"
                                                 : "          cc_circle_n(" + g.F(pc + 13) + ", L);\n";
                const std::string tail = "          cc_extrusion_n(" + g.F(pc + 15) + ", L, pz_);\n"
                                         "          CC_EACH { L[g].w = vsub(L[g].w, vbc<V>(" + g.F(pc + 16) + ")); const Val t_ = L[g]; L[g] = " +
                                         g.transform_from(pc + 17, "t_") + "; }\n        }\n";
                const std::string fused = "        {\n" + coord_load + "          V pz_[G];\n          CC_EACH { L[g] = " + to +
                                          "; pz_[g] = L[g].z; }\n" + profile + tail;
                o << fused;
                if (columns_mode && (size_t)op_index < cols.split_prim.size() && cols.split_prim[(size_t)op_index]) {
                    // columns: the profile half once per column, extrusion / offset / inverse transform per cell (same calls, same operands)
                    const std::string k = std::to_string(n_carried++);
                    split_fused = fused;
                    split_a = "        {\n          CC_EACH L[g] = " + to + ";\n" + profile + "          CC_EACH cc_col_store(cr, " + k + "u, L[g]);\n        }\n";
                    split_b = "        {\n          V pz_[G];\n          CC_EACH { const Val p_ = " + to + "; pz_[g] = p_.z; L[g] = cc_col_load<V>(cr, " + k +
                              "u); }\n" + tail;
                    const std::string scaled = g.value(pc + 26) == 1.0f ? "w_" : "vmul(w_, vbc<V>(" + g.F(pc + 26) + "))";
                    split_sweep = "        {\n          V pz_[G];\n          CC_EACH { const Val p_ = " + to + "; pz_[g] = p_.z; Lw[g] = cc_col_load<V>(cr, " + k +
                                  "u).w; }\n          cc_extrusion_dist(" + g.F(pc + 15) + ", Lw, pz_, range);\n          CC_EACH { const V w_ = vsub(Lw[g], vbc<V>(" +
                                  g.F(pc + 16) + ")); Lw[g] = " + scaled + "; }\n        }\n";
                }
            }
            break;
        }
        case MOP_RECTANGLE: o << "        cc_rectangle_n(" << g.args(pc, 1, 2) << ", L);\n"; break;
        case MOP_CIRCLE: o << "        cc_circle_n(" << g.F(pc + 1) << ", L);\n"; break;
        case MOP_SPHERE: o << "        cc_sphere_n(" << g.F(pc + 1) << ", L);\n"; break;
        case MOP_REGPOLY: o << "        CC_EACH L[g] = cc_op_regpoly(" << g.args(pc, 1, 5) << ", L[g]);\n"; break;
        case MOP_POLYGON: {
            const uint32_t n = (uint32_t)(*reinterpret_cast<const float *>(&c[pc + 1]));
            const uint32_t off = c[pc + 2];
            const int k = g.n_tables++;
            const uint32_t words = CC_POLY_TABLE_WORDS(n);
            g.consts << "__constant__ float cc_poly_" << k << "[" << words << "] = {";
            for (uint32_t i = 0; i < words; ++i) g.consts << (i ? ", " : "") << g.C(off + i);
            g.consts << "};\n";
            o << "        CC_EACH L[g] = cc_op_polygon_table(cc_poly_" << k << ", " << n << "u, L[g]);\n";
            break;
        }
        case MOP_HALF_SPACE: o << "        CC_EACH L[g] = cc_op_half_space(L[g]);\n"; break;
        case MOP_REV_TO: o << "        CC_EACH L[g] = cc_op_rev_to(L[g]);\n"; break;
        case MOP_TWIST_TO: o << "        CC_EACH L[g] = cc_op_twist_to(" << g.args(pc, 1, 2) << ", L[g]);\n"; break;
        case MOP_T_INIT:
        case MOP_T_INIT_M:
            o << "        {\n" << coord_load << "          CC_EACH L[g] = "
              << g.transform_to(pc + 1, coord_smem ? "px[g]" : "gx[g]", coord_smem ? "py[g]" : "gy[g]", coord_smem ? "pz[g]" : "gz[g]")
              << ";\n        }\n";
            break;
        case MOP_T_TO:
        case MOP_T_TO_M:
            o << "        CC_EACH { const Val t_ = L[g]; L[g] = " << g.transform_to(pc + 1, "t_.x", "t_.y", "t_.z") << "; }\n";
            break;
        case MOP_T_FROM:
        case MOP_T_FROM_M:
            o << "        CC_EACH { const Val t_ = L[g]; L[g] = " << g.transform_from(pc + 1, "t_") << "; }\n";
            break;
        case MOP_MIRROR: o << "        CC_EACH L[g].x = vneg(L[g].x);\n"; break;
        case MOP_SYM_TO: o << "        CC_EACH L[g].x = vabs(L[g].x);\n"; break;
        case MOP_OFFSET: o << "        CC_EACH L[g].w = vsub(L[g].w, vbc<V>(" << g.F(pc + 1) << "));\n"; break;
        case MOP_SHELL: o << "        CC_EACH L[g] = cc_op_shell(" << g.F(pc + 1) << ", L[g]);\n"; break;
        case MOP_REPETITION: o << "        CC_EACH L[g] = cc_op_repetition(" << g.args(pc, 1, 3) << ", L[g]);\n"; break;
        case MOP_CREP_TO: o << "        CC_EACH L[g] = cc_op_crep_to(" << g.args(pc, 1, 2) << ", L[g]);\n"; break;
        case MOP_CREP_FROM:
            o << "        CC_EACH L[g] = cc_op_crep_from(" << g.args(pc, 1, 2) << ", L[g], " << B << ");\n";
            break;
        case MOP_GEAR: o << "        CC_EACH L[g] = cc_op_gear(" << g.args(pc, 1, 5) << ", L[g]);\n"; break;
        case MOP_EXTRUSION:
            o << "        { V cz[G]; CC_EACH cz[g] = " << B << ".z; cc_extrusion_n(" << g.F(pc + 1) << ", L, cz); }\n";
            break;
        case MOP_REV_FROM: o << "        CC_EACH L[g] = cc_revolution_from(L[g], " << B << ");\n"; break;
        case MOP_TWIST_FROM:
            o << "        CC_EACH L[g] = cc_op_twist_from(" << g.args(pc, 1, 5) << ", L[g], " << B << ");\n";
            break;
        case MOP_SYM_FROM: o << "        CC_EACH L[g] = cc_op_sym_from(L[g], " << B << ");\n"; break;
        case MOP_UNION: o << "        CC_EACH L[g] = cc_op_union(L[g], " << B << ");\n"; break;
        case MOP_UNION_R:
            o << "        CC_EACH L[g] = " << (out_of_line ? "cc_rounded_union_fn(" : "cc_rounded_union(") << g.F(pc + 1)
              << ", L[g], " << B << ");\n";
            break;
        case MOP_ISECT: o << "        CC_EACH L[g] = cc_op_isect(L[g], " << B << ");\n"; break;
        case MOP_ISECT_R: o << "        CC_EACH L[g] = cc_op_isect_r(" << g.F(pc + 1) << ", L[g], " << B << ");\n"; break;
        case MOP_SUB: o << "        CC_EACH L[g] = cc_op_sub(L[g], " << B << ");\n"; break;
        case MOP_SUB_R: o << "        CC_EACH L[g] = cc_op_sub_r(" << g.F(pc + 1) << ", L[g], " << B << ");\n"; break;
        default:
            *err = "internal: unknown micro-op " + std::to_string(op);
            return CC_ERR_INVALID_PROGRAM;
        }
        if (lazy) op_core[(size_t)op_index] = o.str().substr(core_at);
        {
            bool d = true;  // what L holds after this op
            switch (op) {
            case MOP_T_INIT: case MOP_T_INIT_M: case MOP_T_TO: case MOP_T_TO_M: case MOP_MIRROR: case MOP_SYM_TO:
            case MOP_REV_TO: case MOP_TWIST_TO: case MOP_CREP_TO: case MOP_REPETITION: d = false; break;
            case MOP_LOAD: d = dist_iv[(size_t)op_use[op_index]] != 0; break;
            case MOP_NOP: case MOP_RETURN: d = dist_after.empty() ? false : dist_after.back() != 0; break;
            default: break;
            }
            dist_after.push_back(d);
            if (op_def[op_index] >= 0) dist_iv[(size_t)op_def[op_index]] = d;
        }
        if (op == MOP_RETURN) break;
        if (stop_after >= 0 && ++n_emitted > stop_after) break;
        if (tree_union && columns_mode)
            // the two operands may have run in different bodies (one ahead of the loop, one inside): L holds
            // the running operand's value whenever that one keeps a part, never the slot operand's
            o << "        } else if (!(mask & " << parts.union_b[(size_t)op_index] << "u)) {\n        CC_EACH L[g] = " << B << ";\n        }\n";
        else if (tree_union) o << "        }\n";
        if (op_def[op_index] >= 0) {
            const int d = op_def[op_index];
            if (iv[d].last_read == iv[d].def) {
                // never read: nothing to keep
            } else if (iv[d].cell < 0) {
                if (parts_mode || columns_mode) {
                    hoisted << "        Val I" << d << "[G];\n";
                    o << "        CC_EACH I" << d << "[g] = L[g];\n";
                } else {
                    o << "        Val I" << d << "[G]; CC_EACH I" << d << "[g] = L[g];\n";
                }
                if (crosses[d]) o << "        CC_EACH st.I" << d << "[g] = L[g];\n";
            } else if (iv[d].z_only) {
                o << "        CC_EACH cc_slot_store_z(CC_CELL(" << iv[d].cell << ", g), L[g].z);\n";
            } else {
                o << "        CC_EACH cc_slot_store(CC_CELL(" << iv[d].cell << ", g), L[g]);\n";
            }
        }
        if (!columns_mode && my_part >= 0 &&
            ((size_t)op_index + 1 >= parts.part_of_op.size() || parts.part_of_op[(size_t)op_index + 1] != my_part))
            o << "          if (pw) pw[" << my_part << "] = L[0].w;  // the part's value (brick centres)\n        }\n";
        if (columns_mode) {
            // every micro-op in its own block, under its part's bit (warp-uniform; neighbours with the same
            // condition fuse); what the loop reads from the column pass travels through the column buffer
            // (one `if` per run of micro-ops with the same condition; -2 = nothing open, -1 = unconditional)
            auto put = [&](std::ostringstream &os, int &open, int part, const std::string &t) {
                if (open != part) {
                    if (open >= 0) os << "        }\n";
                    if (part >= 0) os << "        if (mask & " << (1u << part) << "u) {\n";
                    open = part;
                }
                os << "        {\n" << t << "        }\n";
            };
            const uint8_t ph = col_phase(op_index);
            const std::string text = o.str();
            put(full, full_open, my_part, text);
            std::string text_loop = text;  // (the cut primitive: its per-cell half in place of the fused block, the slot store behind it stays)
            if (!split_fused.empty()) text_loop.replace(text_loop.find(split_fused), split_fused.size(), split_b);
            if (my_part >= 0 && ((size_t)op_index + 1 >= parts.part_of_op.size() || parts.part_of_op[(size_t)op_index + 1] != my_part))
                put(full, full_open, my_part, "        if (pw) pw[" + std::to_string(my_part) + "] = L[0].w;  // the part's value (brick centres)\n");
            if (carried_l.empty()) { carried_l.assign(cols.phase.size(), -1); carried_interval.assign(iv.size(), -1); }
            if (ph & 1) {
                ahead << "        {\n" << (split_a.empty() ? text : split_a);
                if (cols.save_l[(size_t)op_index]) {
                    carried_l[(size_t)op_index] = (int)n_carried;
                    ahead << "        CC_EACH cc_col_store(cr, " << n_carried++ << "u, L[g]);\n";
                }
                const int d = op_def[op_index];
                if (d >= 0 && iv[d].carried && !(ph & 2)) {
                    carried_interval[(size_t)d] = (int)n_carried;
                    ahead << "        CC_EACH cc_col_store(cr, " << n_carried++ << "u, L[g]);\n";
                }
                ahead << "        }\n";
            }
            if (ph & 2) {
                if (!deferrable(op)) defer_checks = false;
                const int from = cols.restore_from[(size_t)op_index];
                if (from >= 0) {
                    const int from_part = (size_t)from < parts.part_of_op.size() && parts_mode ? parts.part_of_op[(size_t)from] : -1;
                    put(in_loop, loop_open, from_part, "        CC_EACH L[g] = cc_col_load<V>(cr, " + std::to_string(carried_l[(size_t)from]) + "u);\n");
                }
                std::string fetch;
                const int u = op_use[op_index];
                if (u >= 0 && iv[u].carried)  // (shadows the register of the same name: this body never defines it)
                    fetch = "        Val I" + std::to_string(u) + "[G]; CC_EACH I" + std::to_string(u) + "[g] = cc_col_load<V>(cr, " +
                            std::to_string(carried_interval[(size_t)u]) + "u);\n";
                put(in_loop, loop_open, my_part, fetch + text_loop);
            }
            if ((ph & 2) && lazy) {
                // the sweep's text of this op, the same control flow as the per-cell body's
                std::ostringstream t;
                const int from = cols.restore_from[(size_t)op_index];
                int restored = -1;  // column value restored as the profile of this op's extrusion
                if (from >= 0) {
                    const std::string k = std::to_string(carried_l[(size_t)from]);
                    const int from_part = (size_t)from < parts.part_of_op.size() && parts_mode ? parts.part_of_op[(size_t)from] : -1;
                    const std::string load = "CC_EACH L[g] = cc_col_load<V>(cr, " + k + "u);\n";
                    l_dist = dist_after[(size_t)from] != 0;
                    if (!l_dist) {
                        l_recipe = load;
                        put(sweep, sweep_open, from_part, "        " + load);
                    } else if (op == MOP_EXTRUSION) {
                        restored = carried_l[(size_t)from];
                        l_paths.clear();
                        put(sweep, sweep_open, from_part, "        CC_EACH Lw[g] = cc_col_load<V>(cr, " + k + "u).w;\n");
                    } else {
                        const int leaf = new_leaf(load);
                        l_paths = Paths{Path{leaf, {}}};
                        put(sweep, sweep_open, from_part, "        CC_EACH Lw[g] = cc_col_load<V>(cr, " + k + "u).w;\n        " + set_id(leaf));
                    }
                }
                // the operand: a distance (Bw, Bi and its paths) or a point (Bp and its recipe)
                const int u = op_use[op_index];
                const bool b_dist = u >= 0 && dist_iv[(size_t)u];
                std::string Bw, Bi, Bp, b_recipe;
                Paths b_paths;
                if (u >= 0) {
                    const std::string us = std::to_string(u), is = std::to_string(op_index);
                    if (iv[u].carried) {
                        const std::string k = std::to_string(carried_interval[(size_t)u]);
                        if (b_dist) {
                            const int leaf = new_leaf("CC_EACH L[g] = cc_col_load<V>(cr, " + k + "u);\n");
                            b_paths = Paths{Path{leaf, {}}};
                            t << "        V Iw" << us << "[G], Ii" << us << "[G]; CC_EACH { Iw" << us << "[g] = cc_col_load<V>(cr, " << k << "u).w; Ii" << us
                              << "[g] = vbc<V>(" << leaf << ".0f); }\n";
                            Bw = "Iw" + us + "[g]", Bi = "Ii" + us + "[g]";
                        } else {
                            t << "        Val I" << us << "[G]; CC_EACH I" << us << "[g] = cc_col_load<V>(cr, " << k << "u);\n";
                            Bp = "I" + us + "[g]";
                            b_recipe = "CC_EACH L[g] = cc_col_load<V>(cr, " + k + "u);\n";
                        }
                    } else if (b_dist) {
                        b_paths = iv_paths[(size_t)u];
                        if (iv[u].cell < 0) {
                            Bw = "Iw" + us + "[g]", Bi = "Ii" + us + "[g]";
                        } else {
                            t << "        V Bw" << is << "[G], Bi" << is << "[G]; CC_EACH cc_slot_load_wi_opaque(CC_CELL(" << iv[u].cell << ", g), Bw" << is
                              << "[g], Bi" << is << "[g]);\n";
                            Bw = "Bw" + is + "[g]", Bi = "Bi" + is + "[g]";
                        }
                    } else {
                        b_recipe = iv_recipe[(size_t)u];
                        if (iv[u].cell < 0) {
                            Bp = "I" + us + "[g]";
                        } else {  // (the per-cell body's fetch)
                            t << "        Val B" << is << "[G]; CC_EACH "
                              << (op == MOP_EXTRUSION ? "cc_slot_load_z_opaque(CC_CELL(" : "cc_slot_load_opaque(CC_CELL(") << iv[u].cell << ", g), B" << is
                              << "[g]" << (op == MOP_EXTRUSION ? ".z" : "") << ");\n";
                            Bp = "B" + is + "[g]";
                        }
                    }
                }
                t << tree_union_open;
                auto leaves_of = [](const Paths &p) { std::vector<int> r; for (const Path &x : p) r.push_back(x.leaf); return r; };
                const std::string from_w = g.value(pc + 10) == 1.0f ? "Lw[g]" : "vmul(Lw[g], vbc<V>(" + g.F(pc + 10) + "))";
                switch (op) {
                case MOP_NOP: break;
                case MOP_LOAD:
                    if (b_dist) {
                        t << "        CC_EACH { Lw[g] = " << Bw << "; Li[g] = " << Bi << "; }\n";
                        l_paths = b_paths;
                    } else {
                        t << "        CC_EACH L[g] = " << Bp << ";\n";
                        l_recipe = b_recipe;
                    }
                    l_dist = b_dist;
                    break;
                case MOP_T_INIT: case MOP_T_INIT_M:
                    t << op_core[(size_t)op_index];
                    l_recipe = op_core[(size_t)op_index];
                    l_dist = false;
                    break;
                case MOP_T_TO: case MOP_T_TO_M: case MOP_MIRROR: case MOP_SYM_TO:
                    if (l_dist || l_recipe.empty()) lazy = false;
                    t << op_core[(size_t)op_index];
                    l_recipe += op_core[(size_t)op_index];
                    break;
                case MOP_SPHERE: {
                    if (l_dist || l_recipe.empty()) lazy = false;
                    const int leaf = new_leaf(l_recipe + op_core[(size_t)op_index]);
                    t << "        cc_sphere_dist(" << g.F(pc + 1) << ", L, Lw, range);\n        " << set_id(leaf);
                    l_paths = Paths{Path{leaf, {}}};
                    l_dist = true;
                    break;
                }
                case MOP_EXTRUSION: {
                    if (restored < 0 || u < 0 || b_dist || b_recipe.empty()) lazy = false;
                    const int leaf = new_leaf("{\n        Val Q[G];\n        {\n" + b_recipe + "        CC_EACH Q[g] = L[g];\n        }\n        CC_EACH L[g] = cc_col_load<V>(cr, " +
                                              std::to_string(restored) + "u);\n        { V cz[G]; CC_EACH cz[g] = Q[g].z; cc_extrusion_n(" + g.F(pc + 1) + ", L, cz); }\n        }\n");
                    t << "        { V cz[G]; CC_EACH cz[g] = " << Bp << ".z; cc_extrusion_dist(" << g.F(pc + 1) << ", Lw, cz, range); }\n        " << set_id(leaf);
                    l_paths = Paths{Path{leaf, {}}};
                    l_dist = true;
                    break;
                }
                case MOP_PRIM_CIRCLE: case MOP_PRIM_RECT: case MOP_PRIM_CIRCLE_M: case MOP_PRIM_RECT_M: {
                    if (split_sweep.empty()) {
                        lazy = false;
                        break;
                    }
                    const int leaf = new_leaf(split_b);
                    t << split_sweep << "        " << set_id(leaf);
                    l_paths = Paths{Path{leaf, {}}};
                    l_dist = true;
                    break;
                }
                case MOP_OFFSET:
                    if (!l_dist) lazy = false;
                    t << "        CC_EACH Lw[g] = vsub(Lw[g], vbc<V>(" << g.F(pc + 1) << "));\n";
                    break;
                case MOP_T_FROM: case MOP_T_FROM_M:
                    if (!l_dist) lazy = false;
                    if (from_w != "Lw[g]") t << "        CC_EACH Lw[g] = " << from_w << ";\n";
                    for (Path &p : l_paths) p.chain.push_back(op_index);
                    break;
                case MOP_UNION: case MOP_ISECT: case MOP_SUB: {
                    if (!l_dist || !b_dist || l_paths.empty() || b_paths.empty()) {
                        lazy = false;
                        break;
                    }
                    for (int a : leaves_of(l_paths))
                        for (int b : leaves_of(b_paths))
                            if (a == b) lazy = false;  // a value reaching the root along two paths
                    const std::string pred = op == MOP_UNION ? "vlt(Lw[g], " + Bw + ")" : op == MOP_ISECT ? "vlt(vneg(Lw[g]), vneg(" + Bw + "))"
                                                                                                         : "vlt(vneg(Lw[g]), " + Bw + ")";
                    const std::string other = op == MOP_SUB ? "vneg(" + Bw + ")" : Bw;
                    t << "        CC_EACH { const auto m_ = " << pred << "; Lw[g] = vsel(m_, Lw[g], " << other << "); Li[g] = vsel(m_, Li[g], " << Bi << "); }\n";
                    for (Path p : b_paths) {
                        if (op == MOP_SUB) p.chain.push_back(~op_index);
                        l_paths.push_back(p);
                    }
                    break;
                }
                default:
                    lazy = false;
                    break;
                }
                if (tree_union) t << "        } else if (!(mask & " << parts.union_b[(size_t)op_index] << "u)) {\n        CC_EACH { Lw[g] = " << Bw << "; Li[g] = " << Bi << "; }\n        }\n";
                const int d = op_def[op_index];
                if (d >= 0 && iv[d].last_read != iv[d].def) {
                    const std::string ds = std::to_string(d);
                    if ((dist_iv[(size_t)d] != 0) != l_dist) lazy = false;
                    if (l_dist) {
                        iv_paths[(size_t)d] = l_paths;
                        if (iv[d].cell < 0) {
                            sweep_hoisted << "        V Iw" << ds << "[G], Ii" << ds << "[G];\n";
                            t << "        CC_EACH { Iw" << ds << "[g] = Lw[g]; Ii" << ds << "[g] = Li[g]; }\n";
                        } else {
                            t << "        CC_EACH cc_slot_store_wi(CC_CELL(" << iv[d].cell << ", g), Lw[g], Li[g]);\n";
                        }
                    } else {
                        iv_recipe[(size_t)d] = l_recipe;
                        if (iv[d].cell < 0) {
                            sweep_hoisted << "        Val I" << ds << "[G];\n";
                            t << "        CC_EACH I" << ds << "[g] = L[g];\n";
                        } else if (iv[d].z_only) {
                            t << "        CC_EACH cc_slot_store_z(CC_CELL(" << iv[d].cell << ", g), L[g].z);\n";
                        } else {
                            t << "        CC_EACH cc_slot_store(CC_CELL(" << iv[d].cell << ", g), L[g]);\n";
                        }
                    }
                }
                put(sweep, sweep_open, my_part, t.str());
            }
        }
        pc += CC_HDR_LEN(h);
    }

    std::ostringstream s;
    s << "// generated by libcodecad_b200 (cc_jit.cpp) from " << dec.info.n_micro_ops << " micro-ops\n"
      << "#define CC_THREADS " << cfg.threads << "\n"
      << (no_pack ? "#define CC_OPT_PACKED 0\n" : "") << extra_defines()
      << (columns_mode ? "#define CC_COL_VALUES " + std::to_string(std::max(1u, n_carried)) + "\n#define CC_COL_AXIS " + std::to_string(cols.axis) + "\n"
                       : std::string())
      << "#include \"cc_ops.cuh\"\n#include \"cc_body.cuh\"\n#include \"cc_render.cuh\"\n"
      << "#define PTS " << pts << "\n"
      << "typedef cc_pts<PTS>::V V;\nconstexpr int G = cc_pts<PTS>::G;\ntypedef cc_val<V> Val;\n"
      << "#define CC_EACH _Pragma(\"unroll\") for (int g = 0; g < G; ++g)\n"
      << "#define CC_CELL(cell, g) (sm + ((cell) * PTS + (g) * cc_lane<V>::N) * CC_THREADS)\n"
      << "#define CC_JIT_SMEM_BYTES " << (size_t)n_cells * pts * cfg.threads * 16 << "\n"
      << g.consts.str();
    if (g.n_params) s << "__constant__ float cc_par[" << g.n_params << "] = {" << g.params.str() << "};\n";
    if (columns_mode) {
        // rows of initial transforms whose z coefficient is rounding residue: equal bits at both ends of the column
        // prove the row constant along it (monotone in z); otherwise the column is evaluated cell by cell in full
        std::ostringstream chk;
        {
            std::vector<uint32_t> pcs;  // micro-op index -> pc
            for (uint32_t q = 0; q < c.size() && CC_HDR_OP(c[q]) != MOP_RETURN; q += CC_HDR_LEN(c[q])) pcs.push_back(q);
            for (uint32_t cr : cols.checked_rows) {
                const uint32_t opi = cr / 4, r = cr % 4;
                if (opi >= pcs.size() || !(col_phase((int)opi) & 1)) continue;
                const int part = parts_mode && opi < parts.part_of_op.size() ? parts.part_of_op[opi] : -1;
                const uint32_t m = pcs[opi] + 1;
                chk << "        " << (part >= 0 ? "if (mask & " + std::to_string(1u << part) + "u) " : std::string())
                    << "CC_EACH ok = ok && cc_same_bits(" << g.row_to(m + 3 * r, m + 9 + r, "gx[g]", "gy[g]", "gz[g]") << ", "
                    << g.row_to(m + 3 * r, m + 9 + r, cols.axis == 0 ? "g_last[g]" : "gx[g]", cols.axis == 1 ? "g_last[g]" : "gy[g]",
                                cols.axis == 2 ? "g_last[g]" : "gz[g]") << ");\n";
            }
        }
        if (full_open >= 0) full << "        }\n";
        if (loop_open >= 0) in_loop << "        }\n";
        const std::string zero_l = "        CC_EACH L[g] = Val{vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f)};\n";
        const std::string sig = "(const V (&gx)[G], const V (&gy)[G], const V (&gz)[G]";
        s << "// the full walk: brick centres, bricks with a column that failed the check\n"
          << "struct SceneFull {\n    float4 *sm;\n    unsigned mask;\n    V *pw;\n"
          << "    __device__ __forceinline__ void operator()" << sig << ", Val (&L)[G]) const\n    {\n" << hoisted.str() << zero_l
          << full.str() << "    }\n};\n"
          << "// once per (x, y) column: what cannot see the grid's z; every part (a column crosses many bricks)\n"
          << "struct SceneAhead {\n    float4 *sm;\n    cc_col_ref cr;\n    static constexpr unsigned mask = 0xffffffffu;\n"
          << "    // may one evaluation stand for the whole column?  (g_last: the coordinate along the columns' axis at its far end)\n"
          << "    __device__ __forceinline__ bool invariant" << sig << ", const V (&g_last)[G]) const\n    {\n"
          << "        bool ok = true;\n" << chk.str() << "        return ok;\n    }\n"
          << "    __device__ __forceinline__ void operator()" << sig << ") const\n    {\n" << hoisted.str() << "        Val L[G];\n" << zero_l
          << ahead.str() << "    }\n};\n";
        auto defer_calls = [](std::string &text) {  // the deferred forms: the same calls with the accumulator as a last argument
            for (const char *f : {"cc_extrusion_n(", "cc_circle_n(", "cc_rectangle_n(", "cc_sphere_n("})
                for (size_t at = text.find(f); at != std::string::npos; at = text.find(f, at + 1)) {
                    const size_t close = text.find(");", at);
                    text.insert(close, ", range");
                }
        };
        std::string loop_text = in_loop.str();
        if (column_unit && defer_checks) defer_calls(loop_text);
        s << "// per cell: the rest, reading the column's values" << (column_unit && defer_checks ? "; the range checks go into `range`" : "") << "\n"
          << "struct SceneEval {\n    float4 *sm;\n    unsigned mask;\n    " << (column_unit ? "cc_brick_col_ref" : "cc_col_ref") << " cr;\n"
          << "    __device__ __forceinline__ void operator()" << sig << ", Val (&L)[G]" << (column_unit ? ", unsigned &range" : "") << ") const\n    {\n"
          << (column_unit ? "        (void)range;\n" : "") << hoisted.str() << zero_l << loop_text;
        if (cols.root_restore >= 0) s << "        CC_EACH L[g] = cc_col_load<V>(cr, " << carried_l[(size_t)cols.root_restore] << "u);\n";
        s << "    }\n};\n";
        lazy = lazy && defer_checks;
        std::ostringstream lazy_text;
        if (lazy) {
            if (sweep_open >= 0) sweep << "        }\n";
            if (cols.root_restore >= 0) {
                const std::string load = "CC_EACH L[g] = cc_col_load<V>(cr, " + std::to_string(carried_l[(size_t)cols.root_restore]) + "u);\n";
                l_dist = dist_after[(size_t)cols.root_restore] != 0;
                const int leaf = new_leaf(load);
                l_paths = Paths{Path{leaf, {}}};
                sweep << "        CC_EACH Lw[g] = cc_col_load<V>(cr, " << carried_l[(size_t)cols.root_restore] << "u).w;\n        " << set_id(leaf);
            }
            // every leaf reaches the root, along one path (a second one would have met the first in a union)
            lazy = l_dist && l_paths.size() == leaf_text.size();
        }
        if (lazy) {
            std::vector<const Path *> path_of(leaf_text.size(), nullptr);
            for (const Path &p : l_paths) path_of[(size_t)p.leaf] = &p;
            std::string cases;
            for (size_t k = 0; k < leaf_text.size(); ++k) {
                cases += "        case " + std::to_string(k) + ": {\n        " + leaf_text[k];
                for (int op_at : path_of[k]->chain)
                    cases += op_at >= 0 ? op_core[(size_t)op_at] : "        CC_EACH L[g] = cc_val_neg(L[g]);  // subtrahend (pc " + std::to_string(~op_at) + ")\n";
                cases += "        break;\n        }\n";
            }
            defer_calls(cases);
            lazy_text << "// the lazy gradient (DESIGN.md 4.10), the sweep: the per-cell body's ops on a distance and a leaf id per cell\n"
              << "struct SceneSweep {\n    float4 *sm;\n    unsigned mask;\n    cc_brick_col_ref cr;\n"
              << "    __device__ __forceinline__ void operator()" << sig << ", V (&Lw)[G], V (&Li)[G], unsigned &range) const\n    {\n"
              << "        Val L[G];  // a point\n" << sweep_hoisted.str() << "        CC_EACH { Lw[g] = vbc<V>(0.f); Li[g] = vbc<V>(-1.f); }\n"
              << sweep.str() << "    }\n};\n"
              << "// the replay: leaf k's value from the cell's coordinates and column record, along its path to the root (out of line:\n"
              << "// one copy for both cells of a thread, and nothing of it hoisted into the sweep)\n"
              << "static __device__ __noinline__ SceneVals cc_replay_leaf(int k, const cc_brick_col_ref cr, const ScenePts p)\n{\n"
              << "    SceneVals r;\n    Val (&L)[G] = r.L;\n    const V (&gx)[G] = p.x, (&gy)[G] = p.y, (&gz)[G] = p.z;\n"
              << "    unsigned range = 0;\n    (void)range;\n    switch (k) {\n" << cases
              << "    default:  // (the body's initial zero)\n"
              << "        CC_EACH L[g] = Val{vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f)};\n        break;\n    }\n    return r;\n}\n"
              << "struct SceneReplay {\n    cc_brick_col_ref cr;\n"
              << "    __device__ __forceinline__ void leaf(int k, " << sig.substr(1) << ", Val (&L)[G]) const\n    {\n"
              << "        ScenePts p;\n        CC_EACH { p.x[g] = gx[g]; p.y[g] = gy[g]; p.z[g] = gz[g]; }\n"
              << "        const SceneVals r = cc_replay_leaf(k, cr, p);\n        CC_EACH L[g] = r.L[g];\n    }\n};\n";
        }
        if (tiles)
            s << "// the hierarchy sinks (blocks x linear tiles): the rest per cell, or the full walk for a tile with a flagged column\n"
              << "struct SceneTile {\n    SceneEval loop;\n    SceneFull full;\n    bool use_full;\n"
              << "    __device__ __forceinline__ void locate(const cc_eval_args &a, unsigned tile, unsigned block, const unsigned (&ix)[PTS],\n"
              << "                                           const unsigned (&iy)[PTS], const unsigned (&iz)[PTS])\n    {\n"
              << "        use_full = cc_col_locate<PTS>(a, block, ix, iy, iz, loop.cr);\n"
              << "        if (a.part_masks) loop.mask = full.mask = a.part_masks[tile];  // (cc_tile_centers_body)\n    }\n"
              << "    __device__ __forceinline__ void operator()" << sig << ", Val (&L)[G]) const\n    {\n"
              << "        if (use_full) full(gx, gy, gz, L);\n        else loop(gx, gy, gz, L);\n    }\n};\n";
        else
            s << "// the full walk of one thread's cells, out of line: cc_jit_columns_full and the brick kernel's fallback share it\n"
              << "struct ScenePts {\n    V x[G], y[G], z[G];\n};\nstruct SceneVals {\n    Val L[G];\n};\n"
              << "static __device__ __noinline__ SceneVals cc_full_walk(float4 *sm, unsigned mask, const ScenePts p)\n{\n"
              << "    SceneVals r;\n    const SceneFull e{sm, mask, nullptr};\n    e(p.x, p.y, p.z, r.L);\n    return r;\n}\n"
              << "struct SceneFullCall {\n    float4 *sm;\n    unsigned mask;\n"
              << "    __device__ __forceinline__ void operator()" << sig << ", Val (&L)[G]) const\n    {\n"
              << "        ScenePts p;\n        CC_EACH { p.x[g] = gx[g]; p.y[g] = gy[g]; p.z[g] = gz[g]; }\n"
              << "        const SceneVals r = cc_full_walk(sm, mask, p);\n        CC_EACH L[g] = r.L[g];\n    }\n};\n"
              << lazy_text.str()
              << "// the brick kernel (cc_kernel_body_brick_columns): the rest per cell, or the full walk for a warp in which a range check failed\n"
              << "struct SceneTile {\n    SceneEval loop;\n"
              << "    static constexpr bool deferred = " << (defer_checks ? "CC_DEFER_CHECKS != 0" : "false") << ";\n"
              << (!lazy ? "    __device__ __forceinline__ void operator()" + sig + ", Val (&L)[G], unsigned &range) const { loop(gx, gy, gz, L, range); }\n" :
                  "    __device__ __forceinline__ void operator()" + sig + ", Val (&L)[G], unsigned &range) const\n    {\n"
                  "#if CC_LAZY_GRADIENT && CC_DEFER_CHECKS\n"
                  "        V w[G], id[G];\n        SceneSweep{loop.sm, loop.mask, loop.cr}(gx, gy, gz, w, id, range);\n"
                  "        if (!__any_sync(0xffffffffu, cc_range_flagged(range)))  // (a warp that flags takes the full walk)\n"
                  "            cc_lazy_replay(SceneReplay{loop.cr}, gx, gy, gz, w, id, L);\n"
                  "#else\n        loop(gx, gy, gz, L, range);\n#endif\n    }\n")
              << "    __device__ __forceinline__ void full" << sig << ", Val (&L)[G]) const { SceneFullCall{loop.sm, loop.mask}(gx, gy, gz, L); }\n};\n";
        if (columns_meta) {
            columns_meta->n_values = n_carried;
            columns_meta->checks = !chk.str().empty();
            columns_meta->axis = cols.axis;
            columns_meta->columns = true;
        }
    } else if (!segmented) {
        s << "struct SceneEval {\n    float4 *sm;  // this thread's column of the value cells\n";
        if (parts_mode) s << "    unsigned mask;  // bit k: part k can matter in this brick\n    V *pw;  // brick-centre pass: receives every part's value\n";
        s << "    __device__ __forceinline__ void operator()(const V (&gx)[G], const V (&gy)[G], const V (&gz)[G],\n"
          << "                                               Val (&L)[G]) const\n    {\n" << hoisted.str();
        if (coord_smem)
            s << "        CC_EACH cc_slot_store(CC_CELL(" << coord_cell << ", g), Val{gx[g], gy[g], gz[g], vbc<V>(0.f)});\n";
        s << "        CC_EACH L[g] = Val{vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f)};\n" << o.str() << "    }\n};\n";
    } else {
        seg_text[(size_t)n_segs - 1] = o.str();
        s << "struct State {\n    Val L[G];\n    V gx[G], gy[G], gz[G];\n";
        for (size_t k = 0; k < iv.size(); ++k)
            if (crosses[k]) s << "    Val I" << k << "[G];\n";
        s << "};\n";
        for (int k = 0; k < n_segs; ++k) {
            s << "static __device__ __noinline__ void cc_seg_" << k << "(float4 *sm, State &st)\n{\n"
              << "        Val L[G]; V gx[G], gy[G], gz[G];\n"
              << "        CC_EACH { L[g] = st.L[g]; gx[g] = st.gx[g]; gy[g] = st.gy[g]; gz[g] = st.gz[g]; }\n";
            for (int u : seg_copy_in[(size_t)k]) s << "        Val I" << u << "[G]; CC_EACH I" << u << "[g] = st.I" << u << "[g];\n";
            s << seg_text[(size_t)k] << "        CC_EACH st.L[g] = L[g];\n}\n";
        }
        s << "struct SceneEval {\n    float4 *sm;\n"
          << "    __device__ __forceinline__ void operator()(const V (&gx)[G], const V (&gy)[G], const V (&gz)[G],\n"
          << "                                               Val (&L)[G]) const\n    {\n        State st;\n";
        if (coord_smem)
            s << "        CC_EACH cc_slot_store(CC_CELL(" << coord_cell << ", g), Val{gx[g], gy[g], gz[g], vbc<V>(0.f)});\n";
        s << "        CC_EACH { st.L[g] = Val{vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f), vbc<V>(0.f)}; st.gx[g] = gx[g]; st.gy[g] = gy[g]; "
             "st.gz[g] = gz[g]; }\n";
        for (int k = 0; k < n_segs; ++k) s << "        cc_seg_" << k << "(sm, st);\n";
        s << "        CC_EACH L[g] = st.L[g];\n    }\n};\n";
    }
    const char *names[4] = {"float4", "pymcubes", "classify", "mass"};
    const char *sinks[4] = {"CC_SINK_FLOAT4", "CC_SINK_PYMCUBES", "CC_SINK_CLASSIFY", "CC_SINK_MASS"};
    // min CTAs per SM: caps the registers so that the wanted number of warps stays resident
    std::string bounds = "CC_THREADS";
    if (cfg.min_blocks > 0) bounds += ", " + std::to_string(cfg.min_blocks);
    for (int k = 0; k < 4; ++k)
        if (sink_mask & (1u << k))
        s << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") cc_jit_" << names[k]
          << "(const cc_eval_args a)\n{\n    extern __shared__ float4 cc_cells[];\n    SceneEval e{cc_cells + threadIdx.x};\n"
          << "    cc_kernel_body<PTS, " << sinks[k] << ">(a, e);\n}\n";
    const std::string head = "(const cc_eval_args a)\n{\n    extern __shared__ float4 cc_cells[];\n";
    const char *tile_names[4][2] = {{"", ""}, {"pymcubes", "CC_SINK_PYMCUBES"}, {"classify", "CC_SINK_CLASSIFY"}, {"mass", "CC_SINK_MASS"}};
    if (parts_mode) {
        s << "__constant__ float cc_part_lipschitz[" << parts.n_parts << "] = {";
        for (uint32_t k = 0; k < parts.n_parts; ++k) {
            const float l = parts.lipschitz[k];
            s << (k ? ", " : "");
            if (l - l != 0.0f || l > 1e30f) s << "1e30f";  // no bound: lip * r dwarfs every distance, the part always stays
            else { char buf[48]; std::snprintf(buf, sizeof buf, "%af", (double)l); s << buf; }
        }
        s << "};\n";
    }
    // the functor of the full walk in this unit: SceneFull with the column split, the one SceneEval without
    const std::string full_eval = columns_mode ? "SceneFull" : "SceneEval";
    if (columns_mode)
        s << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") " << (tiles ? "cc_jit_tile_profiles" : "cc_jit_columns_profiles") << head
          << "    SceneAhead e;\n    e.sm = cc_cells + threadIdx.x;\n"
          << "    cc_column_profiles_body<PTS>(a, e);\n}\n";
    if (columns_mode && !tiles) {
        s << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") cc_jit_columns" << head
          << "    SceneTile e;\n    e.loop.sm = cc_cells + threadIdx.x;  // (the part mask: per brick of the CTA's run)\n"
          << "    cc_kernel_body_brick_columns<PTS>(a, e);\n}\n"
          << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") cc_jit_columns_full" << head
          << "    const unsigned n = *a.brick_count;\n    for (unsigned i = blockIdx.x; i < n; i += gridDim.x) {\n"
          << "        const unsigned b = a.brick_list[i];\n"
          << "        SceneFullCall e{cc_cells + threadIdx.x, a.part_masks ? a.part_masks[b] : 0xffffffffu};\n"
          << "        cc_kernel_body_bricks_at<PTS>(a, e, b);\n    }\n}\n";
        if (parts_mode)
            s << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") cc_jit_columns_centers" << head
              << "    V pw[" << parts.n_parts << "];\n    SceneFull e{cc_cells + threadIdx.x, 0xffffffffu, pw};\n"
              << "    cc_part_centers_body<" << parts.n_parts << ">(a, e, pw, cc_part_lipschitz);\n}\n";
    }
    if (parts_mode && !columns_mode && !tiles)
        // main kernel: one 8 x 8 x 16 brick per CTA, its mask decides which parts run; centre pass: a
        // thread evaluates the centres of two bricks (one packed pair), derives the bricks' masks from
        // the parts' values there and their Lipschitz constants, and writes them for the main kernel
        s << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") cc_jit_parts" << head
          << "    SceneEval e{cc_cells + threadIdx.x, a.part_masks[blockIdx.x], nullptr};\n"
          << "    cc_kernel_body_bricks<PTS>(a, e);\n}\n"
          << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") cc_jit_part_centers" << head
          << "    V pw[" << parts.n_parts << "];\n"
          << "    SceneEval e{cc_cells + threadIdx.x, 0xffffffffu, pw};\n"
          << "    cc_part_centers_body<" << parts.n_parts << ">(a, e, pw, cc_part_lipschitz);\n}\n";
    if (tiles) {
        // the hierarchy sinks (blocks x linear tiles): a mask per tile, the per-cell body of the column split
        const char *const *tn = tile_names[tile_kind == CC_SINK_PYMCUBES ? 1 : tile_kind == CC_SINK_CLASSIFY ? 2 : 3];
        if (parts_mode)
            s << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") cc_jit_tile_centers" << head
              << "    V pw[" << parts.n_parts << "];\n    " << full_eval << " e{cc_cells + threadIdx.x, 0xffffffffu, pw};\n"
              << "    cc_tile_centers_body<" << parts.n_parts << ", PTS>(a, e, pw, cc_part_lipschitz);\n}\n";
        if (columns_mode) {
            s << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") cc_jit_tile_" << tn[0] << head
              << "    SceneTile e;\n    e.loop.sm = e.full.sm = cc_cells + threadIdx.x;\n    e.loop.mask = e.full.mask = 0xffffffffu;\n"
              << "    e.full.pw = nullptr;\n    cc_kernel_body<PTS, " << tn[1] << ">(a, e);\n}\n";
        } else {
            s << "struct ScenePartsTile {\n    SceneEval e;\n"
              << "    __device__ __forceinline__ void locate(const cc_eval_args &a, unsigned tile, unsigned, const unsigned (&)[PTS], const unsigned (&)[PTS],\n"
              << "                                           const unsigned (&)[PTS])\n    {\n        e.mask = a.part_masks[tile];\n    }\n"
              << "    __device__ __forceinline__ void operator()(const V (&gx)[G], const V (&gy)[G], const V (&gz)[G], Val (&L)[G]) const { e(gx, gy, gz, L); }\n};\n"
              << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") cc_jit_tile_" << tn[0] << head
              << "    ScenePartsTile t{SceneEval{cc_cells + threadIdx.x, 0xffffffffu, nullptr}};\n"
              << "    cc_kernel_body<PTS, " << tn[1] << ">(a, t);\n}\n";
        }
    }
    if (sink_mask & (1u << CC_SINK_POINTS))
        s << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") cc_jit_points"
          << "(const cc_eval_args a)\n{\n    extern __shared__ float4 cc_cells[];\n    SceneEval e{cc_cells + threadIdx.x};\n"
          << "    cc_kernel_body<PTS, CC_SINK_FLOAT4, SceneEval, true>(a, e);\n}\n";
    // image renderers (cc_render.cuh): one point per thread, their own argument block
    const char *render_names[2] = {"ray_caster", "bitmap"};
    for (int k = 0; k < 2; ++k)
        if (sink_mask & (1u << (CC_SINK_RAY + k))) {
            if (pts != 1) {
                *err = "internal: the image renderers are generated with one point per thread";
                return CC_ERR_INVALID_ARGUMENT;
            }
            s << "extern \"C\" __global__ void __launch_bounds__(" << bounds << ") cc_jit_" << render_names[k]
              << "(const cc_render_args a)\n{\n    extern __shared__ float4 cc_cells[];\n    SceneEval e{cc_cells + threadIdx.x};\n"
              << "    cc_" << render_names[k] << "_body(a, e);\n}\n";
        }
    *src = s.str();
    if (smem_bytes) *smem_bytes = (size_t)n_cells * pts * cfg.threads * 16;
    return CC_OK;
}

}  // namespace

// Default shape of the specialised kernels, measured on B200 (profiles/r1_jit_variants.md):
// two points per thread as one packed lane pair, 512-thread CTAs (warps that start together stay
// close together in the straight-line code and share instruction-cache lines), registers capped
// at 64 so that two CTAs = 32 warps are resident per SM.  Environment overrides for experiments:
// CODECAD_B200_JIT_PTS / _THREADS / _MINB.
// Share of a program's work spent in ops that run lane by lane (no packed form: data-dependent
// loops and early exits).  Such programs gain nothing from a second point per thread but pay its
// registers.
static bool lane_by_lane_dominated(const cc_decoded &dec)
{
    const std::vector<uint32_t> &c = dec.microcode;
    uint64_t heavy = 0;
    for (uint32_t pc = 0; pc < c.size();) {
        const uint32_t h = c[pc], op = CC_HDR_OP(h);
        if (op == MOP_RETURN) break;
        switch (op) {
        // (polygon2d is no longer in this list: its edge loop is branch-free lane-vector code)
        case MOP_REGPOLY: case MOP_TWIST_FROM: heavy += 60; break;
        case MOP_TWIST_TO: case MOP_CREP_TO: case MOP_CREP_FROM: heavy += 40; break;
        case MOP_REPETITION: heavy += 30; break;
        default: break;
        }
        pc += CC_HDR_LEN(h);
    }
    return heavy * 2 > dec.info.flops_min;
}

cc_jit_cfg cc_jit_default_cfg(const cc_decoded &dec, int pts)
{
    cc_jit_cfg c;
    c.pts = lane_by_lane_dominated(dec) ? 1 : 2;
    c.threads = 512;
    c.min_blocks = 2;
    if (const char *t = getenv("CODECAD_B200_JIT_PTS")) c.pts = atoi(t);
    if (pts == 1 || pts == 2 || pts == 4) c.pts = pts;
    if (c.pts != 1 && c.pts != 2 && c.pts != 4) c.pts = 2;
    if (const char *t = getenv("CODECAD_B200_JIT_THREADS")) {
        int n = atoi(t);
        if (n >= 64 && n <= 1024 && n % 32 == 0) c.threads = n;
    }
    if (const char *t = getenv("CODECAD_B200_JIT_MINB")) c.min_blocks = atoi(t);
    // the ordered-compaction sinks scan PTS * warps-per-CTA counters with one warp (cc_body.cuh)
    while (c.pts * (c.threads / 32) > 32) c.threads /= 2;
    if (c.min_blocks * c.threads > 2048) c.min_blocks = 2048 / c.threads;
    // Shared-memory cells for long-lived values.  Two points per thread need 8 registers per live
    // value; what exceeds the 64-register cap ptxas spills to local memory, and with a 344-byte
    // frame per thread the spill lines do not stay in L2 next to the streaming output: 51.5 GB
    // of DRAM writes for 17.2 GB of results (planetary 1024^3).  Up to six values that live for
    // twelve micro-ops or more go to conflict-free shared-memory cells instead (loads through an
    // opaque asm so that the compiler cannot forward the stored registers and keep them live):
    // frame 168 B, DRAM writes 17.7 GB, kernel time +0.9 % (profiles/r1_jit_variants.md).
    c.smem_max_cells = 0;
    c.smem_min_len = 12;
    if (c.pts >= 2) {
        const int ctas = c.min_blocks > 0 ? c.min_blocks : 1;
        const int fit = (int)((220u * 1024u / ctas - 2048u) / ((size_t)c.pts * c.threads * 16));
        c.smem_max_cells = std::max(0, std::min(fit, 6));
        if (const char *t = getenv("CODECAD_B200_JIT_SMEM_CELLS")) c.smem_max_cells = std::max(0, std::min(fit, atoi(t)));
    }
    if (const char *t = getenv("CODECAD_B200_JIT_SMEM_MIN_LEN")) c.smem_min_len = atoi(t);
    c.segment_ops = 320;  // planetary (267 micro-ops) stays one function; the 500-box scene becomes 4
    if (const char *t = getenv("CODECAD_B200_JIT_SEGMENT_OPS")) c.segment_ops = atoi(t);
    return c;
}

// long programs are compiled as segments (generate()); part culling and the column kernels exist for the others
bool cc_jit_is_segmented(const cc_decoded &dec)
{
    const cc_jit_cfg c = cc_jit_default_cfg(dec, 2);
    const int n = (int)dec.info.n_micro_ops + 1;
    return c.segment_ops > 0 && n > c.segment_ops + c.segment_ops / 2;
}

int cc_jit_nvrtc(const std::string &src, std::vector<char> *cubin, std::string *err)
{
    Nvrtc n;
    {
        std::lock_guard<std::mutex> lk(g_nvrtc_mu);  // dlopen + symbol table are set up once
        if (!load_nvrtc(&n, err)) return CC_ERR_CUDA;
    }
    const char *hdr_names[] = {"cc_device_types.h", "cc_math.cuh", "cc_ops.cuh", "cc_body.cuh", "cc_scan.cuh", "cc_render.cuh"};
    std::string hdr_src[6];
    const std::string dir = source_dir();
    for (int i = 0; i < 6; ++i)
        if (!read_file(dir + hdr_names[i], &hdr_src[i])) {
            *err = "cannot read " + dir + hdr_names[i] + " (needed to specialise kernels)";
            return CC_ERR_INVALID_ARGUMENT;
        }
    const char *hdr_ptrs[6] = {hdr_src[0].c_str(), hdr_src[1].c_str(), hdr_src[2].c_str(), hdr_src[3].c_str(),
                               hdr_src[4].c_str(), hdr_src[5].c_str()};
    nvrtcProgram p = nullptr;
    int e = n.CreateProgram(&p, src.c_str(), "cc_scene.cu", 6, hdr_ptrs, hdr_names);
    if (e) {
        *err = std::string("nvrtcCreateProgram: ") + n.GetErrorString(e);
        return CC_ERR_CUDA;
    }
    const char *opts[] = {"--gpu-architecture=sm_100a", "-fmad=false", "--std=c++17", "-lineinfo"};
    e = n.CompileProgram(p, 4, opts);
    if (e) {
        size_t ls = 0;
        n.GetProgramLogSize(p, &ls);
        std::string log(ls, '\0');
        if (ls) n.GetProgramLog(p, &log[0]);
        if (log.size() > 2000) log.resize(2000);
        *err = std::string("nvrtcCompileProgram: ") + n.GetErrorString(e) + "\n" + log;
        n.DestroyProgram(&p);
        return CC_ERR_CUDA;
    }
    size_t sz = 0;
    n.GetCUBINSize(p, &sz);
    cubin->resize(sz);
    n.GetCUBIN(p, cubin->data());
    n.DestroyProgram(&p);
    if (const char *dump = getenv("CODECAD_B200_JIT_DUMP")) {  // debugging: keep source + cubin
        std::ofstream(std::string(dump) + "/cc_scene.cu") << src;
        std::ofstream(std::string(dump) + "/cc_scene.cubin", std::ios::binary).write(cubin->data(), (std::streamsize)sz);
        int major = 0, minor = 0;
        if (n.Version) n.Version(&major, &minor);
        Dl_info info;
        std::fprintf(stderr, "libcodecad_b200: NVRTC %d.%d from %s\n", major, minor,
                     (dladdr((void *)n.CreateProgram, &info) && info.dli_fname) ? info.dli_fname : "?");
    }
    return CC_OK;
}

// ---- cubin cache: in memory (per process) and on disk ----------------------------------------------
// Key = FNV-1a of the generated source, the op-library headers it includes and the compile options,
// so that editing csrc/*.cuh invalidates old entries.  Disk: $CODECAD_B200_CACHE, else
// ~/.cache/codecad_b200; unusable directories are ignored.
namespace {

typedef std::shared_ptr<const std::vector<char>> Cubin;
std::mutex &g_cache_mu = *new std::mutex;
std::map<uint64_t, Cubin> &g_cache = *new std::map<uint64_t, Cubin>;

// On-disk entries carry a header so that a stale, truncated or foreign file with the right name is
// never loaded as a kernel: magic, the source key, the payload length and its FNV-1a checksum.
struct CacheHeader {
    char magic[8];  // "CCB2CUB1"
    uint64_t key, bytes, checksum;
};
uint64_t fnv1a_bytes(const char *p, size_t n)
{
    uint64_t h = 14695981039346656037ull;
    for (size_t i = 0; i < n; ++i) {
        h ^= (unsigned char)p[i];
        h *= 1099511628211ull;
    }
    return h;
}

uint64_t fnv1a(uint64_t h, const std::string &s)
{
    for (unsigned char ch : s) {
        h ^= ch;
        h *= 1099511628211ull;
    }
    return h;
}

uint64_t source_key(const std::string &src)
{
    uint64_t h = 14695981039346656037ull;
    h = fnv1a(h, src);
    const char *hdr_names[] = {"cc_device_types.h", "cc_math.cuh", "cc_ops.cuh", "cc_body.cuh", "cc_scan.cuh", "cc_render.cuh"};
    const std::string dir = source_dir();
    for (const char *n : hdr_names) {
        std::string t;
        if (read_file(dir + n, &t)) h = fnv1a(h, t);
    }
    Nvrtc n;
    std::string err;
    int major = 0, minor = 0;
    {
        std::lock_guard<std::mutex> lk(g_nvrtc_mu);
        if (load_nvrtc(&n, &err) && n.Version) n.Version(&major, &minor);
    }
    return fnv1a(h, "sm_100a -fmad=false c++17 lineinfo nvrtc " + std::to_string(major) + "." + std::to_string(minor));
}

std::string cache_dir()
{
    if (const char *d = getenv("CODECAD_B200_CACHE")) return *d ? std::string(d) : std::string();
    if (const char *h = getenv("HOME")) return std::string(h) + "/.cache/codecad_b200";
    return std::string();
}

std::string cache_path(uint64_t key)
{
    const std::string d = cache_dir();
    if (d.empty()) return d;
    char name[40];
    std::snprintf(name, sizeof name, "/%016llx.cubin", (unsigned long long)key);
    return d + name;
}

void mkdirs(const std::string &d)
{
    for (size_t i = 1; i <= d.size(); ++i)
        if (i == d.size() || d[i] == '/') mkdir(d.substr(0, i).c_str(), 0700);
}

}  // namespace

// source for ONE sink -> cubin, through the caches.  Host-only work: safe on a background thread.
static int build_cubin(const cc_decoded &dec, const cc_jit_cfg &cfg, int sink, Cubin *out, size_t *smem_bytes,
                       cc_columns_meta *meta, bool *cached, std::string *err)
{
    std::string src;
    int rc = generate(dec, cfg, 1u << sink, &src, smem_bytes, err, meta);
    if (rc) return rc;
    const uint64_t key = source_key(src);
    if (cached) *cached = true;
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        auto it = g_cache.find(key);
        if (it != g_cache.end()) {
            *out = it->second;
            return CC_OK;
        }
    }
    auto bin = std::make_shared<std::vector<char>>();
    const std::string path = cache_path(key);
    std::string blob;
    bool from_disk = false;
    if (!path.empty() && read_file(path, &blob) && blob.size() > sizeof(CacheHeader)) {
        CacheHeader hd;
        std::memcpy(&hd, blob.data(), sizeof hd);
        const size_t n = blob.size() - sizeof hd;
        if (std::memcmp(hd.magic, "CCB2CUB1", 8) == 0 && hd.key == key && hd.bytes == n &&
            hd.checksum == fnv1a_bytes(blob.data() + sizeof hd, n)) {
            bin->assign(blob.begin() + sizeof hd, blob.end());
            from_disk = true;
        }
    }
    if (!from_disk) {
        if (cached) *cached = false;
        rc = cc_jit_nvrtc(src, bin.get(), err);
        if (rc) return rc;
        if (!path.empty()) {
            mkdirs(cache_dir());
            const std::string tmp = path + ".tmp" + std::to_string((long)getpid());
            std::ofstream f(tmp.c_str(), std::ios::binary);
            if (f) {
                CacheHeader hd;
                std::memcpy(hd.magic, "CCB2CUB1", 8);
                hd.key = key;
                hd.bytes = bin->size();
                hd.checksum = fnv1a_bytes(bin->data(), bin->size());
                f.write(reinterpret_cast<const char *>(&hd), sizeof hd);
                f.write(bin->data(), (std::streamsize)bin->size());
                f.close();
                if (!f || rename(tmp.c_str(), path.c_str()) != 0) remove(tmp.c_str());
            }
        }
    }
    std::lock_guard<std::mutex> lk(g_cache_mu);
    g_cache[key] = bin;
    *out = bin;
    return CC_OK;
}

// loaded libraries, shared between programs with the same cubin; unreferenced ones are kept (the most
// recent 16) so that re-creating a program for the same scene does not load its code again
namespace {
struct Loaded {
    cudaLibrary_t lib;
    int refs;
    uint64_t stamp;
    Cubin bin;  // keeps the key (the cubin's address) alive
};
std::map<const void *, Loaded> &g_loaded = *new std::map<const void *, Loaded>;
uint64_t g_loaded_clock = 0;

void release_library(cudaLibrary_t lib)
{
    std::lock_guard<std::mutex> lk(g_cache_mu);
    size_t idle = 0;
    for (auto &kv : g_loaded) {
        if (kv.second.lib == lib && kv.second.refs > 0) kv.second.refs -= 1;
        if (kv.second.refs == 0) ++idle;
    }
    while (idle > 16) {
        auto oldest = g_loaded.end();
        for (auto it = g_loaded.begin(); it != g_loaded.end(); ++it)
            if (it->second.refs == 0 && (oldest == g_loaded.end() || it->second.stamp < oldest->second.stamp)) oldest = it;
        if (oldest == g_loaded.end()) break;
        cudaLibraryUnload(oldest->second.lib);
        g_loaded.erase(oldest);
        --idle;
    }
}
}  // namespace

static int load_cubin(cc_program *prog, int sink, const Cubin &bin, const cc_jit_cfg &cfg, size_t smem_bytes,
                      const cc_columns_meta &meta, std::string *err)
{
    static const char *names[CC_N_SINKS] = {"cc_jit_float4", "cc_jit_pymcubes", "cc_jit_classify", "cc_jit_mass",
                                            "cc_jit_ray_caster", "cc_jit_bitmap", "cc_jit_points", "cc_jit_parts", "cc_jit_columns",
                                            "cc_jit_tile_pymcubes", "cc_jit_tile_classify", "cc_jit_tile_mass"};
    // A cubin is loaded once per process: programs with the same specialised source (the same scene
    // uploaded again) share the loaded library.  Loading costs milliseconds per megabyte of code.
    cudaLibrary_t lib = nullptr;
    cudaError_t ce = cudaSuccess;
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        auto it = g_loaded.find(bin.get());
        if (it != g_loaded.end()) {
            lib = it->second.lib;
            it->second.refs += 1;
            it->second.stamp = ++g_loaded_clock;
        }
    }
    if (!lib) {
        ce = cudaLibraryLoadData(&lib, bin->data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
        if (ce != cudaSuccess) {
            *err = std::string("cudaLibraryLoadData: ") + cudaGetErrorString(ce);
            return CC_ERR_CUDA;
        }
        std::lock_guard<std::mutex> lk(g_cache_mu);
        g_loaded[bin.get()] = Loaded{lib, 1, ++g_loaded_clock, bin};
    }
    cudaKernel_t kern = nullptr;
    ce = cudaLibraryGetKernel(&kern, lib, names[sink]);
    if (ce != cudaSuccess) {
        *err = std::string("cudaLibraryGetKernel: ") + cudaGetErrorString(ce);
        release_library(lib);
        return CC_ERR_CUDA;
    }
    // the unit's companion kernels (cc_program::jit_aux)
    const bool parts = prog->dec.parts.enabled;
    const char *aux[3] = {nullptr, nullptr, nullptr};
    if (sink == CC_SINK_PARTS) {
        aux[CC_AUX_CENTERS] = "cc_jit_part_centers";
    } else if (sink == CC_SINK_COLUMNS) {
        aux[CC_AUX_CENTERS] = parts ? "cc_jit_columns_centers" : nullptr;
        aux[CC_AUX_COLUMNS] = "cc_jit_columns_profiles";
        aux[CC_AUX_FULL] = "cc_jit_columns_full";
    } else if (sink == CC_SINK_TILES_PYMCUBES || sink == CC_SINK_TILES_CLASSIFY || sink == CC_SINK_TILES_MASS) {
        aux[CC_AUX_CENTERS] = parts ? "cc_jit_tile_centers" : nullptr;
        aux[CC_AUX_COLUMNS] = meta.columns ? "cc_jit_tile_profiles" : nullptr;
    }
    cudaKernel_t aux_kernel[3] = {nullptr, nullptr, nullptr};
    for (int k = 0; k < 3; ++k)
        if (aux[k] && (ce = cudaLibraryGetKernel(&aux_kernel[k], lib, aux[k])) != cudaSuccess) {
            *err = std::string("cudaLibraryGetKernel(") + aux[k] + "): " + cudaGetErrorString(ce);
            release_library(lib);
            return CC_ERR_CUDA;
        }
    if (prog->jit_library[sink]) release_library((cudaLibrary_t)prog->jit_library[sink]);
    prog->jit_smem[sink] = smem_bytes;
    for (int d = 0; d < CC_MAX_DEVICES; ++d) prog->jit_attr_done[sink][d] = false;
    prog->jit_library[sink] = (void *)lib;
    prog->jit_kernel[sink] = (void *)kern;
    for (int k = 0; k < 3; ++k) prog->jit_aux[sink][k] = (void *)aux_kernel[k];
    prog->jit_meta[sink] = meta;
    prog->jit_cfg[sink] = cfg;
    prog->jit_cubin_bytes += bin->size();
    return CC_OK;
}

// ---- background compilation ------------------------------------------------------------------------
struct cc_jit_job {
    std::thread th;
    std::atomic<int> done{0};
    int rc = CC_OK;
    Cubin bin;
    cc_jit_cfg cfg;
    size_t smem = 0;
    cc_columns_meta meta;
    std::string err;
    double seconds = 0;
    bool cached = false;
};

static void join_job(cc_program *prog, int sink)
{
    cc_jit_job *j = prog->jit_job[sink];
    if (!j) return;
    if (j->th.joinable()) j->th.join();
    delete j;
    prog->jit_job[sink] = nullptr;
}

// Shape of the specialised image renderers: one ray per thread (the state machine of
// cc_render.cuh is scalar) and small CTAs, because a CTA lives as long as its slowest ray.
cc_jit_cfg cc_jit_render_cfg(const cc_decoded &dec)
{
    cc_jit_cfg c = cc_jit_default_cfg(dec, 1);
    c.pts = 1;
    c.threads = CC_RENDER_THREADS;
    c.min_blocks = 4;
    c.smem_max_cells = 0;
    if (const char *t = getenv("CODECAD_B200_JIT_RENDER_MINB")) c.min_blocks = atoi(t);
    return c;
}

// Shape of the brick kernels (part culling, columns): a CTA of 512 threads x 2 points is one 8 x 8 x 16 brick,
// whatever the program's own preference for the linear-tile kernels is.
static cc_jit_cfg cc_jit_brick_cfg(const cc_decoded &dec)
{
    cc_jit_cfg c = cc_jit_default_cfg(dec, 2);
    if (c.pts != 2 || c.threads != 512) {
        c.pts = 2;
        c.threads = 512;
        c.min_blocks = 2;
        c.smem_max_cells = std::min(c.smem_max_cells, 6);
    }
    return c;
}
static cc_jit_cfg cc_jit_cfg_for(const cc_decoded &dec, int sink, int pts)
{
    if (sink == CC_SINK_RAY || sink == CC_SINK_BITMAP) return cc_jit_render_cfg(dec);
    if (sink == CC_SINK_PARTS || sink == CC_SINK_COLUMNS || sink == CC_SINK_TILES_PYMCUBES || sink == CC_SINK_TILES_CLASSIFY ||
        sink == CC_SINK_TILES_MASS)
        return cc_jit_brick_cfg(dec);
    return cc_jit_default_cfg(dec, pts);
}

// synchronous: build + load every sink of the mask
int cc_jit_compile(cc_program *prog, int pts, unsigned sink_mask, double *seconds, std::string *err)
{
    if ((sink_mask & CC_SINK_MASK_ALL) == 0) sink_mask = 15u;  // default: the four grid sinks
    auto t0 = std::chrono::steady_clock::now();
    for (int k = 0; k < CC_N_SINKS; ++k) {
        if (!(sink_mask & (1u << k))) continue;
        join_job(prog, k);
        const cc_jit_cfg cfg = cc_jit_cfg_for(prog->dec, k, pts);
        Cubin bin;
        size_t smem = 0;
        cc_columns_meta meta;
        int rc = build_cubin(prog->dec, cfg, k, &bin, &smem, &meta, nullptr, err);
        if (rc == CC_OK) rc = load_cubin(prog, k, bin, cfg, smem, meta, err);
        if (rc) return rc;
    }
    prog->use_jit = true;
    if (seconds) *seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return CC_OK;
}

// start compiling `sink` on a background thread (no-op if already compiled, running or failed)
void cc_jit_start(cc_program *prog, int sink)
{
    if (prog->jit_kernel[sink] || prog->jit_job[sink] || prog->jit_failed[sink]) return;
    cc_jit_job *j = new cc_jit_job;
    j->cfg = cc_jit_cfg_for(prog->dec, sink, 0);
    prog->jit_job[sink] = j;
    const cc_decoded *dec = &prog->dec;  // immutable; outlives the thread (destroy joins it)
    j->th = std::thread([j, dec, sink]() {
        auto t0 = std::chrono::steady_clock::now();
        j->rc = build_cubin(*dec, j->cfg, sink, &j->bin, &j->smem, &j->meta, &j->cached, &j->err);
        j->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        j->done.store(1, std::memory_order_release);
    });
}

// If the background job of `sink` has finished (or `wait`), load its kernel.  Returns 1 when the
// specialised kernel is usable, 0 when not (yet), negative on a compile/load error (reported once;
// the interpreter stays in use).
int cc_jit_poll(cc_program *prog, int sink, bool wait, std::string *err)
{
    if (prog->jit_kernel[sink]) return 1;
    cc_jit_job *j = prog->jit_job[sink];
    if (!j) return 0;
    if (!wait && !j->done.load(std::memory_order_acquire)) return 0;
    if (j->th.joinable()) j->th.join();
    int rc = j->rc;
    if (rc == CC_OK) rc = load_cubin(prog, sink, j->bin, j->cfg, j->smem, j->meta, &j->err);
    prog->jit_seconds += j->seconds;
    if (rc != CC_OK) {
        if (err) *err = j->err;
        prog->jit_failed[sink] = true;
    }
    delete j;
    prog->jit_job[sink] = nullptr;
    return rc == CC_OK ? 1 : rc;
}

void cc_jit_release(cc_program *prog)
{
    for (int k = 0; k < CC_N_SINKS; ++k) {
        join_job(prog, k);
        if (prog->jit_library[k]) release_library((cudaLibrary_t)prog->jit_library[k]);
        prog->jit_library[k] = nullptr;
        prog->jit_kernel[k] = nullptr;
    }
    prog->jit_cubin_bytes = 0;
}

// MaxDynamicSharedMemorySize is kept per device: set it the first time a device launches the kernel (the companion
// kernels share the value cells' layout, hence the size)
static int ensure_smem_attr(const cc_program *prog, int sink, int dev_index)
{
    cc_program *p = const_cast<cc_program *>(prog);
    if (p->jit_attr_done[sink][dev_index] || p->jit_smem[sink] == 0) return 0;
    for (void *k : {p->jit_kernel[sink], p->jit_aux[sink][0], p->jit_aux[sink][1], p->jit_aux[sink][2]})
        if (k) {
            cudaError_t ce = cudaFuncSetAttribute((const void *)k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->jit_smem[sink]);
            if (ce != cudaSuccess) return (int)ce;
        }
    p->jit_attr_done[sink][dev_index] = true;
    return 0;
}

int cc_jit_launch(const cc_program *prog, int sink, const cc_eval_args &a, void *stream, int dev_index)
{
    const uint32_t grid = a.n_blocks * a.tiles_per_block;
    if (grid == 0) return 0;
    if (int e = ensure_smem_attr(prog, sink, dev_index)) return e;
    void *args[] = {(void *)&a};
    return (int)cudaLaunchKernel((const void *)prog->jit_kernel[sink], dim3(grid), dim3(prog->jit_cfg[sink].threads),
                                 args, prog->jit_smem[sink], (cudaStream_t)stream);
}

int cc_jit_launch_units(const cc_program *prog, int sink, const cc_eval_args &a, uint64_t n_units, int sm_count, void *stream,
                        int dev_index, int *n_launches, bool centers_only)
{
    *n_launches = 0;
    if (n_units == 0) return 0;
    if (int e = ensure_smem_attr(prog, sink, dev_index)) return e;
    void *const *aux = prog->jit_aux[sink];
    const uint32_t threads = (uint32_t)prog->jit_cfg[sink].threads;
    const size_t smem = prog->jit_smem[sink];
    void *args[] = {(void *)&a};
    auto run = [&](const void *kernel, uint64_t grid) {
        ++*n_launches;
        return cudaLaunchKernel(kernel, dim3((unsigned)grid), dim3(threads), args, smem, (cudaStream_t)stream);
    };
    // the centres and the column pass take two bricks / tiles / columns per thread (one packed pair)
    const uint64_t pair = 2 * threads;
    cudaError_t ce;
    if (aux[CC_AUX_CENTERS] && a.part_masks) {
        if ((ce = run(aux[CC_AUX_CENTERS], (n_units + pair - 1) / pair)) != cudaSuccess || centers_only) return (int)ce;
    }
    if (aux[CC_AUX_COLUMNS] && a.columns) {
        const uint64_t ncol = std::max(1u, a.n_blocks) * columns_along(prog->jit_meta[sink].axis, a.nx, a.ny, a.nz);
        if ((ce = run(aux[CC_AUX_COLUMNS], (ncol + pair - 1) / pair)) != cudaSuccess) return (int)ce;
    }
    // (the column brick kernel: one CTA per run of a.brick_run bricks along the columns' axis)
    const uint64_t grid = sink == CC_SINK_COLUMNS ? brick_runs(prog->jit_meta[sink].axis, a) : n_units;
    if ((ce = run(prog->jit_kernel[sink], grid)) != cudaSuccess) return (int)ce;
    if (aux[CC_AUX_FULL] && a.column_flags) ce = run(aux[CC_AUX_FULL], (uint64_t)std::max(1, 2 * sm_count));
    return (int)ce;
}

int cc_jit_source(const cc_decoded &dec, int pts, unsigned sink_mask, std::string *src, std::string *err)
{
    if ((sink_mask & CC_SINK_MASK_ALL) == 0) sink_mask = 15u;
    if (sink_mask & ((1u << CC_SINK_RAY) | (1u << CC_SINK_BITMAP)))
        return generate(dec, cc_jit_render_cfg(dec), sink_mask, src, nullptr, err);
    if (sink_mask & ((1u << CC_SINK_PARTS) | (1u << CC_SINK_COLUMNS) | (1u << CC_SINK_TILES_PYMCUBES) | (1u << CC_SINK_TILES_CLASSIFY) |
                     (1u << CC_SINK_TILES_MASS)))
        return generate(dec, cc_jit_brick_cfg(dec), sink_mask, src, nullptr, err);
    return generate(dec, cc_jit_default_cfg(dec, pts), sink_mask, src, nullptr, err);
}

int cc_jit_launch_render(const cc_program *prog, int sink, const cc_render_args &a, void *stream, int dev_index)
{
    if (int e = ensure_smem_attr(prog, sink, dev_index)) return e;
    const uint32_t threads = (uint32_t)prog->jit_cfg[sink].threads;
    const uint32_t tiles = ((a.w + 7) / 8) * ((a.h + 3) / 4);  // one warp each (cc_render.cuh)
    const uint32_t grid = (tiles + threads / 32 - 1) / (threads / 32);
    if (grid == 0) return 0;
    void *args[] = {(void *)&a};
    return (int)cudaLaunchKernel((const void *)prog->jit_kernel[sink], dim3(grid), dim3(threads), args,
                                 prog->jit_smem[sink], (cudaStream_t)stream);
}
