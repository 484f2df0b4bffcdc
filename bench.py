#!/usr/bin/env python3
"""Headline benchmark: dense SDF grid_eval throughput (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--grid 1024] [--dump-outputs DIR]

One *step* = one pass of the grid_eval kernel (float4 gradient+distance output, the
reference's INDEX3 layout) over the whole 1024^3 grid of the planetary-gearbox scene
(BASELINE.json configs[3]; 467 node instructions, tests/golden/scenes.npz, compiled by the
reference's own node compiler).  With N ranks the grid is cut into N contiguous x-slabs,
one per GPU, no collective on the data path (strong scaling: total work fixed).

Our arm prints ONE JSON line with
  value     Gpts/s, kernel time only (CUDA events on the library's compute stream, max over
            ranks), program and output resident in HBM;
  e2e       same metric through the public host API codecad_b200.grid_eval(): program words
            uploaded, result delivered into pinned HOST memory (D2H inside the timed region);
  roofline  FP32-issue roofline of the interpreter kernel (SURVEY.md 8(d)): algorithmic
            flop/point (static minimum over data-dependent branches, loader's count) x points /
            kernel time, against SMs x 128 lanes x 2 x max SM clock;
  cpu_baseline  the CPU oracle (oracle/, a restatement of the reference's OpenCL path) on a
            bounded sample of the same grid, all host threads.
`--impl reference` times the reference-side CPU implementation alone: oracle/_ref (the
reference's own .cl sources compiled for the host) when it was built, else the oracle port.
`--dump-outputs DIR` writes a fixed sample of the grid the last timed step computed to DIR
(dump_grid_sample), so that two builds run with the same arguments can be compared point for point.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SCENE = "cfg_planetary"
METRIC = "Gpts/s SDF grid_eval at 1024^3"


def load_scene():
    from scenes import load_scenes
    return load_scenes()[SCENE]


# ---- clocks ------------------------------------------------------------------------------

class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, window=None):
        """window = (t0, t1) host times: only the samples taken inside it count."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, s in self.samples:
            if window is not None and not (window[0] <= t <= window[1]):
                continue
            parts = [p.strip() for p in s.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # keep the samples taken under load (upper half of the observed clocks)
        if sm:
            sm_sorted = sorted(sm)
            med = sm_sorted[len(sm_sorted) // 2]
        else:
            med = None
        return {"sm_mhz": med, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- distributed plumbing ------------------------------------------------------------------

def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # one process per GPU: keep this rank's host buffers on the NUMA node next to its GPU (N = 1
    # keeps every core: the CPU baseline legs run there)
    if world > 1:
        try:
            from codecad_b200 import _lib as _cc
            _cc.bind_host_to_device(local)
        except Exception:  # noqa: BLE001
            pass
    import torch
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local, torch, dist


def barrier(torch, dist):
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(torch, dist, value):
    if dist is None:
        return value
    t = torch.tensor([value], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def min_over_ranks(torch, dist, value):
    if dist is None:
        return value
    t = torch.tensor([value], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return float(t.item())


def gather_over_ranks(torch, dist, value):
    if dist is None:
        return [value]
    t = torch.tensor([value], dtype=torch.float64, device="cuda")
    parts = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, t)
    return [float(p.item()) for p in parts]


def sum_over_ranks(torch, dist, value):
    if dist is None:
        return value
    t = torch.tensor([value], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


# ---- CPU side ---------------------------------------------------------------------------------

def cpu_sample_run(scene, n, target_seconds, steps=1, impl="auto"):
    """Time the CPU path on x-planes of the n^3 grid; returns dict for the JSON line."""
    import oracle
    kind = "port"
    evaluator = oracle.grid_eval
    if impl in ("auto", "reference"):
        try:
            from oracle import ref as oracle_ref
            if oracle_ref.available():
                evaluator = oracle_ref.grid_eval
                kind = "reference"
        except Exception:  # noqa: BLE001 - _ref not built: use the port
            pass
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every core it may run on
    try:
        usable = len(os.sched_getaffinity(0))
    except AttributeError:
        usable = os.cpu_count() or 1
    oracle.set_num_threads(usable)   # same libgomp instance serves oracle/_ref
    threads = oracle.num_threads()
    corner, step = scene.grid(n)
    # probe one plane stripe to size the sample
    t0 = time.perf_counter()
    evaluator(scene.words, corner, step, (1, 64, n), x_offset=n // 2)
    per_point = (time.perf_counter() - t0) / (64 * n)
    planes = int(max(1, min(n, target_seconds / max(per_point * n * n, 1e-9))))
    times = []
    for s in range(steps):
        x0 = (n // 2 + s * planes) % max(1, n - planes + 1)
        t0 = time.perf_counter()
        evaluator(scene.words, corner, step, (planes, n, n), x_offset=x0)
        times.append(time.perf_counter() - t0)
    pts = planes * n * n
    best = min(times)
    mean = sum(times) / len(times)
    return {
        "value": pts / mean / 1e9, "unit": "Gpts/s", "cores": threads, "kind": kind,
        "sample": "%d x-planes (%d x %d x %d = %.3g points) of the %d^3 planetary grid per step, "
                  "%d step(s), mean %.2f s/step (best %.2f s)" % (planes, planes, n, n, pts, n, steps, mean, best),
        "ms_per_step": mean * 1e3, "points_per_step": pts, "sample_fraction": pts / float(n) ** 3,
        "compile_flags": ("g++ -std=c++17 -O2 -mavx2 -mfma -ffp-contract=off -fno-fast-math -fopenmp (oracle/build_ref.py: the "
                          "reference's own .cl sources, one work-item at a time)" if kind == "reference" else
                          "gcc -O3 -mavx2 -mfma -ffp-contract=off -fno-fast-math -fopenmp (oracle/sdf_oracle.c)"),
    }


def run_reference(args):
    """--impl reference: CPU implementation of the path, rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    scene = load_scene()
    # untimed warm-up steps share the sizing probe; keep the whole run within a few minutes
    per_step = max(2.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    for _ in range(min(args.warmup, 1)):
        cpu_sample_run(scene, args.grid, 1.0, 1, "reference")
    r = cpu_sample_run(scene, args.grid, per_step, args.steps, "reference")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "Gpts/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.grid, 1),
        "cpu_baseline": {"value": r["value"], "unit": "Gpts/s", "cores": r["cores"], "kind": r["kind"],
                         "sample": r["sample"], "sample_fraction": r["sample_fraction"], "compile_flags": r["compile_flags"]},
        "e2e": {"value": r["value"], "unit": "Gpts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def mass_properties_leg():
    """Second half of BASELINE.json's metric ("mass_properties ms vs host CL"): configs[2], the
    airfoil scene, volume/centroid/inertia at resolution 0.25 with 64^3 blocks, wall clock
    through the public codecad_b200.mass_properties() call (program cached, result on the host);
    beside it the CPU oracle driving the reference's host algorithm on the box's cores."""
    import codecad_b200
    from codecad_b200.cl_util.buffer import ProgramBuffer
    from oracle import host
    from scenes import load_scenes
    a = load_scenes()["cfg_airfoil"]
    scene = a.compiled()
    res, grid = 0.25, 64
    t0 = time.perf_counter()
    first = codecad_b200.mass_properties(scene, res, grid)          # interpreter tier (compile in background)
    first_ms = (time.perf_counter() - t0) * 1e3
    n_ready, _ = scene.program_buffer().wait_specialized(ProgramBuffer.SINK_MASS)
    times = []
    for _ in range(5):
        t0 = time.perf_counter()
        got = codecad_b200.mass_properties(scene, res, grid)
        times.append((time.perf_counter() - t0) * 1e3)
    t0 = time.perf_counter()
    vol, cen, _ = host.mass_properties(a.words, a.box_a, a.box_b, res, grid)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    import oracle
    return {"workload": "examples/airfoil.py mass_properties(resolution=0.25, grid_size=64)",
            "ms": sorted(times)[len(times) // 2], "ms_best": min(times), "ms_first_call_interpreter_tier": first_ms,
            "tier": "specialised" if n_ready else "interpreter",
            "cpu_ms": cpu_ms, "cpu_cores": oracle.num_threads(), "cpu_kind": "port",
            "volume": got.volume, "volume_rel_diff_vs_cpu": abs(got.volume - vol) / vol,
            "centroid_abs_diff_vs_cpu": max(abs(g - w) for g, w in zip(got.centroid, cen)),
            "first_equals_steady": first.volume == got.volume}


def subdivision_leg():
    """configs[1]: examples/csg_example.py adaptive subdivision at 512^3 effective resolution
    (resolution = 100/512) with 16^3 blocks (SURVEY.md 8(a8): 11 936 leaf blocks); wall clock of
    the public codecad_b200.subdivision() call against the CPU oracle's host algorithm."""
    import codecad_b200
    from codecad_b200.cl_util.buffer import ProgramBuffer
    from oracle import host
    from scenes import load_scenes
    c = load_scenes()["cfg_csg_example"]
    scene = c.compiled()
    res, grid = 100.0 / 512, 16
    codecad_b200.subdivision(scene, res, True, grid)
    n_ready, _ = scene.program_buffer().wait_specialized(ProgramBuffer.SINK_CLASSIFY)
    times, times_list = [], []
    for _ in range(5):
        t0 = time.perf_counter()
        blocks = codecad_b200.subdivision(scene, res, True, grid)[2]   # arrays on the host, tuples built on demand
        times.append((time.perf_counter() - t0) * 1e3)
        as_list = list(blocks)                                         # the reference's list of 5-tuples
        times_list.append((time.perf_counter() - t0) * 1e3)
    t0 = time.perf_counter()
    _, want = host.subdivision(c.words, c.box_a, c.box_b, c.dimension, res, True, grid)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    import oracle
    same = sorted(tuple(b[3]) for b in blocks) == sorted(tuple(b[3]) for b in want)
    return {"workload": "examples/csg_example.py subdivision(resolution=100/512, grid_size=16)",
            "ms": sorted(times)[len(times) // 2], "ms_best": min(times), "leaf_blocks": len(blocks),
            "ms_with_python_tuple_list": sorted(times_list)[len(times_list) // 2],
            "tier": "specialised" if n_ready else "interpreter", "cpu_ms": cpu_ms, "cpu_cores": oracle.num_threads(),
            "cpu_kind": "port", "leaf_blocks_identical_to_cpu": bool(same)}


def mesh_export_leg():
    """configs[1], second half: mesh export of examples/csg_example.py at 512^3 effective resolution
    (feature_size / 2 = 100/512) with the reference's default 128^3 blocks: subdivision + batched
    PyMCubes-layout evaluation + marching cubes on the device (cc_mesh_blocks), triangles delivered
    to host memory.  No CPU number beside it: PyMCubes is not installed and the pure-Python oracle
    of this step is only usable on small blocks (tests/test_gpu_mesh.py)."""
    from codecad_b200 import CompiledScene
    from codecad_b200.cl_util.buffer import ProgramBuffer
    from codecad_b200.rendering import mesh_arrays
    from scenes import load_scenes
    c = load_scenes()["cfg_csg_example"]
    scene = CompiledScene(c.words, 3, c.box_a, c.box_b, 2 * 100.0 / 512, "csg_example@512")
    mesh_arrays(scene, 128)
    scene.program_buffer().wait_specialized(ProgramBuffer.SINK_PYMCUBES | ProgramBuffer.SINK_CLASSIFY)
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        vertices, block, boxes = mesh_arrays(scene, 128)
        times.append((time.perf_counter() - t0) * 1e3)
    return {"workload": "examples/csg_example.py triangular_mesh at 512^3 effective resolution, 128^3 blocks",
            "ms": sorted(times)[1], "ms_best": min(times), "leaf_blocks": len(boxes), "triangles": int(len(vertices)),
            "points_evaluated": int(len(boxes)) * 128 ** 3, "d2h_bytes": int(vertices.nbytes + block.nbytes)}


def ray_caster_leg():
    """SURVEY.md 8(f) rank 4: rendering.image.render_pil_image of the planetary assembly at the
    reference's default 1024x768 (what its tests/test_image.py renders per shape): wall clock of the
    public call (program cached, pixels on the host) and the kernel's own time, beside the CPU
    oracle's restatement of ray_caster.cl on the box's cores; the two images must be identical."""
    import numpy as np
    import oracle
    from oracle import render as oracle_render
    from codecad_b200.rendering import ray_caster
    from scenes import load_scenes
    s = load_scenes()["cfg_planetary"]
    scene = s.compiled()
    size = (1024, 768)
    cam = ray_caster.get_camera_params(scene.bounding_box(), size, None)
    from codecad_b200.cl_util.buffer import ProgramBuffer
    t0 = time.perf_counter()
    ray_caster.render(scene, size=size, *cam)                        # interpreter tier (compile in background)
    first_ms = (time.perf_counter() - t0) * 1e3
    n_ready, _ = scene.program_buffer().wait_specialized(ProgramBuffer.SINK_RAY)
    times, stats = [], {}
    for _ in range(5):
        t0 = time.perf_counter()
        got = ray_caster.render(scene, size=size, stats=stats, *cam)
        times.append((time.perf_counter() - t0) * 1e3)
    t0 = time.perf_counter()
    want = oracle_render.ray_cast(s.words, s.box_a, s.box_b, size)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    return {"workload": "examples/planetary.py render_image 1024x768 (ray caster: primary + shadow rays, AO, floor)",
            "ms": sorted(times)[len(times) // 2], "ms_best": min(times), "kernel_ms": stats["ms"],
            "evaluations": stats["evaluations"], "evaluations_per_pixel": stats["evaluations"] / (size[0] * size[1]),
            "geval_per_s": stats["evaluations"] / stats["ms"] / 1e6, "tier": "specialised" if n_ready else "interpreter",
            "ms_first_call_interpreter_tier": first_ms,
            "cpu_ms": cpu_ms, "cpu_cores": oracle.num_threads(), "cpu_kind": "port",
            "image_identical_to_cpu": bool(np.array_equal(got, want))}


def polygon_leg():
    """SURVEY.md 8(f) rank 4: rendering.polygon2d.polygon of the involute gear at 1/16 of its feature
    size with 32x32 boxes (hundreds of boxes, ~10 k outline vertices): device part in two launches,
    beside the CPU oracle (per-box grid_eval + process_polygon + the same chain following)."""
    import oracle
    from oracle import host
    from codecad_b200 import CompiledScene
    from codecad_b200.rendering import polygon2d
    from scenes import load_scenes
    s = load_scenes()["dsdf2d_gear"]
    fs = s.feature_size / 16
    scene = CompiledScene(s.words, 2, s.box_a, s.box_b, fs, "gear@1/16")
    list(polygon2d.polygon(scene, 32))
    times = []
    for _ in range(5):
        t0 = time.perf_counter()
        got = list(polygon2d.polygon(scene, 32))
        times.append((time.perf_counter() - t0) * 1e3)
    t0 = time.perf_counter()
    want = host.polygon(s.words, s.box_a, s.box_b, fs, 32)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    canon = lambda cs: sorted(tuple(c[c.index(min(c)):] + c[:c.index(min(c))]) for c in ([tuple(v) for v in c] for c in cs))
    return {"workload": "tests/data.py gear: polygon() at feature_size/16, 32x32 boxes",
            "ms": sorted(times)[len(times) // 2], "ms_best": min(times), "outlines": len(got),
            "vertices": sum(len(c) for c in got), "cpu_ms": cpu_ms, "cpu_cores": oracle.num_threads(), "cpu_kind": "port",
            "outlines_identical_to_cpu": canon(got) == canon(want)}


def _timed_events(L, _lib, fn, steps):
    e0, e1 = ctypes.c_void_p(), ctypes.c_void_p()
    _lib.check(L.cc_event_record(ctypes.byref(e0)))
    for _ in range(steps):
        fn()
    _lib.check(L.cc_event_record(ctypes.byref(e1)))
    _lib.check(L.cc_event_wait(e1))
    ms = ctypes.c_float()
    _lib.check(L.cc_event_elapsed_ms(e0, e1, ctypes.byref(ms)))
    L.cc_event_destroy(e0)
    L.cc_event_destroy(e1)
    return ms.value


def config_grid_leg(name, label, n, slab_planes, rank, world, torch, dist, info, sm_max_mhz, hbm_peak, steps, out_buffer):
    """Dense grid_eval of one BASELINE.json scene on an n^3 grid cut into x-slabs (one per rank):
    kernel time by CUDA events, max over ranks; FP32 and HBM-store roofline fractions of the launch.
    slab_planes: x-planes per rank (None = n / world)."""
    import importlib
    from codecad_b200 import _lib
    from codecad_b200.cl_util.buffer import ProgramBuffer
    from scenes import load_scenes
    ge = importlib.import_module("codecad_b200.grid_eval")
    L = _lib.lib()
    scene = load_scenes()[name]
    corner, step = scene.grid(n)
    if slab_planes is None:
        x0, x1 = ge.slab_range(n, rank, world)
    else:
        x0, x1 = rank * slab_planes, (rank + 1) * slab_planes
    nx = x1 - x0
    prog = ProgramBuffer(scene.words)
    pinfo = prog.info
    forest = int(pinfo.n_forest_leaves) > 0      # dense grids of union forests use the culling kernel: nothing to compile
    n_ready, spec_s = (0, 0.0) if forest else prog.wait_specialized(ProgramBuffer.SINK_FLOAT4)
    c3 = _lib.f3(corner)
    assert nx * n * n * 16 <= out_buffer.size

    def step_fn():
        _lib.check(L.cc_grid_eval(prog.handle, c3, float(step), nx, n, n, x0, 0, out_buffer.device_ptr, None))

    for _ in range(2):
        step_fn()
    _lib.check(L.cc_synchronize())
    barrier(torch, dist)
    ms = max_over_ranks(torch, dist, _timed_events(L, _lib, step_fn, steps)) / steps
    barrier(torch, dist)
    tier = "forest (per-tile exact culling, csrc/cc_forest.cu)" if forest else ("specialised" if n_ready else "interpreter")
    if (n_ready and not forest and int(pinfo.column_invariant_percent) > 0 and os.environ.get("CODECAD_B200_COLUMNS", "1") != "0"
            and (nx if int(pinfo.column_axis) == 0 else n) >= 8):
        tier = ("specialised, column kernels (%d %% of the arithmetic once per %s-column, csrc/cc_body.cuh)"
                % (int(pinfo.column_invariant_percent), "xyz"[int(pinfo.column_axis)]))
    prog.release()
    pts_rank = float(nx) * n * n
    pts_all = pts_rank * world
    peak = info.sm_count * 128 * 2 * sm_max_mhz * 1e6 / 1e12
    tflops = pts_rank * int(pinfo.flops_min) / (ms * 1e-3) / 1e12
    gbs = pts_rank * 16 / (ms * 1e-3) / 1e9
    f_exec = load_executed_flops().get(name)
    roof = {"fp32_tflops": tflops, "fp32_frac": tflops / peak, "hbm_gbs": gbs, "hbm_frac": gbs / hbm_peak,
            "bound": "fp32" if tflops / peak >= gbs / hbm_peak else "hbm"}
    if forest:
        # the reference's flop count no longer describes the work: most primitives are skipped (exactly)
        roof.update({"bound": "hbm", "fp32_tflops_reference_formulation": tflops, "fp32_frac_reference_formulation": tflops / peak,
                     "note": "algorithmic flops are those of evaluating every primitive at every point, as the reference "
                             "does; the kernel proves per 16^3 tile which primitives cannot change a bit and skips them, so the "
                             "bound that remains is the 16 B/point store"})
        del roof["fp32_tflops"], roof["fp32_frac"]
    return {"workload": label, "scene": name, "grid": [nx * world, n, n], "x_planes_per_rank": nx,
            "value": pts_all / (ms * 1e-3) / 1e9, "unit": "Gpts/s", "ms_per_step": ms, "steps": steps,
            "tier": tier, "specialize_s": spec_s, "micro_ops": int(pinfo.n_micro_ops),
            "flop_per_point": int(pinfo.flops_min), "flop_per_point_executed": f_exec,
            "fp32_frac_executed_branch": (None if f_exec is None or forest else pts_rank * f_exec / (ms * 1e-3) / 1e12 / peak),
            "roofline": roof}


def sharded_hierarchy_legs(rank, world, torch, dist):
    """SURVEY.md 8(e) in front of the driver: mass_properties (configs[2], airfoil, resolution 0.25,
    64^3 blocks) and subdivision (configs[1], csg_example at 100/512 with 16^3 blocks) sharded over
    the ranks.  The hits of the level that feeds the most expensive level are dealt round-robin; the
    only data that crosses NVLink is the 40-int64 exact accumulator of the ten integrals (one NCCL
    all-reduce).  Every rank then also computes the UNSHARDED result on its own GPU: the sharded
    one must be bit-identical."""
    import importlib
    import codecad_b200
    from codecad_b200.cl_util.buffer import ProgramBuffer
    from scenes import load_scenes
    mpm = importlib.import_module("codecad_b200.mass_properties")
    sub = importlib.import_module("codecad_b200.subdivision")
    S = load_scenes()
    out = {}

    # ---- mass_properties ----
    a = S["cfg_airfoil"]
    scene = a.compiled()
    res, grid = 0.25, 64
    st = {}
    codecad_b200.mass_properties(scene, res, grid, group=True if dist else None)
    scene.program_buffer().wait_specialized(ProgramBuffer.SINK_MASS)
    codecad_b200.mass_properties(scene, res, grid, group=True if dist else None)
    times = []
    for _ in range(5):
        barrier(torch, dist)
        t0 = time.perf_counter()
        got = codecad_b200.mass_properties(scene, res, grid, group=True if dist else None, stats=st)
        times.append(max_over_ranks(torch, dist, (time.perf_counter() - t0) * 1e3))
    # the all-reduce alone (40 int64 on the GPU, the same call the leg makes)
    ar_us = None
    if dist:
        limbs = np.arange(40, dtype=np.int64)
        mpm.allreduce_limbs(limbs)
        barrier(torch, dist)
        t0 = time.perf_counter()
        for _ in range(20):
            mpm.allreduce_limbs(limbs)
        ar_us = max_over_ranks(torch, dist, (time.perf_counter() - t0) / 20 * 1e6)
    whole = codecad_b200.mass_properties(scene, res, grid)          # unsharded, this rank's GPU
    same = (got.volume == whole.volume and tuple(got.centroid) == tuple(whole.centroid)
            and np.array_equal(got.inertia_tensor, whole.inertia_tensor))
    cells = gather_over_ranks(torch, dist, float(st["cells"]))
    dealt = gather_over_ranks(torch, dist, float(st["dealt_blocks"]))
    out["mass_properties"] = {
        "workload": "examples/airfoil.py mass_properties(resolution=0.25, grid_size=64), sharded over %d rank(s)" % world,
        "ms": sorted(times)[len(times) // 2], "ms_best": min(times), "nccl_allreduce_us": ar_us,
        "allreduce_bytes": 320 if dist else 0,
        "cells_per_rank": [int(c) for c in cells], "dealt_blocks_per_rank": [int(d) for d in dealt],
        "imbalance_max_over_mean": max(cells) / (sum(cells) / len(cells)),
        "volume": got.volume, "identical_to_unsharded": bool(min_over_ranks(torch, dist, 1.0 if same else 0.0) == 1.0)}

    # ---- subdivision ----
    c = S["cfg_csg_example"]
    scene = c.compiled()
    res, grid = 100.0 / 512, 16
    codecad_b200.subdivision(scene, res, True, grid, rank=rank, world=world)
    scene.program_buffer().wait_specialized(ProgramBuffer.SINK_CLASSIFY)
    times = []
    for _ in range(5):
        barrier(torch, dist)
        t0 = time.perf_counter()
        mine = codecad_b200.subdivision(scene, res, True, grid, rank=rank, world=world)[2]
        times.append(max_over_ranks(torch, dist, (time.perf_counter() - t0) * 1e3))
    whole = codecad_b200.subdivision(scene, res, True, grid)[2]
    counts = gather_over_ranks(torch, dist, float(len(mine)))
    # union over the ranks, put back into the order one GPU lists the blocks
    if dist:
        cap = int(max(counts))
        pad = np.full((cap, 3), -1, dtype=np.int64)
        pad[:len(mine)] = mine.int_corners
        t = torch.from_numpy(pad).cuda()
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        union = np.concatenate([p.cpu().numpy()[:int(n)] for p, n in zip(parts, counts)])
    else:
        union = mine.int_corners
    from codecad_b200.geometry import BoundingBox, as_vector
    box = BoundingBox(as_vector(c.box_a), as_vector(c.box_b)).expanded_additive(res / 2)
    plan = sub.calculate_block_sizes(box, 3, res, grid, True)
    merged = sub.sort_leaf_corners(union, plan)
    same = np.array_equal(merged, whole.int_corners)
    out["subdivision"] = {
        "workload": "examples/csg_example.py subdivision(resolution=100/512, grid_size=16), sharded over %d rank(s)" % world,
        "ms": sorted(times)[len(times) // 2], "ms_best": min(times), "leaf_blocks": int(len(merged)),
        "leaf_blocks_per_rank": [int(n) for n in counts],
        "imbalance_max_over_mean": max(counts) / max(1e-9, sum(counts) / len(counts)),
        "identical_to_unsharded": bool(min_over_ranks(torch, dist, 1.0 if same else 0.0) == 1.0)}
    return out


def d2h_probe(L, _lib, device_ptr, host_array, nbytes, torch, dist):
    """Bare cudaMemcpyAsync of the rank's result slab into its pinned host buffer, all ranks at once:
    what the PCIe / host-memory path delivers without any kernel in the way (attributes the e2e leg)."""
    _lib.check(L.cc_memcpy_d2h_async(host_array.ctypes.data, device_ptr, nbytes, None))
    _lib.check(L.cc_synchronize())
    barrier(torch, dist)
    t0 = time.perf_counter()
    _lib.check(L.cc_memcpy_d2h_async(host_array.ctypes.data, device_ptr, nbytes, None))
    _lib.check(L.cc_synchronize())
    dt = time.perf_counter() - t0
    barrier(torch, dist)
    return nbytes / dt / 1e9, nbytes / max_over_ranks(torch, dist, dt) / 1e9


DUMP_POINTS = 1 << 20   # 16 MB of float4 values + 24 MB of their grid indices


class _CudaArray:
    """A device allocation of the library seen through the CUDA array interface: torch.as_tensor() wraps it without a
    copy (the library allocates with the runtime API, in the primary context torch uses too)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (int(ptr), False),
                                         "strides": None, "version": 2}


def dump_grid_sample(out_dir, L, _lib, out_buffer, x0, x1, n, rank, torch, dist):
    """--dump-outputs: the float4 values (gradient x, y, z, distance) the last step left in the output grid, at a
    fixed sample of its points: all of them when the n^3 grid has at most DUMP_POINTS, else DUMP_POINTS flat indices
    drawn with seed 0 (sorted, duplicates dropped).  Writes grid_eval.npy, float32 [M][4], and grid_eval_index.npy,
    float64 [M][3], the x, y, z grid indices of those points.  Each rank gathers on its GPU the sample points of its
    slab [x0, x1) (out_buffer holds plane x0 first); rank 0 writes the files."""
    total = n ** 3
    if total <= DUMP_POINTS:
        flat = np.arange(total, dtype=np.int64)
    else:
        flat = np.unique(np.random.default_rng(0).integers(0, total, DUMP_POINTS, dtype=np.int64))
    lo, hi = x0 * n * n, x1 * n * n
    mine = (flat >= lo) & (flat < hi)
    _lib.check(L.cc_synchronize())
    slab = torch.as_tensor(_CudaArray(out_buffer.device_ptr.value, ((x1 - x0) * n * n, 4)), device="cuda")
    values = torch.zeros((len(flat), 4), dtype=torch.float32, device="cuda")
    values[torch.from_numpy(mine).cuda()] = slab[torch.from_numpy(flat[mine] - lo).cuda()]
    if dist is not None:
        # each point was filled by the one rank whose slab holds it and is zero elsewhere: an integer sum of the bits
        # over the ranks is that rank's value
        dist.all_reduce(values.view(torch.int32))
    values = values.cpu().numpy()
    if rank == 0:
        xs, yz = np.divmod(flat, n * n)
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "grid_eval.npy"), values)
        np.save(os.path.join(out_dir, "grid_eval_index.npy"), np.stack([xs, yz // n, yz % n], axis=1).astype(np.float64))


def single_process_leg(n_devices):
    """One process, n GPUs (cc_init_devices): the unmodified module calls — the reference's user is a
    single Python script — fan out inside the library.  Prints one JSON object."""
    import importlib
    import codecad_b200
    from codecad_b200 import _lib
    from codecad_b200.cl_util.buffer import ProgramBuffer, _Pinned
    from codecad_b200.geometry import FLOAT4
    from scenes import load_scenes
    S = load_scenes()
    _lib.init(0)
    a = S["cfg_airfoil"].compiled()
    res, grid = 0.25, 64
    codecad_b200.mass_properties(a, res, grid)
    a.program_buffer().wait_specialized(ProgramBuffer.SINK_MASS)
    one = codecad_b200.mass_properties(a, res, grid)
    t1 = []
    for _ in range(5):
        t0 = time.perf_counter()
        codecad_b200.mass_properties(a, res, grid)
        t1.append((time.perf_counter() - t0) * 1e3)
    c = S["cfg_csg_example"].compiled()
    one_sub = codecad_b200.subdivision(c, 100.0 / 512, True, 16)[2]
    # dense grid into host memory: 512 x-planes of the 1024^3 planetary grid
    p = S["cfg_planetary"]
    corner, step = p.grid(1024)
    planes = 256
    pin = _Pinned(planes * 1024 * 1024 * 16)
    host = pin.array(FLOAT4, (planes, 1024, 1024))
    pc = p.compiled()
    ge = importlib.import_module("codecad_b200.grid_eval")
    ge.grid_eval(pc, corner, step, (planes, 1024, 1024), out=host)
    pc.program_buffer().wait_specialized(ProgramBuffer.SINK_FLOAT4)
    t0 = time.perf_counter()
    ge.grid_eval(pc, corner, step, (planes, 1024, 1024), out=host)
    g1 = time.perf_counter() - t0
    check1 = host[::37, ::129, ::257].copy()

    _lib.init_devices(list(range(n_devices)))
    st = {}
    codecad_b200.mass_properties(a, res, grid)
    alln = codecad_b200.mass_properties(a, res, grid, stats=st)
    tn = []
    for _ in range(5):
        t0 = time.perf_counter()
        codecad_b200.mass_properties(a, res, grid)
        tn.append((time.perf_counter() - t0) * 1e3)
    all_sub = codecad_b200.subdivision(c, 100.0 / 512, True, 16)[2]
    ge.grid_eval(pc, corner, step, (planes, 1024, 1024), out=host)
    t0 = time.perf_counter()
    ge.grid_eval(pc, corner, step, (planes, 1024, 1024), out=host)
    gn = time.perf_counter() - t0
    same_grid = bool(np.array_equal(host[::37, ::129, ::257], check1))
    same_mp = (alln.volume == one.volume and tuple(alln.centroid) == tuple(one.centroid)
               and np.array_equal(alln.inertia_tensor, one.inertia_tensor))
    pts = planes * 1024.0 * 1024.0
    print(json.dumps({
        "devices": _lib.active_devices(),
        "mass_properties": {"ms_1gpu": sorted(t1)[2], "ms": sorted(tn)[2], "identical_to_1gpu": bool(same_mp),
                            "cells_busiest_device": st.get("cells_busiest_device"),
                            "cells_idlest_device": st.get("cells_idlest_device")},
        "subdivision": {"leaf_blocks": len(all_sub),
                        "identical_to_1gpu": bool(np.array_equal(all_sub.int_corners, one_sub.int_corners))},
        "grid_eval_to_host": {"grid": [planes, 1024, 1024], "gpts_1gpu": pts / g1 / 1e9, "gpts": pts / gn / 1e9,
                              "identical_to_1gpu": same_grid},
    }))
    return 0


def load_executed_flops():
    """scene -> executed-branch algorithmic flop/point (profiles/executed_flops.json)."""
    try:
        data = json.load(open(os.path.join(ROOT, "profiles", "executed_flops.json")))["scenes"]
        return {k: float(v["flop_per_point_executed"]) for k, v in data.items()}
    except Exception:  # noqa: BLE001
        return {}


def load_issued_flops(tier, n):
    """FP32 operations the kernel actually ISSUED per point (FFMA = 2), from one ncu capture of this kernel at
    this grid size (profiles/bench_issued.json; smsp__sass_thread_inst_executed_op_{ffma,fmul,fadd}_pred_on):
    the kernel's own cheaper formulation (matrices instead of quaternions, zero coefficients dropped),
    hence less than the algorithmic count.  Replayed, not measured in this run."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "bench_issued.json"))).get("%s_%d" % (tier, n))
    except Exception:  # noqa: BLE001
        return None


def workload_config(n, world):
    return {
        "workload": "examples/planetary.py Planetary(11,60,13,41,18,53).make_assembly().shape(): "
                    "dense grid_eval %d^3, float4 (gradient, distance) per point" % n,
        "scene": SCENE, "grid": [n, n, n], "node_instructions": 467,
        "sharding": "x-slabs, %d rank(s), no data-path collective" % world,
        "cache": "output %.1f GB per step streams through the 126 MB L2, no reuse between steps; "
                 "the only input is the %d-word program" % (n ** 3 * 16 / 1e9, 1424),
    }


# ---- our arm ------------------------------------------------------------------------------------

def _stdout_to_stderr():
    """Everything libraries print to stdout (NCCL's version banner under torchrun, ...) goes to
    stderr; the one JSON line is written to the returned descriptor, the original stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return real


def _emit(fd, line):
    os.write(fd, (json.dumps(line) + "\n").encode())


def run_ours(args):
    out_fd = _stdout_to_stderr()
    rank, world, local, torch, dist = dist_setup(args.gpus)
    import importlib
    from codecad_b200 import _lib
    ge = importlib.import_module("codecad_b200.grid_eval")  # (the package re-exports a function of that name)
    from codecad_b200.cl_util import Buffer
    from codecad_b200.cl_util.buffer import ProgramBuffer, _Pinned
    from codecad_b200.geometry import FLOAT4

    L = _lib.init(local)
    info = _lib.device_info()
    scene = load_scene()
    n = args.grid
    corner, step = scene.grid(n)
    x0, x1 = ge.slab_range(n, rank, world)
    nx = x1 - x0
    my_points = nx * n * n

    prog = ProgramBuffer(scene.words)
    pinfo = prog.info
    c3 = _lib.f3(corner)
    # Tiered execution is the library default: the interpreter serves launches while the
    # scene-specialised kernel compiles in the background.  The headline is measured in steady
    # state, i.e. after the switch; the interpreter tier is timed separately below.
    n_ready, specialize_s = prog.wait_specialized(ProgramBuffer.SINK_FLOAT4)
    tier = "specialised" if n_ready else "interpreter"
    # assemblies: the specialised kernels of dense grids skip, per brick, the parts that cannot be nearest
    parts_active = bool(n_ready) and int(pinfo.n_parts_bounded) > 0 and os.environ.get("CODECAD_B200_PARTS", "1") != "0"
    # extrusions: what cannot see the grid coordinate along the extrusion axis is evaluated once per column
    columns_active = (bool(n_ready) and int(pinfo.column_invariant_percent) > 0 and os.environ.get("CODECAD_B200_COLUMNS", "1") != "0"
                      and (nx if int(pinfo.column_axis) == 0 else n) >= 8)
    kernel_key = "columns" if columns_active else "parts" if parts_active else tier
    # Kernel-only leg at N > 1: equal x-slabs.  (CODECAD_B200_BENCH_BALANCED_SLABS=1 cuts slabs of about equal WORK
    # instead — codecad_b200.grid_eval.balanced_slabs, the brick masks' cost estimate; on the planetary grid the
    # estimate moves the cuts by one layer of eight planes at most, so it is not the default.  The end-to-end leg
    # keeps equal slabs either way: it is bound by the bytes each rank copies to its host.)
    slabs = [ge.slab_range(n, r, world) for r in range(world)]
    if world > 1 and parts_active and os.environ.get("CODECAD_B200_BENCH_BALANCED_SLABS", "0") == "1":
        slabs = ge.balanced_slabs(prog, corner, step, (n, n, n), world)
    kx0, kx1 = slabs[rank]
    knx = kx1 - kx0
    out = Buffer(FLOAT4, (max(nx, knx), n, n))   # slab output stays resident in HBM

    def kernel_step():
        _lib.check(L.cc_grid_eval(prog.handle, c3, float(step), knx, n, n, kx0, 0, out.device_ptr, None))

    def timed(fn, steps):
        e0, e1 = ctypes.c_void_p(), ctypes.c_void_p()
        _lib.check(L.cc_event_record(ctypes.byref(e0)))
        for _ in range(steps):
            fn()
        _lib.check(L.cc_event_record(ctypes.byref(e1)))
        _lib.check(L.cc_event_wait(e1))
        ms = ctypes.c_float()
        _lib.check(L.cc_event_elapsed_ms(e0, e1, ctypes.byref(ms)))
        L.cc_event_destroy(e0)
        L.cc_event_destroy(e1)
        return ms.value

    # ---- kernel-only throughput ----
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for _ in range(max(args.warmup, 3)):
        kernel_step()
    _lib.check(L.cc_synchronize())
    barrier(torch, dist)
    L.cc_reset_counters()
    t_begin = time.time()
    ms_total = timed(kernel_step, args.steps)
    _lib.check(L.cc_synchronize())
    t_end = time.time()
    barrier(torch, dist)
    launches, _ = _lib.counters()
    clk = None
    if rank == 0:
        # nvidia-smi samples every 100 ms (started ahead of the warm-up: its first line takes longer than that); the K
        # timed steps may last no longer than one period, so the same step keeps running, untimed, until the load
        # window holds a handful of samples — the window reported is then the timed region plus that continuation
        t_load = t_end
        while len([1 for t, _s in clocks.samples if t_begin <= t <= t_load]) < 5 and t_load - t_end < 2.0:
            kernel_step()
            _lib.check(L.cc_synchronize())
            t_load = time.time()
        clk = clocks.stop((t_begin, t_load))
        clk["window_s"] = {"timed_region": t_end - t_begin, "same_steps_continued_untimed": t_load - t_end}
    if args.dump_outputs:
        # on rank 0 the buffer was last written by the untimed steps that continued the timed ones for the clock
        # samples: the same launch on the same inputs, whose result does not depend on how often it ran
        dump_grid_sample(args.dump_outputs, L, _lib, out, kx0, kx1, n, rank, torch, dist)
    ms_total = max_over_ranks(torch, dist, ms_total)
    ms_step = ms_total / args.steps
    total_points = float(n) ** 3
    value = total_points / (ms_step * 1e-3) / 1e9
    launches_total = int(sum_over_ranks(torch, dist, float(launches)))

    # ---- the interpreter tier alone (what runs before the specialised kernel is ready) ----
    interp = None
    if n_ready:
        prog.use_specialized(False)
        kernel_step()
        _lib.check(L.cc_synchronize())
        barrier(torch, dist)
        i_steps = max(1, min(args.steps, 2))
        i_ms = max_over_ranks(torch, dist, timed(kernel_step, i_steps)) / i_steps
        barrier(torch, dist)
        interp = {"value": total_points / (i_ms * 1e-3) / 1e9, "unit": "Gpts/s", "ms_per_step": i_ms,
                  "steps": i_steps, "kernel": "cc_eval_kernel<PTS,const,FLOAT4>"}
        if parts_active:
            # the interpreter walks the loader's segment table with the same per-brick masks (csrc/cc_parts.cu);
            # the full walk (every micro-op at every point) is timed beside it
            interp["kernel"] = "cc_parts_eval_kernel + cc_parts_centers_kernel (interpreter, per-brick part culling)"
            old_parts = _lib.check(L.cc_set_parts_mode(0))
            kernel_step()
            _lib.check(L.cc_synchronize())
            barrier(torch, dist)
            f_ms = max_over_ranks(torch, dist, timed(kernel_step, 1))
            barrier(torch, dist)
            _lib.check(L.cc_set_parts_mode(old_parts))
            interp["full_walk"] = {"value": total_points / (f_ms * 1e-3) / 1e9, "unit": "Gpts/s", "ms_per_step": f_ms,
                                   "kernel": "cc_eval_kernel<PTS,const,FLOAT4>"}
        prog.use_specialized(True)

    # ---- end to end: fresh program upload + result into pinned host memory ----
    e2e = None
    try:
        pin = _Pinned(my_points * 16)
        host = pin.array(FLOAT4, (nx, n, n))

        def e2e_step():
            p = ProgramBuffer(scene.words)              # H2D: decoded program
            _lib.check(L.cc_grid_eval_to_host(p.handle, c3, float(step), nx, n, n, x0, 0, host.ctypes.data))
            p.release()

        e2e_steps = max(1, min(args.steps, 3))
        e2e_step()                                      # warm-up (page-touches the pinned buffer)
        barrier(torch, dist)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        barrier(torch, dist)
        dt = max_over_ranks(torch, dist, time.perf_counter() - t0) / e2e_steps
        e2e = {"value": total_points / dt / 1e9, "unit": "Gpts/s",
               "h2d_bytes_per_step": int(pinfo.n_micro_words * 4 * world),
               "d2h_bytes_per_step": int(total_points * 16),
               "ms_per_step": dt * 1e3, "steps": e2e_steps,
               "api": "codecad_b200 cc_grid_eval_to_host: program upload + slab-pipelined kernel/D2H into pinned host memory"}
        # the same bytes with no kernel in the way: what the PCIe / host-memory path alone delivers
        try:
            mine_gbs, agg_gbs = d2h_probe(L, _lib, out.device_ptr, host, my_points * 16, torch, dist)
            e2e["d2h_probe"] = {"gbs_this_rank": mine_gbs, "gbs_all_ranks": agg_gbs * world,
                                "e2e_gbs_all_ranks": total_points * 16 / dt / 1e9,
                                "note": "bare cudaMemcpyAsync of every rank's slab into its pinned buffer, all ranks "
                                        "at once, same job: e2e is bound by this path when the two agree"}
        except Exception as exc:  # noqa: BLE001
            e2e["d2h_probe"] = {"error": str(exc)[:200]}
        del host, pin
    except Exception as exc:  # noqa: BLE001
        e2e = {"value": None, "unit": "Gpts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
               "error": str(exc)[:200]}

    # ---- the other BASELINE.json configs as dense grids, and the sharded hierarchy paths: every
    #      rank takes part (slabs / shares), rank 0 reports ----
    sm_max_all = max_over_ranks(torch, dist, float((clk or {}).get("sm_max_mhz") or info.sm_clock_khz / 1e3))
    try:
        hbm_peak_all = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0)
    except Exception:  # noqa: BLE001
        hbm_peak_all = 6650.0
    configs = {}
    if not args.no_configs:
        out.release()
        big = Buffer(FLOAT4, (256, 2048, 2048))   # 17.2 GB: the slab one GPU of eight owns at 2048^3
        plan = [
            ("C1_menger_256", "cfg_menger_sponge", "examples/menger_sponge.py dense grid_eval 256^3 (BASELINE configs[0])", 256, None, 20),
            ("C2_csg_dense_1024", "cfg_csg_example", "examples/csg_example.py dense grid_eval 1024^3 (store-bandwidth probe)", 1024, None, 5),
            ("C3_airfoil_dense_1024", "cfg_airfoil", "examples/airfoil.py dense grid_eval 1024^3", 1024, None, 2),
            ("C5_synthetic500_2048", "cfg_synthetic500",
             "synthetic deep-CSG scene (500 rounded boxes, smooth unions) grid_eval at 2048^3, 256 x-planes per GPU "
             "(the slab each of 8 GPUs owns; the full 2048^3 grid at N = 8) (BASELINE configs[4])", 2048, 256, 5),
        ]
        for key, name, label, n_c, slab, k in plan:
            try:
                configs[key] = config_grid_leg(name, label, n_c, slab, rank, world, torch, dist, info, sm_max_all,
                                               hbm_peak_all, k, big)
            except Exception as exc:  # noqa: BLE001
                configs[key] = {"error": str(exc)[:300]}
        if "value" in configs.get("C5_synthetic500_2048", {}):
            configs["C5_synthetic500_2048"]["full_2048_cubed"] = bool(world == 8)
        big.release()
    sharded = None
    try:
        sharded = sharded_hierarchy_legs(rank, world, torch, dist)
    except Exception as exc:  # noqa: BLE001
        sharded = {"error": str(exc)[:300]}

    # ---- one process driving all N GPUs (rank 0 spawns it while the other ranks wait on the store) ----
    single = None
    if world > 1 and not args.no_configs:
        store = None
        try:
            import torch.distributed.distributed_c10d as c10d
            store = c10d._get_default_store()
        except Exception:  # noqa: BLE001
            store = None
        _lib.check(L.cc_synchronize())
        barrier(torch, dist)
        if rank == 0:
            try:
                env = {k: v for k, v in os.environ.items()
                       if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "OMP_NUM_THREADS")}
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--single-process-leg", str(world)],
                                   capture_output=True, text=True, timeout=600, env=env)
                lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
                single = json.loads(lines[-1]) if (r.returncode == 0 and lines) else {"error": (r.stderr or r.stdout)[-300:]}
            except Exception as exc:  # noqa: BLE001
                single = {"error": str(exc)[:300]}
            if store is not None:
                store.set("single_process_leg_done", "1")
        elif store is not None:
            store.wait(["single_process_leg_done"])
        barrier(torch, dist)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the interpreter kernel ----
    sm_max_mhz = (clk or {}).get("sm_max_mhz") or info.sm_clock_khz / 1e3
    peak_tflops = info.sm_count * 128 * 2 * sm_max_mhz * 1e6 / 1e12
    flops_pt = int(pinfo.flops_min)
    # per launch (= per rank-step): this rank's points / its kernel time; ranks are symmetric
    achieved = (total_points / world) * flops_pt / (ms_step * 1e-3) / 1e12
    if interp:
        interp["roofline_frac"] = (total_points / world) * flops_pt / (interp["ms_per_step"] * 1e-3) / 1e12 / peak_tflops
        if "full_walk" in interp:
            interp["full_walk"]["roofline_frac"] = ((total_points / world) * flops_pt / (interp["full_walk"]["ms_per_step"] * 1e-3)
                                                    / 1e12 / peak_tflops)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "bench_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get("%s_%d" % (kernel_key, n))
        except Exception:  # noqa: BLE001
            traffic = None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    executed = load_executed_flops()
    roofline = {
        "bound": "fp32", "achieved": achieved, "peak": peak_tflops, "unit": "TFLOP/s",
        "frac": achieved / peak_tflops, "traffic": traffic,
        "traffic_source": "replayed from profiles/bench_traffic.json (one ncu --set full capture of this kernel at this "
                          "grid size, dram__bytes_read.sum + dram__bytes_write.sum per launch); not measured in this run",
        "kernel": ("cc_jit_columns + cc_jit_columns_profiles%s (scene-specialised, packed FFMA2 lanes; the 2-D profiles under the "
                   "extrusions once per %s-column, the rest per cell%s)"
                   % (" + cc_jit_columns_centers" if parts_active else "", "xyz"[int(pinfo.column_axis)],
                      ", per-brick part culling" if parts_active else "") if columns_active
                   else "cc_jit_parts + cc_jit_part_centers (scene-specialised, packed FFMA2 lanes, per-brick part culling)" if parts_active
                   else "cc_jit_float4 (scene-specialised, packed FFMA2 lanes)" if n_ready else "cc_eval_kernel<PTS,const,FLOAT4>"),
        "culling": (None if not parts_active else
                    "the scene is an assembly of %d parts under sharp unions; per 8x8x16 brick the kernel evaluates every part at the "
                    "brick centre, bounds it over the brick by its Lipschitz constant and skips the parts that cannot be the nearest "
                    "anywhere in the brick (bit-identical results, tests/test_gpu_parts.py).  `achieved` counts the flops of the full "
                    "walk the reference does, so `frac` exceeds 1; `issued` is what the kernel executes" % int(pinfo.n_parts)),
        "columns": (None if not columns_active else
                    "%d %% of the program's arithmetic (loader estimate) cannot depend on the grid's %s: 2-D profiles under extrusions.  "
                    "One kernel evaluates those micro-ops once per column and writes the values the rest reads into a column buffer, "
                    "the brick kernel evaluates only the rest per cell (bit-identical, tests/test_gpu_columns.py; DESIGN.md 4.10)"
                    % (int(pinfo.column_invariant_percent), "xyz"[int(pinfo.column_axis)])),
        "flop_per_point": flops_pt,
        "flop_per_point_executed": executed.get(SCENE),
        "achieved_executed_branch": (None if SCENE not in executed else
                                     (total_points / world) * executed[SCENE] / (ms_step * 1e-3) / 1e12),
        "frac_executed_branch": (None if SCENE not in executed else
                                 (total_points / world) * executed[SCENE] / (ms_step * 1e-3) / 1e12 / peak_tflops),
        "executed_source": "profiles/executed_flops.json (instrumented CPU oracle, 64^3 stratified subsample of this grid, "
                           "tools/measure_executed_flops.py; SURVEY.md 8(d)); `achieved`/`frac` use the static minimum",
        "issued": load_issued_flops(kernel_key, n),
        "peak_source": "derived: %d SMs x 128 FP32 lanes x 2 x %.0f MHz (no FP32 figure in MEASURED_PEAKS.json)"
                       % (info.sm_count, sm_max_mhz),
        "note": "algorithmic flop/point = static minimum over data-dependent branches with the "
                "SURVEY.md 8(a3) counting rules (FMA = 2; compare/select/abs free; libm-class calls not counted)",
        "hbm": {"achieved_gbs": (total_points / world) * 16 / (ms_step * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                "frac": (total_points / world) * 16 / (ms_step * 1e-3) / 1e9 / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback"},
    }

    # ---- CPU baseline (rank 0, N = 1 only) ----
    cpu = None
    if world == 1 and not args.no_cpu:
        r = cpu_sample_run(scene, n, 12.0, 1, "auto")
        cpu = {"value": r["value"], "unit": "Gpts/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
               "sample_fraction": r["sample_fraction"], "compile_flags": r["compile_flags"]}

    mass = subdiv = mesh = rays = outline = None
    if world == 1 and not args.no_cpu:
        try:
            mass = mass_properties_leg()
        except Exception as exc:  # noqa: BLE001
            mass = {"error": str(exc)[:200]}
        try:
            subdiv = subdivision_leg()
        except Exception as exc:  # noqa: BLE001
            subdiv = {"error": str(exc)[:200]}
        try:
            mesh = mesh_export_leg()
        except Exception as exc:  # noqa: BLE001
            mesh = {"error": str(exc)[:200]}
        try:
            rays = ray_caster_leg()
        except Exception as exc:  # noqa: BLE001
            rays = {"error": str(exc)[:200]}
        try:
            outline = polygon_leg()
        except Exception as exc:  # noqa: BLE001
            outline = {"error": str(exc)[:200]}

    line = {
        "metric": METRIC, "value": value, "unit": "Gpts/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(n, world), x_slabs=[list(sl) for sl in slabs],
                       x_slab_rule=("equal work by the brick masks' cost estimate (cc_grid_eval_cost_profile)" if slabs != [
                           ge.slab_range(n, r, world) for r in range(world)] else "equal plane counts")),
        "clocks": clk, "e2e": e2e,
        "gpu_launches": launches_total, "roofline": roofline, "cpu_baseline": cpu,
        "tier": tier, "specialize_s": specialize_s, "interpreter_tier": interp, "mass_properties": mass, "subdivision": subdiv, "mesh_export": mesh,
        "ray_caster": rays, "polygon2d": outline,
        "configs": configs, "sharded": sharded, "single_process_multi_gpu": single,
        "device": info.name.decode(),
    }
    _emit(out_fd, line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--grid", type=int, default=1024)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config dense grids and the single-process leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed sample of the grid the last timed step computed to DIR as .npy files")
    ap.add_argument("--single-process-leg", type=int, default=0, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU arm's grid; --impl reference has none")
    if args.single_process_leg:
        return single_process_leg(args.single_process_leg)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
