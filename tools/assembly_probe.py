#!/usr/bin/env python3
"""The assembly mass properties (DESIGN.md 4.11) against the routes a caller has without them, on assemblies of 8, 16
and 32 parts from tests/programs.py: extruded hexagons and cylinders on a grid, each touching its neighbours, with a
few of them pushed into a neighbour.  Writes OUT_DIR/assembly_probe.json with the card's name and power limit.

    python tools/assembly_probe.py OUT_DIR [--reps 5] [--pair-seconds 10]

Per assembly:
  one_pass_ms        cc_assembly_mass_properties_exact, median of repetitions alternated with the standalone route
  standalone_t2_ms   n mass_limbs calls on the same box and plan, specialised kernels built and warmed (median)
  standalone_t1_ms   the same on the interpreter (median)
  pairs_isect        the intersection program of a pair through mass_limbs on the interpreter: pairs measured within
                     --pair-seconds, their total and mean time (what n (n - 1) / 2 of them would cost is not stated)
  parts_identical    every part's limbs equal its standalone call's
"""
import argparse
import importlib
import json
import math
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import programs as P  # noqa: E402
from codecad_b200 import _lib  # noqa: E402
from codecad_b200.cl_util.buffer import ProgramBuffer  # noqa: E402
from codecad_b200.geometry import Vector  # noqa: E402
from codecad_b200.subdivision import calculate_block_sizes  # noqa: E402

mpm = importlib.import_module("codecad_b200.mass_properties")
R, H = 1.0, 1.0  # part radius (cylinder; hexagon circumradius) and half height


def assembly(n):
    """n parts on a square grid of pitch 2R (neighbours touch), hexagons and cylinders alternating; every fifth part is
    pushed 0.3 R into its neighbour along x"""
    side = math.ceil(math.sqrt(n))
    hexagon = [(R * math.cos(math.pi / 3 * i), R * math.sin(math.pi / 3 * i)) for i in range(6)]
    parts = []
    for k in range(n):
        i, j = k % side, k // side
        centre = (2 * R * i - (0.3 * R if k % 5 == 4 else 0.0), 2 * R * j, 0.0)
        proto = P.Part.polygon(hexagon, H) if k % 2 == 0 else P.Part.cylinder(R, H)
        parts.append(P.Part.placed(proto, centre))
    lo = (-R - 0.5, -R - 0.5, -H - 0.5)
    hi = (2 * R * (side - 1) + R + 0.5, 2 * R * ((n - 1) // side) + R + 0.5, H + 0.5)
    return parts, lo, hi


def intersection_program(a, b):
    return np.array(a.words(0) + P.ins("_store", 0) + b.words(1) + P.ins("intersection", 0, -1.0) + P.ins("_return"), np.float32)


def timed(fn):
    _lib.check(_lib.lib().cc_synchronize())
    t0 = time.perf_counter()
    out = fn()
    _lib.check(_lib.lib().cc_synchronize())
    return (time.perf_counter() - t0) * 1e3, out


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def probe(n, reps, pair_seconds, grid=64):
    parts, lo, hi = assembly(n)
    progs = [ProgramBuffer(P.program(p)) for p in parts]
    # leaf cells ~ 1.7 x area x grid / res^2 (the near band of the level above, in blocks of grid^3): about 2e8
    area = sum(2 * (3 * math.sqrt(3) / 2 if k % 2 == 0 else math.pi) * R * R + 2 * H * (6 if k % 2 == 0 else 2 * math.pi) * R
               for k in range(n))
    res = math.sqrt(1.7 * area * grid / 2e8)
    a, b = Vector(*lo), Vector(*hi)
    plan = calculate_block_sizes((a, b), 3, res, grid, overlap=False)
    L = _lib.lib()
    row = {"parts": n, "resolution": res, "grid": grid, "levels": len(plan)}

    old = _lib.check(L.cc_set_jit_mode(2))  # tier 2: build every part's specialised kernels, then warm
    ms, (limbs, exps, st) = timed(lambda: mpm.assembly_limbs(progs, a, res, plan))
    row["stats"] = st
    std = [mpm.mass_limbs(p, a, res, plan) for p in progs]
    row["parts_identical"] = bool(all(np.array_equal(limbs[k], std[k][0]) for k in range(n)))
    row["standalone_cells"] = sum(s[2]["cells"] for s in std)
    one, t2 = [], []
    for _ in range(reps):
        one.append(timed(lambda: mpm.assembly_limbs(progs, a, res, plan))[0])
        t2.append(timed(lambda: [mpm.mass_limbs(p, a, res, plan) for p in progs])[0])
    row["standalone_t2_ms"] = statistics.median(t2)
    _lib.check(L.cc_set_jit_mode(0))  # tier 1: the interpreter
    t1 = []
    for _ in range(reps):
        one.append(timed(lambda: mpm.assembly_limbs(progs, a, res, plan))[0])
        t1.append(timed(lambda: [mpm.mass_limbs(p, a, res, plan) for p in progs])[0])
    row["standalone_t1_ms"] = statistics.median(t1)
    row["one_pass_ms"] = statistics.median(one)  # (its own kernel on either setting: both rounds count)
    row["one_pass_ms_all"] = one
    # the intersection-program route, interpreter, pairs in order until the time is used up
    pairs = [(i, j) for i in range(n) for j in range(i + 1, n)]
    spent, done = 0.0, []
    for i, j in pairs:
        prog = ProgramBuffer(intersection_program(parts[i], parts[j]))
        ms, _ = timed(lambda: mpm.mass_limbs(prog, a, res, plan))
        done.append(ms)
        spent += ms / 1e3
        if spent > pair_seconds:
            break
    row["pairs_isect"] = {"measured": len(done), "of": len(pairs), "total_ms": sum(done), "mean_ms": statistics.mean(done)}
    overlapping = [(i, j) for i, j in pairs if limbs[mpm.pair_index(n, i, j)].any()]
    row["overlapping_pairs"] = overlapping
    _lib.check(L.cc_set_jit_mode(old))
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--pair-seconds", type=float, default=10.0)
    ap.add_argument("--parts", type=int, nargs="*", default=[8, 16, 32])
    args = ap.parse_args()
    _lib.init(0)
    info = _lib.device_info()
    out = {"card": card(), "device": info.name.decode(), "rows": []}
    for n in args.parts:
        out["rows"].append(probe(n, args.reps, args.pair_seconds))
        print(json.dumps(out["rows"][-1]), flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "assembly_probe.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
