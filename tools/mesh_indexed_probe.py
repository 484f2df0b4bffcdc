#!/usr/bin/env python3
"""End-to-end time of the welded mesh (indexed_mesh) against the triangle soup (mesh_arrays) on the
same blocks.  After a warm-up (which also waits for the specialised kernels), the two alternate for
--calls calls each; prints the median and spread of each, the triangles, vertices and bytes copied
to the host, and the card's name and power limit.

Workloads: csg_example at 512^3 effective resolution with 128^3 blocks (the benchmark's mesh
workload, DESIGN.md 4.4), and the planetary assembly at feature size 0.5."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from codecad_b200 import CompiledScene, _lib  # noqa: E402
from codecad_b200.cl_util.buffer import ProgramBuffer  # noqa: E402
from codecad_b200.rendering import indexed_mesh, mesh_arrays  # noqa: E402
from scenes import load_scenes  # noqa: E402

WORKLOADS = [("cfg_csg_example", 2 * 100.0 / 512, 128), ("cfg_planetary", 0.5, 128)]


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True)
    return out.stdout.strip()


def timed(fn):
    t0 = time.perf_counter()
    result = fn()  # the arrays are on the host when it returns
    return (time.perf_counter() - t0) * 1e3, result


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--calls", type=int, default=20)
    args = ap.parse_args()
    _lib.init(0)
    print("card:", card())
    scenes = load_scenes()
    for name, feature, grid in WORKLOADS:
        c = scenes[name]
        scene = CompiledScene(c.words, 3, c.box_a, c.box_b, feature, name)
        soup = lambda: mesh_arrays(scene, grid)  # noqa: E731
        welded = lambda: indexed_mesh(scene, grid)  # noqa: E731
        soup()
        scene.program_buffer().wait_specialized(ProgramBuffer.SINK_PYMCUBES | ProgramBuffer.SINK_CLASSIFY)
        for _ in range(2):
            soup()
            welded()
        times = {"mesh_arrays": [], "indexed_mesh": []}
        for _ in range(args.calls):
            ms, r = timed(soup)
            times["mesh_arrays"].append(ms)
            n_tri, n_blocks = len(r[1]), len(r[2])
            del r
            ms, r = timed(welded)
            times["indexed_mesh"].append(ms)
            n_vert, n_tri_w = len(r[0]), len(r[1])
            del r
        print("%s, feature size %g, %d^3 blocks: %d blocks" % (name, feature, grid, n_blocks))
        print("  mesh_arrays : %d triangles, %.1f MB to the host (76 B per triangle)" % (n_tri, n_tri * 76 / 1e6))
        b = n_vert * 24 + n_tri_w * 16
        print("  indexed_mesh: %d triangles, %d vertices, %.1f MB to the host (%.1f B per triangle)"
              % (n_tri_w, n_vert, b / 1e6, b / max(n_tri_w, 1)))
        for k, v in times.items():
            v = np.array(v)
            print("  %-13s median %.2f ms, min %.2f, max %.2f over %d calls" % (k, np.median(v), v.min(), v.max(), len(v)))


if __name__ == "__main__":
    main()
