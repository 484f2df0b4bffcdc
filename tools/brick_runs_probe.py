#!/usr/bin/env python3
"""The column brick kernel (DESIGN.md 4.10) at several run lengths (CODECAD_B200_BRICK_RUN: bricks one CTA walks along
the columns' axis; 1 is one brick per CTA) in one process: planetary 1024^3 (z-columns) and airfoil 1024^3
(y-columns), timed alternately with CUDA events around the whole call (column pass, brick centres, brick kernel, full
walk), every run length's grid (computed into a buffer filled with 0xff bytes) compared with runs of 1 bit for bit on
the device, the warps that fell back, and the bricks that flagged columns sent to the full walk.

    python tools/brick_runs_probe.py [--grid 1024] [--rounds 10] [--runs 1,4,8,16,64]
"""
import argparse
import ctypes
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=1024)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--runs", default="1,4,8,16,64")
    args = ap.parse_args()
    runs = [int(r) for r in args.runs.split(",")]
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip())
    import torch
    from codecad_b200 import _lib
    from scenes import load_scenes
    _lib.init(0)
    L = _lib.lib()
    _lib.check(L.cc_set_jit_mode(2))
    scenes = load_scenes()
    n = args.grid
    ref = torch.empty(n ** 3 * 16, dtype=torch.uint8, device="cuda")
    out = torch.empty_like(ref)

    def launch(prog, corner, step, dst, run):
        os.environ["CODECAD_B200_BRICK_RUN"] = str(run)
        c3 = (ctypes.c_float * 3)(*[float(v) for v in corner])
        _lib.check(L.cc_grid_eval(prog.handle, c3, float(step), n, n, n, 0, 0, ctypes.c_void_p(dst.data_ptr()), None))

    def timed(prog, corner, step, run):
        e0, e1, ms = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_float()
        _lib.check(L.cc_event_record(ctypes.byref(e0)))
        launch(prog, corner, step, out, run)
        _lib.check(L.cc_event_record(ctypes.byref(e1)))
        _lib.check(L.cc_event_wait(e1))
        _lib.check(L.cc_event_elapsed_ms(e0, e1, ctypes.byref(ms)))
        L.cc_event_destroy(e0)
        L.cc_event_destroy(e1)
        return ms.value

    print("| scene | run | ms median | ms min..max | vs run 1 | same bits as run 1 | fallback warps | flagged bricks |")
    print("|---|---|---|---|---|---|---|---|")
    for name in ("cfg_planetary", "cfg_airfoil"):
        s = scenes[name]
        corner, step = s.grid(n)
        prog = s.compiled().program_buffer()
        launch(prog, corner, step, out, 1)     # (jit mode 2: builds what the launch routes to, and waits)
        _lib.check(L.cc_synchronize())
        times = {r: [] for r in runs}
        for _ in range(args.rounds):
            for r in runs:
                times[r].append(timed(prog, corner, step, r))
        base = float(np.median(times[runs[0]]))
        for r in runs:
            dst = ref if r == runs[0] else out
            dst.fill_(255)              # a cell the launch skips keeps 0xff bytes, not the previous run length's value
            torch.cuda.synchronize()    # (the library launches on its own stream)
            L.cc_reset_counters()
            launch(prog, corner, step, dst, r)
            _lib.check(L.cc_synchronize())
            fb, fl = _lib.check_fallbacks(), _lib.flagged_bricks()
            same = "(itself)" if r == runs[0] else ("yes" if torch.equal(out, ref) else "NO")
            t = np.array(times[r])
            print("| %s | %d | %.3f | %.3f..%.3f | %+.1f %% | %s | %d | %d |" % (
                name, r, np.median(t), t.min(), t.max(), 100.0 * (np.median(t) / base - 1.0), same, fb, fl))
            sys.stdout.flush()
    os.environ.pop("CODECAD_B200_BRICK_RUN", None)


if __name__ == "__main__":
    main()
