#!/usr/bin/env python3
"""The column brick kernel's sweep (DESIGN.md 4.10) with its extrusions' min / max against the selects (CC_SWEEP_MINMAX=0)
in one process: planetary 1024^3 and airfoil 1024^3 (a voting body: no sweep), timed alternately with CUDA events around
the whole call (column pass, brick centres, brick kernel, full walk).  The min / max grid (computed into a buffer filled
with 0xff bytes) is compared bit for bit on the device with the selects' one, and the warps that fell back to the full
walk are counted.

    python tools/sweep_minmax_probe.py [--grid 1024] [--rounds 10]
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

BUILDS = (("selects", "CC_SWEEP_MINMAX=0"), ("min/max", None))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=1024)
    ap.add_argument("--rounds", type=int, default=10)
    args = ap.parse_args()
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

    def launch(prog, corner, step, dst):
        c3 = (ctypes.c_float * 3)(*[float(v) for v in corner])
        _lib.check(L.cc_grid_eval(prog.handle, c3, float(step), n, n, n, 0, 0, ctypes.c_void_p(dst.data_ptr()), None))

    def timed(prog, corner, step):
        e0, e1, ms = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_float()
        _lib.check(L.cc_event_record(ctypes.byref(e0)))
        launch(prog, corner, step, out)
        _lib.check(L.cc_event_record(ctypes.byref(e1)))
        _lib.check(L.cc_event_wait(e1))
        _lib.check(L.cc_event_elapsed_ms(e0, e1, ctypes.byref(ms)))
        L.cc_event_destroy(e0)
        L.cc_event_destroy(e1)
        return ms.value

    print("| scene | sweep | ms median | ms min..max | vs selects | Gpts/s | same bits | fallback warps |")
    print("|---|---|---|---|---|---|---|---|")
    for name in ("cfg_planetary", "cfg_airfoil"):
        s = scenes[name]
        corner, step = s.grid(n)
        progs = {}
        for build, defines in BUILDS:
            if defines:
                os.environ["CODECAD_B200_JIT_DEFINES"] = defines
            progs[build] = s.compiled().program_buffer()
            launch(progs[build], corner, step, out)     # (jit mode 2: builds what the launch routes to, and waits)
            _lib.check(L.cc_synchronize())
            os.environ.pop("CODECAD_B200_JIT_DEFINES", None)
        times = {b: [] for b in progs}
        for _ in range(args.rounds):
            for b in progs:
                times[b].append(timed(progs[b], corner, step))
        first = BUILDS[0][0]
        base = float(np.median(times[first]))
        for b, _ in BUILDS:
            dst = ref if b == first else out
            dst.fill_(255)              # a cell the launch skips keeps 0xff bytes
            torch.cuda.synchronize()    # (the library launches on its own stream)
            L.cc_reset_counters()
            launch(progs[b], corner, step, dst)
            _lib.check(L.cc_synchronize())
            fb = _lib.check_fallbacks()
            same = "(itself)" if b == first else ("yes" if torch.equal(out, ref) else "NO")
            t = np.array(times[b])
            print("| %s | %s | %.3f | %.3f..%.3f | %+.1f %% | %.1f | %s | %d |" % (
                name, b, np.median(t), t.min(), t.max(), 100.0 * (np.median(t) / base - 1.0), n ** 3 / np.median(t) / 1e6, same, fb))
            sys.stdout.flush()


if __name__ == "__main__":
    main()
