#!/usr/bin/env python3
"""The column brick kernel (DESIGN.md 4.10) in its four variants — the pair of a thread's cells in one column (A,
CC_COL_PAIR) and one deferred range check per warp (B, CC_DEFER_CHECKS), each on or off — built side by side in one
process: planetary 1024^3 (z-columns) and airfoil 1024^3 (y-columns), timed alternately with CUDA events around the
whole call (column pass, brick centres, brick kernel, full walk), every variant's grid compared with off/off bit for
bit on the device, the warps that fell back, and the seconds each variant's first call took (specialisation).

    python tools/column_pairs_probe.py [--grid 1024] [--rounds 10]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

VARIANTS = [("off/off", "CC_COL_PAIR=0,CC_DEFER_CHECKS=0"), ("A", "CC_COL_PAIR=1,CC_DEFER_CHECKS=0"),
            ("B", "CC_COL_PAIR=0,CC_DEFER_CHECKS=1"), ("A+B", "CC_COL_PAIR=1,CC_DEFER_CHECKS=1")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=1024)
    ap.add_argument("--rounds", type=int, default=10)
    args = ap.parse_args()
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip())
    import ctypes
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

    print("| scene | variant | ms median | ms min..max | vs off/off | same bits as off/off | fallback warps | specialise s |")
    print("|---|---|---|---|---|---|---|---|")
    for name in ("cfg_planetary", "cfg_airfoil"):
        s = scenes[name]
        corner, step = s.grid(n)
        progs, spec = {}, {}
        for label, defines in VARIANTS:
            os.environ["CODECAD_B200_JIT_DEFINES"] = defines
            prog = s.compiled().program_buffer()
            t0 = time.perf_counter()
            launch(prog, corner, step, out)     # (jit mode 2: builds what the launch routes to, and waits)
            _lib.check(L.cc_synchronize())
            spec[label] = time.perf_counter() - t0
            progs[label] = prog
        os.environ.pop("CODECAD_B200_JIT_DEFINES", None)
        times = {label: [] for label, _ in VARIANTS}
        for _ in range(args.rounds):
            for label, _ in VARIANTS:
                times[label].append(timed(progs[label], corner, step))
        base = float(np.median(times["off/off"]))
        for label, _ in VARIANTS:
            L.cc_reset_counters()
            launch(progs[label], corner, step, ref if label == "off/off" else out)
            _lib.check(L.cc_synchronize())
            fb = _lib.check_fallbacks()
            same = "(itself)" if label == "off/off" else ("yes" if torch.equal(out, ref) else "NO")
            t = np.array(times[label])
            print("| %s | %s | %.2f | %.2f..%.2f | %+.1f %% | %s | %d | %.1f |" % (
                name, label, np.median(t), t.min(), t.max(), 100.0 * (np.median(t) / base - 1.0), same, fb, spec[label]))
            sys.stdout.flush()


if __name__ == "__main__":
    main()
