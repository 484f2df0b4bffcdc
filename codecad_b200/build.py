"""Build libcodecad_b200.so in-tree with nvcc for sm_100a.

    python -m codecad_b200.build [--force] [--verbose]

-fmad=false / -ffp-contract=off are part of the numerical contract (csrc/cc_math.cuh):
all fused multiply-adds are explicit.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libcodecad_b200.so")
SOURCES = ["cc_kernels.cu", "cc_parts.cu", "cc_assembly.cu", "cc_forest.cu", "cc_mesh.cu", "cc_polygon.cu", "cc_program.cpp", "cc_api.cpp", "cc_jit.cpp"]
HEADERS = ["cc_internal.h", "cc_microcode.h", "cc_math.cuh", "cc_ops.cuh", "cc_interp.cuh", "cc_body.cuh", "cc_render.cuh", "cc_device_types.h", "cc_mc_table.h", "cc_scan.cuh",
           os.path.join("..", "..", "include", "codecad_b200.h")]

COMPILE_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math",
]
OBJ_DIR = os.path.join(HERE, "build")


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _deps():
    return [os.path.join(CSRC, f) for f in HEADERS] + [os.path.abspath(__file__)]


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in SOURCES] + _deps()
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """One object per source, compiled in parallel and only when stale (objects live in the
    git-ignored codecad_b200/build/), then linked into the in-tree shared library."""
    if not force and not needs_build():
        try:
            build_pylist()
        except Exception:  # noqa: BLE001
            pass
        return SO
    nvcc = find_nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    newest_header = max(os.path.getmtime(d) for d in _deps())
    jobs, objs = [], []
    for f in SOURCES:
        src = os.path.join(CSRC, f)
        obj = os.path.join(OBJ_DIR, os.path.splitext(f)[0] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), newest_header):
            cmd = [nvcc] + COMPILE_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            jobs.append((f, subprocess.Popen(cmd)))
    failed = [f for f, p in jobs if p.wait() != 0]
    if failed:
        raise RuntimeError("nvcc failed for " + ", ".join(failed))
    subprocess.run([nvcc, "-shared", "-o", SO] + objs + ["-ldl"], check=True)
    try:
        build_pylist(force)
    except Exception as exc:  # noqa: BLE001 - optional accelerator of a Python-side conversion
        print("codecad_b200/_cc_pylist.so not built:", exc)
    return SO


def build_pylist(force=False):
    """The small CPython helper (csrc/cc_pylist.c): host-only, plain gcc."""
    import sysconfig
    src = os.path.join(CSRC, "cc_pylist.c")
    so = os.path.join(HERE, "_cc_pylist.so")
    if not force and os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(src):
        return so
    subprocess.run(["gcc", "-O2", "-shared", "-fPIC", "-I", sysconfig.get_paths()["include"], "-o", so, src], check=True)
    return so


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
    print(build_pylist(force="--force" in sys.argv))
