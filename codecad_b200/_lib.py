"""ctypes binding of libcodecad_b200.so (include/codecad_b200.h).

The product path goes through this module only.  If the shared library is missing or no
CUDA device is usable, every entry point raises: there is no CPU or PyTorch fallback.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("CODECAD_B200_LIB") or os.path.join(_HERE, "libcodecad_b200.so")

c_float_p = ctypes.POINTER(ctypes.c_float)
c_u32_p = ctypes.POINTER(ctypes.c_uint32)
c_u8_p = ctypes.POINTER(ctypes.c_uint8)
c_void_pp = ctypes.POINTER(ctypes.c_void_p)

LAYOUT_INDEX3_FLOAT4 = 0
LAYOUT_PYMCUBES_FLOAT = 1


class CodecadB200Error(RuntimeError):
    pass


class DeviceInfo(ctypes.Structure):
    _fields_ = [("device", ctypes.c_int), ("sm_count", ctypes.c_int), ("sm_clock_khz", ctypes.c_int),
                ("l2_bytes", ctypes.c_int), ("total_mem", ctypes.c_size_t), ("name", ctypes.c_char * 64)]


class ProgramInfo(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint32) for n in (
        "n_words", "n_instructions", "n_micro_ops", "n_micro_words", "n_wire_registers",
        "n_slots", "n_fused", "flops_min", "flops_max", "n_forest_leaves", "forest_depth", "n_parts", "n_parts_bounded",
        "column_invariant_percent", "column_axis")]


class Level(ctypes.Structure):
    _fields_ = [("cell_size", ctypes.c_int64), ("nx", ctypes.c_uint32), ("ny", ctypes.c_uint32),
                ("nz", ctypes.c_uint32)]


# every exported symbol of include/codecad_b200.h: name -> (restype, argtypes)
_V = ctypes.c_void_p
_I = ctypes.c_int
_U = ctypes.c_uint32
_F = ctypes.c_float
SIGNATURES = {
    "cc_init": (_I, [_I]),
    "cc_init_devices": (_I, [ctypes.POINTER(ctypes.c_int), _I]),
    "cc_active_devices": (_I, []),
    "cc_shutdown": (None, []),
    "cc_device_count": (_I, []),
    "cc_last_error": (ctypes.c_char_p, []),
    "cc_get_device_info": (_I, [ctypes.POINTER(DeviceInfo)]),
    "cc_device_pci_bus_id": (_I, [_I, ctypes.c_char_p, _I]),
    "cc_synchronize": (_I, []),
    "cc_get_counters": (_I, [ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]),
    "cc_reset_counters": (None, []),
    "cc_get_check_fallbacks": (_I, [ctypes.POINTER(ctypes.c_uint64)]),
    "cc_get_flagged_bricks": (_I, [ctypes.POINTER(ctypes.c_uint64)]),
    "cc_set_tuning": (_I, [_I, _I]),
    "cc_program_create": (_I, [c_float_p, _U, c_void_pp]),
    "cc_program_destroy": (None, [_V]),
    "cc_program_get_info": (_I, [_V, ctypes.POINTER(ProgramInfo)]),
    "cc_program_get_microcode": (_I, [_V, c_u32_p, _U]),
    "cc_program_decode": (_I, [c_float_p, _U, ctypes.POINTER(ProgramInfo), c_u32_p, _U]),
    "cc_program_specialize": (_I, [_V, _I, _U, ctypes.POINTER(ctypes.c_double)]),
    "cc_program_use_specialized": (_I, [_V, _I]),
    "cc_set_jit_mode": (_I, [_I]),
    "cc_set_forest_mode": (_I, [_I]),
    "cc_set_parts_mode": (_I, [_I]),
    "cc_set_columns_mode": (_I, [_I]),
    "cc_grid_eval_cost_profile": (_I, [_V, c_float_p, ctypes.c_float, _U, _U, _U, _U, ctypes.POINTER(ctypes.c_double), _U]),
    "cc_program_get_forest_info": (_I, [_V, c_u32_p]),
    "cc_program_specialize_wait": (_I, [_V, _U, ctypes.POINTER(ctypes.c_double)]),
    "cc_specialize_source": (_I, [c_float_p, _U, _I, _U, ctypes.c_char_p, _U, _I, ctypes.POINTER(ctypes.c_uint64)]),
    "cc_buffer_alloc": (_I, [ctypes.c_size_t, c_void_pp]),
    "cc_buffer_free": (_I, [_V]),
    "cc_host_alloc": (_I, [ctypes.c_size_t, c_void_pp]),
    "cc_host_free": (_I, [_V]),
    "cc_memcpy_h2d_async": (_I, [_V, _V, ctypes.c_size_t, c_void_pp]),
    "cc_memcpy_d2h_async": (_I, [_V, _V, ctypes.c_size_t, c_void_pp]),
    "cc_memset_async": (_I, [_V, _I, ctypes.c_size_t, c_void_pp]),
    "cc_event_record": (_I, [c_void_pp]),
    "cc_event_wait": (_I, [_V]),
    "cc_event_elapsed_ms": (_I, [_V, _V, c_float_p]),
    "cc_event_destroy": (None, [_V]),
    "cc_grid_eval": (_I, [_V, c_float_p, _F, _U, _U, _U, _U, _I, _V, c_void_pp]),
    "cc_grid_eval_to_host": (_I, [_V, c_float_p, _F, _U, _U, _U, _U, _I, _V]),
    "cc_subdivision_step": (_I, [_V, c_float_p, _F, _F, _U, _U, _U, _V, _V, c_void_pp]),
    "cc_mass_properties_step": (_I, [_V, c_float_p, _F, _F, _U, _U, _U, _V, _V, _V, c_void_pp]),
    "cc_subdivide": (_I, [_V, ctypes.POINTER(ctypes.c_double), ctypes.c_double, ctypes.POINTER(Level), _U, _I,
                          _U, _U, ctypes.POINTER(ctypes.POINTER(ctypes.c_int64)), ctypes.POINTER(ctypes.c_uint64)]),
    "cc_mass_properties": (_I, [_V, ctypes.POINTER(ctypes.c_double), ctypes.c_double, ctypes.POINTER(Level), _U,
                                _U, _U, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint64)]),
    "cc_mass_properties_exact": (_I, [_V, ctypes.POINTER(ctypes.c_double), ctypes.c_double, ctypes.POINTER(Level), _U,
                                      _U, _U, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int32),
                                      ctypes.POINTER(ctypes.c_uint64)]),
    "cc_assembly_mass_properties_exact": (_I, [c_void_pp, _U, ctypes.POINTER(ctypes.c_double), ctypes.c_double,
                                               ctypes.POINTER(Level), _U, _U, _U, ctypes.POINTER(ctypes.c_int64),
                                               ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_uint64)]),
    "cc_mass_limbs_to_integrals": (_I, [ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int32),
                                        ctypes.POINTER(ctypes.c_double)]),
    "cc_sort_leaf_corners": (_I, [ctypes.POINTER(ctypes.c_int64), ctypes.c_uint64, ctypes.POINTER(Level), _U]),
    "cc_evaluate_points": (_I, [_V, _V, ctypes.c_uint64, _V, c_void_pp]),
    "cc_ray_caster": (_I, [_V, c_float_p, c_float_p, c_float_p, c_float_p, _F, _F, _F, _F, _F, _U, _U, _U, _V,
                           ctypes.POINTER(ctypes.c_uint64), c_void_pp]),
    "cc_bitmap": (_I, [_V, c_float_p, _F, _U, _U, _V, c_void_pp]),
    "cc_matplotlib_slice": (_I, [_V, c_float_p, _F, _U, _U, _V, c_void_pp]),
    "cc_process_polygon": (_I, [c_float_p, _F, _U, _U, _V, _V, _V, _V, _U, _V, c_void_pp]),
    "cc_polygon_blocks": (_I, [_V, ctypes.POINTER(ctypes.c_double), ctypes.c_double, _U, _U, _U, _V, _V, _V, _V]),
    "cc_polygon_assemble": (_I, [_V, _V, _V, _V, _V, ctypes.c_int64, _U, _U, _U, ctypes.POINTER(ctypes.POINTER(ctypes.c_float)),
                                 ctypes.POINTER(ctypes.POINTER(ctypes.c_uint64)), ctypes.POINTER(ctypes.c_uint64)]),
    "cc_mesh_blocks": (_I, [_V, ctypes.POINTER(ctypes.c_double), ctypes.c_double, _U, _U, _U, _U,
                            ctypes.POINTER(ctypes.POINTER(ctypes.c_double)),
                            ctypes.POINTER(ctypes.POINTER(ctypes.c_uint32)), ctypes.POINTER(ctypes.c_uint64)]),
    "cc_mesh_blocks_indexed": (_I, [_V, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64), ctypes.c_double,
                                    _U, _U, _U, _U,
                                    ctypes.POINTER(ctypes.POINTER(ctypes.c_double)), ctypes.POINTER(ctypes.c_uint64),
                                    ctypes.POINTER(ctypes.POINTER(ctypes.c_uint32)),
                                    ctypes.POINTER(ctypes.POINTER(ctypes.c_uint32)), ctypes.POINTER(ctypes.c_uint64)]),
    "cc_free": (None, [_V]),
}

_lib = None
_initialized_device = None


def load():
    """Load the shared library (no CUDA call yet)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise CodecadB200Error(
                "%s is missing: build it with `python -m codecad_b200.build` "
                "(there is no fallback path)" % SO_PATH)
        L = ctypes.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc < 0:
        raise CodecadB200Error("libcodecad_b200: %s (code %d)" % (load().cc_last_error().decode(), rc))
    return rc


def bind_host_to_device(device):
    """Pin the calling process to the CPU cores (hence the NUMA node) next to CUDA device `device`,
    so that page-locked host buffers allocated afterwards sit on the memory the GPU's PCIe root
    reaches directly.  With one process per GPU and results delivered to host memory this decides
    whether eight ranks share one socket's memory controllers.  Uses the PCI address from sysfs;
    returns the CPU list applied, or None when the topology cannot be read (nothing is changed)."""
    try:
        info = DeviceInfo()
        L = load()
        bus = ctypes.create_string_buffer(32)
        if not hasattr(L, "cc_device_pci_bus_id") or L.cc_device_pci_bus_id(int(device), bus, 32) != 0:
            return None
        path = "/sys/bus/pci/devices/%s/local_cpulist" % bus.value.decode().lower()
        with open(path) as f:
            text = f.read().strip()
        cpus = set()
        for part in text.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return sorted(cpus)
    except Exception:  # noqa: BLE001 - an optimisation, never a failure
        return None


def _devices_from_env():
    """CODECAD_B200_DEVICES: "all", or a comma separated list of CUDA device indices that one
    process should drive (the first one is the primary device)."""
    spec = os.environ.get("CODECAD_B200_DEVICES", "").strip()
    if not spec:
        return None
    if spec.lower() == "all":
        return list(range(load().cc_device_count()))
    return [int(x) for x in spec.split(",") if x.strip()]


def init(device=None):
    """Create the CUDA context on `device` (default: LOCAL_RANK, else 0).  Outside torchrun,
    CODECAD_B200_DEVICES=all (or "0,1,2,3") makes this one process drive several GPUs: the calls
    that shard (mass_properties, subdivision, grid_eval to host) then use all of them."""
    global _initialized_device
    L = load()
    if device is None:
        devices = _devices_from_env() if "LOCAL_RANK" not in os.environ else None
        if devices:
            return init_devices(devices)
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if _initialized_device is None:
        check(L.cc_init(int(device)))
        _initialized_device = int(device)
    elif _initialized_device != int(device):
        raise CodecadB200Error("already initialised on device %d" % _initialized_device)
    return L


def init_devices(devices=None):
    """One process, several GPUs (cc_init_devices): `devices` is a list of CUDA device indices
    (default: all).  devices[0] is the primary device; may follow init(devices[0])."""
    global _initialized_device
    L = load()
    if devices is None:
        devices = list(range(L.cc_device_count()))
    devices = [int(d) for d in devices]
    if not devices:
        raise CodecadB200Error("no CUDA device available; libcodecad_b200 has no CPU fallback")
    if _initialized_device is not None and _initialized_device != devices[0]:
        raise CodecadB200Error("already initialised on device %d" % _initialized_device)
    arr = (ctypes.c_int * len(devices))(*devices)
    check(L.cc_init_devices(arr, len(devices)))
    _initialized_device = devices[0]
    return L


def active_devices():
    return int(load().cc_active_devices())


def lib():
    """Library with an initialised context."""
    return init(_initialized_device)


def device_info():
    info = DeviceInfo()
    check(lib().cc_get_device_info(ctypes.byref(info)))
    return info


def counters():
    a, b = ctypes.c_uint64(), ctypes.c_uint64()
    check(lib().cc_get_counters(ctypes.byref(a), ctypes.byref(b)))
    return a.value, b.value


def check_fallbacks():
    """Warps of the column brick kernel that failed their deferred range check and took the full walk."""
    n = ctypes.c_uint64()
    check(lib().cc_get_check_fallbacks(ctypes.byref(n)))
    return n.value


def flagged_bricks():
    """Bricks of the column brick kernel that a column failing its run-time check sent to the full walk."""
    n = ctypes.c_uint64()
    check(lib().cc_get_flagged_bricks(ctypes.byref(n)))
    return n.value


def f3(v):
    """corner argument: accepts a numpy structured float4 scalar (Vector.as_float4()), or
    any 3/4-sequence; returns a ctypes float[3] rounded to fp32 like as_float4()."""
    a = np.asarray(v)
    if a.dtype.names:
        a = np.array([a["x"], a["y"], a["z"]], dtype=np.float32)
    else:
        a = np.asarray(a, dtype=np.float64).astype(np.float32).ravel()[:3]
    return (ctypes.c_float * 3)(*[float(x) for x in a])


def decode_program(words):
    """Host-only decode of a wire program: (ProgramInfo, microcode uint32 array)."""
    w = np.ascontiguousarray(words, dtype=np.float32)
    info = ProgramInfo()
    n = check(load().cc_program_decode(w.ctypes.data_as(c_float_p), len(w), ctypes.byref(info), None, 0))
    out = np.zeros(n, np.uint32)
    check(load().cc_program_decode(w.ctypes.data_as(c_float_p), len(w), ctypes.byref(info),
                                   out.ctypes.data_as(c_u32_p), n))
    return info, out


def specialize_source(words, points_per_thread=2, compile=False, sink_mask=0):
    """Host-only: CUDA source of the scene-specialised kernels for `words`; with compile=True
    also run NVRTC on it and return (source, cubin_bytes)."""
    w = np.ascontiguousarray(words, dtype=np.float32)
    n = check(load().cc_specialize_source(w.ctypes.data_as(c_float_p), len(w), points_per_thread, sink_mask, None, 0, 0, None))
    buf = ctypes.create_string_buffer(n + 1)
    size = ctypes.c_uint64()
    check(load().cc_specialize_source(w.ctypes.data_as(c_float_p), len(w), points_per_thread, sink_mask, buf, n + 1,
                                      1 if compile else 0, ctypes.byref(size)))
    src = buf.value.decode()
    return (src, int(size.value)) if compile else src
