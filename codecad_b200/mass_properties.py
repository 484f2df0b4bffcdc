"""Volume / centroid / inertia tensor — same signature and result type as the
reference's /root/reference/codecad/mass_properties.py:30-229.  The per-block job loop
(:69-159: one launch, three blocking reads and a Python generator per 64^3 block) is
replaced by cc_mass_properties: every level is one batched launch over all of its blocks,
hit lists and the float64 corner chain stay on the device, and only ten float64 integrals
come back (summed over ranks with an NCCL all-reduce when sharded).
"""
import collections
import ctypes
import functools

import numpy as np

from . import _lib
from .geometry import Vector, as_vector
from .nodes import make_program_buffer
from .subdivision import _levels, calculate_block_sizes


class MassProperties(collections.namedtuple("MassProperties", "volume centroid inertia_tensor")):
    """Volume, centroid and inertia tensor (referenced to the centroid, not the origin)."""

    __slots__ = ()


STAT_NAMES = ("launches", "cells", "blocks", "levels", "dealt_blocks", "devices", "cells_busiest_device",
              "cells_idlest_device")


def mass_limbs(program, box_a, resolution, block_sizes, rank=0, world=1):
    """This rank's share of the ten integrals as the library's exact accumulator: (limbs int64[40],
    exponents int32[10], stats dict).  Limbs of different ranks add up exactly (integers);
    limbs_to_integrals() converts the total."""
    limbs = (ctypes.c_int64 * 40)()
    exps = (ctypes.c_int32 * 10)()
    stats = (ctypes.c_uint64 * 8)()
    a = (ctypes.c_double * 3)(float(box_a[0]), float(box_a[1]), float(box_a[2]))
    _lib.check(_lib.lib().cc_mass_properties_exact(program.handle, a, float(resolution), _levels(block_sizes),
                                                   len(block_sizes), int(rank), int(world), limbs, exps, stats))
    return (np.array(limbs[:], dtype=np.int64), np.array(exps[:], dtype=np.int32),
            dict(zip(STAT_NAMES, (int(v) for v in stats))))


def assembly_limbs(programs, box_a, resolution, block_sizes, rank=0, world=1):
    """The parts of an assembly and the overlaps of every pair of them in one hierarchy pass
    (cc_assembly_mass_properties_exact, DESIGN.md 4.11): this rank's share as exact accumulators, (limbs
    int64[sets][40], exponents int32[10], stats dict).  Row k < n is programs[k], bit for bit what
    mass_limbs(programs[k], ...) returns; the pairs {a < b} follow in lexicographic order (pair_index)."""
    n = len(programs)
    sets = n + n * (n - 1) // 2
    handles = (ctypes.c_void_p * max(n, 1))(*[p.handle if p is not None else None for p in programs])
    limbs = (ctypes.c_int64 * (40 * max(sets, 1)))()
    exps = (ctypes.c_int32 * 10)()
    stats = (ctypes.c_uint64 * 8)()
    a = (ctypes.c_double * 3)(float(box_a[0]), float(box_a[1]), float(box_a[2]))
    _lib.check(_lib.lib().cc_assembly_mass_properties_exact(handles, n, a, float(resolution), _levels(block_sizes),
                                                            len(block_sizes), int(rank), int(world), limbs, exps, stats))
    return (np.array(limbs[:40 * sets], dtype=np.int64).reshape(sets, 40), np.array(exps[:], dtype=np.int32),
            dict(zip(STAT_NAMES, (int(v) for v in stats))))


def pair_index(n, a, b):
    """Row of the pair {a, b} (a != b) among the sets of an assembly of n parts."""
    a, b = min(a, b), max(a, b)
    return n + a * n - a * (a + 1) // 2 + (b - a - 1)


def limbs_to_integrals(limbs, exponents):
    """Exact accumulator -> the ten float64 integrals (one rounding each)."""
    l = (ctypes.c_int64 * 40)(*[int(v) for v in limbs])
    e = (ctypes.c_int32 * 10)(*[int(v) for v in exponents])
    out = (ctypes.c_double * 10)()
    _lib.check(_lib.load().cc_mass_limbs_to_integrals(l, e, out))
    return np.array(out[:], dtype=np.float64)


def mass_integrals(program, box_a, resolution, block_sizes, rank=0, world=1):
    """The ten integrals (one,x,y,z,xx,yy,zz,xy,xz,yz) over this rank's share, + stats
    (launches, cells, blocks, levels)."""
    limbs, exps, stats = mass_limbs(program, box_a, resolution, block_sizes, rank, world)
    return limbs_to_integrals(limbs, exps), tuple(stats[k] for k in STAT_NAMES[:4])


def finish(integrals):
    """mass_properties.py:179-229: integrals -> MassProperties."""
    (integral_one, integral_x, integral_y, integral_z, integral_xx, integral_yy, integral_zz,
     integral_xy, integral_xz, integral_yz) = (float(v) for v in integrals)

    volume = integral_one
    if volume == 0:
        return MassProperties(0, Vector.splat(0), np.zeros((3, 3)))
    centroid = Vector(integral_x, integral_y, integral_z) / integral_one

    sxx = integral_xx - 2 * centroid.x * integral_x + centroid.x * centroid.x * integral_one
    syy = integral_yy - 2 * centroid.y * integral_y + centroid.y * centroid.y * integral_one
    szz = integral_zz - 2 * centroid.z * integral_z + centroid.z * centroid.z * integral_one
    sxy = integral_xy - centroid.x * integral_y - centroid.y * integral_x + centroid.x * centroid.y * integral_one
    sxz = integral_xz - centroid.x * integral_z - centroid.z * integral_x + centroid.x * centroid.z * integral_one
    syz = integral_yz - centroid.y * integral_z - centroid.z * integral_y + centroid.y * centroid.z * integral_one
    I_xx, I_yy, I_zz = syy + szz, sxx + szz, sxx + syy
    I_xy, I_xz, I_yz = -sxy, -sxz, -syz
    inertia_tensor = np.array([[I_xx, I_xy, I_xz], [I_xy, I_yy, I_yz], [I_xz, I_yz, I_zz]])
    return MassProperties(volume, centroid, inertia_tensor)


def mass_properties(shape, resolution, grid_size=None, group=None, stats=None):
    """mass_properties.py:30.  With `group` (a torch.distributed process group, or True
    for the default group) the hierarchy is sharded over its ranks and the exact accumulator
    of the ten integrals is all-reduced (40 int64): every rank returns the same result, and it
    is bit-identical to the unsharded one.  One process that drives several GPUs
    (_lib.init_devices / CODECAD_B200_DEVICES) shards inside the library with no argument here.
    `stats` (a dict) receives this rank's counters."""
    if grid_size is None:
        grid_size = 64

    assert shape.dimension() == 3, "2D objects are not supported yet"
    assert resolution > 0, "Non-positive resolution makes no sense"
    assert grid_size > 1, "Grid needs to be at least 2x2x2"
    assert grid_size ** 5 <= 2 ** 32, "Centroid coordinate sums would overflow"

    program_buffer = make_program_buffer(shape)
    bb = shape.bounding_box()
    box_a, box_b = as_vector(bb[0]), as_vector(bb[1])
    block_sizes = calculate_block_sizes((box_a, box_b), 3, resolution, grid_size, overlap=False)

    rank, world = 0, 1
    if group is not None:
        import torch.distributed as dist
        pg = None if group is True else group
        rank, world = dist.get_rank(pg), dist.get_world_size(pg)

    limbs, exps, st = mass_limbs(program_buffer, box_a, resolution, block_sizes, rank, world)
    if stats is not None:
        stats.update(st)
    if world > 1:
        limbs = allreduce_limbs(limbs, None if group is True else group)
    return finish(limbs_to_integrals(limbs, exps))


class AssemblyMassProperties(collections.namedtuple("AssemblyMassProperties", "parts interference")):
    """`parts`: a MassProperties per shape, in the order given; `interference`: {(i, j): MassProperties} of the
    overlap of shapes i < j, for the pairs whose overlap has a non-zero volume."""

    __slots__ = ()


def assembly_mass_properties(shapes, resolution, grid_size=None, group=None, stats=None):
    """mass_properties() of every shape of an assembly, and of the overlap of every pair of them (the
    interference check), in one hierarchy pass over the union of the shapes' bounding boxes.  Part k is
    exactly mass_properties() of shapes[k] on that box.  `group` and `stats` as for mass_properties()."""
    if grid_size is None:
        grid_size = 64
    shapes = list(shapes)
    assert 1 <= len(shapes) <= 32, "an assembly has 1 to 32 parts"
    assert all(s.dimension() == 3 for s in shapes), "2D objects are not supported yet"
    assert resolution > 0, "Non-positive resolution makes no sense"
    assert grid_size > 1, "Grid needs to be at least 2x2x2"
    assert grid_size ** 5 <= 2 ** 32, "Centroid coordinate sums would overflow"

    programs = [make_program_buffer(s) for s in shapes]
    boxes = [s.bounding_box() for s in shapes]
    box_a = functools.reduce(Vector.min, (as_vector(b[0]) for b in boxes))
    box_b = functools.reduce(Vector.max, (as_vector(b[1]) for b in boxes))
    block_sizes = calculate_block_sizes((box_a, box_b), 3, resolution, grid_size, overlap=False)

    rank, world = 0, 1
    if group is not None:
        import torch.distributed as dist
        pg = None if group is True else group
        rank, world = dist.get_rank(pg), dist.get_world_size(pg)

    limbs, exps, st = assembly_limbs(programs, box_a, resolution, block_sizes, rank, world)
    if stats is not None:
        stats.update(st)
    if world > 1:
        limbs = allreduce_limbs(limbs, None if group is True else group)
    n = len(shapes)
    parts = [finish(limbs_to_integrals(limbs[k], exps)) for k in range(n)]
    interference = {}
    for a in range(n):
        for b in range(a + 1, n):
            mp = finish(limbs_to_integrals(limbs[pair_index(n, a, b)], exps))
            if mp.volume != 0:
                interference[(a, b)] = mp
    return AssemblyMassProperties(parts, interference)


def allreduce_limbs(limbs, group=None):
    """Sum the exact accumulators (40 int64) over the ranks — the only data that crosses NVLink on
    this path.  Integer sums are exact and order-independent, so every rank converts the same total.
    NCCL needs the tensor on the GPU; gloo (CPU tests) does not."""
    import torch
    import torch.distributed as dist
    t = torch.from_numpy(np.ascontiguousarray(limbs, dtype=np.int64))
    if dist.get_backend(group) == "nccl":
        t = t.cuda()
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy()


def allreduce_integrals(integrals, group=None):
    """Sum the ten float64 partial integrals over the ranks (the only data that crosses
    NVLink on this path).  NCCL needs the tensor on the GPU; gloo (CPU tests) does not."""
    import torch
    import torch.distributed as dist
    t = torch.from_numpy(np.ascontiguousarray(integrals, dtype=np.float64))
    if dist.get_backend(group) == "nccl":
        t = t.cuda()
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy()
