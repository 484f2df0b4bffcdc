"""codecad_b200 — B200-native implementation of codecad's data-parallel SDF hot path.

Drop-in for the reference's OpenCL layer and the three modules built on it:

    reference module                     replaced by
    codecad/cl_util/                     codecad_b200.cl_util   (ctypes -> libcodecad_b200.so)
    codecad/grid_eval.py + .cl           codecad_b200.grid_eval
    codecad/subdivision.py + .cl         codecad_b200.subdivision
    codecad/mass_properties.py + .cl     codecad_b200.mass_properties

The shape / node API of the reference (codecad.shapes, codecad.nodes) is used unchanged:
`codecad_b200.dropin.install()` makes an unmodified reference checkout import these
modules in place of its own (see INTEGRATION.md).  Everything that computes runs in the
CUDA library; importing this package does not touch the GPU, the first call does.
"""
from . import opcodes  # noqa: F401
from .geometry import BoundingBox, Vector  # noqa: F401
from .mass_properties import AssemblyMassProperties, MassProperties, assembly_mass_properties, mass_properties  # noqa: F401
from .subdivision import calculate_block_sizes, subdivision  # noqa: F401
from .grid_eval import evaluate_points, grid_eval, grid_eval_pymcubes  # noqa: F401
from .nodes import CompiledScene, make_program, make_program_buffer  # noqa: F401

__all__ = [
    "BoundingBox", "Vector", "MassProperties", "mass_properties", "AssemblyMassProperties", "assembly_mass_properties",
    "calculate_block_sizes",
    "subdivision", "grid_eval", "grid_eval_pymcubes", "CompiledScene", "make_program",
    "make_program_buffer",
]
