"""Callers of the hot path that the reference keeps under codecad/rendering and that were widened
into (SURVEY.md 8(f)): mesh export (rank 1), and the other consumers of evaluate() / grid_eval
(rank 4): ray-cast and bitmap pictures, 2-D boundary polygons, the slice viewer's field.  The rest of the reference's
rendering package (matplotlib viewers, SVG / BOM writers, CLI) is host-side Python and stays there."""
from .mesh import triangular_mesh, mesh_arrays, indexed_mesh, indexed_mesh_blocks  # noqa: F401
from .stl_renderer import render_stl, write_binary_stl  # noqa: F401
from .mesh_files import render_3mf, write_3mf, write_ply  # noqa: F401
from . import bitmap, image, matplotlib_slice, polygon2d, ray_caster  # noqa: F401
