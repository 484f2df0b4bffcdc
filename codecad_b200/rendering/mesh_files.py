"""Indexed mesh files: binary PLY and 3MF, written on the host from the welded mesh of
`indexed_mesh` (shared vertices, triangles as vertex indices, consistently oriented)."""
import zipfile

import numpy as np

from .mesh import indexed_mesh


def _indexed(vertices, triangles):
    v = np.ascontiguousarray(vertices, dtype="<f8").reshape(-1, 3)
    t = np.ascontiguousarray(triangles, dtype="<u4").reshape(-1, 3)
    if len(t) and int(t.max()) >= len(v):
        raise ValueError("triangle index out of range")
    return v, t


def write_ply(filename, vertices, triangles):
    """Binary little-endian PLY: float64 vertices, faces as a uint8 count and three uint32 indices."""
    v, t = _indexed(vertices, triangles)
    header = ("ply\nformat binary_little_endian 1.0\ncomment codecad_b200\n"
              "element vertex %d\nproperty double x\nproperty double y\nproperty double z\n"
              "element face %d\nproperty list uchar uint vertex_indices\nend_header\n" % (len(v), len(t)))
    faces = np.zeros(len(t), dtype=np.dtype([("n", "u1"), ("v", "<u4", 3)]))
    faces["n"] = 3
    faces["v"] = t
    with open(filename, "wb") as f:
        f.write(header.encode("ascii"))
        f.write(v.tobytes())
        f.write(faces.tobytes())
    return len(t)


_CONTENT_TYPES = (
    '<?xml version="1.0" encoding="UTF-8"?>\n'
    '<Types xmlns="http://schemas.openxmlformats.org/package/2006/content-types">'
    '<Default Extension="rels" ContentType="application/vnd.openxmlformats-package.relationships+xml"/>'
    '<Default Extension="model" ContentType="application/vnd.ms-package.3dmanufacturing-3dmodel+xml"/>'
    '</Types>\n')
_RELS = (
    '<?xml version="1.0" encoding="UTF-8"?>\n'
    '<Relationships xmlns="http://schemas.openxmlformats.org/package/2006/relationships">'
    '<Relationship Target="/3D/3dmodel.model" Id="rel0" '
    'Type="http://schemas.microsoft.com/3dmanufacturing/2013/01/3dmodel"/>'
    '</Relationships>\n')
MODEL_NS = "http://schemas.microsoft.com/3dmanufacturing/core/2015/02"


def write_3mf(filename, vertices, triangles):
    """3MF package (a zip: [Content_Types].xml, _rels/.rels, 3D/3dmodel.model) holding one mesh
    object in millimetres and one build item.  Coordinates are written as the shortest decimal that
    reads back as the same float64."""
    v, t = _indexed(vertices, triangles)
    parts = ['<?xml version="1.0" encoding="UTF-8"?>\n<model unit="millimeter" xml:lang="en-US" xmlns="%s">\n'
             '<resources>\n<object id="1" type="model">\n<mesh>\n<vertices>\n' % MODEL_NS]
    parts.extend('<vertex x="%r" y="%r" z="%r"/>\n' % (x, y, z) for x, y, z in v.tolist())
    parts.append('</vertices>\n<triangles>\n')
    parts.extend('<triangle v1="%d" v2="%d" v3="%d"/>\n' % (a, b, c) for a, b, c in t.tolist())
    parts.append('</triangles>\n</mesh>\n</object>\n</resources>\n<build>\n<item objectid="1"/>\n</build>\n</model>\n')
    with zipfile.ZipFile(filename, "w", compression=zipfile.ZIP_DEFLATED) as z:
        z.writestr("[Content_Types].xml", _CONTENT_TYPES)
        z.writestr("_rels/.rels", _RELS)
        z.writestr("3D/3dmodel.model", "".join(parts))
    return len(t)


def render_3mf(obj, filename):
    """The 3-D shape's welded mesh as a 3MF file; returns the number of triangles."""
    vertices, triangles, _, _ = indexed_mesh(obj)
    return write_3mf(filename, vertices, triangles)
