"""The min / max form of cc_extrusion_dist (DESIGN.md 4.10) is exact only where a warp whose range test flags throws its
values away: the generated source must call it in the lazy gradient's sweep alone, and run the sweep only in a build
that defers the range checks to the warp's vote."""
import re

import pytest

from codecad_b200 import _lib

SINK_PARTS, SINK_COLUMNS, SINK_TILES = 7, 8, (9, 10, 11)


def _struct(src, name):
    body = src[src.index("struct " + name + " {"):]
    return body[:body.index("\n};\n")]


@pytest.mark.parametrize("name", ["cfg_planetary", "x_gear3d", "col_assembly", "colr_00", "cfg_airfoil", "col_hole_grid"])
def test_extrusion_dist_only_in_the_deferred_sweep(scenes, name):
    for sink in (SINK_COLUMNS,) + SINK_TILES + (SINK_PARTS,):
        try:
            src = _lib.specialize_source(scenes[name].words, 2, sink_mask=1 << sink)
        except _lib.CodecadB200Error:
            continue        # (no parts: no parts unit)
        calls = len(re.findall(r"\bcc_extrusion_dist\(", src))
        if "struct SceneSweep {" not in src:
            assert calls == 0, (name, sink)
            continue
        assert sink == SINK_COLUMNS and calls and calls == len(re.findall(r"\bcc_extrusion_dist\(", _struct(src, "SceneSweep")))
        tile = _struct(src, "SceneTile")
        guarded = tile[tile.index("#if CC_LAZY_GRADIENT && CC_DEFER_CHECKS\n"):tile.index("#else\n")]
        assert "SceneSweep{" in guarded and "SceneSweep" not in tile.replace(guarded, "")
        assert "static constexpr bool deferred = CC_DEFER_CHECKS != 0;" in tile
