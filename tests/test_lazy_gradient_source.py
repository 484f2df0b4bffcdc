"""The generated source of the column brick kernel's lazy gradient (DESIGN.md 4.10): which per-cell bodies take the
sweep and the replay, and that every leaf the sweep can leave at the root has a replay case."""
import re

import pytest

from codecad_b200 import _lib

SINK_PARTS, SINK_COLUMNS, SINK_TILES = 7, 8, (9, 10, 11)
EAGER_TILE = "Val (&L)[G], unsigned &range) const { loop(gx, gy, gz, L, range); }"


def _struct(src, name):
    body = src[src.index("struct " + name + " {"):]
    return body[:body.index("\n};\n")]


@pytest.mark.parametrize("name", ["cfg_planetary", "x_gear3d", "col_assembly", "colr_00"])
def test_deferring_bodies_are_lazy(scenes, name):
    src = _lib.specialize_source(scenes[name].words, 2, sink_mask=1 << SINK_COLUMNS)
    assert "#if CC_LAZY_GRADIENT && CC_DEFER_CHECKS" in _struct(src, "SceneTile") and EAGER_TILE not in src
    sweep = _struct(src, "SceneSweep")
    assert "cc_extrusion_dist(" in sweep and not re.search(r"\bcc_(extrusion|circle|rectangle|sphere)_n\(", sweep)
    assert "Lw" not in _struct(src, "SceneEval")
    # every id the sweep assigns has its case, and every case is an id the sweep assigns
    ids = {int(k) for k in re.findall(r"= vbc<V>\((\d+)\.0f\)", sweep)}
    replay = src[src.index("cc_replay_leaf("):]
    cases = {int(k) for k in re.findall(r"\n\s*case (\d+): \{", replay[:replay.index("\n}\n")])}
    assert ids and ids == cases == set(range(len(cases)))


@pytest.mark.parametrize("name", ["cfg_airfoil", "col_hole_grid", "col_bolt_circle", "col_crossed_extrusions",
                                  "col_revolved_and_extruded", "colr_05"])
def test_other_bodies_stay_eager(scenes, name):
    src = _lib.specialize_source(scenes[name].words, 2, sink_mask=1 << SINK_COLUMNS)
    assert "SceneSweep" not in src and "cc_replay_leaf" not in src and "CC_LAZY_GRADIENT" not in src
    assert EAGER_TILE in _struct(src, "SceneTile")


@pytest.mark.parametrize("name", ["cfg_planetary", "col_assembly", "colr_00"])
def test_tile_and_parts_units_are_not_lazy(scenes, name):
    words = scenes[name].words
    for sink in SINK_TILES + (SINK_PARTS,):
        try:
            src = _lib.specialize_source(words, 2, sink_mask=1 << sink)
        except _lib.CodecadB200Error:
            continue        # (no parts: no parts unit)
        assert "SceneSweep" not in src and "cc_replay_leaf" not in src and "_dist(" not in src
