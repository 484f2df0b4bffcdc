"""The generated source of the column brick kernel (DESIGN.md 4.10): its per-cell body defers the range checks of its
ops to one vote per warp only when every micro-op in it is pure arithmetic, and no other unit defers them."""
import re

import pytest

from codecad_b200 import _lib

SINK_PARTS, SINK_COLUMNS, SINK_TILES = 7, 8, (9, 10, 11)
CALLS = re.compile(r"\bcc_(?:extrusion|circle|rectangle|sphere)_n\((.*?)\);")


def _deferred(text):
    return [c for c in CALLS.findall(text) if c.endswith(", range")]


def _voting(text):
    return [c for c in CALLS.findall(text) if not c.endswith(", range")]


def _per_cell_body(src):
    body = src[src.index("struct SceneEval {"):]
    return body[:body.index("\n};\n")]


def test_planetary_columns_unit_defers(scenes):
    src = _lib.specialize_source(scenes["cfg_planetary"].words, 2, sink_mask=1 << SINK_COLUMNS)
    body = _per_cell_body(src)
    assert "static constexpr bool deferred = CC_DEFER_CHECKS != 0;" in src
    assert len(_deferred(body)) >= 30 and not _voting(body)
    assert "cc_brick_col_ref cr;" in body
    # the full walk keeps its votes, and is one out-of-line function for the fallback and cc_jit_columns_full
    assert not _deferred(src[:src.index("struct SceneEval {")])
    assert src.count("__noinline__ SceneVals cc_full_walk(") == 1
    assert "SceneFullCall e{" in src[src.index("cc_jit_columns_full"):]


@pytest.mark.parametrize("name", ["cfg_airfoil", "col_hole_grid", "col_bolt_circle", "col_crossed_extrusions",
                                  "col_revolved_and_extruded"])
def test_a_body_with_other_ops_keeps_its_votes(scenes, name):
    """repetitions, circular repetitions, regular polygons, revolutions in the per-cell body: no deferral"""
    src = _lib.specialize_source(scenes[name].words, 2, sink_mask=1 << SINK_COLUMNS)
    body = _per_cell_body(src)
    assert "static constexpr bool deferred = false;" in src
    assert _voting(body) and not _deferred(src)


@pytest.mark.parametrize("name", ["cfg_planetary", "cfg_airfoil", "col_assembly", "colr_05"])
def test_tile_and_parts_units_do_not_defer(scenes, name):
    words = scenes[name].words
    for sink in SINK_TILES + (SINK_PARTS,):
        try:
            src = _lib.specialize_source(words, 2, sink_mask=1 << sink)
        except _lib.CodecadB200Error:
            continue        # (no parts: no parts unit)
        assert not _deferred(src) and "cc_brick_col_ref" not in src and "cc_full_walk" not in src
