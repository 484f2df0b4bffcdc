"""The generated source of the column brick kernel (DESIGN.md 4.10): the columns unit walks runs of bricks and takes
each brick's part mask from its run, and the parts and tile units keep one brick or tile per CTA."""
import pytest

from codecad_b200 import _lib

SINK_PARTS, SINK_COLUMNS, SINK_TILES = 7, 8, (9, 10, 11)


def _kernel(src, name):
    body = src[src.index(" " + name + "(const cc_eval_args a)"):]
    return body[:body.index("\n}\n")]


@pytest.mark.parametrize("name", ["cfg_planetary", "cfg_airfoil", "col_assembly"])
def test_columns_unit_walks_runs(scenes, name):
    src = _lib.specialize_source(scenes[name].words, 2, sink_mask=1 << SINK_COLUMNS)
    k = _kernel(src, "cc_jit_columns")
    assert "cc_kernel_body_brick_columns<PTS>(a, e);" in k
    assert "part_masks" not in k and "blockIdx" not in k       # (the body reads the run's masks)
    assert "a.part_masks[b]" in _kernel(src, "cc_jit_columns_full")


@pytest.mark.parametrize("name", ["cfg_planetary", "col_assembly"])
def test_parts_and_tile_units_keep_one_brick_per_cta(scenes, name):
    words = scenes[name].words
    src = _lib.specialize_source(words, 2, sink_mask=1 << SINK_PARTS)
    k = _kernel(src, "cc_jit_parts")
    assert "a.part_masks[blockIdx.x]" in k and "cc_kernel_body_bricks<PTS>(a, e);" in k
    for sink in SINK_TILES:
        src = _lib.specialize_source(words, 2, sink_mask=1 << sink)
        assert "cc_kernel_body<PTS, CC_SINK_" in src and "cc_kernel_body_brick_columns" not in src
