"""CPU test of the assembly restatement (tests/assembly_oracle.py) that the GPU tests of the assembly mass properties
compare against: one part is oracle.host.mass_properties to the bit, a part given twice overlaps itself exactly, and
parts apart do not overlap."""
import numpy as np

import programs as P
from assembly_oracle import assembly_mass_properties, pair_index
from oracle import host


def test_one_part_is_the_host_mass_properties(scenes):
    s = scenes["cfg_csg_example"]
    got = assembly_mass_properties([s.words], s.box_a, s.box_b, 1.0, 16)
    assert got.shape == (1, 10)
    vol, cen, inertia = host.mass_properties(s.words, s.box_a, s.box_b, 1.0, 16)
    g_vol, g_cen, g_inertia = host.finish_mass_properties(got[0])
    assert g_vol == vol and tuple(g_cen) == tuple(cen) and np.array_equal(g_inertia, inertia)


def test_a_part_twice_overlaps_itself(scenes):
    s = scenes["mp_drunk_box"]
    got = assembly_mass_properties([s.words, s.words], s.box_a, s.box_b, 0.1, 8)
    assert got.shape == (3, 10)
    assert np.array_equal(got[0], got[1]) and np.array_equal(got[pair_index(2, 0, 1)], got[0])
    assert got[0][0] > 0


def test_parts_apart_do_not_overlap():
    words = [P.program(P.Part.placed(P.Part.box(1.0, 1.5, 1.0), c)) for c in ((-3.0, 0.0, 0.0), (3.0, 0.5, 0.0), (0.0, 4.0, 1.0))]
    got = assembly_mass_properties(words, (-4.5, -2.0, -1.5), (4.5, 6.0, 2.5), 0.125, 8)
    assert got.shape == (6, 10)
    assert all(got[k][0] > 0 for k in range(3))
    assert not got[3:].any()
    # the boxes are 2 x 3 x 2 and the grid's cells resolve them: their volumes are near 12
    assert np.allclose(got[:3, 0], 12.0, rtol=0.1)
