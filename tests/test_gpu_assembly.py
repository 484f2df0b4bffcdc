"""Mass properties of an assembly's parts and of every pair's overlap in one hierarchy pass (DESIGN.md 4.11,
cc_assembly_mass_properties_exact): every part is bit for bit the standalone call on the same box and plan, the pairs
are bit for bit the parts where the contract says so and agree with the CPU restatement (tests/assembly_oracle.py)
elsewhere, shares add up exactly, and a level cut into several launches changes nothing."""
import importlib

import numpy as np
import pytest

import programs as P
from assembly_oracle import assembly_mass_properties as oracle_assembly
from exact_mass import buffers as _buffers, integrals as _integrals, lipschitz_parts, part_box as _part_box, plan as _plan

pytestmark = pytest.mark.gpu

mpm = importlib.import_module("codecad_b200.mass_properties")


@pytest.fixture(scope="module")
def cb():
    import codecad_b200
    from codecad_b200 import _lib
    _lib.init(0)
    return codecad_b200


@pytest.fixture(params=[0, 2], ids=["interpreter", "specialised"])
def jit(cb, request):
    """the standalone calls' tiers: the interpreter only, or the specialised kernels (built at first use, waited for)"""
    from codecad_b200 import _lib
    old = _lib.check(_lib.lib().cc_set_jit_mode(request.param))
    yield request.param
    _lib.check(_lib.lib().cc_set_jit_mode(old))


def _union_box(scenes_list):
    a = tuple(min(s.box_a[i] for s in scenes_list) for i in range(3))
    b = tuple(max(s.box_b[i] for s in scenes_list) for i in range(3))
    return a, b


# ---- groups of parts -------------------------------------------------------------------------------------------------

FIXTURE_GROUPS = {
    "solids": (["dsdf3d_box", "dsdf3d_sphere", "dsdf3d_torus", "mp_cylinder", "mp_drunk_box"], 0.05, 16),
    "large": (["cfg_csg_example", "cfg_airfoil", "dsdf3d_torus", "mp_cylinder", "mp_drunk_box"], 0.5, 16),
}


def _cloud(seed, n, spread=2.5, size=1.5):
    rng = np.random.default_rng(seed)
    return P.primitive_cloud(rng, n, (0.0, 0.0, 0.0), spread, size)


def _program_groups():
    ties = P.leaves(P.near_tie_assembly(0.0, n=3, gap=0.25, length=6.0))  # (quads 0.3 wide: neighbours overlap)
    cloud = _cloud(7, 8)
    return {
        "near_tie_quads": ([P.program(p) for p in ties], _part_box(ties), 0.05, 16),
        "primitive_cloud": ([P.program(p) for p in cloud], _part_box(cloud), 0.05, 16),
    }


def _group(scenes, name):
    if name in FIXTURE_GROUPS:
        names, res, grid = FIXTURE_GROUPS[name]
        ss = [scenes[n] for n in names]
        box_a, box_b = _union_box(ss)
        return [s.words for s in ss], box_a, box_b, res, grid
    words, (box_a, box_b), res, grid = _program_groups()[name]
    return words, box_a, box_b, res, grid


ALL_GROUPS = sorted(FIXTURE_GROUPS) + ["near_tie_quads", "primitive_cloud"]


@pytest.mark.parametrize("group", ALL_GROUPS)
def test_parts_are_bit_exact(cb, scenes, jit, group):
    words, box_a, box_b, res, grid = _group(scenes, group)
    progs = _buffers(words)
    a, _, plan = _plan(box_a, box_b, res, grid)
    limbs, exps, st = mpm.assembly_limbs(progs, a, res, plan)
    n = len(progs)
    assert limbs.shape == (n + n * (n - 1) // 2, 40)
    for k, p in enumerate(progs):
        want, w_exps, _ = mpm.mass_limbs(p, a, res, plan)
        assert np.array_equal(exps, w_exps)
        assert np.array_equal(limbs[k], want), "part %d differs from its standalone call" % k
        assert want[:4].any(), "part %d is empty: the group does not test it" % k  # (limbs 0..3: the volume)
    # the groups overlap around the origin: some pair has a volume
    assert any(limbs[n:, :4].any(axis=1))


def test_pairs_are_bit_exact_where_the_contract_says_so(cb, scenes):
    A, B = scenes["mp_drunk_box"].words, scenes["dsdf3d_sphere"].words
    box_a, box_b = _union_box([scenes["mp_drunk_box"], scenes["dsdf3d_sphere"]])
    a, _, plan = _plan(box_a, box_b, 0.05, 16)
    pa, pb = _buffers([A, B])
    single, exps, _ = mpm.assembly_limbs([pa], a, 0.05, plan)
    want, w_exps, _ = mpm.mass_limbs(pa, a, 0.05, plan)
    assert single.shape == (1, 40) and np.array_equal(single[0], want) and np.array_equal(exps, w_exps)
    twice, _, _ = mpm.assembly_limbs([pa, pa], a, 0.05, plan)
    assert np.array_equal(twice[0], want) and np.array_equal(twice[1], want) and np.array_equal(twice[2], want)
    aba, _, _ = mpm.assembly_limbs([pa, pb, pa], a, 0.05, plan)
    n = 3
    assert np.array_equal(aba[mpm.pair_index(n, 0, 2)], want)
    assert np.array_equal(aba[mpm.pair_index(n, 0, 1)], aba[mpm.pair_index(n, 1, 2)])
    assert aba[mpm.pair_index(n, 0, 1)].any()


ORACLE_GROUPS = [(["dsdf3d_box", "dsdf3d_sphere", "mp_drunk_box"], 0.05, 8), (["dsdf3d_torus", "mp_cylinder", "dsdf3d_sphere"], 0.2, 8)]


@pytest.mark.parametrize("names,res,grid", ORACLE_GROUPS)
def test_pairs_match_the_restatement(cb, scenes, names, res, grid):
    ss = [scenes[n] for n in names]
    box_a, box_b = _union_box(ss)
    want = oracle_assembly([s.words for s in ss], box_a, box_b, res, grid)
    a, _, plan = _plan(box_a, box_b, res, grid)
    limbs, exps, _ = mpm.assembly_limbs(_buffers([s.words for s in ss]), a, res, plan)
    got = _integrals(limbs, exps)
    assert got.shape == want.shape
    # the bar of the mass tests between the exact accumulator and Kahan sums, relative to each integral's scale: the
    # largest volume times the box's largest coordinate to the integral's order (moments about the origin of parts
    # centred there cancel to rounding noise)
    m = max(abs(v) for v in box_a + box_b)
    scale = want[:, 0].max() * np.array([1.0, m, m, m] + [m * m] * 6)
    assert np.all(np.abs(got - want) <= 1e-12 * scale)
    assert (want[len(ss):, 0] > 0).any()


@pytest.mark.parametrize("kind", ["two", "three"])
def test_inclusion_exclusion(cb, kind):
    parts = lipschitz_parts(kind)
    box_a, box_b = _part_box(parts)
    res = 0.03
    a, _, plan = _plan(box_a, box_b, res, 16)
    progs = _buffers([P.program(p) for p in parts])
    limbs, exps, _ = mpm.assembly_limbs(progs, a, res, plan)
    n = len(parts)
    sets = _integrals(limbs, exps)
    union, u_exps, _ = mpm.mass_limbs(_buffers([P.program(P.balanced(parts))])[0], a, res, plan)
    u = mpm.limbs_to_integrals(union, u_exps)
    pairs = [mpm.pair_index(n, i, j) for i in range(n) for j in range(i + 1, n)]
    combined = sets[:n].sum(axis=0) - sets[pairs].sum(axis=0)
    assert sets[mpm.pair_index(n, 0, 1)][0] > 0
    if kind == "three":
        assert sets[mpm.pair_index(n, 1, 2)][0] == 0 and sets[mpm.pair_index(n, 0, 2)][0] > 0
    assert combined[0] == pytest.approx(u[0], rel=1e-12)
    m = max(abs(v) for v in box_a + box_b)
    assert np.allclose(combined[1:4], u[1:4], rtol=1e-12, atol=1e-12 * u[0] * m)
    # the second moments (the inertia): the same bar, one more coordinate
    assert np.allclose(combined[4:], u[4:], rtol=1e-12, atol=1e-12 * u[0] * m * m)


def test_disjoint_parts(cb):
    parts = [P.Part.placed(P.Part.box(1.0, 1.5, 1.0), c) for c in ((-3.0, 0.0, 0.0), (3.0, 0.5, 0.0))]
    parts.append(P.Part.placed(P.Part.cylinder(1.0, 1.0), (0.0, 4.0, 1.0)))
    box_a, box_b = (-4.5, -2.0, -1.5), (4.5, 6.0, 2.5)
    res = 0.04
    a, _, plan = _plan(box_a, box_b, res, 16)
    limbs, exps, _ = mpm.assembly_limbs(_buffers([P.program(p) for p in parts]), a, res, plan)
    assert not limbs[3:].any(), "parts apart overlap nowhere"
    union, u_exps, _ = mpm.mass_limbs(_buffers([P.program(P.balanced(parts))])[0], a, res, plan)
    u = mpm.limbs_to_integrals(union, u_exps)
    total = _integrals(limbs[:3], exps).sum(axis=0)
    assert total[0] == pytest.approx(u[0], rel=1e-12)
    assert np.allclose(total[1:4], u[1:4], rtol=1e-12, atol=1e-12 * u[0] * 6.0)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_shares_add_up_exactly(cb, scenes, world):
    words, box_a, box_b, res, grid = _group(scenes, "solids")
    progs = _buffers(words)
    a, _, plan = _plan(box_a, box_b, res, grid)
    whole, exps, _ = mpm.assembly_limbs(progs, a, res, plan)
    total = np.zeros_like(whole)
    for rank in range(world):
        limbs, e, _ = mpm.assembly_limbs(progs, a, res, plan, rank, world)
        assert np.array_equal(e, exps)
        total += limbs
    assert np.array_equal(total, whole)


def test_a_level_cut_into_several_launches(cb):
    """32 parts: 528 sets of counters a block, so the counter budget cuts a level of small blocks into several launches;
    every part is its standalone call and every pair the pair of a two-part group, whose levels are not cut."""
    parts = _cloud(11, 32, spread=3.0, size=1.2)
    box_a, box_b = _part_box(parts)
    res, grid = 0.03, 4
    a, _, plan = _plan(box_a, box_b, res, grid)
    progs = _buffers([P.program(p) for p in parts])
    limbs, exps, st = mpm.assembly_limbs(progs, a, res, plan)
    levels_run = st["levels"]
    assert st["launches"] > levels_run, "no level was cut: %s" % st
    for k, p in enumerate(progs):
        assert np.array_equal(limbs[k], mpm.mass_limbs(p, a, res, plan)[0]), k
    n = len(parts)
    overlapping = [(i, j) for i in range(n) for j in range(i + 1, n) if limbs[mpm.pair_index(n, i, j)].any()]
    assert overlapping
    for i, j in overlapping[:4]:
        two, _, st2 = mpm.assembly_limbs([progs[i], progs[j]], a, res, plan)
        assert st2["launches"] <= st2["levels"]
        assert np.array_equal(two[2], limbs[mpm.pair_index(n, i, j)]), (i, j)


def test_errors(cb, scenes):
    from codecad_b200 import _lib
    s = scenes["mp_sphere"]
    a, _, plan = _plan(s.box_a, s.box_b, 0.1, 8)
    prog = s.compiled().program_buffer()
    for progs in ([], [prog] * 33, [prog, None]):
        with pytest.raises(_lib.CodecadB200Error):
            mpm.assembly_limbs(progs, a, 0.1, plan)


def test_shape_level_call(cb, scenes):
    names = ["dsdf3d_box", "mp_drunk_box", "dsdf3d_sphere", "dsdf3d_torus"]
    shapes = [scenes[n].compiled() for n in names]
    stats = {}
    got = cb.assembly_mass_properties(shapes, 0.1, 16, stats=stats)
    assert isinstance(got, cb.AssemblyMassProperties) and len(got.parts) == len(shapes) and stats["launches"] > 0
    box_a, box_b = _union_box([scenes[n] for n in names])
    a, _, plan = _plan(box_a, box_b, 0.1, 16)
    limbs, exps, _ = mpm.assembly_limbs([s.program_buffer() for s in shapes], a, 0.1, plan)
    n = len(shapes)
    for k in range(n):
        want = mpm.finish(mpm.limbs_to_integrals(limbs[k], exps))
        assert got.parts[k].volume == want.volume and tuple(got.parts[k].centroid) == tuple(want.centroid)
        assert np.array_equal(got.parts[k].inertia_tensor, want.inertia_tensor)
    pairs = {(i, j) for i in range(n) for j in range(i + 1, n) if limbs[mpm.pair_index(n, i, j)].any()}
    assert set(got.interference) == pairs and (0, 1) in pairs
    for (i, j), mp in got.interference.items():
        assert mp.volume == mpm.finish(mpm.limbs_to_integrals(limbs[mpm.pair_index(n, i, j)], exps)).volume
        assert 0 < mp.volume <= min(got.parts[i].volume, got.parts[j].volume) * (1 + 1e-12)
