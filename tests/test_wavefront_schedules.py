"""The fixtures of the wavefront-schedule matrix (tests/schedule_lib.py) on the CPU: each lands on the traversal-stack class it is meant to
exercise, the hand-built chain trees are valid trees of their scene (the oracle answers every query and renders every sample through them
exactly as through the SweepBuilder's tree), the pack chain reaches TokenHierarchy.MaxLayer, and `schedule` always puts the switches back."""
import numpy as np
import pytest

from echorenderer_b200 import _native, host, scenes, structs
from tests import oracle_lib, schedule_lib


@pytest.fixture(scope="module")
def chains():
    swept = schedule_lib.chain_cornell()
    return swept, {per_node: schedule_lib.chain_qbvh(swept, per_node) for per_node in (1, 2)}


def test_stack_class_boundaries():
    """the device's rounding: a pack chain's entries go up to the smallest depth with 3 * depth + 1 >= entries, a plain scene's are 3 * depth + 1"""
    assert [schedule_lib.stack_class(e) for e in (1, 46, 47, 48, 49, 94, 95, 96, 97, 190, 191, 193)] == [48, 48, 96, 96, 96, 96, 192, 192, 192, 192, None, None]
    assert [schedule_lib.stack_class(3 * depth + 1) for depth in (15, 16, 31, 32, 63, 64)] == [48, 96, 96, 192, 192, None]


def test_entries_of_the_existing_fixtures(cornell, textured_small):
    assert schedule_lib.stack_entries(cornell) == 19
    assert schedule_lib.stack_entries(textured_small) == 34
    assert schedule_lib.stack_entries(host.prepare(scenes.instanced_scene(grid=4, rings=12, segments=14, nested=False))) == 35
    assert schedule_lib.stack_entries(host.prepare(scenes.instanced_scene(grid=4, rings=12, segments=14, nested=True))) == 51
    assert schedule_lib.stack_entries(host.prepare(scenes.instanced_scene())) == 60
    assert schedule_lib.stack_entries(host.prepare(scenes.many_packs_scene())) == 67


def test_every_fixture_lands_on_its_class(cornell, textured_small, chains):
    _, chain = chains
    plain = {48: cornell, 96: chain[2], 192: chain[1]}
    packs = {48: host.prepare(scenes.instanced_scene(grid=4, rings=12, segments=14, nested=False)),
             96: host.prepare(scenes.instanced_scene(grid=4, rings=12, segments=14, nested=True)), 192: schedule_lib.deep_pack_scene(5)}
    for expected, prepared in list(plain.items()) + list(packs.items()) + [(48, textured_small)]:
        assert schedule_lib.stack_class(schedule_lib.stack_entries(prepared)) == expected
    assert all(p.packs is None for p in plain.values()) and all(p.packs is not None for p in packs.values())
    assert textured_small.packs is None and textured_small.textures is not None  # INST without packs
    assert [schedule_lib.stack_class(schedule_lib.stack_entries(schedule_lib.deep_pack_scene(layers))) for layers in (3, 4)] == [96, 96]


def test_chain_trees_have_the_shape_they_claim(chains):
    swept, chain = chains
    count = len(swept.triangles) + len(swept.spheres)
    for per_node, prepared in chain.items():
        nodes = prepared.nodes
        tokens = nodes["token4"][nodes["token4"] != structs.TOKEN_EMPTY]
        kinds = structs.token_type(tokens)
        assert sorted(structs.token_index(tokens[kinds != structs.TOKEN_TYPE_NODE])) == list(range(count))  # every primitive exactly once
        assert list(structs.token_index(tokens[kinds == structs.TOKEN_TYPE_NODE])) == list(range(1, len(nodes)))  # one chain
        assert prepared.max_depth == len(nodes) + 1
        assert prepared.bound_radius == swept.bound_radius
        assert prepared.triangles is swept.triangles and prepared.light_nodes is swept.light_nodes
    assert len(chain[1].nodes) == count - 1 and len(chain[2].nodes) == count // 2


@pytest.mark.parametrize("per_node", [1, 2])
def test_chain_trees_answer_queries_like_the_swept_tree(chains, per_node):
    swept, chain = chains
    rays = scenes.random_rays(swept.bounds, 20_000, seed=29)
    shadow = scenes.random_rays(swept.bounds, 20_000, seed=31, occlusion=True)
    expected, through = oracle_lib.OracleScene(swept), oracle_lib.OracleScene(chain[per_node])
    hits = expected.trace(rays)
    assert (hits["token"] != structs.TOKEN_EMPTY).mean() > 0.3
    assert np.array_equal(through.trace(rays).view(np.uint32), hits.view(np.uint32))
    occluded = expected.occlude(shadow)
    assert 0.02 < occluded.mean() < 0.98
    assert np.array_equal(through.occlude(shadow), occluded)


@pytest.mark.parametrize("per_node", [1, 2])
def test_chain_trees_render_like_the_swept_tree(chains, per_node):
    """bit for bit with equal statistics rows, at 64 x 64, 4 spp and bounce limit 24; the chain only costs more node visits"""
    swept, chain = chains
    params = structs.render_params(64, 64, 16, extend=4, bounce_limit=24, seed=6)
    tiles = scenes.tile_grid(64, 64, 16)
    expected, expected_stats = oracle_lib.OracleScene(swept).render_tiles(params, tiles)
    image, stats = oracle_lib.OracleScene(chain[per_node]).render_tiles(params, tiles)
    assert expected[..., :3].mean() > 0.01
    assert np.array_equal(image.view(np.uint32), expected.view(np.uint32))
    for name in structs.STATS_FIELDS[:12]:
        assert int(stats[name][0]) == int(expected_stats[name][0]), name
    assert int(stats["nodeVisits"][0]) > int(expected_stats["nodeVisits"][0])


def test_deep_pack_scene_reaches_five_instance_layers():
    prepared = schedule_lib.deep_pack_scene(5)
    oracle = oracle_lib.OracleScene(prepared)
    hits, layers = oracle.trace_hierarchy(scenes.random_rays(prepared.bounds, 20_000, seed=37))
    hit = hits["token"] != structs.TOKEN_EMPTY
    assert layers["instanceCount"].max() == structs.MAX_INSTANCE_LAYERS
    assert set(np.unique(layers["instanceCount"][hit])) == {0, 1, 2, 3, 4, 5}
    image, _ = oracle.render_tiles(structs.render_params(32, 32, 16, extend=2, bounce_limit=12, seed=3), scenes.tile_grid(32, 32, 16))
    assert image[..., :3].mean() > 0.01


def test_schedule_restores_every_switch_when_its_body_raises():
    for name in schedule_lib.SCHEDULES:
        with pytest.raises(RuntimeError):
            with schedule_lib.schedule(name, 1 << 18):
                switches = schedule_lib.schedule_switches(name, 1 << 18)
                assert {option: _native.get_option(option) for option in switches} == switches
                raise RuntimeError("inside the schedule")
        assert {option: _native.get_option(option) for option in schedule_lib.DEFAULTS} == schedule_lib.DEFAULTS
    with pytest.raises(_native.EchoNativeError):
        _native.get_option("NO_SUCH_SWITCH")
    with pytest.raises(ValueError):
        schedule_lib.schedule_switches("no_such_schedule")
