"""echo_b200_build_packs on the B200: every pack's QBVH and light tree equal the host mirror's byte for byte (fed with the restated
placement rows of pack_build_lib.py), and a scene built with PreparedScene(build_packs_on_device=True) renders and traces exactly as one
given the standalone call's arrays."""
import numpy as np
import pytest

from echorenderer_b200 import PreparedScene, _native, build_packs_device, host, scenes, structs
from tests import oracle_lib
from tests import pack_build_lib as lib_expected

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bench_instanced():
    return host.prepare(scenes.instanced_scene(grid=48))


@pytest.fixture(scope="module")
def many_packs():
    return host.prepare(scenes.many_packs_scene(pack_count=520, seed=11))


def check_device_build(prepared):
    expected, _ = lib_expected.expected_packs(prepared)
    built = build_packs_device(prepared)
    lib_expected.assert_same_packs(built.packs, built.nodes, built.light_nodes, built.emitter_tokens, built.emitter_bitpaths, built.power, expected)
    return built


def test_nested_scene_same_bytes():
    check_device_build(host.prepare(scenes.instanced_scene(grid=4, rings=12, segments=12)))


def test_bench_instanced_scene_same_bytes(bench_instanced):
    assert len(bench_instanced.instances) >= 2304
    check_device_build(bench_instanced)


def test_many_packs_same_bytes(many_packs):
    assert len(many_packs.packs) >= 500
    check_device_build(many_packs)
    stats = _native.last_pack_build()
    assert stats["rounds"] == 4 and stats["rebuilt_packs"] == 0


def test_refusals():
    prepared = host.prepare(scenes.instanced_scene(grid=3, rings=8, segments=8))
    prepared.packs = prepared.packs.copy()
    prepared.packs[1]["triangleCount"], prepared.packs[1]["sphereCount"] = 1, 0
    with pytest.raises(_native.EchoNativeError) as error:
        build_packs_device(prepared)
    assert error.value.status == _native.ERR_INVALID


def test_flat_builds_refuse_packs():
    prepared = host.prepare(scenes.instanced_scene(grid=3, rings=8, segments=8))
    with pytest.raises(ValueError, match="build_packs_on_device"):
        PreparedScene(prepared, build_tree_on_device=True)
    with pytest.raises(_native.EchoNativeError):
        PreparedScene(prepared, build_light_tree_on_device=True)


def arrays_of(prepared, built):
    """`prepared` with the standalone call's arrays in place of host.prepare's."""
    result = host.PreparedArrays.__new__(host.PreparedArrays)
    result.__dict__.update(prepared.__dict__)
    result.packs, result.nodes, result.max_depth = built.packs, built.nodes, built.max_depth
    result.light_nodes, result.emitter_tokens, result.emitter_bitpaths = built.light_nodes, built.emitter_tokens, built.emitter_bitpaths
    return result


@pytest.mark.parametrize("description", ["instanced", "many_packs"])
def test_rendering_matches_the_standalone_arrays(description):
    prepared = host.prepare(scenes.instanced_scene(grid=4, rings=12, segments=12) if description == "instanced" else scenes.many_packs_scene(pack_count=60, seed=4))
    built = build_packs_device(prepared)
    given = arrays_of(prepared, built)

    with PreparedScene(prepared, build_packs_on_device=True) as on_device, PreparedScene(given) as standalone:
        assert on_device.built_packs == (len(built.nodes), len(built.light_nodes), len(built.emitter_tokens), pytest.approx(built.power, abs=0))

        params = structs.render_params(64, 64, 16, extend=4, bounce_limit=8)
        tiles = scenes.tile_grid(64, 64, 16)
        image, stats = on_device.render_tiles(params, tiles)
        expected, expected_stats = standalone.render_tiles(params, tiles)
        assert image.tobytes() == expected.tobytes()
        assert stats.tobytes() == expected_stats.tobytes()

        rays = scenes.random_rays(prepared.bounds, 50000, seed=17)
        hits, layers = on_device.trace_hierarchy(rays)
        expected_hits, expected_layers = standalone.trace_hierarchy(rays)
        assert hits.tobytes() == expected_hits.tobytes() and layers.tobytes() == expected_layers.tobytes()
        shadow = scenes.random_rays(prepared.bounds, 50000, seed=18, occlusion=True)
        assert np.array_equal(on_device.occlude_hierarchy(shadow), standalone.occlude_hierarchy(shadow))

        # per-sample radiance against the oracle on the same arrays (test_gpu_instancing.py's check)
        oracle = oracle_lib.OracleScene(given)
        pixels = np.stack(np.meshgrid(np.arange(0, 64, 7), np.arange(0, 64, 9)), axis=-1).reshape(-1, 2).astype(np.int32)
        index = np.arange(len(pixels), dtype=np.uint32) % 4
        radiance = on_device.evaluate_samples(params, pixels, index)
        reference = oracle.evaluate_samples(params, pixels, index)
        assert np.allclose(radiance, reference, rtol=1e-4, atol=1e-5)
