"""The stratified sample sequence (ECHO_DISTRIBUTION_STRATIFIED) on the device: the sequence itself (debug op 103), every evaluator and render
entry point bit for bit against the oracle, epoch sharding, the variance it saves and its refusals."""
import numpy as np
import pytest

from echorenderer_b200 import EchoNativeError, PreparedScene, _native, host, scenes, structs
from tests import oracle_lib, stratified_oracle
from tests.test_gpu_render import relative_rmse, sample_grid
from tests.test_stratified import oracle_values

pytestmark = pytest.mark.gpu
STRATIFIED = structs.DISTRIBUTION_STRATIFIED


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


def device_stratified(seed, pixel, sample, extend, dimension, two_d):
    """debug op 103 over element pairs: (n, 2) values"""
    n = len(seed)
    a = np.stack([seed, pixel], axis=-1).astype(np.uint32).reshape(-1).view(np.float32)
    b = np.stack([sample, extend], axis=-1).astype(np.uint32).reshape(-1).view(np.float32)
    c = np.stack([dimension, two_d], axis=-1).astype(np.uint32).reshape(-1).view(np.float32)
    out = np.zeros(2 * n, dtype=np.float32)
    _native.check(_native.library().echo_b200_debug_math(0, 103, _native.pointer(a), _native.pointer(b), _native.pointer(c), 2 * n, _native.pointer(out)))
    return out.reshape(n, 2)


def test_device_sequence_is_bit_identical_to_the_oracle():
    rng = np.random.default_rng(3)
    extends = np.array([1, 2, 3, 4, 6, 7, 16, 17, 64, 100, 256, 1000, 4096, 65537, 1 << 20, 1 << 23], dtype=np.uint32)
    count = 12000
    seed = rng.integers(0, 2 ** 32, count, dtype=np.uint64).astype(np.uint32)
    pixel = rng.integers(0, 2 ** 32, count, dtype=np.uint64).astype(np.uint32)
    sample = rng.integers(0, 2 ** 32, count, dtype=np.uint64).astype(np.uint32)
    extend = extends[rng.integers(0, len(extends), count)]
    dimension = rng.integers(0, 800, count).astype(np.uint32)
    two_d = rng.integers(0, 2, count).astype(np.uint32)
    got = device_stratified(seed, pixel, sample, extend, dimension, two_d)
    for i in range(count):
        want = oracle_values(int(seed[i]), int(pixel[i]), [int(sample[i])], int(extend[i]), int(dimension[i]), bool(two_d[i]))[0]
        want = np.array([want[0], want[1]] if two_d[i] else [want, 0.0], dtype=np.float32)
        assert np.array_equal(bits(got[i]), bits(want)), (i, seed[i], pixel[i], sample[i], extend[i], dimension[i], two_d[i])
    bad = device_stratified(np.array([1, 1], np.uint32), np.array([2, 2], np.uint32), np.array([3, 3], np.uint32), np.array([0, (1 << 23) + 1], np.uint32),
                            np.array([0, 0], np.uint32), np.array([0, 1], np.uint32))
    assert np.isnan(bad).all()


@pytest.mark.parametrize("fixture,bounce_limit", [("cornell", 128), ("mixed_small", 8), ("lights_small", 128), ("terrain_small", 16), ("coated_small", 12),
                                                  ("directional_small", 12), ("textured_small", 12), ("environment_small", 12), ("cubemap_small", 12)])
def test_samples_match_oracle(fixture, bounce_limit, request):
    prepared = request.getfixturevalue(fixture)
    oracle = stratified_oracle.scene(prepared)
    width, height = 96, 64
    params = structs.render_params(width, height, 16, extend=4, bounce_limit=bounce_limit, seed=7, evaluator=STRATIFIED)
    pixel_xy, sample_index = sample_grid(width, height, 8)  # two epochs of four

    with PreparedScene(prepared) as scene:
        actual = scene.evaluate_samples(params, pixel_xy, sample_index)

    expected = oracle.evaluate_samples(params, pixel_xy, sample_index)
    assert expected.max() > 0
    assert np.array_equal(actual.view(np.uint32), expected.view(np.uint32))


@pytest.mark.parametrize("extend", [4, 6, 7, 16])
@pytest.mark.parametrize("fixture", ["cornell", "instanced"])
def test_samples_match_oracle_at_every_grid_shape(fixture, extend):
    prepared = host.prepare(scenes.cornell_box() if fixture == "cornell" else scenes.instanced_scene(grid=3, rings=8, segments=10))
    oracle = stratified_oracle.scene(prepared)
    width, height = 48, 32
    params = structs.render_params(width, height, 16, extend=extend, bounce_limit=24, seed=13, evaluator=STRATIFIED)
    pixel_xy, sample_index = sample_grid(width, height, 2 * extend)
    sample_index = sample_index + np.uint32(3 * extend)  # epochs 3 and 4

    with PreparedScene(prepared) as scene:
        actual = scene.evaluate_samples(params, pixel_xy, sample_index)

    expected = oracle.evaluate_samples(params, pixel_xy, sample_index)
    assert np.array_equal(actual.view(np.uint32), expected.view(np.uint32))


def render_pair(prepared, params, tiles):
    oracle = stratified_oracle.scene(prepared)
    with PreparedScene(prepared) as scene:
        actual, stats = scene.render_tiles(params, tiles)
    expected, expected_stats = oracle.render_tiles(params, tiles)
    assert np.array_equal(actual.view(np.uint32), expected.view(np.uint32))
    for name in structs.STATS_FIELDS[:12]:
        assert int(stats[name][0]) == int(expected_stats[name][0]), name
    return stats


def test_render_tiles_fixed_and_adaptive_epochs(cornell, mixed_small):
    width, height = 80, 48
    tiles = scenes.tile_grid(width, height, 32)
    stats = render_pair(mixed_small, structs.render_params(width, height, 32, extend=8, min_epoch=2, max_epoch=2, bounce_limit=16, seed=3, evaluator=STRATIFIED), tiles)
    assert int(stats["sampleEvaluated"][0]) == width * height * 16
    tiles = scenes.tile_grid(32, 32, 16)
    stats = render_pair(cornell, structs.render_params(32, 32, 16, extend=8, min_epoch=1, max_epoch=6, noise_threshold=0.3, seed=5, evaluator=STRATIFIED), tiles)
    assert 32 * 32 * 8 < int(stats["sampleEvaluated"][0]) < 32 * 32 * 48


def test_render_tiles_deep_cornell_reaches_the_tail_kernel(cornell):
    """bounce limit 128: the last few thousand paths of every batch are finished by tail_kernel"""
    render_pair(cornell, structs.render_params(64, 64, 16, extend=16, bounce_limit=128, seed=9, evaluator=STRATIFIED), scenes.tile_grid(64, 64, 16))


def test_render_tiles_narrow_path(cornell):
    """NARROW_LIMIT above every ray count: every bounce on the one-thread-per-ray kernels"""
    try:
        _native.set_option("NARROW_LIMIT", 1 << 30)
        render_pair(cornell, structs.render_params(48, 48, 16, extend=6, bounce_limit=24, seed=4, evaluator=STRATIFIED), scenes.tile_grid(48, 48, 16))
    finally:
        _native.set_option("NARROW_LIMIT", 1 << 20)


def test_counted_pass_with_the_flag_matches_the_oracle(cornell):
    params = structs.render_params(48, 32, 16, extend=4, bounce_limit=16, seed=2, evaluator=STRATIFIED | structs.EVALUATOR_COUNT_VISITS)
    render_pair(cornell, params, scenes.tile_grid(48, 32, 16))


@pytest.mark.parametrize("evaluator", [structs.EVALUATOR_ALBEDO | structs.EVALUATOR_DIVERGE_ONCE, structs.EVALUATOR_ALBEDO,
                                       structs.EVALUATOR_NORMAL_DEPTH, structs.EVALUATOR_NORMAL_DEPTH | structs.EVALUATOR_DIVERGE_ONCE,
                                       structs.EVALUATOR_NAIVE])
def test_auxiliary_and_naive_evaluators_match_oracle(evaluator, mixed_small):
    oracle = stratified_oracle.scene(mixed_small)
    width, height = 64, 48
    params = structs.render_params(width, height, 16, extend=6, bounce_limit=40, seed=7, evaluator=evaluator | STRATIFIED)
    pixel_xy, sample_index = sample_grid(width, height, 6)
    expected = np.zeros((len(sample_index), 4), dtype=np.float32)
    oracle.lib.oracle_evaluate_samples4(oracle.handle, oracle_lib.ptr(params), oracle_lib.ptr(pixel_xy), oracle_lib.ptr(sample_index), len(sample_index),
                                        oracle_lib.ptr(expected), 4, 0)
    tiles = scenes.tile_grid(width, height, 16)
    expected_tiles, _ = oracle.render_tiles(params, tiles)

    with PreparedScene(mixed_small) as scene:
        actual = scene.evaluate_samples(params, pixel_xy, sample_index, channels=4)
        actual_tiles, _ = scene.render_tiles(params, tiles)

    assert np.array_equal(actual.view(np.uint32), expected.view(np.uint32))
    assert np.array_equal(actual_tiles.view(np.uint32), expected_tiles.view(np.uint32))


def test_epoch_sharding(cornell):
    """two "ranks" render epochs [0, 2) and [2, 4) into frames that are summed and resolved: the one-call render of all four epochs"""
    import torch
    from echorenderer_b200 import shard_epochs
    oracle = stratified_oracle.scene(cornell)
    width, height, tile, epochs, world = 80, 48, 16, 4, 2
    tiles = scenes.tile_grid(width, height, tile)

    with PreparedScene(cornell) as scene:
        stream = torch.cuda.current_stream().cuda_stream
        frames = []
        for rank in range(world):
            first, count = shard_epochs(epochs, rank, world)
            block = structs.render_params(width, height, tile, extend=4, min_epoch=count, max_epoch=count, seed=6, epoch_offset=first, evaluator=STRATIFIED)
            frame = torch.zeros(height * width * 4, dtype=torch.float32, device="cuda")
            scene.render_frame_device(block, tiles, frame.data_ptr(), stream)
            frames.append(frame)
        total = frames[0] + frames[1]
        scene.frame_resolve_device(total.data_ptr(), width, height, stream)
        torch.cuda.synchronize()
        reduced = total.cpu().numpy().reshape(height, width, 4)

    everything = structs.render_params(width, height, tile, extend=4, min_epoch=epochs, max_epoch=epochs, seed=6, evaluator=STRATIFIED)
    expected, _ = oracle.render_tiles(everything, tiles)
    whole = scenes.assemble_tiles(expected, tiles, width, height, tile)
    assert np.allclose(reduced[..., :3], whole[..., :3], rtol=2e-6, atol=1e-7)


def test_stratified_cornell_is_closer_to_the_converged_image(cornell):
    """Cornell box 128 x 128 at extend 64 (one epoch), relative RMSE against a 4096-spp uniform device render of another seed. Measured on a
    B200: 0.0427 stratified against 0.0563 uniform, a ratio of 0.76. The bound, 0.9, leaves room for the reference's own noise."""
    size = 128
    tiles = scenes.tile_grid(size, size, 16)
    with PreparedScene(cornell) as scene:
        reference, _ = scene.render_tiles(structs.render_params(size, size, 16, extend=256, min_epoch=16, max_epoch=16, seed=99), tiles)
        errors = {}
        for evaluator in (0, STRATIFIED):
            image, _ = scene.render_tiles(structs.render_params(size, size, 16, extend=64, seed=5, evaluator=evaluator), tiles)
            errors[evaluator] = relative_rmse(image[..., :3], reference[..., :3])
    ratio = errors[STRATIFIED] / errors[0]
    print(f"stratified / uniform relative RMSE at 64 spp: {errors[STRATIFIED]:.4f} / {errors[0]:.4f} = {ratio:.3f}")
    assert ratio < 0.9, errors


def test_refusals(cornell):
    tiles = scenes.tile_grid(32, 32, 16)
    with PreparedScene(cornell) as scene:
        for extend in ((1 << 23) + 1, 1 << 24):
            params = structs.render_params(32, 32, 16, extend=extend, evaluator=STRATIFIED)
            with pytest.raises(EchoNativeError) as refused:
                scene.render_tiles(params, tiles)
            assert refused.value.status == _native.ERR_INVALID
            with pytest.raises(EchoNativeError) as refused:
                scene.evaluate_samples(params, np.zeros((1, 2), np.int32), np.zeros(1, np.uint32))
            assert refused.value.status == _native.ERR_INVALID
