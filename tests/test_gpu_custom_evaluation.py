"""The host-driven EvaluationOperation of include/echo_b200_evaluation.h on the GPU: its draws and camera rays against the oracle, its
Accumulator and epoch loop against a Python restatement of EvaluationOperation.cs, StandardNaiveEvaluator composed in torch from the
device queries against echo_b200_render_tiles (byte for byte), the frame form, two evaluations at once, and every refusal."""
import ctypes

import numpy as np
import pytest
import torch

from echorenderer_b200 import EchoNativeError, EvaluationOperation, EvaluationProfile, PreparedScene, RenderTexture, _native, host, scenes, structs
from tests import oracle_lib, stratified_oracle
from tests.custom_evaluators_lib import HashEvaluator, TorchNaiveEvaluator, hash_samples

pytestmark = pytest.mark.gpu

STRAT = structs.DISTRIBUTION_STRATIFIED


def spawn(evaluation, count):
    """(rays, pixels int32[count, 2], sample indices uint32[count]) of the open epoch"""
    rays = torch.empty((count, 8), dtype=torch.float32, device="cuda")
    pixels = torch.empty((count, 2), dtype=torch.int32, device="cuda")
    samples = torch.empty(count, dtype=torch.int32, device="cuda")
    evaluation.spawn_device(rays.data_ptr(), pixels.data_ptr(), samples.data_ptr())
    return rays.cpu().numpy().view(structs.RAY).reshape(-1), pixels.cpu().numpy(), samples.cpu().numpy().view(np.uint32)


def inside_pixels(params, tiles):
    size, width, height = int(params["tileSize"][0]), int(params["width"][0]), int(params["height"][0])
    return {(x * size + i, y * size + j) for x, y in tiles for j in range(size) for i in range(size) if x * size + i < width and y * size + j < height}


def check_slot_layout(params, tiles, pixels, samples, epoch):
    """slot = active-pixel position x extend + s, the samples of an epoch in order, every pixel of the tiles inside the image once"""
    extend, offset = int(params["extend"][0]), int(params["epochOffset"][0])
    grouped = pixels.reshape(-1, extend, 2)
    assert np.all(grouped == grouped[:, :1])
    assert np.array_equal(samples.reshape(-1, extend), np.tile((offset + epoch - 1) * extend + np.arange(extend, dtype=np.uint32), (len(grouped), 1)))
    assert {tuple(p) for p in grouped[:, 0]} == inside_pixels(params, tiles) and len(grouped) == len(inside_pixels(params, tiles))


@pytest.mark.parametrize("stratified", [False, True])
def test_draws_equal_the_oracle(cornell, stratified):
    width, seed, extend = 20, 9, 6
    params = structs.render_params(width, 12, 8, extend=extend, min_epoch=2, max_epoch=2, seed=seed, epoch_offset=3, evaluator=STRAT if stratified else 0)
    tiles = np.array([[0, 0], [2, 1], [1, 1]], dtype=np.int32)  # the last two cross the image's right and bottom edges
    out = np.zeros(2, dtype=np.float32)
    uniform, strat = oracle_lib.library(), stratified_oracle.library()

    def expected(pixel, sample, dimension, two_d):
        if stratified:
            strat.oracle_stratified_value(seed, pixel, int(sample), extend, dimension, 1 if two_d else 0, out.ctypes.data_as(ctypes.c_void_p))
            return out.copy() if two_d else out[:1].copy()
        values = [uniform.oracle_sample_value(seed, pixel, int(sample), dimension + k) for k in range(2 if two_d else 1)]
        return np.array(values, dtype=np.float32)

    with PreparedScene(cornell) as scene, scene.evaluation(params, tiles) as evaluation:
        for epoch in (1, 2):
            count = evaluation.next_epoch()
            _, pixels, samples = spawn(evaluation, count)
            check_slot_layout(params, tiles, pixels, samples, epoch)
            index = pixels[:, 1] * width + pixels[:, 0]
            for dimension in range(12):
                for components in (1, 2):
                    draws = torch.empty(count * components, dtype=torch.float32, device="cuda")
                    evaluation.draw_device(dimension, components, draws.data_ptr())
                    got = draws.cpu().numpy().reshape(count, components)
                    want = np.stack([expected(int(p), s, dimension, components == 2) for p, s in zip(index, samples)])
                    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (epoch, dimension, components)
            evaluation.accumulate_device(torch.zeros((count, 4), dtype=torch.float32, device="cuda").data_ptr())
        assert evaluation.next_epoch() == 0


@pytest.mark.parametrize("stratified", [False, True])
@pytest.mark.parametrize("camera", ["perspective", "thin_lens", "orthographic", "cylindrical"])
def test_camera_rays_equal_the_oracle(camera, stratified):
    description = scenes.cornell_box()
    if camera == "perspective":
        description.camera = scenes.perspective_camera((0, 5, -18.025444), field_of_view=42.0, lens_radius=0.0)
    elif camera == "thin_lens":
        description.camera = scenes.perspective_camera((0, 5, -18.025444), field_of_view=42.0, lens_radius=0.3, focal_distance=16.0)
    elif camera == "orthographic":
        description.camera = scenes.orthographic_camera((0, 5, -4), (0, 0, 0), width=9.0)
    else:
        description.camera = scenes.cylindrical_camera((0, 5, 0), (10, 30, 0))
    prepared = host.prepare(description)
    oracle = stratified_oracle.scene(prepared) if stratified else oracle_lib.OracleScene(prepared)
    params = structs.render_params(40, 24, 16, extend=5, seed=4, epoch_offset=2, evaluator=STRAT if stratified else 0)
    tiles = np.array([[0, 0], [2, 0], [1, 1], [2, 1]], dtype=np.int32)  # 40 x 24: tiles of the last column and row cross the edges

    with PreparedScene(prepared) as scene, scene.evaluation(params, tiles) as evaluation:
        count = evaluation.next_epoch()
        rays, pixels, samples = spawn(evaluation, count)
        check_slot_layout(params, tiles, pixels, samples, 1)
        without = torch.empty((count, 8), dtype=torch.float32, device="cuda")
        evaluation.spawn_device(without.data_ptr())  # the pixel and sample outputs are optional
        assert np.array_equal(without.cpu().numpy().view(structs.RAY).reshape(-1).view(np.uint8), rays.view(np.uint8))
    expected = oracle.spawn_rays(params, pixels, samples)
    assert np.array_equal(rays.view(np.uint8), expected.view(np.uint8))


def reference_operation(params, tiles, evaluate):
    """EvaluationOperation.cs:100-141 per pixel with oracle_lib.accumulate: (tiles, stats, epochs per pixel, tiles after epoch 1)"""
    size, width, height = int(params["tileSize"][0]), int(params["width"][0]), int(params["height"][0])
    extend, offset = int(params["extend"][0]), int(params["epochOffset"][0])
    min_epoch, max_epoch, threshold = int(params["minEpoch"][0]), int(params["maxEpoch"][0]), np.float32(params["noiseThreshold"][0])
    out, preview = np.zeros((len(tiles), size, size, 4), dtype=np.float32), np.zeros((len(tiles), size, size, 4), dtype=np.float32)
    evaluated = rejected = pixels = 0
    epochs = {}
    for t, (tx, ty) in enumerate(tiles):
        for j in range(size):
            for i in range(size):
                x, y = tx * size + i, ty * size + j
                if x >= width or y >= height:
                    continue
                pixels += 1
                taken, epoch = [], 0
                while True:
                    epoch += 1
                    taken.append(evaluate(np.full(extend, y * width + x), (offset + epoch - 1) * extend + np.arange(extend)))
                    mean, noise, count = oracle_lib.accumulate(np.concatenate(taken))
                    if epoch == 1:
                        preview[t, j, i] = mean
                    if not (epoch < max_epoch and (epoch < min_epoch or (count >= 2 and np.float32(noise) > threshold))):
                        break
                samples = np.concatenate(taken)
                evaluated += len(samples)
                with np.errstate(invalid="ignore"):  # inf + -inf: the NaN sum Accumulator.Add rejects
                    rejected += int((~np.isfinite((samples[:, 0] + samples[:, 1]) + (samples[:, 2] + samples[:, 3]))).sum())
                out[t, j, i] = mean
                epochs[(x, y)] = epoch
    return out, (evaluated, rejected, pixels), epochs, preview


def operation_rows(stats):
    return int(stats["sampleEvaluated"][0]), int(stats["sampleRejected"][0]), int(stats["pixelEvaluated"][0])


def test_accumulator_and_epochs_equal_evaluation_operation(cornell):
    width = 24
    params = structs.render_params(width, 20, 8, extend=8, min_epoch=2, max_epoch=6, noise_threshold=0.03, seed=3, epoch_offset=1)
    tiles = np.array([[0, 0], [1, 0], [2, 0], [0, 2], [2, 2]], dtype=np.int32)  # the last row crosses the bottom edge
    expected, rows, epochs, preview = reference_operation(params, tiles, hash_samples)
    assert set(epochs.values()) >= {2, 6} and len(set(epochs.values())) >= 3  # some pixels stop at minEpoch, some run to maxEpoch
    assert rows[1] > 0

    evaluator = HashEvaluator(width)
    with PreparedScene(cornell) as scene, scene.evaluation(params, tiles) as evaluation:
        epoch = 0
        while True:
            count = evaluation.next_epoch()
            if count == 0:
                break
            epoch += 1
            assert count == 8 * sum(1 for e in epochs.values() if e >= epoch)
            evaluation.accumulate_device(evaluator.evaluate(scene, evaluation, count, 0))
            if epoch == 1:  # a progressive preview between epochs
                early, early_stats = evaluation.finish()
                assert np.array_equal(early.view(np.uint32), preview.view(np.uint32))
                assert operation_rows(early_stats)[2] == rows[2]
        got, stats = evaluation.finish()
    assert epoch == 6
    assert np.array_equal(got.view(np.uint32), expected.view(np.uint32))
    assert operation_rows(stats) == rows
    assert int(stats["kernelLaunches"][0]) > 0
    assert all(int(stats[name][0]) == 0 for name in structs.STATS_FIELDS[3:12])


def instanced_nested():
    return host.prepare(scenes.instanced_scene(grid=3, rings=8, segments=10, nested=True))


@pytest.fixture(scope="module")
def naive_scenes(cornell, textured_small):
    return {"cornell": cornell, "textured": textured_small, "instanced": instanced_nested()}


def naive_params(mode, stratified, evaluator=0):
    flag = STRAT if stratified else 0
    if mode == "adaptive":
        return structs.render_params(48, 40, 16, extend=4, min_epoch=1, max_epoch=4, noise_threshold=0.2, bounce_limit=8, seed=11, evaluator=evaluator | flag)
    return structs.render_params(48, 40, 16, extend=4, min_epoch=2, max_epoch=2, bounce_limit=8, seed=11, epoch_offset=3, evaluator=evaluator | flag)


def run_evaluation(scene, params, tiles, evaluator, stream=0, frame=None):
    with scene.evaluation(params, tiles, stream=stream) as evaluation:
        while True:
            count = evaluation.next_epoch()
            if count == 0:
                break
            evaluation.accumulate_device(evaluator.evaluate(scene, evaluation, count, stream))
        result = evaluation.finish(None if frame is None else frame.data_ptr())
    evaluator.status()
    return result


@pytest.mark.parametrize("mode", ["adaptive", "offset"])
@pytest.mark.parametrize("stratified", [False, True])
@pytest.mark.parametrize("name", ["cornell", "textured", "instanced"])
def test_naive_evaluator_in_torch_renders_the_tiles_of_render_tiles(naive_scenes, name, stratified, mode):
    prepared = naive_scenes[name]
    params = naive_params(mode, stratified)
    tiles = scenes.tile_grid(48, 40, 16)  # 3 x 3 tiles, the last row and column crossing the edges
    with PreparedScene(prepared) as scene:
        expected, expected_stats = scene.render_tiles(naive_params(mode, stratified, structs.EVALUATOR_NAIVE), tiles)
        got, stats = run_evaluation(scene, params, tiles, TorchNaiveEvaluator(prepared.packs is not None, 8))
        assert scene.bounds_violations() in (None, 0)
    assert np.array_equal(got.view(np.uint32), expected.view(np.uint32))
    assert operation_rows(stats) == operation_rows(expected_stats)
    assert np.abs(expected).max() > 0


def test_evaluation_operation_runs_a_device_evaluator(cornell):
    destination = RenderTexture(40, 24, tile_size=16)
    expected = RenderTexture(40, 24, tile_size=16)
    with PreparedScene(cornell) as scene:
        from echorenderer_b200 import StandardNaiveEvaluator
        builtin = EvaluationOperation(scene, EvaluationProfile(evaluator=StandardNaiveEvaluator(bounce_limit=8), extend=4, max_epoch=3, seed=2), expected)
        builtin.execute()
        operation = EvaluationOperation(scene, EvaluationProfile(evaluator=TorchNaiveEvaluator(False, 8), extend=4, max_epoch=3, seed=2), destination)
        operation.execute()
    assert np.array_equal(destination.pixels.view(np.uint32), expected.pixels.view(np.uint32))
    assert operation.total_samples == builtin.total_samples and operation.statistics_report()["Pixel/Evaluated"] == 40 * 24


def test_frame_form_adds_what_render_frame_device_adds(cornell):
    width, height = 48, 40
    tiles = scenes.tile_grid(width, height, 16)
    params = naive_params("adaptive", False)
    with PreparedScene(cornell) as scene:
        expected = torch.zeros((height * width, 4), dtype=torch.float32, device="cuda")
        got = torch.zeros((height * width, 4), dtype=torch.float32, device="cuda")
        expected[:7] = 0.25  # the frames add to what is there
        got[:7] = 0.25
        torch.cuda.synchronize()  # render_frame_device runs on the scene's own stream
        scene.render_frame_device(naive_params("adaptive", False, structs.EVALUATOR_NAIVE), tiles, expected.data_ptr())
        run_evaluation(scene, params, tiles, TorchNaiveEvaluator(False, 8), frame=got)
        torch.cuda.synchronize()
        assert torch.equal(got.view(torch.int32), expected.view(torch.int32))
        scene.frame_resolve_device(expected.data_ptr(), width, height)
        scene.frame_resolve_device(got.data_ptr(), width, height)
        torch.cuda.synchronize()
        assert torch.equal(got.view(torch.int32), expected.view(torch.int32)) and float(got.abs().max()) > 0


def test_two_evaluations_on_two_streams_interleaved(cornell):
    tiles = scenes.tile_grid(48, 40, 16)
    first, second = naive_params("adaptive", False), naive_params("offset", True)
    with PreparedScene(cornell) as scene:
        alone = [run_evaluation(scene, p, t, TorchNaiveEvaluator(False, 8)) for p, t in ((first, tiles), (second, tiles[::-1].copy()))]

        streams = [torch.cuda.Stream(), torch.cuda.Stream()]
        evaluators = [TorchNaiveEvaluator(False, 8), TorchNaiveEvaluator(False, 8)]
        evaluations = [scene.evaluation(first, tiles, stream=streams[0].cuda_stream), scene.evaluation(second, tiles[::-1].copy(), stream=streams[1].cuda_stream)]
        running = [True, True]
        while any(running):
            counts = [e.next_epoch() if r else 0 for e, r in zip(evaluations, running)]
            pending = [(k, evaluators[k].evaluate(scene, evaluations[k], counts[k], streams[k].cuda_stream)) for k in range(2) if counts[k]]
            for k, samples in pending:
                evaluations[k].accumulate_device(samples)
            running = [c > 0 for c in counts]
        together = [e.finish() for e in evaluations]
        for e in evaluations:
            e.close()
    for (tiles_alone, stats_alone), (tiles_together, stats_together) in zip(alone, together):
        assert np.array_equal(tiles_together.view(np.uint32), tiles_alone.view(np.uint32))
        assert operation_rows(stats_together) == operation_rows(stats_alone)


def refused(call, message):
    with pytest.raises(EchoNativeError) as error:
        call()
    assert error.value.status == _native.ERR_INVALID, str(error.value)
    assert message in str(error.value), str(error.value)


def test_refusals(cornell):
    good = structs.render_params(32, 32, 16, extend=4)
    tiles = scenes.tile_grid(32, 32, 16)

    def with_(**fields):
        params = good.copy()
        for name, value in fields.items():
            params[name] = value
        return params

    with PreparedScene(cornell) as scene:
        create = lambda params, t=tiles: scene.evaluation(params, t).close()  # noqa: E731
        for bad in (dict(width=0), dict(height=-1), dict(tileSize=0), dict(extend=0), dict(maxEpoch=0), dict(minEpoch=3, maxEpoch=2)):
            refused(lambda: create(with_(**bad)), "invalid EchoRenderParams")
        refused(lambda: create(with_(evaluator=STRAT, extend=(1 << 23) + 1, tileSize=1), np.zeros((1, 2), np.int32)), "ECHO_DISTRIBUTION_STRATIFIED takes an extend of 1 to 2^23")
        for evaluator in (structs.EVALUATOR_NAIVE, structs.EVALUATOR_ALBEDO, structs.EVALUATOR_DIVERGE_ONCE, structs.EVALUATOR_COUNT_VISITS, STRAT | 0x800):
            refused(lambda: create(with_(evaluator=evaluator)), "evaluator 0 or ECHO_DISTRIBUTION_STRATIFIED")
        refused(lambda: create(with_(tileSize=1024, extend=2049), np.zeros((1, 2), np.int32)), "at most 2^31 slots")
        refused(lambda: create(with_(tileSize=1024, extend=1), np.zeros((1025, 2), np.int32)), "at most 2^31 slots")
        refused(lambda: create(good, np.array([[0, -1]], np.int32)), "a tile position is negative")

        lib = _native.library()
        handle, count = ctypes.c_void_p(), ctypes.c_uint64()
        assert lib.echo_b200_evaluation_create(scene.handle, None, _native.pointer(tiles), len(tiles), None, ctypes.byref(handle)) == _native.ERR_INVALID
        assert lib.echo_b200_evaluation_create(scene.handle, _native.pointer(good), None, len(tiles), None, ctypes.byref(handle)) == _native.ERR_INVALID
        assert lib.echo_b200_evaluation_create(scene.handle, _native.pointer(good), _native.pointer(tiles), len(tiles), None, None) == _native.ERR_INVALID
        assert lib.echo_b200_evaluation_create(None, _native.pointer(good), _native.pointer(tiles), len(tiles), None, ctypes.byref(handle)) == _native.ERR_INVALID
        assert b"scene is null" in lib.echo_b200_last_error()
        for call in (lambda: lib.echo_b200_evaluation_next_epoch(None, ctypes.byref(count)), lambda: lib.echo_b200_evaluation_spawn_device(None, None, None, None),
                     lambda: lib.echo_b200_evaluation_draw_device(None, 0, 1, None), lambda: lib.echo_b200_evaluation_accumulate_device(None, None),
                     lambda: lib.echo_b200_evaluation_finish(None, None, None, None), lambda: lib.echo_b200_evaluation_destroy(None)):
            assert call() == _native.ERR_INVALID and b"evaluation is null" in lib.echo_b200_last_error()

        buffer = torch.zeros(32 * 32 * 4 * 8 + 4, dtype=torch.float32, device="cuda")
        address = buffer.data_ptr()
        with scene.evaluation(good, tiles) as evaluation:
            refused(lambda: evaluation.spawn_device(address), "no epoch is open")
            refused(lambda: evaluation.draw_device(0, 1, address), "no epoch is open")
            refused(lambda: evaluation.accumulate_device(address), "no epoch is open")
            assert evaluation.next_epoch() == 32 * 32 * 4
            refused(lambda: evaluation.next_epoch(), "has not been accumulated")
            refused(lambda: evaluation.finish(), "an epoch is open")
            for components in (0, 3):
                refused(lambda: evaluation.draw_device(5, components, address), "components is 1 (Next1D) or 2 (Next2D)")
            refused(lambda: evaluation.draw_device(5, 1, 0), "d_out is null")
            refused(lambda: evaluation.spawn_device(0), "d_rays is null")
            refused(lambda: evaluation.accumulate_device(address + 4), "not 16-byte aligned")
            evaluation.draw_device(0xFFFFFFFF, 2, address)  # any dimension
            evaluation.accumulate_device(address)
            refused(lambda: evaluation.accumulate_device(address), "no epoch is open")
            refused(lambda: evaluation.spawn_device(address), "no epoch is open")
            evaluation.finish()  # between epochs: a preview
            assert evaluation.next_epoch() == 0 and evaluation.next_epoch() == 0
            evaluation.finish()

        uncommitted = ctypes.c_void_p()
        _native.check(lib.echo_b200_scene_create(ctypes.byref(uncommitted), 0))
        try:
            assert lib.echo_b200_evaluation_create(uncommitted, _native.pointer(good), _native.pointer(tiles), len(tiles), None, ctypes.byref(handle)) == _native.ERR_INVALID
            assert b"scene is not committed" in lib.echo_b200_last_error()
        finally:
            lib.echo_b200_scene_destroy(uncommitted)
        torch.cuda.synchronize()
        assert scene.bounds_violations() in (None, 0)


def test_multi_device_scene_is_refused(cornell):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    with PreparedScene(cornell, devices=[0, 1]) as scene:
        refused(lambda: scene.evaluation(structs.render_params(32, 32, 16, extend=4), scenes.tile_grid(32, 32, 16)), "single-device scene")
