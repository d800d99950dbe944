"""Every wavefront schedule of render.cu against the oracle: the persistent, narrow and tail kernels, several batches per call and the counted
pass, at all three traversal-stack classes (48, 96, 192 entries), for plain scenes, a textured scene (INST without packs) and scenes with
packs (tests/schedule_lib.py proves on the CPU that each fixture lands on its class).

The renders have more paths than two resident waves of the persistent kernels, on one pipeline and one batch, so that under the
`persistent` schedule the first bounces really replace work. Tiles and statistics rows must equal the oracle's bit for bit."""
import functools

import numpy as np
import pytest

from echorenderer_b200 import PreparedScene, _native, host, scenes, structs
from tests import oracle_lib, schedule_lib, stratified_oracle
from tests.test_gpu_render import sample_grid

pytestmark = pytest.mark.gpu

WIDTH, HEIGHT, TILE, EXTEND, BOUNCES = 160, 128, 16, 16, 16
PATHS = WIDTH * HEIGHT * EXTEND
TILES = scenes.tile_grid(WIDTH, HEIGHT, TILE)
DISTRIBUTIONS = {"uniform": 0, "stratified": structs.DISTRIBUTION_STRATIFIED}

# fixture: the stack class it lands on
FIXTURES = {"cornell": 48, "cornell_chain96": 96, "cornell_chain192": 192, "textured": 48, "flat_packs": 48, "nested_packs": 96, "deep_packs": 192}
DEEP = ["cornell_chain96", "cornell_chain192", "nested_packs", "deep_packs"]


@functools.lru_cache(maxsize=None)
def prepared(name):
    if name == "cornell":
        return host.prepare(scenes.cornell_box())
    if name.startswith("cornell_chain"):
        return schedule_lib.chain_qbvh(schedule_lib.chain_cornell(), 1 if name.endswith("192") else 2)
    if name == "textured":
        return host.prepare(scenes.textured_scene())
    if name.endswith("_packs") and name != "deep_packs":
        return host.prepare(scenes.instanced_scene(grid=4, rings=12, segments=14, nested=name == "nested_packs"))
    return schedule_lib.deep_pack_scene(5)


def params(distribution, evaluator=structs.EVALUATOR_PATH_TRACED):
    return structs.render_params(WIDTH, HEIGHT, TILE, extend=EXTEND, bounce_limit=BOUNCES, seed=5, evaluator=evaluator | DISTRIBUTIONS[distribution])


def oracle(name, distribution):
    return stratified_oracle.scene(prepared(name)) if distribution == "stratified" else oracle_lib.OracleScene(prepared(name))


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def device_scenes():
    opened = {}

    def get(name):
        if name not in opened:
            opened[name] = PreparedScene(prepared(name))
        return opened[name]

    yield get
    for scene in opened.values():
        scene.close()


@pytest.fixture(scope="module")
def oracle_renders():
    """the oracle's tiles and statistics, once per (fixture, distribution)"""
    return functools.lru_cache(maxsize=None)(lambda name, distribution: oracle(name, distribution).render_tiles(params(distribution), TILES))


@pytest.fixture(autouse=True)
def switches_back_at_defaults():
    yield
    assert {name: _native.get_option(name) for name in schedule_lib.DEFAULTS} == schedule_lib.DEFAULTS


def test_the_render_is_large_enough_for_work_replacement():
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert PATHS > 2 * sms * 8 * 128
    assert schedule_lib.schedule_switches("narrow")["BATCH_PATHS"] >= PATHS and schedule_lib.schedule_switches("persistent")["RENDER_WORKERS"] == 1
    assert all(schedule_lib.stack_class(schedule_lib.stack_entries(prepared(name))) == size for name, size in FIXTURES.items())


@pytest.mark.parametrize("distribution", list(DISTRIBUTIONS))
@pytest.mark.parametrize("schedule", schedule_lib.SCHEDULES)
@pytest.mark.parametrize("fixture", list(FIXTURES))
def test_schedule_matrix(fixture, schedule, distribution, device_scenes, oracle_renders):
    expected, expected_stats = oracle_renders(fixture, distribution)
    with schedule_lib.schedule(schedule, PATHS):
        image, stats = device_scenes(fixture).render_tiles(params(distribution), TILES)
    assert expected[..., :3].max() > 0
    assert np.array_equal(bits(image), bits(expected))
    for name in structs.STATS_FIELDS[:12]:
        assert int(stats[name][0]) == int(expected_stats[name][0]), name
    assert int(stats["sampleEvaluated"][0]) == PATHS


@pytest.mark.parametrize("fixture", list(FIXTURES))
def test_schedules_take_effect(fixture, device_scenes):
    """in lock step the launches are exact: persistent and narrow launch the same kernels per bounce, the tail schedule one kernel after the camera rays"""
    launches = {}
    for name in ("narrow", "persistent", "tail"):
        with schedule_lib.schedule(name, PATHS):
            _, stats = device_scenes(fixture).render_tiles(params("uniform"), TILES)
        launches[name] = int(stats["kernelLaunches"][0])
    assert launches["persistent"] == launches["narrow"]
    assert launches["tail"] < launches["narrow"]


@pytest.mark.parametrize("fixture", list(FIXTURES))
def test_per_sample_bits(fixture, device_scenes):
    pixel_xy, sample_index = sample_grid(WIDTH, HEIGHT, 2, stride=2)
    sample_params = params("uniform")
    expected = oracle(fixture, "uniform").evaluate_samples(sample_params, pixel_xy, sample_index)
    assert expected.max() > 0
    for name in ("persistent", "narrow", "tail"):
        with schedule_lib.schedule(name, len(sample_index)):
            actual = device_scenes(fixture).evaluate_samples(sample_params, pixel_xy, sample_index)
        assert np.array_equal(bits(actual), bits(expected)), name


@pytest.mark.parametrize("fixture", list(FIXTURES))
def test_counted_pass(fixture, device_scenes, oracle_renders):
    """ECHO_EVALUATOR_COUNT_VISITS takes the counted one-thread-per-query kernels on every bounce: the same tiles, and node / triangle /
    sphere / light-node visits equal to the oracle's counters"""
    expected, expected_stats = oracle_renders(fixture, "uniform")
    scene = device_scenes(fixture)
    image, stats = scene.render_tiles(params("uniform"), TILES)
    counted, counted_stats = scene.render_tiles(params("uniform", structs.EVALUATOR_COUNT_VISITS), TILES)
    assert np.array_equal(bits(counted), bits(image)) and np.array_equal(bits(counted), bits(expected))
    for name in structs.STATS_FIELDS[:12]:
        assert int(counted_stats[name][0]) == int(stats[name][0]) == int(expected_stats[name][0]), name
    for name in structs.STATS_VISIT_FIELDS:
        assert int(counted_stats[name][0]) == int(expected_stats[name][0]), name
    assert int(counted_stats["nodeVisits"][0]) > 0 and int(counted_stats["triangleVisits"][0]) > 0


@pytest.mark.parametrize("evaluator", [structs.EVALUATOR_ALBEDO | structs.EVALUATOR_DIVERGE_ONCE, structs.EVALUATOR_NORMAL_DEPTH, structs.EVALUATOR_NAIVE])
@pytest.mark.parametrize("fixture", DEEP)
def test_auxiliary_and_naive_at_deep_stacks(fixture, evaluator, device_scenes):
    target = oracle(fixture, "uniform")
    sample_params = structs.render_params(WIDTH, HEIGHT, TILE, extend=4, bounce_limit=24, seed=7, evaluator=evaluator)
    pixel_xy, sample_index = sample_grid(WIDTH, HEIGHT, 2, stride=2)
    expected = np.zeros((len(sample_index), 4), dtype=np.float32)
    target.lib.oracle_evaluate_samples4(target.handle, oracle_lib.ptr(sample_params), oracle_lib.ptr(pixel_xy), oracle_lib.ptr(sample_index), len(sample_index),
                                        oracle_lib.ptr(expected), 4, 0)
    actual = device_scenes(fixture).evaluate_samples(sample_params, pixel_xy, sample_index, channels=4)
    assert expected[:, :3].max() > 0
    assert np.array_equal(bits(actual), bits(expected))


@pytest.mark.parametrize("fixture", ["cornell", "nested_packs"])
def test_persistent_queue_count_edges(fixture, device_scenes):
    """the persistent kernels with queues from one ray to one more than their resident lanes (ECHO_MIN_BLOCKS / ECHO_INST_MIN_BLOCKS CTAs of
    128 per SM): every prefix of one sample list, each sample equal to the oracle's"""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    lanes = (6 if prepared(fixture).packs is not None else 7) * 128 * sms
    counts = [1, 2, 31, 32, 33, 127, 128, 129, lanes - 1, lanes, lanes + 1]
    pixel_xy, sample_index = sample_grid(WIDTH, HEIGHT, 8)
    pixel_xy, sample_index = pixel_xy[:counts[-1]], sample_index[:counts[-1]]
    assert len(sample_index) == counts[-1]
    sample_params = params("uniform")
    expected = oracle(fixture, "uniform").evaluate_samples(sample_params, pixel_xy, sample_index)
    with schedule_lib.schedule("persistent"):
        for n in counts:
            actual = device_scenes(fixture).evaluate_samples(sample_params, pixel_xy[:n], sample_index[:n])
            assert np.array_equal(bits(actual), bits(expected[:n])), n
