"""The host-driven EvaluationOperation of include/echo_b200_evaluation.h without a GPU: the header on its own, the exported and bound
symbols, the C# declarations of INTEGRATION.md, clean refusal of a NULL scene or evaluation, and EvaluationOperation's epoch loop for a
DeviceEvaluator, run against a fake Evaluation."""
import ctypes
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from echorenderer_b200 import DeviceEvaluator, EvaluationOperation, EvaluationProfile, PreparedScene, RenderTexture, _native, scene as scene_module, structs
from tests.test_abi import declared_functions, have_gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_compiles_as_c99():
    source = ('#include "echo_b200_evaluation.h"\n'
              'int32_t (*next)(EchoEvaluation*, uint64_t*) = echo_b200_evaluation_next_epoch;\n'
              'int main(void) { EchoEvaluation* e = 0; uint64_t count = 0; return next && e == 0 && count == 0 ? 0 : 1; }\n')
    with tempfile.TemporaryDirectory() as directory:
        path, binary = os.path.join(directory, "header.c"), os.path.join(directory, "header.o")
        open(path, "w").write(source)
        subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-c", "-I", os.path.join(ROOT, "include"), path, "-o", binary], check=True)


def test_evaluation_symbols_are_declared_bound_and_exported():
    declared = declared_functions("echo_b200_evaluation.h")
    assert declared == set(_native.EVALUATION_EXPORTS) and len(declared) == 7
    assert not declared & (set(_native.EXPORTS) | set(_native.QUERY_EXPORTS) | set(_native.DEVICE_QUERY_EXPORTS))
    lib = _native.library()
    for name in declared:
        assert hasattr(lib, name), name
        assert getattr(lib, name).argtypes is not None, f"{name} has no ctypes signature"


def test_integration_document_declares_every_evaluation_call():
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    for name in _native.EVALUATION_EXPORTS:
        assert re.search(rf"\[DllImport\(Library\)\] public static extern \w+ {name}\(", text), name


@pytest.mark.skipif(have_gpu(), reason="checks the no-device behaviour")
def test_every_evaluation_call_refuses_a_null_scene_or_evaluation():
    lib = _native.library()
    params = structs.render_params(32, 32, 16, extend=4)
    tiles = np.zeros((1, 2), dtype=np.int32)
    buffer = ctypes.create_string_buffer(4096)  # stands for every device buffer: the calls must refuse before touching one
    b = ctypes.addressof(buffer)

    handle = ctypes.c_void_p()
    assert lib.echo_b200_evaluation_create(None, _native.pointer(params), _native.pointer(tiles), 1, None, ctypes.byref(handle)) == _native.ERR_INVALID
    assert b"scene is null" in lib.echo_b200_last_error() and not handle.value

    count = ctypes.c_uint64()
    calls = [
        lambda: lib.echo_b200_evaluation_next_epoch(None, ctypes.byref(count)),
        lambda: lib.echo_b200_evaluation_spawn_device(None, b, b, b),
        lambda: lib.echo_b200_evaluation_draw_device(None, 4, 2, b),
        lambda: lib.echo_b200_evaluation_accumulate_device(None, b),
        lambda: lib.echo_b200_evaluation_finish(None, b, None, b),
        lambda: lib.echo_b200_evaluation_destroy(None),
    ]
    for call in calls:
        assert call() == _native.ERR_INVALID
        assert b"evaluation is null" in lib.echo_b200_last_error()


class FakeEvaluation:
    """Records the calls EvaluationOperation makes of an Evaluation; its epochs have the given slot counts."""

    def __init__(self, scene, params, tile_xy, stream=0):
        self.calls = [("create", int(params["tileSize"][0]), int(params["evaluator"][0]), len(tile_xy), stream)]
        self.tile_xy = np.asarray(tile_xy).reshape(-1, 2)
        self.tile_size = int(params["tileSize"][0])
        self.counts = list(FakeEvaluation.counts)
        FakeEvaluation.made.append(self)

    def next_epoch(self):
        count = self.counts.pop(0) if self.counts else 0
        self.calls.append(("next_epoch", count))
        return count

    def accumulate_device(self, samples):
        self.calls.append(("accumulate", samples))

    def finish(self, frame_pointer=None):
        self.calls.append(("finish",))
        tiles = np.zeros((len(self.tile_xy), self.tile_size, self.tile_size, 4), dtype=np.float32)
        for k in range(len(tiles)):
            tiles[k] = k + 1
        stats = np.zeros(1, dtype=structs.STATS)
        stats["sampleEvaluated"], stats["sampleRejected"], stats["pixelEvaluated"], stats["kernelLaunches"] = 96, 3, 20, 7
        return tiles, stats

    def close(self):
        self.calls.append(("close",))

    def __enter__(self):
        return self

    def __exit__(self, *_):
        self.close()


class CountingEvaluator(DeviceEvaluator):
    def __init__(self):
        self.seen = []

    def evaluate(self, scene, evaluation, count, stream):
        self.seen.append((scene, evaluation, count, stream))
        evaluation.calls.append(("evaluate", count))
        return 0x1000 + count  # the device address the operation hands to accumulate


@pytest.mark.parametrize("stratified", [False, True])
def test_evaluation_operation_runs_the_epoch_loop_of_a_device_evaluator(monkeypatch, stratified):
    monkeypatch.setattr(scene_module, "Evaluation", FakeEvaluation)
    monkeypatch.setattr(FakeEvaluation, "counts", [64, 40, 8], raising=False)
    monkeypatch.setattr(FakeEvaluation, "made", [], raising=False)
    scene = object.__new__(PreparedScene)  # no native scene: PreparedScene.evaluation only hands itself to the Evaluation
    evaluator = CountingEvaluator()
    destination = RenderTexture(20, 12, tile_size=8)
    operation = EvaluationOperation(scene, EvaluationProfile(evaluator=evaluator, extend=8, stratified=stratified), destination, stream=1234)
    operation.statistics["sampleEvaluated"] = 4  # statistics add up over executions

    assert operation.execute() is destination
    (evaluation,) = FakeEvaluation.made
    expected_flags = structs.DISTRIBUTION_STRATIFIED if stratified else 0
    assert evaluation.calls == [("create", 8, expected_flags, 6, 1234),
                                ("next_epoch", 64), ("evaluate", 64), ("accumulate", 0x1000 + 64),
                                ("next_epoch", 40), ("evaluate", 40), ("accumulate", 0x1000 + 40),
                                ("next_epoch", 8), ("evaluate", 8), ("accumulate", 0x1000 + 8),
                                ("next_epoch", 0), ("finish",), ("close",)]
    assert [(s, e, c, st) for s, e, c, st in evaluator.seen] == [(scene, evaluation, c, 1234) for c in (64, 40, 8)]

    # tile k (in the operation's tile order) was filled with k + 1 and lands at its position, clipped to the texture
    for k, (x, y) in enumerate(operation.tile_positions):
        block = destination.pixels[y * 8:min(y * 8 + 8, 12), x * 8:min(x * 8 + 8, 20)]
        assert block.size and np.all(block == k + 1)
    report = operation.statistics_report()
    assert operation.total_samples == 100 and report["Sample/Rejected"] == 3 and report["Pixel/Evaluated"] == 20 and int(operation.statistics["kernelLaunches"][0]) == 7


def test_a_device_evaluator_is_abstract():
    with pytest.raises(NotImplementedError):
        DeviceEvaluator().evaluate(None, None, 1, 0)
