"""Samples/s of a host's own evaluator run through include/echo_b200_evaluation.h, beside the built-in evaluator it restates, on one GPU.

Per scene (the Cornell box and the instanced scene, 512 x 512, extend 16, bounce limit 8, one epoch), in one process:
  render_tiles      echo_b200_render_tiles with ECHO_EVALUATOR_NAIVE: host wall time of the synchronous call, median of --repeat after
                    one warm-up call
  composed          StandardNaiveEvaluator composed in torch from the device queries (tests/custom_evaluators_lib.py), through an
                    Evaluation on the legacy default stream: host wall time from create to finish, synchronised, median of --repeat
                    after one warm-up run
  operation_share   the share of one composed run spent in the Evaluation's own calls (next_epoch, spawn_device, draw_device,
                    accumulate_device): CUDA events around each call on the evaluation's stream, summed, over the composed run's time
  identical         whether the two tile sets are equal bit for bit; refused_query: the lowest query the device checks refused, if any
The card's name and power limit are read in the same run. Prints one JSON line per scene; writes them to --out when given.

    python variants/custom_evaluation_rates.py [--repeat 3] [--out PATH]
"""
import argparse
import contextlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from echorenderer_b200 import EchoNativeError, PreparedScene, host, scenes, structs  # noqa: E402
from variants.pack_build_times import card  # noqa: E402

SIZE, EXTEND, BOUNCES = 512, 16, 8
SCENES = {"cornell": scenes.cornell_box, "instanced": scenes.instanced_scene}


def composed_run(scene, params, tiles, instanced, events=None):
    """one EvaluationOperation with the torch evaluator: (tiles, stats, seconds, the queries' status: None or the lowest refusal);
    `events` collects (call, start, end) when given"""
    import torch
    from tests.custom_evaluators_lib import TorchNaiveEvaluator

    @contextlib.contextmanager
    def timer(name):
        if events is None:
            yield
            return
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        yield
        end.record()
        events.append((name, start, end))

    evaluator = TorchNaiveEvaluator(instanced, BOUNCES, timer=timer)
    torch.cuda.synchronize()
    started = time.perf_counter()
    with scene.evaluation(params, tiles) as evaluation:
        while True:
            with timer("next_epoch"):
                count = evaluation.next_epoch()
            if count == 0:
                break
            samples = evaluator.evaluate(scene, evaluation, count, 0)
            with timer("accumulate"):
                evaluation.accumulate_device(samples)
        result, stats = evaluation.finish()
    torch.cuda.synchronize()
    seconds = time.perf_counter() - started
    try:
        evaluator.status()
        refused = None
    except EchoNativeError as error:  # a refused query got the record of a miss: reported beside the rates, not hidden
        refused = str(error)
    return result, stats, seconds, refused


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--repeat", type=int, default=3)
    parser.add_argument("--out")
    args = parser.parse_args()

    name, limit = card()
    lines = []
    tiles = scenes.tile_grid(SIZE, SIZE, 16)

    for label, build in SCENES.items():
        prepared = host.prepare(build())
        instanced = prepared.packs is not None
        builtin = structs.render_params(SIZE, SIZE, 16, extend=EXTEND, bounce_limit=BOUNCES, evaluator=structs.EVALUATOR_NAIVE)
        params = structs.render_params(SIZE, SIZE, 16, extend=EXTEND, bounce_limit=BOUNCES)
        with PreparedScene(prepared) as scene:
            expected, expected_stats = scene.render_tiles(builtin, tiles)
            times = []
            for _ in range(args.repeat):
                started = time.perf_counter()
                scene.render_tiles(builtin, tiles)
                times.append(time.perf_counter() - started)
            builtin_seconds = sorted(times)[len(times) // 2]

            composed_run(scene, params, tiles, instanced)
            runs = [composed_run(scene, params, tiles, instanced) for _ in range(args.repeat)]
            got, stats, _, refused = runs[0]
            composed_seconds = sorted(run[2] for run in runs)[len(runs) // 2]

            events = []
            _, _, profiled_seconds, _ = composed_run(scene, params, tiles, instanced, events)
            own = {}
            for call, start, end in events:
                own[call] = own.get(call, 0.0) + start.elapsed_time(end)

        samples = int(stats["sampleEvaluated"][0])
        record = {"scene": label, "size": SIZE, "extend": EXTEND, "bounce_limit": BOUNCES, "samples": samples,
                  "render_tiles_ms": round(builtin_seconds * 1e3, 3), "render_tiles_samples_per_s": round(int(expected_stats["sampleEvaluated"][0]) / builtin_seconds),
                  "composed_ms": round(composed_seconds * 1e3, 3), "composed_samples_per_s": round(samples / composed_seconds),
                  "composed_over_render_tiles": round(composed_seconds / builtin_seconds, 2),
                  "operation_ms": {call: round(ms, 3) for call, ms in own.items()},
                  "operation_share": round(sum(own.values()) / (profiled_seconds * 1e3), 4),
                  "identical": bool(np.array_equal(got.view(np.uint32), expected.view(np.uint32))), "refused_query": refused,
                  "gpu": name, "power_limit": limit, "repeat": args.repeat}
        lines.append(json.dumps(record))
        print(lines[-1], flush=True)

    if args.out:
        with open(args.out, "w") as out:
            out.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
