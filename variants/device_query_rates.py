"""Rates of the device-buffer PreparedScene queries (include/echo_b200_query_device.h) on one GPU, beside the host-buffer calls they
mirror, on the scenes and hits of variants/scene_query_rates.py (c3 mixed materials, c4 many lights, up to 16 Mi camera-ray hits).

Per scene and call, in one process:
  device_ms          the _device call on tensors already resident on the GPU, end to end including the checks on the device:
                     CUDA events around --repeat back-to-back calls on one stream after one warm-up call, divided by --repeat
  checked_kernel_ms  the device time of its checked query kernel, one call under torch.profiler (CUDA activities)
  kernel_ms          the device time of the unchecked kernel the host-buffer call launches, one call under torch.profiler
  host_ms            the host-buffer call, host wall time, median of --repeat after one warm-up call
The card's name and power limit are read in the same run. Prints one JSON line per scene and call; writes them to --out when given.

    python variants/device_query_rates.py [--repeat 10] [--hits 16777216] [--out PATH]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from echorenderer_b200 import PreparedScene, _native, host, structs  # noqa: E402
from variants.pack_build_times import card  # noqa: E402
from variants.scene_query_rates import KERNELS, SCENES, calls, kernel_milliseconds, query_inputs  # noqa: E402


def device_calls(scene, x, stream):
    """the device forms of scene_query_rates.calls on resident copies of the same inputs, and the status word they lower"""
    import torch

    def up(array, dtype):
        return torch.from_numpy(np.ascontiguousarray(array, dtype=dtype).view(np.uint8).reshape(-1).copy()).cuda()

    def out(count, dtype):
        return torch.empty(count * np.dtype(dtype).itemsize, dtype=torch.uint8, device="cuda")

    n = len(x["rays"])
    d = {"rays": up(x["rays"], structs.RAY), "hits": up(x["hits"], structs.HIT), "bounce": up(x["bounce"], np.float32), "incident": up(x["incident"], np.float32),
         "points": up(x["points"], structs.SURFACE), "pick": up(x["pick"], np.float32), "tokens": up(x["tokens"], np.uint32), "layers": up(x["layers"], structs.TOKEN_HIERARCHY),
         "radiant": up(x["radiant"], np.float32), "towards": up(x["towards"], np.float32), "directions": up(x["rays"]["direction"], np.float32),
         "contacts": out(n, structs.CONTACT), "scatter": out(n, structs.SCATTER), "rgba": out(n * 4, np.float32), "picked": out(n, np.uint32),
         "picked_layers": out(n, structs.TOKEN_HIERARCHY), "pmf": out(n, np.float32), "sample": out(n, structs.LIGHT_SAMPLE), "rgb": out(n * 3, np.float32)}
    p = {k: v.data_ptr() for k, v in d.items()}
    word = torch.full((1,), -1, dtype=torch.int64, device="cuda")
    w, s = word.data_ptr(), stream.cuda_stream
    functions = {
        "interact": lambda: scene.interact_device(p["rays"], p["hits"], None, n, p["contacts"], w, stream=s),
        "scatter_sample": lambda: scene.scatter_sample_device(p["rays"], p["hits"], None, p["bounce"], n, p["scatter"], w, stream=s),
        "scatter_evaluate": lambda: scene.scatter_evaluate_device(p["rays"], p["hits"], None, p["incident"], n, p["rgba"], w, stream=s),
        "pick": lambda: scene.pick_device(p["points"], p["pick"], n, p["picked"], p["picked_layers"], p["pmf"], w, stream=s),
        "probability_mass": lambda: scene.probability_mass_device(p["tokens"], p["layers"], p["points"], n, p["pmf"], w, stream=s),
        "sample": lambda: scene.sample_device(p["tokens"], p["layers"], p["points"], p["radiant"], n, p["sample"], w, stream=s),
        "probability_density": lambda: scene.probability_density_device(p["tokens"], p["layers"], p["points"], p["towards"], n, p["pmf"], w, stream=s),
        "evaluate_infinite": lambda: scene.evaluate_infinite_device(p["directions"], n, False, p["rgb"], w, stream=s),
    }
    return functions, word, d


def main():
    import torch

    parser = argparse.ArgumentParser()
    parser.add_argument("--repeat", type=int, default=10)
    parser.add_argument("--hits", type=int, default=1 << 24)
    parser.add_argument("--out")
    args = parser.parse_args()

    name, limit = card()
    lines = []

    for label, build in SCENES.items():
        prepared = host.prepare(build())
        with PreparedScene(prepared) as scene:
            inputs = query_inputs(scene, prepared, args.hits)
            n = len(inputs["rays"])
            stream = torch.cuda.Stream()
            functions, word, _keep = device_calls(scene, inputs, stream)

            device = {}
            with torch.cuda.stream(stream):
                for call, function in functions.items():
                    function()
                    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    start.record(stream)
                    for _ in range(args.repeat):
                        function()
                    end.record(stream)
                    end.synchronize()
                    device[call] = start.elapsed_time(end) / args.repeat
            _native.query_status(word.item())

            def on_stream(function):
                def run():
                    with torch.cuda.stream(stream):
                        function()
                    stream.synchronize()
                return run

            checked = kernel_milliseconds({call: on_stream(f) for call, f in functions.items()})

            host_functions = calls(scene, inputs)
            timed = {}
            for call, function in host_functions.items():
                function()
                times = []
                for _ in range(args.repeat):
                    started = time.perf_counter()
                    function()
                    times.append(time.perf_counter() - started)
                timed[call] = sorted(times)[len(times) // 2]
            unchecked = kernel_milliseconds(host_functions)

        for call in functions:
            rate = lambda ms: round(n / (ms / 1e3)) if ms > 0 else None  # noqa: E731
            record = {"scene": label, "call": call, "queries": n, "kernel": KERNELS[call],
                      "device_ms": round(device[call], 4), "device_queries_per_s": rate(device[call]),
                      "checked_kernel_ms": round(checked[call], 4), "checked_kernel_queries_per_s": rate(checked[call]),
                      "kernel_ms": round(unchecked[call], 4), "kernel_queries_per_s": rate(unchecked[call]),
                      "host_ms": round(timed[call] * 1e3, 3), "host_queries_per_s": rate(timed[call] * 1e3),
                      "checked_over_unchecked_kernel": round(checked[call] / unchecked[call], 4) if unchecked[call] > 0 else None,
                      "gpu": name, "power_limit": limit, "repeat": args.repeat}
            lines.append(json.dumps(record))
            print(lines[-1], flush=True)

    if args.out:
        with open(args.out, "w") as out:
            out.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
