"""Rates of the batched PreparedScene queries (include/echo_b200_query.h) on one GPU, on

  c3   scenes.mixed_material_scene()   (Dielectric, Conductor GGX, Oren-Nayar blobs)
  c4   scenes.many_lights_scene()      (10 k emissive triangles: Pick / ProbabilityMass walk a deep light tree)

The queries are made at up to 16 Mi camera-ray hits: pinhole rays through 13 jittered positions per pixel of a 1920 x 1080 frame (a third of them escape) from
the scene's camera, traced with trace_batch, the hits kept. Each call then runs on those hits or on what the calls before it
returned: interact, scatter_sample, scatter_evaluate (towards the sampled directions), pick (from the contacts), probability_mass /
sample / probability_density (of the picked lights) and evaluate_infinite (along the camera directions).

Two passes per scene, in one process. The timed pass reports queries/s end to end through the host-buffer call (host wall time of
the synchronous call, median of --repeat after one warm-up call: host validation, upload, kernel, download). The profiled pass runs
every call once under torch.profiler with CUDA activities and reports the device time of its query kernel. The card's name and
power limit are read in the same run. Prints one JSON line per scene and call; writes them to --out only when it is given.

    python variants/scene_query_rates.py [--repeat 3] [--hits 16777216] [--out PATH]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from echorenderer_b200 import PreparedScene, host, scenes, structs  # noqa: E402
from variants.pack_build_times import card  # noqa: E402

SCENES = {"c3": scenes.mixed_material_scene, "c4": scenes.many_lights_scene}
KERNELS = {"interact": "query_interact_kernel", "scatter_sample": "query_scatter_sample_kernel", "scatter_evaluate": "query_scatter_evaluate_kernel",
           "pick": "query_pick_kernel", "probability_mass": "query_mass_kernel", "sample": "query_sample_kernel",
           "probability_density": "query_pdf_kernel", "evaluate_infinite": "query_infinite_kernel"}


def camera_rays(camera, width=1920, height=1080, jitters=13, seed=1):
    """pinhole rays of the scene's camera (Entity.InverseTransform rows, forwardLength) through jittered pixel positions"""
    rng = np.random.default_rng(seed)
    matrix = camera["transform"][0].reshape(3, 4).astype(np.float64)
    ys, xs = np.meshgrid(np.arange(height), np.arange(width), indexing="ij")
    xs, ys = np.repeat(xs.reshape(-1), jitters), np.repeat(ys.reshape(-1), jitters)
    u = (xs + rng.random(len(xs))) / width - 0.5
    v = (ys + rng.random(len(ys))) / height - 0.5
    local = np.stack([u * (width / height), v, np.full(len(u), float(camera["forwardLength"][0]))], axis=1)
    direction = local @ matrix[:, :3].T
    rays = np.zeros(len(u), dtype=structs.RAY)
    rays["origin"] = matrix[:, 3].astype(np.float32)
    rays["direction"] = (direction / np.linalg.norm(direction, axis=1, keepdims=True)).astype(np.float32)
    rays["distance"], rays["ignore"] = np.inf, structs.TOKEN_EMPTY
    return rays


def query_inputs(scene, prepared, count):
    rays = camera_rays(prepared.description.camera)
    hits = scene.trace(rays)
    keep = np.flatnonzero(hits["token"] != structs.TOKEN_EMPTY)[:count]
    rays, hits = np.ascontiguousarray(rays[keep]), np.ascontiguousarray(hits[keep])
    rng = np.random.default_rng(7)
    n = len(rays)
    inputs = {"rays": rays, "hits": hits, "bounce": rng.random((n, 2), dtype=np.float32), "pick": rng.random(n, dtype=np.float32),
              "radiant": rng.random((n, 2), dtype=np.float32)}
    contacts = scene.interact(rays, hits)
    scattered = scene.scatter_sample(rays, hits, inputs["bounce"])
    incident = scattered["incident"].copy()
    incident[~(scattered["pdf"] > 0)] = rays["direction"][~(scattered["pdf"] > 0)]  # the impossible samples look back along the ray
    points = np.zeros(n, dtype=structs.SURFACE)
    points["position"], points["normal"] = contacts["position"], contacts["normal"]
    tokens, layers, _ = scene.pick(points, inputs["pick"])
    sampled = scene.sample(tokens, points, inputs["radiant"], layers)
    towards = sampled["incident"].copy()
    towards[~(sampled["pdf"] > 0)] = incident[~(sampled["pdf"] > 0)]
    inputs.update(incident=incident, points=points, tokens=tokens, layers=layers, towards=towards)
    return inputs


def calls(scene, x):
    return {
        "interact": lambda: scene.interact(x["rays"], x["hits"]),
        "scatter_sample": lambda: scene.scatter_sample(x["rays"], x["hits"], x["bounce"]),
        "scatter_evaluate": lambda: scene.scatter_evaluate(x["rays"], x["hits"], x["incident"]),
        "pick": lambda: scene.pick(x["points"], x["pick"]),
        "probability_mass": lambda: scene.probability_mass(x["tokens"], x["points"], x["layers"]),
        "sample": lambda: scene.sample(x["tokens"], x["points"], x["radiant"], x["layers"]),
        "probability_density": lambda: scene.probability_density(x["tokens"], x["points"], x["towards"], x["layers"]),
        "evaluate_infinite": lambda: scene.evaluate_infinite(x["rays"]["direction"]),
    }


def kernel_milliseconds(functions):
    """device time of each call's query kernel, one call each under torch.profiler (CUDA activities)"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    result = {}
    for name, function in functions.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            function()
            torch.cuda.synchronize()
        total = 0.0
        for event in prof.events():
            if KERNELS[name] in event.name and event.device_type.name == "CUDA":
                total += event.device_time_total if hasattr(event, "device_time_total") else event.cuda_time_total
        result[name] = total / 1e3
    return result


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--repeat", type=int, default=3)
    parser.add_argument("--hits", type=int, default=1 << 24)
    parser.add_argument("--out")
    args = parser.parse_args()

    name, limit = card()
    lines = []

    for label, build in SCENES.items():
        prepared = host.prepare(build())
        with PreparedScene(prepared) as scene:
            inputs = query_inputs(scene, prepared, args.hits)
            functions = calls(scene, inputs)
            n = len(inputs["rays"])

            timed = {}
            for call, function in functions.items():
                function()
                times = []
                for _ in range(args.repeat):
                    started = time.perf_counter()
                    function()
                    times.append(time.perf_counter() - started)
                timed[call] = sorted(times)[len(times) // 2]

            kernels = kernel_milliseconds(functions)

        for call in functions:
            record = {"scene": label, "call": call, "queries": n, "e2e_ms": round(timed[call] * 1e3, 3), "queries_per_s": round(n / timed[call]),
                      "kernel_ms": round(kernels[call], 3), "kernel_queries_per_s": round(n / (kernels[call] / 1e3)) if kernels[call] > 0 else None,
                      "gpu": name, "power_limit": limit, "repeat": args.repeat}
            lines.append(json.dumps(record))
            print(lines[-1], flush=True)

    if args.out:
        with open(args.out, "w") as out:
            out.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
