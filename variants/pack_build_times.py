"""Build times of every pack of an instanced scene, three ways, on the bench's instanced scene (instanced_scene(grid=48): 2 304 placements of
two packs) and on many_packs_scene(520 packs, three layers of placements):

  mirror     host.prepare: the host mirror's SweepBuilder and LightTree, pack by pack (libecho_host.so)
  hooks      host.prepare with the per-pack device builds as its tree_builder / light_tree_builder (two device calls per pack)
  packs      echo_b200_build_packs: one call, rounds of packs of equal height, a QBVH forest and a light forest per round

Each arm runs once to warm up, then `--repeat` times; the line reports the median call time (host wall time of a synchronised call) and,
for the device arms, the levels read back (each one a synchronising read-back of the level loop). The card's name and power limit are read
in the same run. Prints one JSON line per scene and arm, and also writes them to --out when it is given.

    python variants/pack_build_times.py [--repeat 3] [--out PATH]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from echorenderer_b200 import _native, host, scene, scenes  # noqa: E402


def card():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, check=True).stdout.strip()
        name, limit = [v.strip() for v in line.split(",")]
        return name, limit
    except Exception as error:  # the numbers stay valid without it
        return f"unknown ({error})", "unknown"


def median_time(function, repeat):
    function()
    times = []
    for _ in range(repeat):
        started = time.perf_counter()
        result = function()
        times.append((time.perf_counter() - started) * 1e3)
    times.sort()
    return times[len(times) // 2], result


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--repeat", type=int, default=3)
    parser.add_argument("--out", default=None)
    args = parser.parse_args()
    name, limit = card()

    descriptions = {"instanced_grid48": scenes.instanced_scene(grid=48), "many_packs_520": scenes.many_packs_scene(pack_count=520, seed=11)}
    lines = []
    for label, description in descriptions.items():
        prepared = host.prepare(description)
        packs = len(prepared.packs)

        mirror_ms, _ = median_time(lambda: host.prepare(description), args.repeat)

        levels = {"qbvh": 0, "light": 0}

        def tree(triangles, spheres, boxes):
            result = scene.build_qbvh_device(triangles, spheres, instance_bounds=boxes)
            levels["qbvh"] += _native.last_build()["binary_levels"]
            return result

        def light(source, rows):
            result = scene.build_light_tree_device(source, rows)
            levels["light"] += _native.last_light_build()["levels"]
            return result

        def hooked():
            levels["qbvh"] = levels["light"] = 0
            return host.prepare(description, tree_builder=tree, light_tree_builder=light)

        hooks_ms, _ = median_time(hooked, args.repeat)
        hook_levels = dict(levels)

        packs_ms, built = median_time(lambda: scene.build_packs_device(prepared), args.repeat)
        stats = _native.last_pack_build()

        for arm, ms, extra in (("mirror", mirror_ms, {}),
                               ("hooks", hooks_ms, {"qbvh_levels_read_back": hook_levels["qbvh"], "light_levels_read_back": hook_levels["light"],
                                                    "device_calls": 2 * packs}),
                               ("packs", packs_ms, {"qbvh_levels_read_back": stats["qbvh_levels"], "light_levels_read_back": stats["light_levels"],
                                                    "read_backs": stats["read_backs"], "rounds": stats["rounds"], "device_build_ms": stats["build_ms"],
                                                    "launches": stats["launches"], "device_calls": 1})):
            line = {"scene": label, "packs": packs, "placements": len(prepared.instances), "arm": arm, "call_ms": round(ms, 3), **extra,
                    "what": "median host wall time of a synchronised call; mirror and hooks include host.prepare's layout work, packs is the build call alone",
                    "gpu": name, "power_limit": limit}
            print(json.dumps(line), flush=True)
            lines.append(line)

    if args.out:
        with open(args.out, "w") as handle:
            for line in lines:
                handle.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
