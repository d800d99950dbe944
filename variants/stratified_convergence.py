"""Image error against time for the two sample sequences: the uniform one (the default) and the stratified one
(ECHO_DISTRIBUTION_STRATIFIED, EvaluationProfile(stratified=True)), on

  c1   Cornell box 512 x 512, bounce limit 128 (the whole frame)
  c3   scenes.mixed_material_scene(), 1920 x 1080 camera, bounce limit 8: the centred 512 x 256 pixels (32 x 16 tiles of 16)
  c4   scenes.many_lights_scene(), 1920 x 1080 camera, bounce limit 128: the same centred crop

For each scene one high-spp reference is rendered with the uniform sequence and its own seed (--reference-spp, default 4096, in epochs of
256), the same for both arms. Each arm then renders at 16, 64 and 256 spp (one epoch of that many samples) and reports the relative RMSE
of the RGB against the reference and samples/s from the host wall time of the synchronised render call (median of --repeat calls after one
warm-up). The reference's own noise is part of every error, so the 256-spp errors are biased slightly upwards. From a least-squares fit
of log error against log spp per arm, `equal_error` gives the spp and the milliseconds each arm needs to reach the uniform arm's 64-spp
error at its 64-spp rate. The card's name and power limit are read in the same run. Prints one JSON line per scene / arm / spp and one per
scene / arm for the equal-error estimate, and also writes them to --out when it is given.

    python variants/stratified_convergence.py [--repeat 3] [--reference-spp 4096] [--out PATH]
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

SPPS = (16, 64, 256)
ARMS = {"uniform": structs.EVALUATOR_PATH_TRACED, "stratified": structs.DISTRIBUTION_STRATIFIED}


def centred_tiles(width, height, crop_width, crop_height, tile):
    tiles = scenes.tile_grid(width, height, tile)
    x0, y0 = (width - crop_width) // 2 // tile, (height - crop_height) // 2 // tile
    keep = (tiles[:, 0] >= x0) & (tiles[:, 0] < x0 + crop_width // tile) & (tiles[:, 1] >= y0) & (tiles[:, 1] < y0 + crop_height // tile)
    return np.ascontiguousarray(tiles[keep])


def relative_rmse(actual, expected):
    return float(np.sqrt(np.mean((actual - expected) ** 2)) / np.sqrt(np.mean(expected ** 2)))


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--repeat", type=int, default=3)
    parser.add_argument("--reference-spp", type=int, default=4096)
    parser.add_argument("--out", default=None)
    args = parser.parse_args()
    name, limit = card()
    tile = 16

    configurations = [
        ("c1", scenes.cornell_box, 512, 512, 128, None),
        ("c3", scenes.mixed_material_scene, 1920, 1080, 8, (512, 256)),
        ("c4", scenes.many_lights_scene, 1920, 1080, 128, (512, 256)),
    ]
    lines = []

    def emit(record):
        record.update(card=name, power_limit=limit)
        line = json.dumps(record)
        print(line, flush=True)
        lines.append(line)

    for label, build, width, height, bounce, crop in configurations:
        prepared = host.prepare(build())
        tiles = centred_tiles(width, height, *crop, tile) if crop else scenes.tile_grid(width, height, tile)
        pixels = len(tiles) * tile * tile

        with PreparedScene(prepared) as scene:
            epochs = max(1, args.reference_spp // 256)
            reference_params = structs.render_params(width, height, tile, extend=min(256, args.reference_spp), min_epoch=epochs, max_epoch=epochs,
                                                     bounce_limit=bounce, seed=1000)
            reference, _ = scene.render_tiles(reference_params, tiles)
            reference = reference[..., :3].astype(np.float64)
            measured = {}

            for arm, evaluator in ARMS.items():
                for spp in SPPS:
                    params = structs.render_params(width, height, tile, extend=spp, bounce_limit=bounce, seed=7, evaluator=evaluator)
                    image, _ = scene.render_tiles(params, tiles)  # warm-up; also the image the error is taken of
                    times = []
                    for _ in range(args.repeat):
                        started = time.perf_counter()
                        scene.render_tiles(params, tiles)
                        times.append(time.perf_counter() - started)
                    seconds = sorted(times)[len(times) // 2]
                    error = relative_rmse(image[..., :3].astype(np.float64), reference)
                    rate = pixels * spp / seconds
                    measured[(arm, spp)] = (error, rate)
                    emit(dict(scene=label, arm=arm, spp=spp, pixels=pixels, bounce_limit=bounce, reference_spp=epochs * min(256, args.reference_spp),
                              relative_rmse=round(error, 6), ms=round(seconds * 1e3, 3), samples_per_s=round(rate)))

            target = measured[("uniform", 64)][0]
            for arm in ARMS:
                x = np.log([float(s) for s in SPPS])
                y = np.log([measured[(arm, s)][0] for s in SPPS])
                slope, intercept = np.polyfit(x, y, 1)
                spp = float(np.exp((np.log(target) - intercept) / slope))
                rate = measured[(arm, 64)][1]
                emit(dict(scene=label, arm=arm, equal_error=round(target, 6), error_slope=round(float(slope), 4), spp_needed=round(spp, 2),
                          ms_needed=round(spp * pixels / rate * 1e3, 3), samples_per_s_at_64=round(rate)))

    if args.out:
        with open(args.out, "w") as file:
            file.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
