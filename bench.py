#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the hot path (see DESIGN.md "Measurement").

Default run (`python bench.py [--gpus N --steps K --warmup W]`, what the driver launches) prints ONE JSON line:

* headline = BASELINE.json configs[1] (C2): 1 M-triangle synthetic QBVH (+10 k spheres), 16 Mi fully incoherent rays per GPU,
  one closest-hit pass + one occlusion pass per step. `value` = Mrays/s with the inputs resident in HBM, `e2e` = the same
  through the host-buffer C ABI (page-locked host memory from echo_b200_host_alloc; `e2e_pageable` = ordinary host memory),
  `roofline` from the device visit counters, `cpu_baseline` = the oracle port on the box's host cores. Every rank traces its own
  batch: weak scaling, no data-path collective.
* `render` = the path tracer, measured the way the reference reports it (samples/s = Evaluate calls / wall time of the
  evaluation operation, Processes/ScheduledRender.cs:226-234), each record with its own roofline (algorithmic bytes per sample
  from one counted pass, SURVEY.md 8d), cpu_baseline (oracle on a crop) and plugin-call e2e (echo_b200_render_tiles into host memory):
    - `c1` (N = 1 only): the Cornell box 512x512, 16 spp per step, bounce limit 128 (BASELINE configs[0], the reference's CPU-runnable case)
    - `c3` (N = 1 only): mixed materials 1920x1080, 64 spp per step (C3's own epoch), bounce limit 8
    - `c4` (N = 1 only): 10 000 emissive triangles 1920x1080, 64 spp per step, bounce limit 128 (light-tree NEE)
    - `c5` (every N): ~10 M triangles 3840x2160, 256 spp per step (C5's own epoch), bounce limit 128, tiles sharded over the ranks
      (strong scaling), the accumulation frames merged by one NCCL all-reduce per 1024-spp render = every 4th step.

`--workload trace` / `--workload render --scene ...` run one part alone (A/B scripts in variants/). `--impl reference` times the
oracle port (the reference is C#/.NET and cannot run here) on the host cores with the same line shape.
Only this file's cpu_baseline / --impl reference legs execute oracle/ (as the timed CPU stand-in for the reference's C# path).

`--dump-outputs DIR` writes what the timed path returned in its last timed step as DIR/<name>.npy (float32 / float64, under 64 MB):
the C2 hits (a miss with distance -1) and occlusion flags of a fixed sample of rank 0's rays, and the resolved frame of every render record at a fixed sample
of its pixels. The inputs depend only on the arguments, so two builds can be compared output for output. A render's host thread
picks the kernel of a bounce from the ray counts it has seen so far (csrc/render.cu, evaluate_paths), so a stalled run can differ
from another one in a few pixels of a frame (measured on one B200 at 1000 W: C3); compare frames with a tolerance.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the tree it runs from may be read-only: nothing is written there
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from echorenderer_b200 import host, scenes, structs  # noqa: E402

MRAYS = 1e6
PATH_STATE_BYTES = 68  # wavefront path state per path (DESIGN.md "Data layout in HBM"): the S of SURVEY.md 8(d)'s B_sample


def parse():
    parser = argparse.ArgumentParser()
    parser.add_argument("--gpus", type=int, default=1)
    parser.add_argument("--steps", type=int, default=5)
    parser.add_argument("--warmup", type=int, default=3)
    parser.add_argument("--impl", default="b200", choices=["b200", "reference"])
    parser.add_argument("--workload", default="all", choices=["all", "trace", "render"],
                        help="all (default): the C2 headline plus the `render` records (C1, C3, C4 at N = 1, C5 at every N); trace / render: one part alone")
    parser.add_argument("--rays", type=int, default=1 << 24, help="rays per pass per GPU (C2: 16 Mi)")
    parser.add_argument("--quads", type=int, nargs=2, default=[1000, 500], help="terrain quads (C2: 1000 x 500 = 1 M triangles)")
    parser.add_argument("--cpu-sample", type=int, default=1 << 24,
                        help="rays per pass of the bounded CPU baseline sample (default: the whole 16 Mi-ray batch, ~1 s on 16 threads = ~13 core-seconds)")
    parser.add_argument("--width", type=int, default=1920)
    parser.add_argument("--height", type=int, default=1080)
    parser.add_argument("--spp", type=int, default=16, help="--workload render: samples per pixel per step (one epoch)")
    parser.add_argument("--scene", default="mixed", choices=["cornell", "mixed", "lights", "large", "instanced", "textured"],
                        help="--workload render scene: C1 / C3 / C4 / C5 / 2 304 placements of two packs (SURVEY.md 8f rank 2) / textured")
    parser.add_argument("--instanced", action="store_true", help="trace workload: the instanced scene instead of the C2 terrain (same ray recipe)")
    parser.add_argument("--bounce-limit", type=int, default=8, help="--workload render: PathTracedEvaluator.BounceLimit (C3: 8; reference default 128)")
    parser.add_argument("--tree", default="sah", choices=["sah", "device"],
                        help="trace workload: the SweepBuilder mirror's tree (default) or the device-built linear BVH (echo_b200_build_qbvh)")
    parser.add_argument("--shard", default="tiles", choices=["tiles", "samples"],
                        help="render, N > 1: tile sharding (blocks of the tile sequence dealt round-robin) or sample sharding (every rank renders spp / N samples of every tile)")
    parser.add_argument("--shard-by", default="position", choices=["position", "sequence"],
                        help="tile sharding: tile (x, y) -> rank (x + y) mod N (default: every rank samples the whole image, balanced shards) or blocks of the tile sequence")
    parser.add_argument("--shard-block", type=int, default=64, help="--shard-by sequence: consecutive tiles of the sequence per block (block b -> rank b mod N)")
    parser.add_argument("--pattern", default="hilbert", choices=["hilbert", "ordered"],
                        help="render: tile sequence, the HilbertCurvePattern of EvaluationProfile.Pattern (reference default) or an OrderedPattern")
    parser.add_argument("--reduce-every", type=int, default=1, help="--workload render: steps (epochs) accumulated on the device between frame all-reduces")
    parser.add_argument("--render-steps", type=int, default=None, help="default run: timed steps of each `render` record (default: --steps; at most --steps when given)")
    parser.add_argument("--render-warmup", type=int, default=1, help="default run: warm-up steps of each `render` record (a C5 step is seconds long)")
    parser.add_argument("--no-render", action="store_true", help="default run: skip the `render` records")
    parser.add_argument("--no-cpu-baseline", action="store_true")
    parser.add_argument("--no-tree-build", action="store_true", help="skip the device tree build record (device SweepBuilder beside the host mirror)")
    parser.add_argument("--no-secondary", action="store_true", help="skip the secondary-ray batch reported beside the headline (SURVEY.md 8d)")
    parser.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (rank 0; --impl b200)")
    args = parser.parse_args()
    if args.steps < 1:
        parser.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        parser.error("--dump-outputs records the outputs of the device path (--impl b200)")
    return args


DUMP_SAMPLES = 1 << 19  # rays per C2 output (12 MiB in all); a render frame keeps half as many pixels (RGBA, 4 MiB): 28 MiB for the default run


def dump_sample(count, limit):
    """A fixed, seeded choice of `limit` of `count` indices, ascending (every index when there are no more than `limit`)."""
    if count <= limit:
        return np.arange(count)
    return np.sort(np.argsort(scenes.uniform(5, np.arange(count, dtype=np.uint64)), kind="stable")[:limit])


def dump_outputs(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, array in arrays.items():
        assert array.dtype in (np.float32, np.float64) and np.isfinite(array).all(), name
        np.save(os.path.join(directory, f"{name}.npy"), array)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as file:
            return float(json.load(file)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed `ncu --set full` capture of this
    command (profiles/ncu_traffic.json); null when no capture has been recorded."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        with open(path) as file:
            return json.load(file).get(key)
    return None


def measured_on_chip_peaks(device):
    """L2 read bandwidth and L1 sector (LSU wavefront) rate measured live by the library's own microbenchmark kernels
    (echo_b200_debug_measure_peak, csrc/peaks.cu): the ceilings the traversal kernel actually runs against, since its working set
    (72 MB of nodes) lives in L2 and its loads are divergent 32-byte sector fetches. None when the library has no such entry."""
    from echorenderer_b200 import _native
    try:
        return _native.measure_peaks(device)
    except (AttributeError, _native.EchoNativeError):
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe). nvidia-smi needs a moment to
    start, so the sampler is started before the warm-up and `mark()`s delimit the timed region; samples are stamped on arrival."""
    QUERY = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.lines, self.process, self.index, self.window = [], None, index, [None, None]

    def __enter__(self):
        try:
            self.process = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "20"],
                                            stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            deadline = time.time() + 3.0
            while not self.lines and time.time() < deadline:
                time.sleep(0.02)
        except OSError:
            self.process = None
        return self

    def _read(self):
        for line in self.process.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self, which):
        self.window[which] = time.time()

    def __exit__(self, *_):
        if self.process:
            self.process.terminate()
            try:
                self.process.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.process.kill()

    def summary(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        begin, end = self.window
        rows = []
        for stamp, line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                rows.append((stamp, float(parts[0]), float(parts[1]), [n for n, f in zip(names, parts[4:8]) if f.lower().startswith("active")]))
            except ValueError:
                continue
        inside = [r for r in rows if begin is not None and end is not None and begin - 0.03 <= r[0] <= end + 0.03]
        scope = "timed region"
        if not inside:  # region shorter than the sampling period: fall back to every sample taken under load (warm-up + timed)
            inside, scope = [r for r in rows if begin is None or r[0] >= begin - 1.0], "warm-up + timed region"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        reasons = sorted({reason for r in inside for reason in r[3]})
        return {"sm_mhz": float(np.median([r[1] for r in inside])), "sm_max_mhz": max(r[2] for r in inside), "reasons": reasons,
                "samples": len(inside), "scope": scope}


class Context:
    """torch / NCCL plumbing of one rank: device, stream, barrier and max-over-ranks."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.distributed = self.world > 1
        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)
        if self.distributed:
            dist.init_process_group("nccl", device_id=self.device)
        self.stream = torch.cuda.current_stream().cuda_stream

    def barrier(self):
        if self.distributed:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, value):
        if not self.distributed:
            return value
        tensor = self.torch.tensor([value], dtype=self.torch.float64, device=self.device)
        self.dist.all_reduce(tensor, op=self.dist.ReduceOp.MAX)
        return float(tensor.item())

    def sum_over_ranks(self, value):
        if not self.distributed:
            return value
        tensor = self.torch.tensor([value], dtype=self.torch.float64, device=self.device)
        self.dist.all_reduce(tensor)
        return float(tensor.item())

    def gather(self, value):
        if not self.distributed:
            return [value]
        tensor = self.torch.tensor([value], dtype=self.torch.float64, device=self.device)
        out = [self.torch.zeros_like(tensor) for _ in range(self.world)]
        self.dist.all_gather(out, tensor)
        return [float(t.item()) for t in out]

    def close(self):
        if self.distributed:
            self.dist.destroy_process_group()


def instanced_bench_scene():
    return scenes.instanced_scene(grid=48, rings=128, segments=130)


def build_trace_inputs(args, rank):
    description = instanced_bench_scene() if getattr(args, "instanced", False) else scenes.terrain_scene(args.quads[0], args.quads[1], 10000)
    tree = None
    if getattr(args, "tree", "sah") == "device" and not getattr(args, "instanced", False):
        from echorenderer_b200 import build_qbvh_device
        build_qbvh_device(description.triangles[:64], description.spheres[:0], device=int(os.environ.get("LOCAL_RANK", "0")))  # context + module load
        started = time.perf_counter()
        tree = build_qbvh_device(description.triangles, description.spheres, device=int(os.environ.get("LOCAL_RANK", "0")))
        args.tree_build_seconds = time.perf_counter() - started
    started = time.perf_counter()
    prepared = host.prepare(description, tree=tree)
    args.prepare_seconds = time.perf_counter() - started
    # every rank traces its own batch (distinct seeds per rank)
    rays = scenes.random_rays(prepared.bounds, args.rays, seed=11 + 1000 * rank)
    shadow = rays.copy()
    low, high = prepared.bounds
    diagonal = float(np.linalg.norm(np.asarray(high, np.float64) - np.asarray(low, np.float64)))
    shadow["distance"] = scenes.uniform(17 + 1000 * rank, np.arange(args.rays, dtype=np.uint64)) * np.float32(diagonal)
    return prepared, rays, shadow


def tree_build_record(prepared, device):
    """The device-side SweepBuilder (echo_b200_build_qbvh, csrc/sweep.cu) on the headline's geometry beside the host mirror of the reference's
    recursive build: the whole call from host buffers, its phases, and whether the two node arrays are the same bytes. Not part of `value`."""
    from echorenderer_b200 import _native, build_qbvh_device
    triangles, spheres = prepared.triangles, prepared.spheres
    build_qbvh_device(triangles[:64], spheres[:0], device=device)  # context + module load
    calls = []
    for _ in range(3):
        started = time.perf_counter()
        nodes, depth = build_qbvh_device(triangles, spheres, device=device)
        calls.append(((time.perf_counter() - started) * 1e3, _native.last_build()))
    call_ms, phases = min(calls, key=lambda pair: pair[0])
    started = time.perf_counter()
    expected, expected_depth = host.build_qbvh(triangles, spheres)
    host_ms = (time.perf_counter() - started) * 1e3
    return {"what": "the reference's SweepBuilder tree (SweepBuilder.cs + the QBVH collapse) built level-synchronously on the device: echo_b200_build_qbvh from host buffers, best of 3 calls",
            "primitives": int(len(triangles) + len(spheres)), "nodes": int(len(nodes)), "quad_depth": int(depth), "call_ms": call_ms, **phases,
            "host_mirror_ms": host_ms, "host_mirror_threads": os.cpu_count(), "identical_to_host_mirror": bool(depth == expected_depth and nodes.tobytes() == expected.tobytes())}


def light_tree_build_record(prepared, device):
    """The device-side LightTree.Build (echo_b200_build_light_tree, csrc/lightbuild.cu) on a scene's emitters beside the host mirror of the
    reference's recursive build: the whole call from host buffers, its phases, and whether nodes and emitter map are the same bytes."""
    from echorenderer_b200 import _native, build_light_tree_device
    description = prepared.description
    build_light_tree_device(description, device=device)  # context + module load
    calls = []
    for _ in range(3):
        started = time.perf_counter()
        nodes, tokens, paths, power = build_light_tree_device(description, device=device)
        calls.append(((time.perf_counter() - started) * 1e3, _native.last_light_build()))
    call_ms, phases = min(calls, key=lambda pair: pair[0])
    started = time.perf_counter()
    expected_nodes, expected_tokens, expected_paths, _ = host.build_light_tree(description)
    host_ms = (time.perf_counter() - started) * 1e3
    identical = nodes.tobytes() == expected_nodes.tobytes() and tokens.tobytes() == expected_tokens.tobytes() and paths.tobytes() == expected_paths.tobytes()
    return {"what": "the reference's light tree (LightCollection.CreateBounds + LightTree.Build + AddToMap) built level-synchronously on the device: echo_b200_build_light_tree from host buffers, best of 3 calls; "
                    "a node's two sweeps are chains of non-associative cone unions, one thread each, so the time is a few chain lengths",
            "candidates": int(len(description.triangles) + len(description.spheres) + len(description.point_lights)), "emitters": int(len(tokens)), "nodes": int(len(nodes)),
            "call_ms": call_ms, **phases, "host_mirror_ms": host_ms, "host_mirror_threads": 1, "identical_to_host_mirror": bool(identical)}


def secondary_batch(scene, prepared, rays, d_hits, ctx, args):
    """The second batch SURVEY.md §8(d) asks to report beside the headline: rays leaving the surfaces the first batch hit
    (cosine-hemisphere directions, ignore = hit token, as TraceQuery.SpawnTrace does), tiled up to the size of the first batch.
    Reported separately; it is not part of `value`."""
    torch, device, stream = ctx.torch, ctx.device, ctx.stream
    hits = d_hits.cpu().numpy().view(structs.HIT)
    spawned = scenes.secondary_rays(prepared, rays, hits)
    if len(spawned) == 0:
        return None
    unique = len(spawned)
    spawned = np.tile(spawned, (len(rays) + unique - 1) // unique)[:len(rays)]
    n = len(spawned)
    shadow = spawned.copy()
    low, high = prepared.bounds
    diagonal = float(np.linalg.norm(np.asarray(high, np.float64) - np.asarray(low, np.float64)))
    shadow["distance"] = scenes.uniform(29, np.arange(n, dtype=np.uint64)) * np.float32(diagonal)

    d_rays = torch.from_numpy(spawned.view(np.uint8).reshape(-1)).to(device)
    d_shadow = torch.from_numpy(shadow.view(np.uint8).reshape(-1)).to(device)
    d_out = torch.empty(n * 16, dtype=torch.uint8, device=device)
    d_flags = torch.empty(n, dtype=torch.uint8, device=device)
    d_counts = torch.zeros(6, dtype=torch.int64, device=device)
    scene.trace_device(d_rays.data_ptr(), n, d_out.data_ptr(), stream, d_counts.data_ptr())
    scene.occlude_device(d_shadow.data_ptr(), n, d_flags.data_ptr(), stream, d_counts.data_ptr() + 24)
    torch.cuda.synchronize()
    counts = d_counts.cpu().numpy().astype(np.float64) / n
    hit_rate = float(np.mean(d_out.cpu().numpy().view(structs.HIT)["token"] != structs.TOKEN_EMPTY))

    for _ in range(args.warmup):
        scene.trace_device(d_rays.data_ptr(), n, d_out.data_ptr(), stream)
        scene.occlude_device(d_shadow.data_ptr(), n, d_flags.data_ptr(), stream)
    events = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    trace_ms = occlude_ms = 0.0
    torch.cuda.synchronize()
    for _ in range(args.steps):
        events[0].record()
        scene.trace_device(d_rays.data_ptr(), n, d_out.data_ptr(), stream)
        events[1].record()
        scene.occlude_device(d_shadow.data_ptr(), n, d_flags.data_ptr(), stream)
        events[2].record()
        torch.cuda.synchronize()
        trace_ms += events[0].elapsed_time(events[1]) / args.steps
        occlude_ms += events[1].elapsed_time(events[2]) / args.steps
    trace_ms, occlude_ms = ctx.max_over_ranks(trace_ms), ctx.max_over_ranks(occlude_ms)
    bytes_trace = 32 + 16 + 128 * counts[0] + 36 * counts[1] + 16 * counts[2]
    bytes_occlude = 32 + 1 + 128 * counts[3] + 36 * counts[4] + 16 * counts[5]
    return {"rays_per_pass_per_gpu": n, "distinct_rays": unique, "hit_rate": hit_rate,
            "closest_hit": {"mrays_per_s": n / (trace_ms * 1e-3) / MRAYS, "ms_per_launch": trace_ms, "algorithmic_bytes_per_query": bytes_trace,
                            "achieved_gbs": bytes_trace * n / (trace_ms * 1e-3) / 1e9,
                            "visits_per_query": {"nodes": counts[0], "triangles": counts[1], "spheres": counts[2]}},
            "occlusion": {"mrays_per_s": n / (occlude_ms * 1e-3) / MRAYS, "ms_per_launch": occlude_ms, "algorithmic_bytes_per_query": bytes_occlude,
                          "achieved_gbs": bytes_occlude * n / (occlude_ms * 1e-3) / 1e9,
                          "visits_per_query": {"nodes": counts[3], "triangles": counts[4], "spheres": counts[5]}}}


def cpu_baseline_trace(prepared, rays, shadow, sample, threads=0):
    """The oracle (C++ restatement of the reference's CPU path) on a bounded sample, all host threads."""
    from tests import oracle_lib
    oracle = oracle_lib.OracleScene(prepared)
    sample = min(sample, len(rays))
    cores = threads or os.cpu_count() or 1
    oracle.trace(rays[:4096], threads=cores)  # warm-up (page in the scene)
    start = time.perf_counter()
    oracle.trace(rays[:sample], threads=cores)
    oracle.occlude(shadow[:sample], threads=cores)
    seconds = time.perf_counter() - start
    whole = "all" if sample == len(rays) else "first"
    return 2 * sample / seconds / MRAYS, cores, seconds, f"{whole} {sample} closest-hit + {sample} occlusion queries of the rank-0 batch, {cores} threads"


def crop_tiles(width, height, tile, budget_samples, spp):
    """A centred block of tiles holding about `budget_samples` samples at `spp`: the bounded sample of a frame for the CPU legs."""
    tiles_x, tiles_y = (width + tile - 1) // tile, (height + tile - 1) // tile
    wanted = int(min(max(budget_samples // (tile * tile * spp), 4), tiles_x * tiles_y))
    columns = int(min(tiles_x, max(2, round((wanted * tiles_x / tiles_y) ** 0.5))))
    rows = int(min(tiles_y, max(2, (wanted + columns - 1) // columns)))
    x0, y0 = (tiles_x - columns) // 2, (tiles_y - rows) // 2
    ty, tx = np.meshgrid(np.arange(y0, y0 + rows), np.arange(x0, x0 + columns), indexing="ij")
    return np.stack([tx.reshape(-1), ty.reshape(-1)], axis=-1).astype(np.int32)


def cpu_baseline_render(prepared, width, height, tile, spp, bounce_limit, budget_samples=64_000_000):  # ~10 s on 16 host threads
    """The oracle's EvaluationOperation.Execute on a centred crop of the frame at the same samples per pixel, one tile per
    procedure on all host threads (Processes/Evaluation/EvaluationOperation.cs:83-148)."""
    from tests import oracle_lib
    oracle = oracle_lib.OracleScene(prepared)
    cores = os.cpu_count() or 1
    crop = crop_tiles(width, height, tile, budget_samples, spp)
    params = structs.render_params(width, height, tile, extend=spp, min_epoch=1, max_epoch=1, bounce_limit=bounce_limit)
    start = time.perf_counter()
    _, stats = oracle.render_tiles(params, crop, threads=cores)
    seconds = time.perf_counter() - start
    samples = int(stats["sampleEvaluated"][0])
    return {"value": samples / seconds, "unit": "samples/s", "cores": cores, "kind": "port", "seconds": seconds,
            "sample": f"{len(crop)} central tiles of the {width}x{height} frame at {spp} spp ({samples} samples), oracle port on {cores} threads"}


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path. Echo is C#/.NET 6 and cannot be built or run
    here (no dotnet), so the C++ oracle port stands in, on all host threads; each step is a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return

    if args.workload in ("all", "trace"):
        prepared, rays, shadow = build_trace_inputs(argparse.Namespace(**{**vars(args), "rays": args.cpu_sample}), 0)
        from tests import oracle_lib
        oracle = oracle_lib.OracleScene(prepared)
        cores = os.cpu_count() or 1
        times = []
        for step in range(args.warmup + args.steps):
            start = time.perf_counter()
            oracle.trace(rays, threads=cores)
            oracle.occlude(shadow, threads=cores)
            if step >= args.warmup:
                times.append(time.perf_counter() - start)
        seconds = sum(times)
        value = 2 * len(rays) * args.steps / seconds / MRAYS
        sample = f"{len(rays)} closest-hit + {len(rays)} occlusion queries per step ({'the whole' if len(rays) == args.rays else 'a bounded sample of the'} {args.rays}-ray batch), {cores} threads"
        line = base_line(args, "Mrays/s", value, seconds / args.steps * 1e3, trace_config(args, len(rays)), "f32")
    else:
        prepared = host.prepare(RENDER_SCENES[args.scene][1]())
        from tests import oracle_lib
        oracle = oracle_lib.OracleScene(prepared)
        cores = os.cpu_count() or 1
        params = structs.render_params(args.width, args.height, 16, extend=args.spp, min_epoch=1, max_epoch=1, bounce_limit=args.bounce_limit)
        crop = crop_tiles(args.width, args.height, 16, 144 * 256 * args.spp, args.spp)
        times, samples = [], 0
        for step in range(args.warmup + args.steps):
            start = time.perf_counter()
            _, stats = oracle.render_tiles(params, crop, threads=cores)
            if step >= args.warmup:
                times.append(time.perf_counter() - start)
                samples += int(stats["sampleEvaluated"][0])
        seconds = sum(times)
        value = samples / seconds
        sample = f"{len(crop)} central tiles of the {args.width}x{args.height} frame at {args.spp} spp per step"
        line = base_line(args, "samples/s", value, seconds / args.steps * 1e3, render_config(args, args.scene, args.width, args.height, args.spp, args.bounce_limit), "f32")

    line["impl"] = "reference"
    line["cpu_baseline"] = {"value": line["value"], "unit": line["unit"], "cores": cores, "kind": "port", "sample": sample}
    line["e2e"] = {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    line["gpu_launches"] = 0
    emit(line)


def trace_config(args, rays):
    if getattr(args, "instanced", False):
        return {"workload": "incoherent ray-batch intersection through instanced packs (48 x 48 placements of a 33 k-triangle pack and of a pack of three of those): closest-hit + occlusion",
                "rays_per_pass_per_gpu": rays, "passes_per_step": 2, "parallelism": f"replicated scene x{args.gpus}",
                "l2": "inputs larger than L2 (ray batch 512 MiB + hit buffer 256 MiB per pass vs 126 MB L2)"}
    return {"workload": "C2 incoherent ray-batch intersection: closest-hit + occlusion", "triangles": args.quads[0] * args.quads[1] * 2,
            "spheres": 10000, "rays_per_pass_per_gpu": rays, "passes_per_step": 2, "parallelism": f"replicated scene x{args.gpus}",
            "l2": "inputs larger than L2 (ray batch 512 MiB + hit buffer 256 MiB per pass vs 126 MB L2)"}


RENDER_SCENES = {
    "cornell": ("C1 Cornell box (CornellBox.cs / cornell.echo)", scenes.cornell_box),
    "mixed": ("C3 mixed-material scene (Dielectric, Conductor GGX, Oren-Nayar)", scenes.mixed_material_scene),
    "lights": ("C4 many-lights scene (10 k emissive triangles, light-tree NEE)", scenes.many_lights_scene),
    "large": ("C5 ~10 M-triangle terrain with the C3 material mix", scenes.large_scene),
    "textured": ("image textures in every material slot, normal map, alpha cut-out (SURVEY.md 8f rank 3)", lambda: scenes.textured_scene(rings=128, segments=130)),
    "instanced": ("2 304 placements of two packs (one nests three placements of the other), lights inside the packs", instanced_bench_scene),
}


def render_config(args, scene_key, width, height, spp, bounce_limit, reduce_every=1):
    sharding = f"every rank renders {spp} / {args.gpus} samples of every tile" if args.shard == "samples" else \
        ("tile (x, y) -> rank (x + y) mod N, rendered in sequence order" if args.shard_by == "position" else f"blocks of {args.shard_block} tiles of the sequence dealt round-robin")
    return {"workload": f"{RENDER_SCENES[scene_key][0]}, path tracer bounce limit {bounce_limit}", "width": width, "height": height, "spp_per_step": spp,
            "parallelism": f"scene replicated x{args.gpus}, {sharding}, accumulation frames merged by one NCCL all-reduce every {reduce_every} step(s)",
            "tile_pattern": args.pattern, "l2": "wavefront state (up to ~4 GB per pipeline) larger than L2"}


def base_line(args, unit, value, ms_per_step, config, dtype):
    # trace: every rank traces its own batch (weak); render: one fixed frame sharded by tiles (strong)
    return {"metric": "Mrays/s" if unit == "Mrays/s" else "samples/sec", "value": value, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak" if unit == "Mrays/s" else "strong", "vs_baseline": None,
            "dtype": dtype, "data": "synthetic", "config": config}


_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version banner from C when the box
    sets NCCL_DEBUG=VERSION), so file descriptor 1 points at stderr while the bench runs and emit() writes to the real one."""
    global _STDOUT
    if _STDOUT is None:
        sys.stdout.flush()
        _STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _STDOUT if _STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def note(ctx, message):
    if ctx.rank == 0:
        print(f"[bench {time.strftime('%H:%M:%S')}] {message}", file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# C2: the headline
# ---------------------------------------------------------------------------------------------------------------------

def run_trace(ctx, args):
    from echorenderer_b200 import PreparedScene, _native
    torch, device, stream = ctx.torch, ctx.device, ctx.stream
    peak, peak_source = peaks()

    prepared, rays, shadow = build_trace_inputs(args, ctx.rank)
    scene = PreparedScene(prepared, device=ctx.local_rank)
    n = len(rays)

    # host buffers of the plugin-call leg: page-locked memory from the library's own allocator (what a P/Invoke host would use)
    host_rays, host_shadow = _native.HostBuffer(n, structs.RAY), _native.HostBuffer(n, structs.RAY)
    host_hits, host_occluded = _native.HostBuffer(n, structs.HIT), _native.HostBuffer(n, np.uint8)
    host_rays.array[:] = rays
    host_shadow.array[:] = shadow

    d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1)).to(device)
    d_shadow = torch.from_numpy(shadow.view(np.uint8).reshape(-1)).to(device)
    d_hits = torch.empty(n * 16, dtype=torch.uint8, device=device)
    d_occluded = torch.empty(n, dtype=torch.uint8, device=device)
    d_counts = torch.zeros(6, dtype=torch.int64, device=device)

    # visit counters -> algorithmic bytes per query (SURVEY.md §8d); one untimed counted pass
    scene.trace_device(d_rays.data_ptr(), n, d_hits.data_ptr(), stream, d_counts.data_ptr())
    scene.occlude_device(d_shadow.data_ptr(), n, d_occluded.data_ptr(), stream, d_counts.data_ptr() + 24)
    torch.cuda.synchronize()
    counts = d_counts.cpu().numpy().astype(np.float64) / n
    bytes_trace = 32 + 16 + 128 * counts[0] + 36 * counts[1] + 16 * counts[2]
    bytes_occlude = 32 + 1 + 128 * counts[3] + 36 * counts[4] + 16 * counts[5]

    def step():
        scene.trace_device(d_rays.data_ptr(), n, d_hits.data_ptr(), stream)
        scene.occlude_device(d_shadow.data_ptr(), n, d_occluded.data_ptr(), stream)

    events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]

    with ClockSampler(ctx.local_rank) as clocks:
        for _ in range(args.warmup):
            step()
        ctx.barrier()

        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks.mark(0)
        start.record()
        for first, middle, last in events:
            first.record()
            scene.trace_device(d_rays.data_ptr(), n, d_hits.data_ptr(), stream)
            middle.record()
            scene.occlude_device(d_shadow.data_ptr(), n, d_occluded.data_ptr(), stream)
            last.record()
        stop.record()
        ctx.barrier()
        clocks.mark(1)
        total_ms = ctx.max_over_ranks(start.elapsed_time(stop))

    if args.dump_outputs and ctx.rank == 0:
        keep = torch.from_numpy(dump_sample(n, DUMP_SAMPLES)).to(device)
        hits = d_hits.view(n, 16)[keep].cpu().numpy().view(structs.HIT).reshape(-1)
        # a miss returns the ray's limit, +inf for these rays; the token already marks it, so its distance is stored as -1 (no hit has that)
        distance = np.where(hits["token"] == structs.TOKEN_EMPTY, np.float32(-1.0), hits["distance"])
        dump_outputs(args.dump_outputs, {"trace_token": hits["token"].astype(np.float64), "trace_distance": distance, "trace_uv": hits["uv"],
                                         "occluded": d_occluded[keep].cpu().numpy().astype(np.float32)})

    trace_ms = float(np.mean([a.elapsed_time(b) for a, b, _ in events]))
    occlude_ms = float(np.mean([b.elapsed_time(c) for _, b, c in events]))
    value = ctx.world * 2 * n * args.steps / (total_ms * 1e-3) / MRAYS

    # end to end through the host-buffer C ABI: host rays in, hits / occlusion flags out, every step
    def e2e_leg(rays_pointer, shadow_pointer, hits_pointer, occluded_pointer, steps):
        for _ in range(2):
            scene.trace_pointers(rays_pointer, n, hits_pointer)
        ctx.barrier()
        wall = time.perf_counter()
        for _ in range(steps):
            scene.trace_pointers(rays_pointer, n, hits_pointer)
            scene.occlude_pointers(shadow_pointer, n, occluded_pointer)
        ctx.barrier()
        ms = ctx.max_over_ranks((time.perf_counter() - wall) * 1e3)
        return ctx.world * 2 * n * steps / (ms * 1e-3) / MRAYS, ms / steps

    e2e_value, e2e_ms = e2e_leg(host_rays.address, host_shadow.address, host_hits.address, host_occluded.address, args.steps)
    # the same from ordinary (pageable) host memory: what a `fixed`-pinned managed array is to CUDA
    pageable_hits, pageable_occluded = np.empty(n, dtype=structs.HIT), np.empty(n, dtype=np.uint8)
    pageable_value, pageable_ms = e2e_leg(rays.ctypes.data, shadow.ctypes.data, pageable_hits.ctypes.data, pageable_occluded.ctypes.data, min(args.steps, 3))

    # The ceiling of that leg: the bare copies of one step (H2D of both ray batches, D2H of hits and flags, the two directions on
    # two streams as in the library's pipeline) with no kernel at all, all ranks at the same time — what the host's memory system and
    # the PCIe links deliver when N ranks move their batches at once. `e2e` is reported as a fraction of it.
    pinned = [torch.from_numpy(buffer.array.view(np.uint8).reshape(-1)) for buffer in (host_rays, host_shadow, host_hits, host_occluded)]
    up, down = torch.cuda.Stream(device=device), torch.cuda.Stream(device=device)

    def bare_copies():
        with torch.cuda.stream(up):
            d_rays.copy_(pinned[0], non_blocking=True)
            d_shadow.copy_(pinned[1], non_blocking=True)
        with torch.cuda.stream(down):
            pinned[2].copy_(d_hits, non_blocking=True)
            pinned[3].copy_(d_occluded, non_blocking=True)

    bare_copies()
    ctx.barrier()
    wall = time.perf_counter()
    for _ in range(args.steps):
        bare_copies()
    ctx.barrier()
    copy_ms = ctx.max_over_ranks((time.perf_counter() - wall) * 1e3) / args.steps
    del pinned

    line = base_line(args, "Mrays/s", value, total_ms / args.steps, trace_config(args, n), "f32")
    achieved = bytes_trace * n / (trace_ms * 1e-3) / 1e9
    line["roofline"] = {"bound": "hbm", "kernel": "instanced closest-hit kernel" if args.instanced else "persistent_batch_kernel<48, false> (closest hit)", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_nominal_8tbs": achieved / 8000.0,
                        "traffic": ncu_traffic("closest_hit_dram_bytes_per_launch"), "peak_source": peak_source, "algorithmic_bytes_per_query": bytes_trace, "ms_per_launch": trace_ms,
                        "mrays_per_s": n / (trace_ms * 1e-3) / MRAYS,
                        "visits_per_query": {"nodes": counts[0], "triangles": counts[1], "spheres": counts[2]},
                        "occlusion": {"kernel": "persistent_batch_kernel<48, true>", "traffic": ncu_traffic("occlusion_dram_bytes_per_launch"), "achieved": bytes_occlude * n / (occlude_ms * 1e-3) / 1e9, "algorithmic_bytes_per_query": bytes_occlude,
                                      "ms_per_launch": occlude_ms, "mrays_per_s": n / (occlude_ms * 1e-3) / MRAYS,
                                      "visits_per_query": {"nodes": counts[3], "triangles": counts[4], "spheres": counts[5]}}}

    # what the kernel is actually bound by (ncu, profiles/README.md): divergent 32-byte sector fetches through the L1 data pipe
    # and L2 latency; the 72 MB node array lives in L2, DRAM carries little more than the ray / hit streams. The on-chip ceilings
    # are measured live by the library's microbenchmark kernels and the same algorithmic bytes are set against them.
    on_chip = measured_on_chip_peaks(ctx.local_rank)
    if on_chip:
        tree_bytes = (bytes_trace - 48) * n  # node + primitive bytes: served by L2 / L1, not by DRAM
        line["roofline"].update({
            "bound_measured": "L1/TEX data pipe (divergent sector fetches) + L2 latency, not DRAM (ncu: profiles/README.md)",
            "l2_peak_gbs": on_chip["l2_read_gbs"], "frac_l2": achieved / on_chip["l2_read_gbs"],
            "l2_sector_peak_gbs": on_chip["l2_sector_gbs"], "frac_l2_sectors": tree_bytes / (trace_ms * 1e-3) / 1e9 / on_chip["l2_sector_gbs"],
            "l1_sector_peak_gbs": on_chip["l1_sector_gbs"], "frac_l1_sectors": tree_bytes / (trace_ms * 1e-3) / 1e9 / on_chip["l1_sector_gbs"],
            "fractions": "frac = all algorithmic bytes / HBM copy peak; frac_l2 = the same bytes / coalesced L2 read peak; frac_l2_sectors, frac_l1_sectors = node + primitive bytes "
                         "(what the divergent 32-byte sector fetches carry) / the measured random-sector rate out of L2, out of L1",
            "on_chip_peaks": on_chip})

    line["e2e"] = {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": 2 * n * 32, "d2h_bytes_per_step": n * 16 + n, "ms_per_step": e2e_ms,
                   "host_memory": "page-locked (echo_b200_host_alloc)",
                   "copy_ceiling": {"ms_per_step": copy_ms, "gbs_per_rank": (2 * n * 32 + n * 17) / (copy_ms * 1e-3) / 1e9, "gbs_all_ranks": ctx.world * (2 * n * 32 + n * 17) / (copy_ms * 1e-3) / 1e9,
                                    "what": "the same host<->device copies with no kernels, up and down on two streams, all ranks at once"},
                   "frac_of_copy_ceiling": copy_ms / e2e_ms}
    line["e2e_pageable"] = {"value": pageable_value, "unit": "Mrays/s", "ms_per_step": pageable_ms, "host_memory": "pageable (what a `fixed`-pinned managed array is to CUDA); the library stages it through page-locked buffers, one host thread per pipeline slot"}
    line["gpu_launches"] = 2 * args.steps
    line["clocks"] = clocks.summary()
    line["config"]["tree"] = {"builder": args.tree, "nodes": int(len(prepared.nodes)), "quad_depth": int(prepared.max_depth),
                              "device_build_seconds": getattr(args, "tree_build_seconds", None), "host_prepare_seconds": getattr(args, "prepare_seconds", None)}

    if not args.no_secondary and not args.instanced:
        line["secondary"] = secondary_batch(scene, prepared, rays, d_hits, ctx, args)

    if ctx.rank == 0 and not args.instanced and not args.no_tree_build:
        line["tree_build"] = tree_build_record(prepared, ctx.local_rank)

    if ctx.rank == 0 and not args.no_cpu_baseline:
        cpu_value, cores, seconds, sample = cpu_baseline_trace(prepared, rays, shadow, args.cpu_sample)
        line["cpu_baseline"] = {"value": cpu_value, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample, "seconds": seconds}
        # SURVEY.md 8(d): the single-thread rate too, to set beside the reference's published single-thread figures (BASELINE.md: 1.68 / 2.06 Mrays/s in C#)
        single_value, _, single_seconds, single_sample = cpu_baseline_trace(prepared, rays, shadow, max(4096, min(args.cpu_sample, len(rays)) // 16), threads=1)
        line["cpu_baseline"]["single_thread"] = {"value": single_value, "unit": "Mrays/s", "cores": 1, "sample": single_sample, "seconds": single_seconds}

    for buffer in (host_rays, host_shadow, host_hits, host_occluded):
        buffer.free()
    scene.close()
    return line


# ---------------------------------------------------------------------------------------------------------------------
# the path tracer
# ---------------------------------------------------------------------------------------------------------------------

def bytes_per_sample(stats):
    """SURVEY.md §8(d)'s B_sample from the counters of one counted pass:
       B_sample = sum over bounces [ B_trace + 64 (rest of the hit triangle) + 64 (material) + p_nee (64 D_lt + 36 (emitter) + B_occl) + 2 S ] + 16
    with B_trace = 32 + 16 + 128 N_node + 36 N_tri + 16 N_sph and B_occl = 32 + 1 + the same visit terms. Summed over a pass:
    trace queries x 48 + occlusion queries x 33 + 128 node visits + 36 triangle visits + 16 sphere visits (both kinds of query)
    + 128 per surface hit + 36 per sampled light + 64 per light-tree node visit + 2 S per trace query + 16 per sample."""
    get = lambda name: float(stats[name][0])
    samples = get("sampleEvaluated")
    hits = get("traceQueries") - get("lightEvaluatedInfinite")  # "Light/Evaluated Infinite" counts exactly the trace queries that escaped
    parts = {
        "queries": 48 * get("traceQueries") + 33 * get("occludeQueries"),
        "nodes": 128 * get("nodeVisits"),
        "primitives": 36 * get("triangleVisits") + 16 * get("sphereVisits"),
        "surface": 128 * hits,
        "lights": 36 * get("lightSampled") + 64 * get("lightNodeVisits"),
        "path_state": 2 * PATH_STATE_BYTES * get("traceQueries"),
        "pixel": 16 * samples,
    }
    per_sample = {key: value / samples for key, value in parts.items()}
    counters = {"trace_queries": get("traceQueries") / samples, "occlude_queries": get("occludeQueries") / samples, "node_visits": get("nodeVisits") / samples,
                "triangle_visits": get("triangleVisits") / samples, "sphere_visits": get("sphereVisits") / samples, "light_node_visits": get("lightNodeVisits") / samples,
                "lights_sampled": get("lightSampled") / samples, "surface_hits": hits / samples}
    return sum(per_sample.values()), per_sample, counters


def run_render(ctx, args, scene_key, width, height, spp, bounce_limit, steps, warmup, reduce_every, with_cpu_baseline=True, builder=None):
    """One render record: `steps` epochs of `spp` samples per pixel over the whole frame, the tiles sharded over the ranks, the
    accumulation frames all-reduced and resolved every `reduce_every` steps (one finished render)."""
    from echorenderer_b200 import PreparedScene, _native, hilbert_curve_pattern, shard_tiles
    torch, dist, device, stream = ctx.torch, ctx.dist, ctx.device, ctx.stream
    peak, peak_source = peaks()
    world, rank = ctx.world, ctx.rank
    tile = 16

    note(ctx, f"render {scene_key}: building the scene")
    started = time.perf_counter()
    prepared = host.prepare((builder or RENDER_SCENES[scene_key][1])())
    prepare_seconds = time.perf_counter() - started
    scene = PreparedScene(prepared, device=ctx.local_rank)

    tile_count = ((width + tile - 1) // tile, (height + tile - 1) // tile)
    all_tiles = hilbert_curve_pattern(tile_count) if args.pattern == "hilbert" else scenes.tile_grid(width, height, tile)
    by_samples = args.shard == "samples" and world > 1
    tiles = all_tiles if by_samples else shard_tiles(all_tiles, rank, world, block=args.shard_block, by=args.shard_by)
    extend = max(1, spp // world) if by_samples else spp
    frame = torch.zeros(height * width * 4, dtype=torch.float32, device=device)

    def params_for(index, evaluator=structs.EVALUATOR_PATH_TRACED):
        # sample sharding: rank r renders epoch index * world + r, spp / world samples per pixel
        epoch = index * world + rank if by_samples else index
        return structs.render_params(width, height, tile, extend=extend, min_epoch=1, max_epoch=1, bounce_limit=bounce_limit, seed=1, epoch_offset=epoch, evaluator=evaluator)

    # ---- one counted pass over a spread of this rank's tiles: visit counters -> algorithmic bytes per sample
    note(ctx, f"render {scene_key}: counted pass")
    spread = tiles[::max(1, len(tiles) // 256)][:256]
    scratch = torch.zeros(height * width * 4, dtype=torch.float32, device=device)
    counted = scene.render_frame_device(params_for(0, structs.EVALUATOR_PATH_TRACED | structs.EVALUATOR_COUNT_VISITS), spread, scratch.data_ptr(), stream)
    torch.cuda.synchronize()
    del scratch
    per_sample_bytes, per_sample_parts, per_sample_counters = bytes_per_sample(counted)

    render_ms, reduce_ms, launches, samples = [], [], 0, 0
    reduce_events = []

    def step(index, timed):
        nonlocal launches, samples
        begin = time.perf_counter()
        stats = scene.render_frame_device(params_for(index), tiles, frame.data_ptr(), stream)
        if timed:
            render_ms.append((time.perf_counter() - begin) * 1e3)
            launches += int(stats["kernelLaunches"][0])
            samples += int(stats["sampleEvaluated"][0])
        if (index + 1) % reduce_every == 0 or index + 1 == steps:  # the last step finishes its render
            first, middle, last = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            first.record()
            if ctx.distributed:
                dist.barrier()  # the collective waits for the slowest rank either way; a barrier in front of it separates that wait from the transfer
            middle.record()
            if ctx.distributed:
                dist.all_reduce(frame)  # the accumulation-buffer reduce over NVLink (tile sharding: disjoint pixels, sum with zeros)
            last.record()
            scene.frame_resolve_device(frame.data_ptr(), width, height, stream)
            if index + 1 < steps:
                frame.zero_()  # the next render starts from an empty accumulation frame; the last one stays for --dump-outputs
            if timed:
                reduce_events.append((first, middle, last))
                launches += 2
        return stats

    note(ctx, f"render {scene_key}: {warmup} warm-up + {steps} timed steps")
    with ClockSampler(ctx.local_rank) as clocks:
        for index in range(warmup):
            scene.render_frame_device(params_for(index), tiles, frame.data_ptr(), stream)
        if ctx.distributed:
            dist.all_reduce(frame)  # NCCL sets its channels up for this buffer outside the timed region
        frame.zero_()
        ctx.barrier()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks.mark(0)
        start.record()
        for index in range(steps):
            stats = step(index, True)
        stop.record()
        ctx.barrier()
        clocks.mark(1)
        total_ms = ctx.max_over_ranks(start.elapsed_time(stop))

    if args.dump_outputs and rank == 0:
        keep = torch.from_numpy(dump_sample(width * height, DUMP_SAMPLES // 2)).to(device)
        dump_outputs(args.dump_outputs, {f"frame_{scene_key}": frame.view(-1, 4)[keep].cpu().numpy()})

    reduce_ms = [b.elapsed_time(c) for _, b, c in reduce_events]
    skew_ms = [a.elapsed_time(b) for a, b, _ in reduce_events]
    total_samples = int(ctx.sum_over_ranks(samples))
    total_launches = int(ctx.sum_over_ranks(launches))
    value = total_samples / (total_ms * 1e-3)
    per_rank_ms = ctx.gather(float(np.mean(render_ms)))
    per_rank_worst = ctx.gather(float(np.max(render_ms)))

    # ---- end to end through the plugin call: echo_b200_render_tiles with host buffers (tile positions in, accumulated tiles out)
    note(ctx, f"render {scene_key}: plugin-call leg")
    e2e_steps = max(1, min(steps, 4))
    host_tiles = _native.HostBuffer(len(tiles) * tile * tile * 4, np.float32)
    warm = structs.render_params(width, height, tile, extend=1, min_epoch=1, max_epoch=1, bounce_limit=bounce_limit, seed=1)
    scene.render_tiles_pointers(warm, tiles, host_tiles.address)  # first-call allocations (the library's tile buffer for this many tiles), one sample per pixel
    ctx.barrier()
    wall = time.perf_counter()
    e2e_samples = 0
    for index in range(e2e_steps):
        e2e_stats = scene.render_tiles_pointers(params_for(index), tiles, host_tiles.address)
        e2e_samples += int(e2e_stats["sampleEvaluated"][0])
    ctx.barrier()
    e2e_ms = ctx.max_over_ranks((time.perf_counter() - wall) * 1e3)
    e2e_total = ctx.sum_over_ranks(e2e_samples)
    host_tiles.free()

    achieved = per_sample_bytes * value / world / 1e9  # per GPU: every rank runs the same kernels on its share of the samples
    traffic_per_sample = ncu_traffic(f"{scene_key}_dram_bytes_per_sample")  # DRAM bytes of a whole step / its samples, from the committed ncu capture
    record = {"metric": "samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": total_ms / steps,
              "higher_is_better": True, "scaling": "strong", "dtype": "f32", "data": "synthetic",
              "config": render_config(args, scene_key, width, height, spp, bounce_limit, reduce_every),
              "samples_per_step": total_samples // steps,
              "rank_step_ms": {"min": min(per_rank_ms), "max": max(per_rank_ms), "mean": float(np.mean(per_rank_ms)), "worst_single_step": max(per_rank_worst), "per_rank": per_rank_ms,
                               "what": "host wall time of echo_b200_render_frame_device per step, mean over the timed steps, per rank"},
              "all_reduce": {"count": len(reduce_ms), "ms_mean": float(np.mean(reduce_ms)) if reduce_ms else None, "wait_for_slowest_rank_ms_mean": float(np.mean(skew_ms)) if skew_ms else None,
                             "bytes": int(frame.numel() * 4), "collective": "NCCL all-reduce (sum) of the fp32 accumulation frame" if ctx.distributed else "none (one GPU)"},
              "roofline": {"bound": "hbm", "kernel": "wavefront step (raygen, extend, classify, shade x6, shadow, accumulate), per GPU", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_nominal_8tbs": achieved / 8000.0,
                           "traffic": traffic_per_sample * (total_samples // steps) if traffic_per_sample else None, "traffic_bytes_per_sample": traffic_per_sample,
                           "peak_source": peak_source, "algorithmic_bytes_per_sample": per_sample_bytes,
                           "bytes_per_sample_parts": per_sample_parts, "per_sample_counters": per_sample_counters, "path_state_bytes": PATH_STATE_BYTES,
                           "counted_pass": f"{len(spread)} tiles spread over rank 0's shard at {extend} spp, one-thread-per-query kernels with visit counters (ECHO_EVALUATOR_COUNT_VISITS)",
                           "bound_measured": "latency / L1 sector fetches in extend + shadow, instruction fetch in the shading kernels (ncu: profiles/README.md); DRAM is not the limiter"},
              "e2e": {"value": e2e_total / (e2e_ms * 1e-3), "unit": "samples/s", "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
                      "h2d_bytes_per_step": int(tiles.nbytes) + structs.RENDER_PARAMS.itemsize, "d2h_bytes_per_step": int(len(tiles) * tile * tile * 16) + structs.STATS.itemsize,
                      "call": "echo_b200_render_tiles: tile positions in, accumulated Float4 tiles out into page-locked host memory (echo_b200_host_alloc), per rank"},
              "gpu_launches": total_launches,
              "clocks": clocks.summary(),
              "scene": {"triangles": int(len(prepared.triangles)), "spheres": int(len(prepared.spheres)), "nodes": int(len(prepared.nodes)), "quad_depth": int(prepared.max_depth),
                        "light_tree_nodes": int(len(prepared.light_nodes)), "host_prepare_seconds": prepare_seconds},
              "stats_last_step": {label: int(stats[name][0]) for label, name in zip(structs.STATS_LABELS, structs.STATS_FIELDS)}}

    if rank == 0 and prepared.packs is None and len(prepared.light_nodes) > 1000 and not args.no_tree_build:
        record["light_tree_build"] = light_tree_build_record(prepared, ctx.local_rank)

    if with_cpu_baseline and rank == 0 and not args.no_cpu_baseline:
        note(ctx, f"render {scene_key}: CPU baseline")
        record["cpu_baseline"] = cpu_baseline_render(prepared, width, height, tile, spp, bounce_limit)

    scene.close()
    del frame
    torch.cuda.empty_cache()
    return record


def main():
    args = parse()
    if args.warmup < 3:
        args.warmup = 3  # the contract's floor (W >= 3); the emitted `warmup` is what ran
    quiet_stdout()

    if args.impl == "reference":
        reference_arm(args)
        return

    ctx = Context()

    if args.workload == "render":
        record = run_render(ctx, args, args.scene, args.width, args.height, args.spp, args.bounce_limit, args.steps, args.warmup, args.reduce_every)
        line = base_line(args, "samples/s", record["value"], record["ms_per_step"], record["config"], "f32")
        line.update({key: value for key, value in record.items() if key not in line})
    else:
        note(ctx, "C2 trace batches")
        line = run_trace(ctx, args)

        if args.workload == "all" and not args.no_render and not args.instanced:
            steps = args.steps if args.render_steps is None else max(1, min(args.render_steps, args.steps))
            line["render"] = {"what": "the path tracer measured as the reference reports it (samples/s, ScheduledRender.cs:226-234); records have the shape of a bench line"}
            # ECHO_BENCH_SHRINK=1 (tests/test_gpu_bench.py only): the same code path on scenes and frames that take seconds
            shrink = os.environ.get("ECHO_BENCH_SHRINK") == "1"
            # (key, scene, width, height, spp per step, bounce limit, steps per finished render, builder override)
            c1 = ("c1", "cornell", 128, 128, 4, 128, 1, None) if shrink else ("c1", "cornell", 512, 512, 16, 128, 1, None)
            c3 = ("c3", "mixed", 256, 144, 8, 8, 4, lambda: scenes.mixed_material_scene(rings=24, segments=24)) if shrink else ("c3", "mixed", 1920, 1080, 64, 8, 4, None)
            c4 = ("c4", "lights", 256, 144, 8, 128, 4, lambda: scenes.many_lights_scene(light_count=300, rings=16, segments=16)) if shrink else ("c4", "lights", 1920, 1080, 64, 128, 4, None)
            c5 = ("c5", "large", 384, 208, 16, 128, 4, lambda: scenes.large_scene(160, 80)) if shrink else ("c5", "large", 3840, 2160, 256, 128, 4, None)
            records = [c1, c3, c4, c5] if ctx.world == 1 else [c5]  # C1, C3 and C4 are one-GPU configurations (BASELINE.json); C5 is the sharded one
            for key, scene_key, width, height, spp, bounce_limit, reduce_every, builder in records:
                line["render"][key] = run_render(ctx, args, scene_key, width, height, spp, bounce_limit, steps, args.render_warmup, reduce_every, builder=builder)
            line["gpu_launches"] += sum(record["gpu_launches"] for key, record in line["render"].items() if isinstance(record, dict))

    if ctx.rank == 0:
        emit(line)
    ctx.close()


if __name__ == "__main__":
    main()
