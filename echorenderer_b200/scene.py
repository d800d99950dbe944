"""Host-side mirror of the reference interface for the hot path, on top of the C ABI.

  PreparedScene          Aggregation/Preparation/PreparedScene.cs — Trace / Occlude (batched) and the scene payload
  PathTracedEvaluator    Evaluation/Evaluators/PathTracedEvaluator.cs:33,40 — BounceLimit, Survivability
  EvaluationProfile      Processes/Evaluation/EvaluationProfile.cs:13-75 — Evaluator, Distribution.Extend, Min/MaxEpoch, NoiseThreshold
  RenderTexture          Textures/Evaluation/RenderTexture.cs — tile-based destination (CreateTile / Apply semantics)
  EvaluationOperation    Processes/Evaluation/EvaluationOperation.cs:21-177 — tilePositions, destination, profile, TotalSamples, Execute

Names, argument meaning and error behaviour follow the reference (validation errors raise like EvaluationProfile.Validate,
native failures raise EchoNativeError with the pulled error string). The compute always runs in libecho_b200.so.
"""
import ctypes
from dataclasses import dataclass, field

import numpy as np

from . import _native, structs
from .host import PreparedArrays


class PreparedScene:
    """The flattened scene resident on one B200; the device twin of Echo's PreparedScene."""

    def __init__(self, prepared: PreparedArrays, device: int = 0, devices=None, build_tree_on_device: bool = False, build_light_tree_on_device: bool = False,
                 build_packs_on_device: bool = False):
        """`device`: the CUDA device of a single-device scene. `build_tree_on_device`: the library builds the accelerator itself from
        the uploaded triangles and spheres (echo_b200_scene_build_qbvh: the SweepBuilder's tree, on the device) instead of taking
        `prepared.nodes`; `self.built_tree` = (node count, max depth) then. `build_light_tree_on_device`: likewise the light tree
        (echo_b200_scene_build_light_tree: LightTree.Build on the device) instead of `prepared.light_nodes` and the emitter map;
        `self.built_light_tree` = (node count, emitter count, power) then. Both refuse a scene with packs (ValueError /
        EchoNativeError); `build_packs_on_device`
        builds every pack of one instead, QBVH and light tree, in one call (echo_b200_scene_build_packs) and ignores `prepared`'s nodes,
        light trees and the outputs of its pack records; `self.built_packs` = (node count, light node count, emitter count, power) then. `devices` (a list of device indices) instead replicates the scene
        on several devices of this process (echo_b200_scene_create_multi): trace / occlude split their batches over them and
        render_tiles deals blocks of tiles to them; the *_device methods then do not apply."""
        lib = _native.library()
        self._lib = lib
        self.prepared = prepared
        self.device = device
        self._handle = ctypes.c_void_p()
        if devices is None:
            _native.check(lib.echo_b200_scene_create(ctypes.byref(self._handle), device))
        else:
            mask = 0
            for index in devices:
                mask |= 1 << int(index)
            _native.check(lib.echo_b200_scene_create_multi(ctypes.byref(self._handle), mask))

        try:
            d = prepared.description
            ptr = _native.pointer
            triangles, spheres, materials = prepared.triangles, prepared.spheres, prepared.materials
            _native.check(lib.echo_b200_scene_set_triangles(self._handle, ptr(triangles), len(triangles)))
            _native.check(lib.echo_b200_scene_set_spheres(self._handle, ptr(spheres), len(spheres)))
            instanced = prepared.packs is not None
            if instanced and build_tree_on_device:  # scene_build_qbvh would see one flat scene: set_packs comes after it
                raise ValueError("build_tree_on_device builds the accelerator of a scene without packs: use build_packs_on_device=True")
            if build_packs_on_device and not instanced:
                raise ValueError("build_packs_on_device builds a scene with packs: use build_tree_on_device / build_light_tree_on_device")
            self.built_tree = None
            self.built_packs = None
            if build_tree_on_device:
                count, depth = ctypes.c_uint32(), ctypes.c_uint32()
                _native.check(lib.echo_b200_scene_build_qbvh(self._handle, ctypes.byref(count), ctypes.byref(depth)))
                self.built_tree = (count.value, depth.value)
            elif not build_packs_on_device:  # the pack build installs the nodes after set_packs
                _native.check(lib.echo_b200_scene_set_qbvh(self._handle, ptr(prepared.nodes), len(prepared.nodes), prepared.max_depth))
            _native.check(lib.echo_b200_scene_set_materials(self._handle, ptr(materials), len(materials)))
            if prepared.textures is not None:
                _native.check(lib.echo_b200_scene_set_textures(self._handle, ptr(prepared.textures), len(prepared.textures), ptr(prepared.texels), len(prepared.texels),
                                                                  ptr(prepared.material_textures), len(prepared.material_textures)))
            if prepared.distributions is not None:
                _native.check(lib.echo_b200_scene_set_distributions(self._handle, ptr(prepared.distributions), len(prepared.distributions)))
            if prepared.packs is not None:
                _native.check(lib.echo_b200_scene_set_packs(self._handle, ptr(prepared.packs), len(prepared.packs), ptr(prepared.instances), len(prepared.instances)))
            self.built_light_tree = None
            if build_packs_on_device:
                counts = [ctypes.c_uint32() for _ in range(3)]
                power = ctypes.c_float()
                _native.check(lib.echo_b200_scene_build_packs(self._handle, ptr(prepared.point_lights), len(prepared.point_lights),
                                                              *(ctypes.byref(c) for c in counts), ctypes.byref(power)))
                self.built_packs = (counts[0].value, counts[1].value, counts[2].value, power.value)
            elif build_light_tree_on_device:
                count, emitters, power = ctypes.c_uint32(), ctypes.c_uint32(), ctypes.c_float()
                _native.check(lib.echo_b200_scene_build_light_tree(self._handle, ptr(prepared.point_lights), len(prepared.point_lights),
                                                                   ctypes.byref(count), ctypes.byref(emitters), ctypes.byref(power)))
                self.built_light_tree = (count.value, emitters.value, power.value)
            else:
                _native.check(lib.echo_b200_scene_set_light_tree(self._handle, ptr(prepared.light_nodes), len(prepared.light_nodes),
                                                                 ptr(prepared.emitter_tokens), ptr(prepared.emitter_bitpaths), len(prepared.emitter_tokens),
                                                                 ptr(prepared.point_lights), len(prepared.point_lights)))
            _native.check(lib.echo_b200_scene_set_infinite(self._handle, ptr(d.infinite_lights), len(d.infinite_lights),
                                                           prepared.infinite_threshold, prepared.infinite_pdf))
            _native.check(lib.echo_b200_scene_set_camera(self._handle, ptr(d.camera)))
            _native.check(lib.echo_b200_scene_set_bound_radius(self._handle, prepared.bound_radius))
            _native.check(lib.echo_b200_scene_commit(self._handle))
        except Exception:
            self.close()
            raise

    def bounds_violations(self):
        """Bit set of failed index checks since commit in a -DECHO_BOUNDS_CHECK build of the library (0 = clean); None for a
        release build, which has no checks compiled in."""
        bits = ctypes.c_uint32()
        _native.check(self._lib.echo_b200_debug_bounds_violations(self._handle, ctypes.byref(bits)))
        return None if bits.value == 0xFFFFFFFF else int(bits.value)

    def close(self, quiet=False):
        """Destroys the native scene. A bounds-check build reports failed index checks here by raising — except with
        `quiet` (what __del__ and an __exit__ that is already unwinding an exception use: they must not raise or mask)."""
        if getattr(self, "_handle", None) is not None and self._handle.value:
            violations = None
            try:
                violations = self.bounds_violations()
            except Exception:  # a failed context must not hide the error that led here
                pass
            self._lib.echo_b200_scene_destroy(self._handle)
            self._handle = ctypes.c_void_p()
            if violations and not quiet:
                raise _native.EchoNativeError(-2, f"out-of-bounds index in a kernel: failed checks 0x{violations:x} (echo_scene.cuh CHECK_*)")

    def __del__(self):
        try:
            self.close(quiet=True)
        except Exception:  # interpreter shutdown: the library may already be gone
            pass

    def __enter__(self):
        return self

    def __exit__(self, exception_type, *_):
        self.close(quiet=exception_type is not None)

    @property
    def handle(self):
        return self._handle

    @property
    def gpu_count(self):
        count = ctypes.c_int32()
        _native.check(self._lib.echo_b200_scene_gpu_count(self._handle, ctypes.byref(count)))
        return count.value

    # ---- PreparedScene.Trace / Occlude, batched (PreparedScene.cs:66-86); host numpy buffers ----
    def trace(self, rays, out=None):
        """Closest hit for every TraceQuery in `rays` (structs.RAY). Returns structs.HIT records: on a miss token is
        TOKEN_EMPTY and distance keeps the query's input distance."""
        rays = np.ascontiguousarray(rays, dtype=structs.RAY)
        hits = out if out is not None else np.empty(len(rays), dtype=structs.HIT)
        _native.check(self._lib.echo_b200_trace_batch(self._handle, _native.pointer(rays), len(rays), _native.pointer(hits)))
        return hits

    def occlude(self, rays, out=None):
        """Any hit within `distance` (the OccludeQuery travel) for every query; returns uint8 0/1."""
        rays = np.ascontiguousarray(rays, dtype=structs.RAY)
        occluded = out if out is not None else np.empty(len(rays), dtype=np.uint8)
        _native.check(self._lib.echo_b200_occlude_batch(self._handle, _native.pointer(rays), len(rays), _native.pointer(occluded)))
        return occluded

    # ---- the same with full TokenHierarchy in and out, for instanced scenes (GeometryCollection.cs:123-131,160-168) ----
    def trace_hierarchy(self, rays, ignore_layers=None):
        """Returns (hits, layers): structs.HIT plus the structs.TOKEN_HIERARCHY instance layers of every hit."""
        rays = np.ascontiguousarray(rays, dtype=structs.RAY)
        ignore = None if ignore_layers is None else np.ascontiguousarray(ignore_layers, dtype=structs.TOKEN_HIERARCHY)
        hits = np.empty(len(rays), dtype=structs.HIT)
        layers = np.zeros(len(rays), dtype=structs.TOKEN_HIERARCHY)
        _native.check(self._lib.echo_b200_trace_batch_hierarchy(self._handle, _native.pointer(rays), _native.pointer(ignore) if ignore is not None else None,
                                                                len(rays), _native.pointer(hits), _native.pointer(layers)))
        return hits, layers

    def occlude_hierarchy(self, rays, ignore_layers=None):
        rays = np.ascontiguousarray(rays, dtype=structs.RAY)
        ignore = None if ignore_layers is None else np.ascontiguousarray(ignore_layers, dtype=structs.TOKEN_HIERARCHY)
        occluded = np.empty(len(rays), dtype=np.uint8)
        _native.check(self._lib.echo_b200_occlude_batch_hierarchy(self._handle, _native.pointer(rays), _native.pointer(ignore) if ignore is not None else None,
                                                                  len(rays), _native.pointer(occluded)))
        return occluded

    # ---- raw-pointer variants for pinned host memory / device memory owned by the caller (torch tensors) ----
    def trace_pointers(self, rays_pointer, count, hits_pointer):
        _native.check(self._lib.echo_b200_trace_batch(self._handle, ctypes.c_void_p(rays_pointer), count, ctypes.c_void_p(hits_pointer)))

    def occlude_pointers(self, rays_pointer, count, occluded_pointer):
        _native.check(self._lib.echo_b200_occlude_batch(self._handle, ctypes.c_void_p(rays_pointer), count, ctypes.c_void_p(occluded_pointer)))

    def trace_device(self, rays_pointer, count, hits_pointer, stream=0, counts_pointer=None):
        """Asynchronous launch on `stream` (a cudaStream_t value) over device-resident buffers."""
        if counts_pointer is None:
            _native.check(self._lib.echo_b200_trace_batch_device(self._handle, ctypes.c_void_p(rays_pointer), count, ctypes.c_void_p(hits_pointer), ctypes.c_void_p(stream)))
        else:
            _native.check(self._lib.echo_b200_trace_batch_device_counted(self._handle, ctypes.c_void_p(rays_pointer), count, ctypes.c_void_p(hits_pointer),
                                                                       ctypes.c_void_p(counts_pointer), ctypes.c_void_p(stream)))

    def occlude_device(self, rays_pointer, count, occluded_pointer, stream=0, counts_pointer=None):
        if counts_pointer is None:
            _native.check(self._lib.echo_b200_occlude_batch_device(self._handle, ctypes.c_void_p(rays_pointer), count, ctypes.c_void_p(occluded_pointer), ctypes.c_void_p(stream)))
        else:
            _native.check(self._lib.echo_b200_occlude_batch_device_counted(self._handle, ctypes.c_void_p(rays_pointer), count, ctypes.c_void_p(occluded_pointer),
                                                                         ctypes.c_void_p(counts_pointer), ctypes.c_void_p(stream)))

    # ---- tile rendering ----
    def render_tiles(self, params, tile_xy):
        """One EvaluationOperation worth of tiles -> (tiles[n, tileSize, tileSize, 4] float32, stats record)."""
        tile_xy = np.ascontiguousarray(tile_xy, dtype=np.int32).reshape(-1, 2)
        tile_size = int(params["tileSize"][0])
        out = np.zeros((len(tile_xy), tile_size, tile_size, 4), dtype=np.float32)
        stats = np.zeros(1, dtype=structs.STATS)
        _native.check(self._lib.echo_b200_render_tiles(self._handle, _native.pointer(params), _native.pointer(tile_xy), len(tile_xy),
                                                       _native.pointer(out), _native.pointer(stats)))
        return out, stats

    def render_tiles_pointers(self, params, tile_xy, out_pointer):
        """echo_b200_render_tiles into caller-owned host memory (e.g. a HostBuffer): tile-major Float4s. Returns the stats record."""
        tile_xy = np.ascontiguousarray(tile_xy, dtype=np.int32).reshape(-1, 2)
        stats = np.zeros(1, dtype=structs.STATS)
        _native.check(self._lib.echo_b200_render_tiles(self._handle, _native.pointer(params), _native.pointer(tile_xy), len(tile_xy),
                                                       ctypes.c_void_p(out_pointer), _native.pointer(stats)))
        return stats

    def render_frame_device(self, params, tile_xy, frame_pointer, stream=0):
        """Renders tiles into a device-resident full frame (width*height Float4; xyz = mean, w = 1 where rendered)."""
        tile_xy = np.ascontiguousarray(tile_xy, dtype=np.int32).reshape(-1, 2)
        stats = np.zeros(1, dtype=structs.STATS)
        if int(params["maxEpoch"][0]) == 0:  # a rank whose share of the epochs is empty (shard_epochs): its frame stays zero
            return stats
        _native.check(self._lib.echo_b200_render_frame_device(self._handle, _native.pointer(params), _native.pointer(tile_xy), len(tile_xy),
                                                              ctypes.c_void_p(frame_pointer), _native.pointer(stats), ctypes.c_void_p(stream)))
        return stats

    def frame_resolve_device(self, frame_pointer, width, height, stream=0):
        _native.check(self._lib.echo_b200_frame_resolve_device(self._handle, ctypes.c_void_p(frame_pointer), width, height, ctypes.c_void_p(stream)))

    def evaluate_samples(self, params, pixel_xy, sample_index, channels=3):
        """Diagnostic: one Evaluator.Evaluate per (pixel, sample index) -> radiance[n, 3] (channels=4 keeps the W lane the
        auxiliary evaluators use, e.g. NormalDepth128's depth)."""
        pixel_xy = np.ascontiguousarray(pixel_xy, dtype=np.int32).reshape(-1, 2)
        sample_index = np.ascontiguousarray(sample_index, dtype=np.uint32)
        out = np.zeros((len(sample_index), channels), dtype=np.float32)
        entry = self._lib.echo_b200_debug_evaluate_samples if channels == 3 else self._lib.echo_b200_debug_evaluate_samples4
        _native.check(entry(self._handle, _native.pointer(params), _native.pointer(pixel_xy), _native.pointer(sample_index), len(sample_index), _native.pointer(out)))
        return out


@dataclass(frozen=True)
class PathTracedEvaluator:
    """Evaluation/Evaluators/PathTracedEvaluator.cs:33,40."""
    bounce_limit: int = 128
    survivability: float = 2.5


    @property
    def code(self):
        return structs.EVALUATOR_PATH_TRACED


@dataclass(frozen=True)
class AlbedoEvaluator:
    """Evaluation/Evaluators/AlbedoEvaluator.cs:13-16: the first non-specular surface's albedo (Float4, W = 0)."""
    diverge_once: bool = True
    bounce_limit: int = 128      # unused by this evaluator; kept so every evaluator fills EchoRenderParams the same way
    survivability: float = 2.5

    @property
    def code(self):
        return structs.EVALUATOR_ALBEDO | (structs.EVALUATOR_DIVERGE_ONCE if self.diverge_once else 0)


@dataclass(frozen=True)
class NormalDepthEvaluator:
    """Evaluation/Evaluators/NormalDepthEvaluator.cs:13-18: shading normal + depth (NormalDepth128.ToFloat4)."""
    diverge_once: bool = False
    bounce_limit: int = 128
    survivability: float = 2.5

    @property
    def code(self):
        return structs.EVALUATOR_NORMAL_DEPTH | (structs.EVALUATOR_DIVERGE_ONCE if self.diverge_once else 0)


@dataclass(frozen=True)
class StandardNaiveEvaluator:
    """Evaluation/Evaluators/StandardNaiveEvaluator.cs:13-14: brute-force path tracing (no light sampling, no roulette) — slow
    to converge, but an independent estimator of the same image."""
    bounce_limit: int = 128
    survivability: float = 2.5  # unused

    @property
    def code(self):
        return structs.EVALUATOR_NAIVE


@dataclass(frozen=True)
class EvaluationProfile:
    """Processes/Evaluation/EvaluationProfile.cs:13-75 (Distribution reduced to its Extend and seed)."""
    evaluator: object = field(default_factory=PathTracedEvaluator)
    extend: int = 16                # ContinuousDistribution.Extend, ContinuousDistribution.cs:25
    min_epoch: int = 1
    max_epoch: int = 20
    noise_threshold: float = 0.045
    seed: int = 1

    def validate(self):
        """EvaluationProfile.Validate, EvaluationProfile.cs:65-75."""
        if self.evaluator is None:
            raise ValueError("Evaluator is null")
        if self.extend <= 0:
            raise ValueError("Distribution.Extend out of bounds")
        if self.min_epoch <= 0 or self.max_epoch < self.min_epoch:
            raise ValueError("MinEpoch / MaxEpoch out of bounds")
        if self.noise_threshold < 0:
            raise ValueError("NoiseThreshold out of bounds")


class RenderTexture:
    """Tile-based destination, rows growing upward (Textures/Evaluation/RenderTexture.cs, EvaluationLayer.cs:16-52)."""

    def __init__(self, width, height, tile_size=16):
        if width <= 0 or height <= 0 or tile_size <= 0:
            raise ValueError("size out of bounds")
        self.width, self.height, self.tile_size = width, height, tile_size
        self.pixels = np.zeros((height, width, 4), dtype=np.float32)

    @property
    def tile_count(self):
        return ((self.width + self.tile_size - 1) // self.tile_size, (self.height + self.tile_size - 1) // self.tile_size)

    @property
    def tile_positions(self):
        """profile.Pattern.CreateSequence(destination.size.CeiledDivide(tileSize)) with the default pattern
        (EvaluationOperation.cs:157-160, EvaluationProfile.Pattern = new HilbertCurvePattern())."""
        return hilbert_curve_pattern(self.tile_count)

    def apply(self, tile_position, tile):
        """IEvaluationLayer.Apply for one finished tile (EvaluationLayer.cs:111-121): tiles are immutable once applied."""
        x0, y0 = int(tile_position[0]) * self.tile_size, int(tile_position[1]) * self.tile_size
        w, h = min(self.tile_size, self.width - x0), min(self.tile_size, self.height - y0)
        self.pixels[y0:y0 + h, x0:x0 + w] = tile[:h, :w]


def ordered_pattern(size, horizontal=True):
    """OrderedPattern.CreateSequence (Processes/Evaluation/ITilePattern.cs:20-36): row-major (or column-major) tile positions."""
    sx, sy = int(size[0]), int(size[1])
    if horizontal:
        return np.array([(x, y) for y in range(sy) for x in range(sx)], dtype=np.int32).reshape(-1, 2)
    return np.array([(x, y) for x in range(sx) for y in range(sy)], dtype=np.int32).reshape(-1, 2)


def _sign(v):
    return (v > 0) - (v < 0)


def _half(v):
    return int(v / 2)  # C# integer division truncates toward zero, also for the negative rectangle sides


def _hilbert_2d(position, rect_a, rect_b, out):
    """The generalised Hilbert curve over an arbitrary rectangle (HilbertCurvePattern.Hilbert2D, ITilePattern.cs:143-202)."""
    width, height = abs(rect_a[0] + rect_a[1]), abs(rect_b[0] + rect_b[1])
    da = (_sign(rect_a[0]), _sign(rect_a[1]))  # unit major direction
    db = (_sign(rect_b[0]), _sign(rect_b[1]))  # unit orthogonal direction
    x, y = position

    if height == 1:
        for _ in range(width):
            out.append((x, y))
            x, y = x + da[0], y + da[1]
    elif width == 1:
        for _ in range(height):
            out.append((x, y))
            x, y = x + db[0], y + db[1]
    else:
        a2 = [_half(rect_a[0]), _half(rect_a[1])]
        b2 = [_half(rect_b[0]), _half(rect_b[1])]
        width2, height2 = abs(a2[0] + a2[1]), abs(b2[0] + b2[1])

        if width * 2 > height * 3:
            if width2 % 2 != 0 and width > 2:
                a2 = [a2[0] + da[0], a2[1] + da[1]]
            _hilbert_2d((x, y), a2, rect_b, out)
            _hilbert_2d((x + a2[0], y + a2[1]), (rect_a[0] - a2[0], rect_a[1] - a2[1]), rect_b, out)
        else:
            if height2 % 2 != 0 and height > 2:
                b2 = [b2[0] + db[0], b2[1] + db[1]]
            _hilbert_2d((x, y), b2, a2, out)
            _hilbert_2d((x + b2[0], y + b2[1]), rect_a, (rect_b[0] - b2[0], rect_b[1] - b2[1]), out)
            _hilbert_2d((x + (rect_a[0] - da[0]) + (b2[0] - db[0]), y + (rect_a[1] - da[1]) + (b2[1] - db[1])),
                        (-b2[0], -b2[1]), (-(rect_a[0] - a2[0]), -(rect_a[1] - a2[1])), out)


def hilbert_curve_pattern(size):
    """HilbertCurvePattern.CreateSequence (ITilePattern.cs:72-141), the default `EvaluationProfile.Pattern`
    (EvaluationProfile.cs): one generalised Hilbert curve per quadrant, mirrored so that all four start at the centre of the
    texture, interlaced one position at a time — tiles are handed out from the middle outwards, neighbours close in time."""
    sx, sy = int(size[0]), int(size[1])
    if (sx, sy) == (1, 1):
        return np.zeros((1, 2), dtype=np.int32)

    def corner(cx, cy):
        out = []
        if cx > cy:
            _hilbert_2d((0, 0), (cx, 0), (0, cy), out)
        else:
            _hilbert_2d((0, 0), (0, cy), (cx, 0), out)
        return out

    floor_x, ceil_x, floor_y, ceil_y = sx // 2, (sx + 1) // 2, sy // 2, (sy + 1) // 2
    top_right_size, top_left_size = (ceil_x, floor_y), (floor_x, floor_y)
    bottom_right_size, bottom_left_size = (ceil_x, ceil_y), (floor_x, ceil_y)

    top_left = [(top_left_size[0] - x - 1, top_left_size[1] - y - 1) for x, y in corner(*top_left_size)]
    top_right = [(x + top_left_size[0], top_right_size[1] - y - 1) for x, y in corner(*top_right_size)]
    bottom_left = [(bottom_left_size[0] - x - 1, y + top_left_size[1]) for x, y in corner(*bottom_left_size)]
    bottom_right = [(x + top_left_size[0], y + top_left_size[1]) for x, y in corner(*bottom_right_size)]

    result, cursors = [], [0, 0, 0, 0]
    corners = [top_left, top_right, bottom_left, bottom_right]
    while len(result) < sx * sy:
        for k in range(4):
            if cursors[k] < len(corners[k]):
                result.append(corners[k][cursors[k]])
                cursors[k] += 1
    return np.array(result, dtype=np.int32).reshape(-1, 2)


def shard_tiles(tile_positions, rank, world_size, block=1, by="sequence"):
    """Tile sharding across devices, the static analogue of Operation.Execute's shared procedure counter
    (Common/Compute/Operation.cs:164-177). What a rank renders keeps the order of the caller's sequence (the preview fills in
    as EvaluationProfile.Pattern intends); `by` decides who owns a tile:

    "position"  tile (x, y) belongs to rank (x + y) mod world_size: diagonal stripes one tile wide, so every rank samples every
                region of the image at the same density and the shards cost the same whatever the image holds. Measured on C5
                at 8 GPUs (variants/r2_sweep_c5.py): per-rank step times within 1.5 % of each other, against 7 % for blocks of
                64 consecutive tiles of the Hilbert sequence and 23 % for every 8th tile of it (the HilbertCurvePattern
                interlaces four quadrant curves, so position in the sequence correlates with position in the image).
    "sequence"  the sequence is cut into blocks of `block` consecutive tiles and block b goes to rank (b mod world_size);
                block = 1 deals single tiles round-robin."""
    tile_positions = np.asarray(tile_positions, dtype=np.int32).reshape(-1, 2)
    if by == "position":
        owner = (tile_positions[:, 0].astype(np.int64) + tile_positions[:, 1].astype(np.int64)) % world_size
    elif by == "sequence":
        owner = (np.arange(len(tile_positions)) // max(1, int(block))) % world_size
    else:
        raise ValueError(f"unknown sharding rule {by!r}")
    return np.ascontiguousarray(tile_positions[owner == rank])


def build_qbvh_device(triangles, spheres, device=0, instance_bounds=None):
    """The optional device-side tree build (echo_b200_build_qbvh). Returns (nodes, max_depth) like host.build_qbvh. By default
    (BUILD_ALGORITHM 2, csrc/sweep.cu) the tree IS the SweepBuilder's — the nodes equal host.build_qbvh's byte for byte; inputs that
    chain deeper than the traversal stacks allow, and BUILD_ALGORITHM 1 / 0, give a clustered (PLOC) or Morton-ordered tree instead:
    valid, but not the reference's. instance_bounds: [n, 6] float32 boxes (min xyz, max xyz) of the pack's placements, tokenized
    after the spheres (echo_b200_build_qbvh_instanced), as in host.build_qbvh."""
    lib = _native.library()
    triangles = np.ascontiguousarray(triangles, dtype=structs.TRIANGLE)
    spheres = np.ascontiguousarray(spheres, dtype=structs.SPHERE)
    boxes = np.zeros((0, 6), dtype=np.float32) if instance_bounds is None else np.ascontiguousarray(instance_bounds, dtype=np.float32).reshape(-1, 6)
    total = len(triangles) + len(spheres) + len(boxes)
    nodes = np.empty(max(total - 1, 1), dtype=structs.QBVH_NODE)
    count, depth = ctypes.c_uint32(), ctypes.c_uint32()
    _native.check(lib.echo_b200_build_qbvh_instanced(device, _native.pointer(triangles), len(triangles), _native.pointer(spheres), len(spheres), _native.pointer(boxes), len(boxes),
                                                     _native.pointer(nodes), ctypes.byref(count), ctypes.byref(depth)))
    nodes.resize(count.value, refcheck=False)  # shrinks in place (realloc): no second copy of a 600 MB array
    return nodes, int(depth.value)


def build_light_tree_device(description, instance_lights=None, device=0):
    """The optional device-side light-tree build (echo_b200_build_light_tree, csrc/lightbuild.cu). Takes and returns what
    host.build_light_tree does — (nodes, emitter_tokens, emitter_bitpaths, power) — and the arrays equal that build's byte for byte:
    LightCollection.CreateBounds + LightTree.Build + AddToMap, level by level on the device. `description` needs triangles, spheres,
    materials and point_lights; instance_lights: [n, 12] float32 PreparedInstance.LightBound rows. Pass it to host.prepare as
    `light_tree_builder=scene.build_light_tree_device`."""
    lib = _native.library()
    d = description
    triangles = np.ascontiguousarray(d.triangles, dtype=structs.TRIANGLE)
    spheres = np.ascontiguousarray(d.spheres, dtype=structs.SPHERE)
    materials = np.ascontiguousarray(d.materials, dtype=structs.MATERIAL)
    points = np.ascontiguousarray(d.point_lights, dtype=structs.POINT_LIGHT)
    rows = np.zeros((0, 12), dtype=np.float32) if instance_lights is None else np.ascontiguousarray(instance_lights, dtype=np.float32).reshape(-1, 12)

    # room: an emitter is a point light, a placement, or a primitive whose material is Emissive (LightCollection.cs:99-121)
    emissive = materials["type"] == structs.MATERIAL_EMISSIVE
    lit = lambda index: int(np.count_nonzero(emissive[index[index < len(materials)]])) if len(materials) else 0
    capacity = len(points) + len(rows) + lit(triangles["material"]) + lit(spheres["material"])
    nodes = np.empty(max(2 * capacity, 1), dtype=structs.LIGHT_NODE)
    tokens, paths = np.empty(max(capacity, 1), dtype=np.uint32), np.empty(max(capacity, 1), dtype=np.uint64)
    node_count, emitter_count, power = ctypes.c_uint32(), ctypes.c_uint32(), ctypes.c_float()
    _native.check(lib.echo_b200_build_light_tree(device, _native.pointer(triangles), len(triangles), _native.pointer(spheres), len(spheres), _native.pointer(materials), len(materials),
                                                 _native.pointer(points), len(points), _native.pointer(rows), len(rows), _native.pointer(nodes), len(nodes), ctypes.byref(node_count),
                                                 _native.pointer(tokens), _native.pointer(paths), len(tokens), ctypes.byref(emitter_count), ctypes.byref(power)))
    return nodes[:node_count.value].copy(), tokens[:emitter_count.value].copy(), paths[:emitter_count.value].copy(), float(power.value)


@dataclass
class BuiltPacks:
    """What echo_b200_build_packs returns: the pack records completed (nodeOffset / nodeCount / maxDepth / lightNode* / emitter*),
    every pack's QBVH nodes, light nodes, emitter tokens and bit paths back to back in pack order, and pack 0's light-tree root power."""
    packs: np.ndarray
    nodes: np.ndarray
    light_nodes: np.ndarray
    emitter_tokens: np.ndarray
    emitter_bitpaths: np.ndarray
    power: float

    @property
    def max_depth(self):
        return int(self.packs["maxDepth"].max())


def pack_build_arguments(prepared):
    """The inputs of echo_b200_build_packs from an instanced PreparedArrays: the shared arrays, the pack records with only their input
    ranges kept (geometry, placements, swatch, point lights), and output arrays with room for any result."""
    packs = np.zeros(len(prepared.packs), dtype=structs.PACK)
    for name in ("triangleOffset", "triangleCount", "sphereOffset", "sphereCount", "instanceOffset", "instanceCount", "materialOffset", "pointLightOffset", "pointLightCount"):
        packs[name] = prepared.packs[name]
    triangles = np.ascontiguousarray(prepared.triangles, dtype=structs.TRIANGLE)
    spheres = np.ascontiguousarray(prepared.spheres, dtype=structs.SPHERE)
    materials = np.ascontiguousarray(prepared.materials, dtype=structs.MATERIAL)
    points = np.ascontiguousarray(prepared.point_lights, dtype=structs.POINT_LIGHT)
    instances = np.ascontiguousarray(prepared.instances, dtype=structs.INSTANCE)
    candidates = len(triangles) + len(spheres) + len(instances) + len(points)
    outputs = (np.empty(max(len(triangles) + len(spheres) + len(instances), 1), dtype=structs.QBVH_NODE), np.empty(max(2 * candidates, 1), dtype=structs.LIGHT_NODE),
               np.empty(max(candidates, 1), dtype=np.uint32), np.empty(max(candidates, 1), dtype=np.uint64))
    return (triangles, spheres, materials, points, packs, instances), outputs


def build_packs_device(prepared, device=0):
    """Every pack of an instanced scene built on the device in one call (echo_b200_build_packs, csrc/packbuild.cu): each pack's QBVH
    and light tree equal host.build_qbvh / host.build_light_tree's byte for byte, fed with the placements' rows the device computes
    from the finished child trees. Returns BuiltPacks; the arrays are laid out as host.prepare lays them out."""
    lib = _native.library()
    (triangles, spheres, materials, points, packs, instances), (nodes, light_nodes, tokens, paths) = pack_build_arguments(prepared)
    ptr = _native.pointer
    node_count, light_count, emitter_count, power = ctypes.c_uint32(), ctypes.c_uint32(), ctypes.c_uint32(), ctypes.c_float()
    _native.check(lib.echo_b200_build_packs(device, ptr(triangles), len(triangles), ptr(spheres), len(spheres), ptr(materials), len(materials), ptr(points), len(points),
                                            ptr(packs), len(packs), ptr(instances), len(instances), ptr(nodes), len(nodes), ctypes.byref(node_count),
                                            ptr(light_nodes), len(light_nodes), ctypes.byref(light_count), ptr(tokens), ptr(paths), len(tokens), ctypes.byref(emitter_count),
                                            ctypes.byref(power)))
    return BuiltPacks(packs, nodes[:node_count.value].copy(), light_nodes[:light_count.value].copy(), tokens[:emitter_count.value].copy(),
                      paths[:emitter_count.value].copy(), float(power.value))


def shard_epochs(max_epoch, rank, world_size):
    """Sample sharding across devices (few tiles, many samples; SURVEY.md 8(e)(ii)): rank r renders block r of
    ceil(max_epoch / world_size) consecutive epochs of EVERY tile; returns (epoch_offset, epoch_count) for that rank's
    EchoRenderParams (epochOffset, minEpoch = maxEpoch = epoch_count). The sample index of a path is epoch * extend + i, so the
    blocks are disjoint sample sets. Each device accumulates (mean * epochs, epochs) per pixel (render_frame_device), the frames
    are summed with one all-reduce and frame_resolve divides by the summed weight. A trailing rank can be left with epoch_count 0
    (max_epoch 20 on 8 ranks: rank 7): render_frame_device / render_tiles treat maxEpoch == 0 as nothing to render."""
    per_rank = (max_epoch + world_size - 1) // world_size
    first = min(rank * per_rank, max_epoch)
    return first, max(0, min(per_rank, max_epoch - first))


class EvaluationOperation:
    """Processes/Evaluation/EvaluationOperation.cs:21-177 on the GPU: same public surface (tile_positions, destination,
    profile, total_samples, statistics), Execute renders every tile through libecho_b200 and applies it to the destination."""

    def __init__(self, scene: PreparedScene, profile: EvaluationProfile, destination: RenderTexture, tile_positions=None):
        profile.validate()
        self.scene = scene
        self.profile = profile
        self.destination = destination
        self.tile_positions = destination.tile_positions if tile_positions is None else np.asarray(tile_positions, dtype=np.int32).reshape(-1, 2)
        self.statistics = np.zeros(1, dtype=structs.STATS)

    @property
    def params(self):
        p = self.profile
        return structs.render_params(self.destination.width, self.destination.height, self.destination.tile_size, p.extend, p.min_epoch,
                                     p.max_epoch, p.noise_threshold, p.evaluator.bounce_limit, p.evaluator.survivability, p.seed,
                                     evaluator=p.evaluator.code)

    @property
    def total_samples(self):
        """EvaluationOperation.TotalSamples (:73-81): the "Sample/Evaluated" counter."""
        return int(self.statistics["sampleEvaluated"][0])

    def execute(self):
        tiles, stats = self.scene.render_tiles(self.params, self.tile_positions)
        for position, tile in zip(self.tile_positions, tiles):
            self.destination.apply(position, tile)
        for name in structs.STATS_FIELDS:
            self.statistics[name] += stats[name]
        return self.destination

    def statistics_report(self):
        """label -> count, the labels EvaluatorStatistics.Report uses on this path."""
        return {label: int(self.statistics[name][0]) for label, name in zip(structs.STATS_LABELS, structs.STATS_FIELDS)}
