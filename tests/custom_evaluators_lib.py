"""Evaluators a host writes itself (echorenderer_b200.DeviceEvaluator), for the tests of include/echo_b200_evaluation.h and
variants/custom_evaluation_rates.py. TEST INFRASTRUCTURE ONLY: they need torch, which the package does not import."""
import numpy as np
import torch

from echorenderer_b200 import DeviceEvaluator, _native

EPSILON = np.float32(8e-7)  # FastMath.Epsilon
IS_ZERO = [EPSILON / np.float32(w) for w in (0.212671, 0.715160, 0.072169)]  # RGB128.IsZero: luminance weights, as the kernels divide them


def torch_stream(stream):
    """the torch stream of a cudaStream_t given as an int (0: the legacy default stream, torch's default)"""
    return torch.cuda.ExternalStream(stream) if stream else torch.cuda.default_stream()


class TorchNaiveEvaluator(DeviceEvaluator):
    """StandardNaiveEvaluator (Evaluation/Evaluators/StandardNaiveEvaluator.cs:16-55) composed from the device queries on the
    evaluation's stream: trace (layered on a scene with packs), interact, scatter_sample with the draw at dimension 4 + 2 * depth,
    evaluate_infinite (direct at depth 0), then the fold of naive_kernel, value = scatter * value + emission from the innermost bounce
    outwards, each step a separate float32 operation in the kernel's order. `timer(name)`, when given, is a context manager around the
    Evaluation's own calls (spawn, draws)."""

    def __init__(self, instanced, bounce_limit, timer=None):
        self.instanced = instanced
        self.bounce_limit = bounce_limit
        self.timer = timer
        self.samples = None  # the Float4s of the last epoch, alive until the next call
        self.word = None

    def status(self):
        """raises EchoNativeError when a query of any epoch so far was refused (synchronises)"""
        if self.word is not None:
            _native.query_status(self.word.item())

    def _timed(self, name, call):
        if self.timer is None:
            call()
        else:
            with self.timer(name):
                call()

    def evaluate(self, scene, evaluation, count, stream):
        with torch.cuda.stream(torch_stream(stream)):
            self.samples = self._evaluate(scene, evaluation, count, stream)
        return self.samples.data_ptr()

    def _evaluate(self, scene, evaluation, n, stream):
        cuda = torch.device("cuda")
        if self.word is None:
            self.word = torch.full((1,), -1, dtype=torch.int64, device=cuda)
        w = self.word.data_ptr()

        rays = torch.empty((n, 8), dtype=torch.float32, device=cuda)  # EchoRay
        self._timed("spawn", lambda: evaluation.spawn_device(rays.data_ptr()))
        draws = torch.empty((n, 2), dtype=torch.float32, device=cuda)
        value = torch.zeros((n, 3), dtype=torch.float32, device=cuda)
        bounces = []  # per depth: (paths that bounced, scatter, emission)
        alive = torch.arange(n, device=cuda)
        ray, ignore = rays, None

        for depth in range(self.bounce_limit + 1):
            m = len(alive)
            if m == 0:
                break
            hits = torch.empty((m, 4), dtype=torch.int32, device=cuda)  # EchoHit
            layers = torch.empty((m, 6), dtype=torch.int32, device=cuda) if self.instanced else None  # EchoTokenHierarchy
            if depth == self.bounce_limit:
                hit = torch.zeros(m, dtype=torch.bool, device=cuda)
            else:
                if self.instanced:
                    scene.trace_hierarchy_device(ray.data_ptr(), None if ignore is None else ignore.data_ptr(), m, hits.data_ptr(), layers.data_ptr(), stream=stream)
                else:
                    scene.trace_device(ray.data_ptr(), m, hits.data_ptr(), stream=stream)
                hit = hits[:, 0] != -1

            missed = torch.nonzero(~hit).flatten()
            if len(missed):  # scene.EvaluateInfinite(direction, direct = depth == 0)
                directions = ray[missed, 3:6].contiguous()
                light = torch.empty((len(missed), 3), dtype=torch.float32, device=cuda)
                scene.evaluate_infinite_device(directions.data_ptr(), len(missed), depth == 0, light.data_ptr(), w, stream=stream)
                value[alive[missed]] = light

            found = torch.nonzero(hit).flatten()
            k = len(found)
            if k == 0:
                break
            hit_rays, hit_hits = ray[found].contiguous(), hits[found].contiguous()
            hit_layers = layers[found].contiguous() if self.instanced else None
            layers_pointer = None if hit_layers is None else hit_layers.data_ptr()
            contacts = torch.empty((k, 16), dtype=torch.float32, device=cuda)  # EchoContact
            scene.interact_device(hit_rays.data_ptr(), hit_hits.data_ptr(), layers_pointer, k, contacts.data_ptr(), w, stream=stream)
            self._timed("draw", lambda: evaluation.draw_device(4 + 2 * depth, 2, draws.data_ptr()))
            sample = draws[alive[found]].contiguous()
            scattered = torch.empty((k, 8), dtype=torch.float32, device=cuda)  # EchoScatter
            scene.scatter_sample_device(hit_rays.data_ptr(), hit_hits.data_ptr(), layers_pointer, sample.data_ptr(), k, scattered.data_ptr(), w, stream=stream)

            emission, incident, pdf, content = contacts[:, 12:15], scattered[:, 0:3], scattered[:, 3], scattered[:, 4:7]
            zero = (content[:, 0] < float(IS_ZERO[0])) & (content[:, 1] < float(IS_ZERO[1])) & (content[:, 2] < float(IS_ZERO[2]))
            stop = ~(pdf >= float(EPSILON)) | zero  # "Exit if the BSDF sample is not promising"
            stopped = torch.nonzero(stop).flatten()
            value[alive[found[stopped]]] = emission[stopped]

            go = torch.nonzero(~stop).flatten()
            shade, towards = contacts[go, 6:9], incident[go]
            cosine = (towards[:, 0] * shade[:, 0] + towards[:, 1] * shade[:, 1]) + towards[:, 2] * shade[:, 2]
            scatter = (content[go] / pdf[go].unsqueeze(1)) * cosine.abs().unsqueeze(1)
            bounces.append((alive[found[go]], scatter, emission[go]))

            ray = torch.empty((len(go), 8), dtype=torch.float32, device=cuda)  # query.SpawnTrace(incident)
            ray[:, 0:3], ray[:, 3:6], ray[:, 6] = contacts[go, 0:3], towards, float("inf")
            ray.view(torch.int32)[:, 7] = hit_hits[go, 0]
            ignore = hit_layers[go].contiguous() if self.instanced else None
            alive = alive[found[go]]

        for paths, scatter, emission in reversed(bounces):  # innermost first
            value[paths] = scatter * value[paths] + emission

        out = torch.zeros((n, 4), dtype=torch.float32, device=cuda)
        out[:, 0:3] = value
        return out


def hash_samples(pixel_index, sample_index):
    """A Float4 per (pixel, sample index), with NaN and infinities among them. Pixel % 3 picks how much the samples vary: a little
    around a large mean, or as u^2 or u^8 of a uniform u (relative spreads of 0.9 and 1.9), so that a noise threshold stops some pixels
    at minEpoch, some later and some not before maxEpoch."""
    pixel_index = np.asarray(pixel_index, dtype=np.uint64)
    h = (pixel_index * np.uint64(0x9E3779B1) + np.asarray(sample_index, dtype=np.uint64) * np.uint64(0x85EBCA77) + np.uint64(0x165667B1)) & np.uint64(0xFFFFFFFF)
    for shift, factor in ((15, 0x2C1B3C6D), (12, 0x297A2D39), (15, 1)):
        h ^= h >> np.uint64(shift)
        h = (h * np.uint64(factor)) & np.uint64(0xFFFFFFFF)
    lanes = np.stack([((h >> np.uint64(8 * c)) & np.uint64(0xFF)).astype(np.float32) / np.float32(256.0) for c in range(4)], axis=1)
    kind = (pixel_index % np.uint64(3)).astype(np.int64)[:, None]
    base = np.where(kind == 0, np.float32(0.5) + (pixel_index % np.uint64(7)).astype(np.float32)[:, None], np.float32(0.0)).astype(np.float32)
    spread = np.choose(kind, [np.float32(0.02), np.float32(2.0), np.float32(3.0)]).astype(np.float32)
    power = np.choose(kind, [np.float32(1.0), np.float32(2.0), np.float32(8.0)]).astype(np.float32)
    values = (base + spread * np.power(lanes, power)).astype(np.float32)
    values[h % np.uint64(53) == 0, 0] = np.nan
    values[h % np.uint64(59) == 0, 2] = np.inf
    values[h % np.uint64(61) == 0, 1] = -np.inf
    return values


class HashEvaluator(DeviceEvaluator):
    """hash_samples of each slot's (pixel, sample index) as spawn_device reports them: computed on the host, uploaded"""

    def __init__(self, width):
        self.width = width
        self.samples = None

    def evaluate(self, scene, evaluation, count, stream):
        with torch.cuda.stream(torch_stream(stream)):
            rays = torch.empty((count, 8), dtype=torch.float32, device="cuda")
            pixels = torch.empty((count, 2), dtype=torch.int32, device="cuda")
            samples = torch.empty(count, dtype=torch.int32, device="cuda")
            evaluation.spawn_device(rays.data_ptr(), pixels.data_ptr(), samples.data_ptr())
            pixels, samples = pixels.cpu().numpy(), samples.cpu().numpy().view(np.uint32)
            index = pixels[:, 1].astype(np.uint64) * np.uint64(self.width) + pixels[:, 0].astype(np.uint64)
            self.samples = torch.from_numpy(hash_samples(index, samples)).cuda()
        return self.samples.data_ptr()
