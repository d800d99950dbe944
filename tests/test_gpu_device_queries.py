"""The device-buffer queries of include/echo_b200_query_device.h on torch CUDA tensors: the same bytes as the host-buffer calls on
every parity fixture and two instanced scenes, every refusal of the host-buffer calls replayed through the status word, the edge
table of the shared rules, a direct-lighting evaluator that stays on the device, and capture in a CUDA graph."""
import ctypes

import numpy as np
import pytest
import torch

from echorenderer_b200 import EchoNativeError, PreparedScene, _native, host, scenes, structs
from tests import query_rules_lib
from tests.scene_query_oracle import samples_with_edges, scene as query_oracle_scene, surfaces, unit_vectors
from tests.test_gpu_scene_queries import PARITY, camera_rays, direct_lighting, gpu_count, prepared_scene, query_rays
from tests.test_furnace import RHO, lit_plane, point_light_radiance, polygon_irradiance

pytestmark = pytest.mark.gpu

CLEAR = _native.QUERY_STATUS_CLEAR


def up(array, dtype):
    """a numpy array as a CUDA byte tensor (None stays None)"""
    if array is None:
        return None
    data = np.ascontiguousarray(array, dtype=dtype)
    return torch.from_numpy(data.view(np.uint8).reshape(-1).copy()).cuda()


def down(tensor, dtype, shape=None):
    out = tensor.cpu().numpy().view(dtype)
    return out if shape is None else out.reshape(shape)


def address(tensor):
    return None if tensor is None else tensor.data_ptr()


def empty(count, dtype):
    return torch.empty(max(count * np.dtype(dtype).itemsize, 1), dtype=torch.uint8, device="cuda")


class DeviceQueries:
    """PreparedScene's host-buffer query methods over the _device calls, on the current torch stream: numpy in, numpy out. Every
    call lowers self.status, which status() reads back."""

    def __init__(self, scene):
        self.scene = scene
        self.word = torch.full((1,), -1, dtype=torch.int64, device="cuda")

    def clear(self):
        self.word.fill_(-1)

    def status(self):
        return int(self.word.item()) & CLEAR

    def _call(self, method, *arguments):
        """tensors among `arguments` stand for their addresses, and stay alive until the call is enqueued"""
        addresses = [a.data_ptr() if isinstance(a, torch.Tensor) else a for a in arguments]
        getattr(self.scene, method)(*addresses, self.word.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)

    def interact(self, rays, hits, layers=None):
        out = empty(len(rays), structs.CONTACT)
        self._call("interact_device", up(rays, structs.RAY), up(hits, structs.HIT), up(layers, structs.TOKEN_HIERARCHY), len(rays), out)
        return down(out, structs.CONTACT)

    def scatter_sample(self, rays, hits, samples, layers=None):
        out = empty(len(rays), structs.SCATTER)
        self._call("scatter_sample_device", up(rays, structs.RAY), up(hits, structs.HIT), up(layers, structs.TOKEN_HIERARCHY),
                   up(samples, np.float32), len(rays), out)
        return down(out, structs.SCATTER)

    def scatter_evaluate(self, rays, hits, incident, layers=None):
        out = empty(len(rays) * 4, np.float32)
        self._call("scatter_evaluate_device", up(rays, structs.RAY), up(hits, structs.HIT), up(layers, structs.TOKEN_HIERARCHY),
                   up(incident, np.float32), len(rays), out)
        return down(out, np.float32, (-1, 4))

    def pick(self, points, samples):
        n = len(points)
        tokens, layers, pmf = empty(n, np.uint32), empty(n, structs.TOKEN_HIERARCHY), empty(n, np.float32)
        self._call("pick_device", up(points, structs.SURFACE), up(samples, np.float32), n, tokens, layers, pmf)
        return down(tokens, np.uint32), down(layers, structs.TOKEN_HIERARCHY), down(pmf, np.float32)

    def probability_mass(self, tokens, points, layers=None):
        out = empty(len(tokens), np.float32)
        self._call("probability_mass_device", up(tokens, np.uint32), up(layers, structs.TOKEN_HIERARCHY), up(points, structs.SURFACE), len(tokens), out)
        return down(out, np.float32)

    def sample(self, tokens, points, samples, layers=None):
        out = empty(len(tokens), structs.LIGHT_SAMPLE)
        self._call("sample_device", up(tokens, np.uint32), up(layers, structs.TOKEN_HIERARCHY), up(points, structs.SURFACE),
                   up(samples, np.float32), len(tokens), out)
        return down(out, structs.LIGHT_SAMPLE)

    def probability_density(self, tokens, points, incident, layers=None):
        out = empty(len(tokens), np.float32)
        self._call("probability_density_device", up(tokens, np.uint32), up(layers, structs.TOKEN_HIERARCHY), up(points, structs.SURFACE),
                   up(incident, np.float32), len(tokens), out)
        return down(out, np.float32)

    def evaluate_infinite(self, directions, direct=False):
        out = empty(len(directions) * 3, np.float32)
        self._call("evaluate_infinite_device", up(directions, np.float32), len(directions), direct, out)
        return down(out, np.float32, (-1, 3))


def same_bytes(a, b):
    return all(same_bytes(x, y) for x, y in zip(a, b)) if isinstance(a, tuple) else np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def trace_both(scene, prepared, rays, ignore=None):
    """the hierarchy trace through both forms (the plain trace without packs): (hits, layers) of the host call, checked against the device call"""
    if prepared.packs is None:
        return scene.trace(rays), None
    hits, layers = scene.trace_hierarchy(rays, ignore)
    d_rays, d_ignore = up(rays, structs.RAY), up(ignore, structs.TOKEN_HIERARCHY)
    d_hits, d_layers = empty(len(rays), structs.HIT), empty(len(rays), structs.TOKEN_HIERARCHY)
    scene.trace_hierarchy_device(address(d_rays), address(d_ignore), len(rays), address(d_hits), address(d_layers))
    assert same_bytes(down(d_hits, structs.HIT), hits) and same_bytes(down(d_layers, structs.TOKEN_HIERARCHY), layers)
    occluded = empty(len(rays), np.uint8)
    scene.occlude_hierarchy_device(address(d_rays), address(d_ignore), len(rays), address(occluded))
    assert same_bytes(down(occluded, np.uint8), scene.occlude_hierarchy(rays, ignore))
    return hits, layers


@pytest.mark.parametrize("fixture", PARITY + ["instanced", "many_packs"])
def test_every_device_call_gives_the_host_calls_bytes(fixture, request):
    prepared = prepared_scene(fixture, request)
    rng = np.random.default_rng(17)

    with PreparedScene(prepared) as scene:
        device = DeviceQueries(scene)
        rays = query_rays(prepared, query_oracle_scene(prepared), seed=3)
        hits, layers = trace_both(scene, prepared, rays)
        hit = hits["token"] != structs.TOKEN_EMPTY

        def both(name, *arguments):
            expected, actual = getattr(scene, name)(*arguments), getattr(device, name)(*arguments)
            assert same_bytes(actual, expected), name
            return expected

        contacts = both("interact", rays, hits, layers)
        scattered = both("scatter_sample", rays, hits, samples_with_edges(rng, (len(rays), 2)), layers)
        incident = scattered["incident"].copy()
        impossible = ~(scattered["pdf"] > 0)
        incident[impossible] = unit_vectors(rng, int(impossible.sum()))
        both("scatter_evaluate", rays, hits, incident, layers)

        points = surfaces(contacts["position"][hit], contacts["normal"][hit])
        tokens, light_layers, _ = both("pick", points, samples_with_edges(rng, len(points)))
        both("sample", tokens, points, samples_with_edges(rng, (len(points), 2)), light_layers)
        both("probability_mass", tokens, points, light_layers)
        both("probability_density", tokens, points, unit_vectors(rng, len(points)), light_layers)

        onward = hit & (scattered["pdf"] > 0)
        secondary = np.zeros(int(onward.sum()), dtype=structs.RAY)
        secondary["origin"], secondary["direction"] = contacts["position"][onward], scattered["incident"][onward]
        secondary["distance"], secondary["ignore"] = np.inf, hits["token"][onward]
        found, found_layers = trace_both(scene, prepared, secondary, None if layers is None else layers[onward])
        origins = surfaces(contacts["position"][onward], contacts["normal"][onward])
        both("probability_mass", found["token"], origins, found_layers)  # misses included
        both("probability_density", found["token"], origins, secondary["direction"], found_layers)
        for direct in (False, True):
            both("evaluate_infinite", np.concatenate([rays["direction"][~hit], secondary["direction"]]), direct)
        assert device.status() == CLEAR


def miss_record(name, out):
    """the record a refused query gets: the zeroed record of a miss"""
    if name == "pick":
        return (np.full(1, structs.TOKEN_EMPTY, np.uint32), np.zeros(1, structs.TOKEN_HIERARCHY), np.zeros(1, np.float32))
    record = np.zeros(1, out.dtype) if out.ndim == 1 else np.zeros((1,) + out.shape[1:], out.dtype)
    if name == "interact":
        record["material"] = structs.TOKEN_EMPTY
    return record


def replay(scene, device, name, arguments, index):
    """a call the host-buffer form refuses at `index`, through the device form: the same index and reason, the refused row zeroed,
    every other row what the host call gives for the batch without the refused row"""
    with pytest.raises(EchoNativeError) as error:
        getattr(scene, name)(*arguments)
    message = query_rules_lib.normalise(str(error.value))
    device.clear()
    actual = getattr(device, name)(*arguments)
    status = device.status()
    assert status != CLEAR and status >> 8 == index, (name, status, message)
    assert f"query {index}: {_native.query_reason(status & 0xFF)}" in message, (name, message)

    rows = tuple(actual) if isinstance(actual, tuple) else (actual,)
    assert same_bytes(tuple(r[index:index + 1] for r in rows), miss_record(name, rows[0]) if name == "pick" else (miss_record(name, rows[0]),)), name
    n = len(rows[0])
    valid = [np.delete(a, index, axis=0) if isinstance(a, np.ndarray) and len(a) == n else a for a in arguments]
    expected = getattr(scene, name)(*valid)
    expected = tuple(expected) if isinstance(expected, tuple) else (expected,)
    assert same_bytes(tuple(np.delete(r, index, axis=0) for r in rows), expected), name
    with pytest.raises(EchoNativeError, match=f"query {index}:"):
        _native.query_status(status)


def test_refusals_through_the_status_word(cornell):
    """every case of test_gpu_scene_queries.test_refusals, then the lower of two refusals, NULL buffers, n = 0, an uncommitted scene"""
    instanced = host.prepare(scenes.instanced_scene(grid=3, rings=8, segments=10))
    rays = scenes.random_rays(cornell.bounds, 8, seed=2)
    samples = np.full((8, 2), 0.5, np.float32)
    incident = np.tile(np.float32([0, 1, 0]), (8, 1))
    points = surfaces(np.zeros((8, 3), np.float32), incident)

    def light(kind, index):
        return structs.make_token(structs.TOKEN_TYPE_LIGHT, (kind << structs.LIGHT_INDEX_BITS) | index)

    with PreparedScene(cornell) as scene:
        device = DeviceQueries(scene)
        hits = scene.trace(rays)
        hits[:3] = hits[0]
        hits["token"][:3] = structs.make_token(structs.TOKEN_TYPE_TRIANGLE, 0)
        hits["uv"][:3] = (0.25, 0.25)
        hits["distance"][:3] = 1.0

        def bad_hit(token, uv=(0.25, 0.25)):
            h = hits.copy()
            h["token"][3], h["uv"][3], h["distance"][3] = token, uv, 1.0
            return h

        replay(scene, device, "interact", (rays, bad_hit(structs.make_token(structs.TOKEN_TYPE_TRIANGLE, len(cornell.triangles)))), 3)
        replay(scene, device, "scatter_sample", (rays, bad_hit(structs.make_token(structs.TOKEN_TYPE_SPHERE, len(cornell.spheres) + 2), (0.0, 0.0)), samples), 3)
        replay(scene, device, "interact", (rays, bad_hit(structs.make_token(structs.TOKEN_TYPE_TRIANGLE, 0), (0.5, 1.5))), 3)
        replay(scene, device, "interact", (rays, bad_hit(structs.make_token(structs.TOKEN_TYPE_INSTANCE, 0))), 3)
        nan_rays = rays.copy()
        nan_rays["origin"][5, 1] = np.nan
        replay(scene, device, "interact", (nan_rays, bad_hit(structs.TOKEN_EMPTY)), 5)
        inf_samples = samples.copy()
        inf_samples[6, 0] = np.inf
        replay(scene, device, "scatter_sample", (rays, bad_hit(structs.TOKEN_EMPTY), inf_samples), 6)
        nan_incident = incident.copy()
        nan_incident[2, 2] = np.nan
        replay(scene, device, "scatter_evaluate", (rays, bad_hit(structs.TOKEN_EMPTY), nan_incident), 2)

        layers = np.zeros(8, structs.TOKEN_HIERARCHY)
        layers["instanceCount"][4], layers["instances"][4, 0] = 1, structs.make_token(structs.TOKEN_TYPE_INSTANCE, 0)
        replay(scene, device, "interact", (rays, bad_hit(structs.TOKEN_EMPTY), layers), 4)
        tokens = np.full(8, structs.TOKEN_EMPTY, np.uint32)
        replay(scene, device, "probability_mass", (tokens, points, layers), 4)

        def bad_light(token):
            t = tokens.copy()
            t[1] = token
            return t

        replay(scene, device, "sample", (bad_light(light(structs.LIGHT_TYPE_POINT, len(cornell.point_lights))), points, samples), 1)
        replay(scene, device, "probability_density", (bad_light(light(structs.LIGHT_TYPE_INFINITE, len(cornell.description.infinite_lights))), points, incident), 1)
        replay(scene, device, "probability_mass", (bad_light(structs.make_token(structs.TOKEN_TYPE_TRIANGLE, len(cornell.triangles))), points), 1)
        replay(scene, device, "sample", (bad_light(structs.make_token(structs.TOKEN_TYPE_SPHERE, len(cornell.spheres))), points, samples), 1)
        replay(scene, device, "probability_mass", (bad_light(structs.make_token(structs.TOKEN_TYPE_NODE, 0)), points), 1)
        nan_points = points.copy()
        nan_points["normal"][7, 0] = np.inf
        replay(scene, device, "pick", (nan_points, np.full(8, 0.5, np.float32)), 7)
        replay(scene, device, "pick", (points, np.array([0.5] * 7 + [np.nan], np.float32)), 7)
        directions = np.tile(np.float32([0, 1, 0]), (8, 1))
        directions[0] = (0, 2, 0)
        replay(scene, device, "evaluate_infinite", (directions,), 0)

        # two refused queries report the lower index, also across calls on one status word; valid batches leave it clear
        twice = bad_hit(structs.make_token(structs.TOKEN_TYPE_TRIANGLE, len(cornell.triangles)))
        twice["token"][6] = structs.make_token(structs.TOKEN_TYPE_INSTANCE, 0)
        device.clear()
        device.interact(rays, twice)
        assert device.status() >> 8 == 3
        device.evaluate_infinite(directions[::-1].copy())  # refused at 7: the word keeps 3
        assert device.status() >> 8 == 3
        device.clear()
        device.interact(rays, scene.trace(rays))
        device.pick(points, np.full(8, 0.5, np.float32))
        assert device.status() == CLEAR

        lib, handle = _native.library(), scene.handle
        buffer, word = torch.zeros(4096, dtype=torch.uint8, device="cuda"), device.word
        b, w = buffer.data_ptr(), word.data_ptr()
        assert lib.echo_b200_interact_batch_device(handle, b, b, None, 8, b, None, None) == _native.ERR_INVALID and b"null buffer" in lib.echo_b200_last_error()
        assert lib.echo_b200_light_pick_batch_device(handle, None, b, 8, b, None, b, w, None) == _native.ERR_INVALID and b"null buffer" in lib.echo_b200_last_error()
        assert lib.echo_b200_evaluate_infinite_batch_device(handle, b, 8, 0, b, None, None) == _native.ERR_INVALID
        assert lib.echo_b200_interact_batch_device(handle, None, None, None, 0, None, None, None) == _native.OK  # n == 0 needs no buffers
        assert lib.echo_b200_interact_batch_device(handle, b, b, None, 1 << 56, b, w, None) == _native.ERR_INVALID
        assert lib.echo_b200_trace_batch_hierarchy_device(handle, b, None, 8, b, None, None) == _native.ERR_INVALID and b"no packs" in lib.echo_b200_last_error()
        torch.cuda.synchronize()
        assert not scene.bounds_violations()

    with PreparedScene(instanced) as scene:
        device = DeviceQueries(scene)
        rays = scenes.random_rays(instanced.bounds, 8, seed=4)
        hits, layers = scene.trace_hierarchy(rays)
        layers[3]["instanceCount"], layers[3]["instances"][0] = 1, structs.make_token(structs.TOKEN_TYPE_TRIANGLE, 0)
        replay(scene, device, "interact", (rays, hits, layers), 3)
        layers[3]["instanceCount"] = structs.MAX_INSTANCE_LAYERS + 1
        replay(scene, device, "interact", (rays, hits, layers), 3)
        lib, handle = _native.library(), scene.handle
        assert lib.echo_b200_occlude_batch_hierarchy_device(handle, None, None, 8, None, None) == _native.ERR_INVALID
        assert lib.echo_b200_trace_batch_hierarchy_device(handle, None, None, 0, None, None, None) == _native.OK
        torch.cuda.synchronize()
        assert not scene.bounds_violations()

    lib = _native.library()
    handle = ctypes.c_void_p()
    _native.check(lib.echo_b200_scene_create(ctypes.byref(handle), 0))
    try:
        buffer = torch.zeros(4096, dtype=torch.uint8, device="cuda")
        b = buffer.data_ptr()
        for n in (8, 0):
            assert lib.echo_b200_light_mass_batch_device(handle, b, None, b, n, b, b, None) == _native.ERR_INVALID
            assert b"not committed" in lib.echo_b200_last_error()
            assert lib.echo_b200_trace_batch_hierarchy_device(handle, b, None, n, b, None, None) == _native.ERR_INVALID
    finally:
        lib.echo_b200_scene_destroy(handle)


@pytest.mark.skipif(gpu_count() < 2, reason="needs two GPUs")
def test_multi_device_scene_is_refused():
    prepared = host.prepare(scenes.instanced_scene(grid=3, rings=8, segments=10))
    with PreparedScene(prepared, devices=[0, 1]) as multi:
        buffer = torch.zeros(4096, dtype=torch.uint8, device="cuda")
        b = buffer.data_ptr()
        with pytest.raises(EchoNativeError, match="single-device scene"):
            multi.evaluate_infinite_device(b, 8, False, b, b)
        with pytest.raises(EchoNativeError, match="single-device scene"):
            multi.trace_hierarchy_device(b, None, 8, b, None)


@pytest.mark.parametrize("name", ["instanced", "cornell_box"])
def test_edge_table_is_decided_alike_by_host_and_device(name):
    prepared = host.prepare(scenes.instanced_scene(grid=3, rings=8, segments=10) if name == "instanced" else scenes.cornell_box())
    contact, light, expected_contact, expected_light = query_rules_lib.edge_table(prepared)

    def host_reason(call):
        try:
            call()
            return None
        except EchoNativeError as error:
            return query_rules_lib.normalise(str(error)).split("query 0: ", 1)[1]

    with PreparedScene(prepared) as scene:
        device = DeviceQueries(scene)
        for i, expected in enumerate(expected_contact):
            row = (contact["rays"][i:i + 1], contact["hits"][i:i + 1], contact["values"][i:i + 1], contact["layers"][i:i + 1])
            assert host_reason(lambda: scene.scatter_evaluate(*row)) == expected, i
            device.clear()
            device.scatter_evaluate(*row)
            status = device.status()
            assert (None if status == CLEAR else _native.query_reason(status & 0xFF)) == expected, i
        for i, expected in enumerate(expected_light):
            row = (light["tokens"][i:i + 1], light["points"][i:i + 1], light["values"][i:i + 1], light["layers"][i:i + 1])
            assert host_reason(lambda: scene.probability_density(*row)) == expected, i
            device.clear()
            device.probability_density(*row)
            status = device.status()
            assert (None if status == CLEAR else _native.query_reason(status & 0xFF)) == expected, i
        # the whole table in one call: the lowest refused row
        device.clear()
        device.scatter_evaluate(contact["rays"], contact["hits"], contact["values"], contact["layers"])
        assert device.status() >> 8 == next(i for i, e in enumerate(expected_contact) if e is not None)
        torch.cuda.synchronize()
        assert not scene.bounds_violations()


class Replayed:
    """the numbers a numpy Generator drew, handed out again in the same order"""

    def __init__(self, rng):
        self.rng, self.drawn = rng, []

    def random(self, size, dtype=np.float64):
        value = self.rng.random(size, dtype=dtype)
        self.drawn.append(value)
        return value


def direct_lighting_on_device(scene, rays, numbers, mis):
    """direct_lighting of test_gpu_scene_queries over device tensors: every call on one non-default stream, compaction with
    torch.nonzero, shadow and secondary rays assembled in a tensor viewed as EchoRay, one synchronise at the end. `numbers` are
    the random arrays the numpy version drew, in its order. Returns (radiance float64[n, 3], hit mask, downloaded intermediates)."""
    n = len(rays)
    numbers = list(numbers)
    stream = torch.cuda.Stream()
    word = torch.full((1,), -1, dtype=torch.int64, device="cuda")
    cuda = stream.cuda_stream
    f32 = lambda t: t.view(torch.float32)  # noqa: E731
    out = {}

    with torch.cuda.stream(stream):
        d_rays = up(rays, structs.RAY)
        ray_words = f32(d_rays).view(n, 8)
        hits = empty(n, structs.HIT)
        scene.trace_device(d_rays.data_ptr(), n, hits.data_ptr(), stream=cuda)
        hit_tokens = hits.view(torch.int32).view(n, 4)[:, 0]
        hit = hit_tokens != -1
        contacts = empty(n, structs.CONTACT)
        scene.interact_device(d_rays.data_ptr(), hits.data_ptr(), None, n, contacts.data_ptr(), word.data_ptr(), stream=cuda)
        c = f32(contacts).view(n, 16)
        position, normal, shade = c[:, 0:3], c[:, 3:6], c[:, 6:9].double()
        points = torch.cat([position, normal], dim=1).contiguous()  # EchoSurface
        radiance = torch.zeros((n, 3), dtype=torch.float64, device="cuda")

        lit = torch.nonzero(hit).flatten()
        m = len(lit)
        lit_points = points[lit].contiguous()
        picks = torch.from_numpy(numbers.pop(0)).cuda()
        tokens, pmf = torch.empty(m, dtype=torch.int32, device="cuda"), torch.empty(m, dtype=torch.float32, device="cuda")
        scene.pick_device(lit_points.data_ptr(), picks.data_ptr(), m, tokens.data_ptr(), None, pmf.data_ptr(), word.data_ptr(), stream=cuda)
        radiant = torch.from_numpy(numbers.pop(0)).cuda()
        sampled = torch.empty((m, 8), dtype=torch.float32, device="cuda")
        scene.sample_device(tokens.data_ptr(), None, lit_points.data_ptr(), radiant.data_ptr(), m, sampled.data_ptr(), word.data_ptr(), stream=cuda)
        keep = torch.nonzero((pmf > 0) & (sampled[:, 3] > 0)).flatten()
        k = len(keep)
        light = lit[keep]
        shadow = torch.zeros((k, 8), dtype=torch.float32, device="cuda")  # EchoRay
        shadow[:, 0:3], shadow[:, 3:6], shadow[:, 6] = position[light], sampled[keep, 4:7], sampled[keep, 7]
        shadow.view(torch.int32)[:, 7] = hit_tokens[light]
        occluded = torch.empty(k, dtype=torch.uint8, device="cuda")
        scene.occlude_device(shadow.data_ptr(), k, occluded.data_ptr(), stream=cuda)
        light_rays, light_hits = ray_words[light].contiguous(), hits.view(n, 16)[light].contiguous()
        incident = sampled[keep, 4:7].contiguous()
        f = torch.empty((k, 4), dtype=torch.float32, device="cuda")
        scene.scatter_evaluate_device(light_rays.data_ptr(), light_hits.data_ptr(), None, incident.data_ptr(), k, f.data_ptr(), word.data_ptr(), stream=cuda)
        cosine = (incident.double() * shade[light]).sum(dim=1).abs()
        pdf = pmf[keep].double() * sampled[keep, 3].double()
        fpdf = f[:, 3].double()
        weight = torch.where(pdf * pdf + fpdf * fpdf > 0, pdf * pdf / torch.clamp(pdf * pdf + fpdf * fpdf, min=1e-38), 0.0) if mis else 1.0
        visible = (occluded == 0).double()
        radiance[light] += (sampled[keep, 0:3] * f[:, 0:3]).double() * (cosine * weight * visible / pdf)[:, None]  # float32 product, as numpy forms it
        out.update(hits=hits, contacts=contacts, tokens=tokens, pmf=pmf, sampled=sampled, occluded=occluded, f=f)

        if mis:
            bounce = torch.from_numpy(numbers.pop(0)).cuda()
            bounced = torch.empty((n, 8), dtype=torch.float32, device="cuda")
            scene.scatter_sample_device(d_rays.data_ptr(), hits.data_ptr(), None, bounce.data_ptr(), n, bounced.data_ptr(), word.data_ptr(), stream=cuda)
            onward = torch.nonzero(hit & (bounced[:, 3] > 0)).flatten()
            o = len(onward)
            secondary = torch.zeros((o, 8), dtype=torch.float32, device="cuda")
            secondary[:, 0:3], secondary[:, 3:6], secondary[:, 6] = position[onward], bounced[onward, 0:3], float("inf")
            secondary.view(torch.int32)[:, 7] = hit_tokens[onward]
            found = empty(o, structs.HIT)
            scene.trace_device(secondary.data_ptr(), o, found.data_ptr(), stream=cuda)
            emitted = torch.empty((o, 16), dtype=torch.float32, device="cuda")
            scene.interact_device(secondary.data_ptr(), found.data_ptr(), None, o, emitted.data_ptr(), word.data_ptr(), stream=cuda)
            found_tokens = found.view(torch.int32).view(o, 4)[:, 0].contiguous()  # a miss is ECHO_TOKEN_EMPTY already
            onward_points, onward_incident = points[onward].contiguous(), bounced[onward, 0:3].contiguous()
            mass, density = torch.empty(o, dtype=torch.float32, device="cuda"), torch.empty(o, dtype=torch.float32, device="cuda")
            scene.probability_mass_device(found_tokens.data_ptr(), None, onward_points.data_ptr(), o, mass.data_ptr(), word.data_ptr(), stream=cuda)
            scene.probability_density_device(found_tokens.data_ptr(), None, onward_points.data_ptr(), onward_incident.data_ptr(), o, density.data_ptr(), word.data_ptr(), stream=cuda)
            scatter_pdf = bounced[onward, 3].double()
            light_pdf = mass.double() * density.double()
            weight = torch.where(scatter_pdf ** 2 + light_pdf ** 2 > 0, scatter_pdf ** 2 / torch.clamp(scatter_pdf ** 2 + light_pdf ** 2, min=1e-38), 0.0)
            cosine = (onward_incident.double() * shade[onward]).sum(dim=1).abs()
            radiance[onward] += emitted[:, 12:15].double() * bounced[onward, 4:7].double() * (cosine * weight / scatter_pdf)[:, None]
            out.update(bounced=bounced, found=found, emitted=emitted, mass=mass, density=density, secondary=secondary)

    stream.synchronize()
    _native.query_status(word.item())
    return radiance.cpu().numpy(), hit.cpu().numpy(), {name: t.cpu().numpy() for name, t in out.items()}


def check_intermediates(scene, rays, numbers, got, mis):
    """every downloaded intermediate is what the host-buffer call gives for the same inputs"""
    hits = got["hits"].view(structs.HIT)
    assert same_bytes(hits, scene.trace(rays))
    contacts = got["contacts"].view(structs.CONTACT)
    assert same_bytes(contacts, scene.interact(rays, hits))
    hit = hits["token"] != structs.TOKEN_EMPTY
    points = surfaces(contacts["position"], contacts["normal"])[hit]
    tokens, _, pmf = scene.pick(points, numbers[0])
    assert same_bytes(got["tokens"].view(np.uint32), tokens) and same_bytes(got["pmf"], pmf)
    sampled = scene.sample(tokens, points, numbers[1])
    assert same_bytes(got["sampled"].view(structs.LIGHT_SAMPLE).reshape(-1), sampled)
    keep = (pmf > 0) & (sampled["pdf"] > 0)
    light = np.flatnonzero(hit)[keep]
    assert same_bytes(got["f"], scene.scatter_evaluate(rays[light], hits[light], sampled["incident"][keep]))
    if mis:
        bounced = scene.scatter_sample(rays, hits, numbers[2])
        assert same_bytes(got["bounced"].view(structs.SCATTER).reshape(-1), bounced)
        secondary = got["secondary"].view(structs.RAY).reshape(-1)
        found = scene.trace(secondary)
        assert same_bytes(got["found"].view(structs.HIT), found)
        assert same_bytes(got["emitted"].view(structs.CONTACT).reshape(-1), scene.interact(secondary, found))
        origins = points[np.isin(np.flatnonzero(hit), np.flatnonzero(hit & (bounced["pdf"] > 0)))]
        assert same_bytes(got["mass"], scene.probability_mass(found["token"], origins))
        assert same_bytes(got["density"], scene.probability_density(found["token"], origins, secondary["direction"]))


def test_device_evaluator_one_point_light_is_exact_per_sample():
    light = ((30.0, 20.0, 10.0), (1.0, 3.0, -0.5))
    description = lit_plane([light])
    rays = camera_rays(description, 16, 2, seed=8)
    with PreparedScene(host.prepare(description)) as scene:
        drawn = Replayed(np.random.default_rng(3))
        expected, expected_hit = direct_lighting(scene, rays, drawn, mis=False)
        radiance, hit, got = direct_lighting_on_device(scene, rays, drawn.drawn, mis=False)
        check_intermediates(scene, rays, drawn.drawn, got, mis=False)
        hits = scene.trace(rays)
    assert np.array_equal(hit, expected_hit) and np.allclose(radiance, expected, rtol=1e-12, atol=0)
    points = rays["origin"].astype(np.float64) + rays["direction"].astype(np.float64) * np.where(hit, hits["distance"], 0.0)[:, None]
    assert hit.mean() > 0.8 and np.all(radiance[~hit] == 0)
    assert np.allclose(radiance[hit], point_light_radiance(points[hit], *light), rtol=1e-5, atol=0)


def test_device_evaluator_with_mis_converges_to_lamberts_formula():
    emission = np.array((10.0, 8.0, 6.0))
    corner, side = np.array((-1.0, 3.0, -1.0)), 2.0
    vertices = np.stack([corner, corner + (side, 0, 0), corner + (0, 0, side)])
    materials = np.concatenate([scenes.material(structs.MATERIAL_DIFFUSE, RHO), scenes.material(structs.MATERIAL_EMISSIVE, tuple(emission))])
    triangles = np.concatenate([scenes.plane(0, (20, 20)), scenes.make_triangles(vertices[0:1], vertices[1:2], vertices[2:3], 1)])
    description = lit_plane([])
    description.triangles, description.materials = triangles, materials
    rays = camera_rays(description, 12, 256, seed=10)

    with PreparedScene(host.prepare(description)) as scene:
        drawn = Replayed(np.random.default_rng(4))
        expected, expected_hit = direct_lighting(scene, rays, drawn, mis=True)
        radiance, hit, got = direct_lighting_on_device(scene, rays, drawn.drawn, mis=True)
        check_intermediates(scene, rays, drawn.drawn, got, mis=True)
        hits = scene.trace(rays)
    assert np.array_equal(hit, expected_hit) and np.allclose(radiance, expected, rtol=1e-12, atol=0)
    points = rays["origin"].astype(np.float64) + rays["direction"].astype(np.float64) * np.where(hit, hits["distance"], 0.0)[:, None]
    on_plane = hit & (points[:, 1] < 1e-3)
    assert on_plane.mean() > 0.7
    truth = (np.array(RHO) / np.pi * emission * polygon_irradiance(points[on_plane], vertices)[:, None]).mean(axis=0)
    mean, error = radiance[on_plane].mean(axis=0), radiance[on_plane].std(axis=0) / np.sqrt(on_plane.sum())
    assert np.all(np.abs(mean - truth) < 4 * error), (mean, truth, error)
    assert np.all(error / truth < 0.01)


def test_the_eight_queries_replay_from_a_cuda_graph():
    """captured once warmed up, the calls allocate, copy and synchronise nothing: a graph replay gives the same outputs"""
    prepared = host.prepare(scenes.instanced_scene(grid=3, rings=8, segments=10))
    with PreparedScene(prepared) as scene:
        rays = scenes.random_rays(prepared.bounds, 4096, seed=9)
        hits, layers = scene.trace_hierarchy(rays)
        n = len(rays)
        rng = np.random.default_rng(1)
        contacts = scene.interact(rays, hits, layers)
        points = surfaces(contacts["position"], contacts["normal"])
        tokens, light_layers, _ = scene.pick(points, rng.random(n, np.float32))
        inputs = {"rays": up(rays, structs.RAY), "hits": up(hits, structs.HIT), "layers": up(layers, structs.TOKEN_HIERARCHY), "points": up(points, structs.SURFACE),
                  "tokens": up(tokens, np.uint32), "light_layers": up(light_layers, structs.TOKEN_HIERARCHY), "samples1": up(rng.random(n, np.float32), np.float32),
                  "samples2": up(rng.random((n, 2), np.float32), np.float32), "incident": up(unit_vectors(rng, n), np.float32)}
        outputs = {"contacts": empty(n, structs.CONTACT), "scatter": empty(n, structs.SCATTER), "evaluate": empty(n * 4, np.float32), "picked": empty(n, np.uint32),
                   "picked_layers": empty(n, structs.TOKEN_HIERARCHY), "pick_pmf": empty(n, np.float32), "mass": empty(n, np.float32),
                   "sample": empty(n, structs.LIGHT_SAMPLE), "pdf": empty(n, np.float32), "infinite": empty(n * 3, np.float32)}
        word = torch.full((1,), -1, dtype=torch.int64, device="cuda")
        a, o = {k: v.data_ptr() for k, v in inputs.items()}, {k: v.data_ptr() for k, v in outputs.items()}

        def calls(stream):
            s, w = stream.cuda_stream, word.data_ptr()
            scene.interact_device(a["rays"], a["hits"], a["layers"], n, o["contacts"], w, stream=s)
            scene.scatter_sample_device(a["rays"], a["hits"], a["layers"], a["samples2"], n, o["scatter"], w, stream=s)
            scene.scatter_evaluate_device(a["rays"], a["hits"], a["layers"], a["incident"], n, o["evaluate"], w, stream=s)
            scene.pick_device(a["points"], a["samples1"], n, o["picked"], o["picked_layers"], o["pick_pmf"], w, stream=s)
            scene.probability_mass_device(a["tokens"], a["light_layers"], a["points"], n, o["mass"], w, stream=s)
            scene.sample_device(a["tokens"], a["light_layers"], a["points"], a["samples2"], n, o["sample"], w, stream=s)
            scene.probability_density_device(a["tokens"], a["light_layers"], a["points"], a["incident"], n, o["pdf"], w, stream=s)
            scene.evaluate_infinite_device(a["incident"], n, True, o["infinite"], w, stream=s)

        stream = torch.cuda.Stream()
        with torch.cuda.stream(stream):
            calls(stream)
        stream.synchronize()
        first = {k: v.clone() for k, v in outputs.items()}
        assert int(word.item()) & CLEAR == CLEAR
        for v in outputs.values():
            v.zero_()

        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            calls(stream)
        graph.replay()
        torch.cuda.synchronize()
        for k in outputs:
            assert torch.equal(outputs[k], first[k]), k
        assert int(word.item()) & CLEAR == CLEAR
        assert same_bytes(down(outputs["contacts"], structs.CONTACT), contacts)
