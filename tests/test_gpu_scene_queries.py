"""The batched PreparedScene queries of include/echo_b200_query.h on the device: bit parity with the oracle's batch exports on
every parity fixture and two instanced scenes, agreement with what the renderer's path kernels compute, a direct-lighting
evaluator composed from the calls, every refusal, and multi-device scenes."""
import ctypes

import numpy as np
import pytest

from echorenderer_b200 import EchoNativeError, PreparedScene, _native, host, scenes, structs
from tests import oracle_lib
from tests.scene_query_oracle import OracleQueries, scene as query_oracle_scene, samples_with_edges, surfaces, unit_vectors
from tests.test_furnace import RHO, lit_plane, point_light_radiance, polygon_irradiance
from tests.test_gpu_render import sample_grid

pytestmark = pytest.mark.gpu

PARITY = ["cornell", "mixed_small", "lights_small", "terrain_small", "coated_small", "directional_small", "textured_small", "environment_small", "cubemap_small"]
INFINITE_TOKEN = int(structs.make_token(structs.TOKEN_TYPE_LIGHT, structs.LIGHT_TYPE_INFINITE << structs.LIGHT_INDEX_BITS))


def same_bits(a, b):
    """bit equality, except that a NaN equals any NaN: 0 / 0 is the x86 default NaN on the oracle's side and the canonical NaN on
    the device (LightTree.ProbabilityMass when both children's importance is 0; the renderer drops such a mass as not positive)"""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    if a.dtype.names:
        return all(same_bits(a[name], b[name]) for name in a.dtype.names)
    if a.dtype.kind == "f":
        nan = np.isnan(a)
        if not np.array_equal(nan, np.isnan(b)):
            return False
        a, b = np.where(nan, 0, a).astype(a.dtype), np.where(nan, 0, b).astype(b.dtype)
    return np.array_equal(a.view(np.uint8), b.view(np.uint8))


def prepared_scene(name, request):
    if name == "instanced":
        return host.prepare(scenes.instanced_scene(grid=3, rings=8, segments=10))
    if name == "many_packs":
        return host.prepare(scenes.many_packs_scene(pack_count=24, seed=5))
    return request.getfixturevalue(name)


def trace(scene, prepared, rays, ignore_layers=None):
    """(hits, instance layers or None): the hierarchy call on a scene with packs"""
    if prepared.packs is None:
        return scene.trace(rays), None
    return scene.trace_hierarchy(rays, ignore_layers)


def query_rays(prepared, oracle, seed):
    """camera rays of a 48 x 32 grid and random rays through the bounds, misses included"""
    params = structs.render_params(48, 32, 16, seed=seed)
    pixel_xy, sample_index = sample_grid(48, 32, 2)
    camera = oracle.spawn_rays(params, pixel_xy, sample_index)
    return np.concatenate([camera, scenes.random_rays(prepared.bounds, 3000, seed=seed)])


@pytest.mark.parametrize("fixture", PARITY + ["instanced", "many_packs"])
def test_every_query_is_bit_identical_to_the_oracle(fixture, request):
    prepared = prepared_scene(fixture, request)
    oracle = query_oracle_scene(prepared)
    expected = OracleQueries(oracle)
    rng = np.random.default_rng(17)

    with PreparedScene(prepared) as scene:
        rays = query_rays(prepared, oracle, seed=3)
        hits, layers = trace(scene, prepared, rays)
        hit = hits["token"] != structs.TOKEN_EMPTY
        assert hit.mean() > 0.2

        contacts = scene.interact(rays, hits, layers)
        assert same_bits(contacts, expected.interact(rays, hits, layers))
        assert np.all(contacts["material"][~hit] == structs.TOKEN_EMPTY) and np.all(contacts["lobes"][~hit] == 0)

        bounce = samples_with_edges(rng, (len(rays), 2))
        scattered = scene.scatter_sample(rays, hits, bounce, layers)
        assert same_bits(scattered, expected.scatter_sample(rays, hits, bounce, layers))
        assert (scattered["pdf"][hit] > 0).mean() > 0.1

        incident = scattered["incident"].copy()
        impossible = ~(scattered["pdf"] > 0)
        incident[impossible] = unit_vectors(rng, int(impossible.sum()))
        evaluated = scene.scatter_evaluate(rays, hits, incident, layers)
        assert same_bits(evaluated, expected.scatter_evaluate(rays, hits, incident, layers))

        # light queries from the contacts of the hits
        points = surfaces(contacts["position"][hit], contacts["normal"][hit])
        picks = samples_with_edges(rng, len(points))
        tokens, light_layers, pmf = scene.pick(points, picks)
        expected_tokens, expected_layers, expected_pmf = expected.pick(points, picks)
        assert same_bits(tokens, expected_tokens) and same_bits(light_layers, expected_layers) and same_bits(pmf, expected_pmf)

        radiant = samples_with_edges(rng, (len(points), 2))
        light_samples = scene.sample(tokens, points, radiant, light_layers)
        assert same_bits(light_samples, expected.sample(tokens, points, radiant, light_layers))

        # BSDF-sampled rays from the contacts: masses and densities of the emitters they reach, the infinite lights where they escape
        onward = hit & (scattered["pdf"] > 0)
        secondary = np.zeros(int(onward.sum()), dtype=structs.RAY)
        secondary["origin"], secondary["direction"] = contacts["position"][onward], scattered["incident"][onward]
        secondary["distance"], secondary["ignore"] = np.inf, hits["token"][onward]
        found, found_layers = trace(scene, prepared, secondary, None if layers is None else layers[onward])
        escaped = found["token"] == structs.TOKEN_EMPTY
        origins = surfaces(contacts["position"][onward], contacts["normal"][onward])
        light_tokens = np.where(escaped, np.uint32(INFINITE_TOKEN if len(prepared.description.infinite_lights) else structs.TOKEN_EMPTY), found["token"])
        mass = scene.probability_mass(light_tokens, origins, found_layers)
        assert same_bits(mass, expected.probability_mass(light_tokens, origins, found_layers))
        density = scene.probability_density(light_tokens, origins, secondary["direction"], found_layers)
        assert same_bits(density, expected.probability_density(light_tokens, origins, secondary["direction"], found_layers))

        directions = np.concatenate([rays["direction"][~hit], secondary["direction"][escaped]])
        for direct in (False, True):
            assert same_bits(scene.evaluate_infinite(directions, direct), expected.evaluate_infinite(directions, direct))


@pytest.mark.parametrize("fixture", ["mixed_small", "textured_small"])
def test_contacts_are_the_renderers(fixture, request):
    """The NormalDepthEvaluator reports the shading normal and the distance of the first hit whose BSDF is not purely specular: where
    that is the camera ray's own hit, interact's shadeNormal and the hit distance are what the path kernels computed, bit for bit."""
    prepared = request.getfixturevalue(fixture)
    oracle = query_oracle_scene(prepared)
    width, height = 64, 48
    params = structs.render_params(width, height, 16, extend=2, seed=21, evaluator=structs.EVALUATOR_NORMAL_DEPTH)
    pixel_xy, sample_index = sample_grid(width, height, 2)
    rays = oracle.spawn_rays(params, pixel_xy, sample_index)

    with PreparedScene(prepared) as scene:
        hits = scene.trace(rays)
        contacts = scene.interact(rays, hits)
        scattered = scene.scatter_sample(rays, hits, np.full((len(rays), 2), 0.5, np.float32))
        rendered = scene.evaluate_samples(params, pixel_xy, sample_index, channels=4)

    # a BSDF has one lobe or two non-specular ones, so the sampled lobe says whether all are specular
    diffuse = (hits["token"] != structs.TOKEN_EMPTY) & (contacts["lobes"] > 0) & (scattered["specular"] == 0)
    assert diffuse.mean() > 0.2
    assert same_bits(contacts["shadeNormal"][diffuse], rendered[diffuse, :3])
    assert same_bits(hits["distance"][diffuse], rendered[diffuse, 3])


def power_heuristic(a, b):
    return np.where(a * a + b * b > 0, a * a / np.maximum(a * a + b * b, 1e-38), 0.0)


def direct_lighting(scene, rays, rng, mis):
    """A custom evaluator written against the query interface: the first hit's emission-free direct light, one light sample
    (Pick + Sample + Occlude + BSDF.Evaluate) and, with `mis`, one BSDF sample (Scatter + Trace + Interact) weighted by the power
    heuristic against ProbabilityMass * ProbabilityDensity. Flat scenes. Returns (radiance[n, 3] float64, hit mask)."""
    n = len(rays)
    hits = scene.trace(rays)
    hit = hits["token"] != structs.TOKEN_EMPTY
    contacts = scene.interact(rays, hits)
    points = surfaces(contacts["position"], contacts["normal"])
    radiance = np.zeros((n, 3))
    normal = contacts["shadeNormal"].astype(np.float64)

    tokens, _, pmf = scene.pick(points[hit], rng.random(int(hit.sum()), dtype=np.float32))
    sampled = scene.sample(tokens, points[hit], rng.random((int(hit.sum()), 2), dtype=np.float32))
    keep = (pmf > 0) & (sampled["pdf"] > 0)
    light = np.flatnonzero(hit)[keep]
    shadow = np.zeros(len(light), dtype=structs.RAY)
    shadow["origin"], shadow["direction"] = contacts["position"][light], sampled["incident"][keep]
    shadow["distance"], shadow["ignore"] = sampled["travel"][keep], hits["token"][light]
    visible = scene.occlude(shadow) == 0
    f = scene.scatter_evaluate(rays[light], hits[light], sampled["incident"][keep])
    cosine = np.abs((sampled["incident"][keep] * normal[light]).sum(axis=1))
    pdf = pmf[keep].astype(np.float64) * sampled["pdf"][keep]
    weight = power_heuristic(pdf, f[:, 3].astype(np.float64)) if mis else 1.0
    value = sampled["radiance"][keep] * f[:, :3] * (cosine * weight * visible / pdf)[:, None]
    radiance[light] += value

    if mis:
        bounced = scene.scatter_sample(rays, hits, rng.random((n, 2), dtype=np.float32))
        onward = np.flatnonzero(hit & (bounced["pdf"] > 0))
        secondary = np.zeros(len(onward), dtype=structs.RAY)
        secondary["origin"], secondary["direction"] = contacts["position"][onward], bounced["incident"][onward]
        secondary["distance"], secondary["ignore"] = np.inf, hits["token"][onward]
        found = scene.trace(secondary)
        reached = found["token"] != structs.TOKEN_EMPTY
        emitted = scene.interact(secondary, found)["emission"].astype(np.float64)
        mass = scene.probability_mass(np.where(reached, found["token"], structs.TOKEN_EMPTY), points[onward])
        density = scene.probability_density(np.where(reached, found["token"], structs.TOKEN_EMPTY), points[onward], bounced["incident"][onward])
        scatter_pdf = bounced["pdf"][onward].astype(np.float64)
        weight = power_heuristic(scatter_pdf, mass.astype(np.float64) * density)
        cosine = np.abs((bounced["incident"][onward] * normal[onward]).sum(axis=1))
        radiance[onward] += emitted * bounced["value"][onward] * (cosine * weight / scatter_pdf)[:, None]

    return radiance, hit


def camera_rays(description, size, extend, seed):
    oracle = oracle_lib.OracleScene(host.prepare(description))
    params = structs.render_params(size, size, 8, extend=extend, seed=seed)
    pixel_xy, sample_index = sample_grid(size, size, extend)
    return oracle.spawn_rays(params, pixel_xy, sample_index)


def test_composed_evaluator_one_point_light_is_exact_per_sample():
    light = ((30.0, 20.0, 10.0), (1.0, 3.0, -0.5))
    description = lit_plane([light])
    rays = camera_rays(description, 16, 2, seed=8)
    with PreparedScene(host.prepare(description)) as scene:
        radiance, hit = direct_lighting(scene, rays, np.random.default_rng(3), mis=False)
        hits = scene.trace(rays)
    points = rays["origin"].astype(np.float64) + rays["direction"].astype(np.float64) * np.where(hit, hits["distance"], 0.0)[:, None]
    assert hit.mean() > 0.8 and np.all(radiance[~hit] == 0)
    assert np.allclose(radiance[hit], point_light_radiance(points[hit], *light), rtol=1e-5, atol=0)


def test_composed_evaluator_with_mis_converges_to_lamberts_formula():
    emission = np.array((10.0, 8.0, 6.0))
    corner, side = np.array((-1.0, 3.0, -1.0)), 2.0
    vertices = np.stack([corner, corner + (side, 0, 0), corner + (0, 0, side)])
    materials = np.concatenate([scenes.material(structs.MATERIAL_DIFFUSE, RHO), scenes.material(structs.MATERIAL_EMISSIVE, tuple(emission))])
    triangles = np.concatenate([scenes.plane(0, (20, 20)), scenes.make_triangles(vertices[0:1], vertices[1:2], vertices[2:3], 1)])
    description = lit_plane([])
    description.triangles, description.materials = triangles, materials
    rays = camera_rays(description, 12, 256, seed=10)

    with PreparedScene(host.prepare(description)) as scene:
        radiance, hit = direct_lighting(scene, rays, np.random.default_rng(4), mis=True)
        hits = scene.trace(rays)
    points = rays["origin"].astype(np.float64) + rays["direction"].astype(np.float64) * np.where(hit, hits["distance"], 0.0)[:, None]
    on_plane = hit & (points[:, 1] < 1e-3)
    assert on_plane.mean() > 0.7

    expected = np.array(RHO) / np.pi * emission * polygon_irradiance(points[on_plane], vertices)[:, None]
    mean, truth = radiance[on_plane].mean(axis=0), expected.mean(axis=0)
    error = radiance[on_plane].std(axis=0) / np.sqrt(on_plane.sum())
    assert np.all(np.abs(mean - truth) < 4 * error), (mean, truth, error)
    assert np.all(error / truth < 0.01)


def refused(call, message):
    with pytest.raises(EchoNativeError) as error:
        call()
    assert error.value.status == _native.ERR_INVALID, str(error.value)
    assert message in str(error.value), str(error.value)


def test_refusals(cornell):
    instanced = host.prepare(scenes.instanced_scene(grid=3, rings=8, segments=10))
    rays = scenes.random_rays(cornell.bounds, 8, seed=2)
    samples = np.full((8, 2), 0.5, np.float32)
    incident = np.tile(np.float32([0, 1, 0]), (8, 1))
    points = surfaces(np.zeros((8, 3), np.float32), incident)

    def light(kind, index):
        return structs.make_token(structs.TOKEN_TYPE_LIGHT, (kind << structs.LIGHT_INDEX_BITS) | index)

    with PreparedScene(cornell) as scene:
        hits = scene.trace(rays)
        hits[:3] = hits[0]  # keep the first rows plausible: query 3 is the one made bad below
        hits["token"][:3] = structs.make_token(structs.TOKEN_TYPE_TRIANGLE, 0)
        hits["uv"][:3] = (0.25, 0.25)
        hits["distance"][:3] = 1.0

        def bad_hit(token, uv=(0.25, 0.25)):
            h = hits.copy()
            h["token"][3], h["uv"][3], h["distance"][3] = token, uv, 1.0
            return h

        refused(lambda: scene.interact(rays, bad_hit(structs.make_token(structs.TOKEN_TYPE_TRIANGLE, len(cornell.triangles)))), "query 3: triangle index out of range")
        refused(lambda: scene.scatter_sample(rays, bad_hit(structs.make_token(structs.TOKEN_TYPE_SPHERE, len(cornell.spheres) + 2), (0.0, 0.0)), samples), "query 3: sphere index out of range")
        refused(lambda: scene.interact(rays, bad_hit(structs.make_token(structs.TOKEN_TYPE_TRIANGLE, 0), (0.5, 1.5))), "query 3: triangle hit uv outside [0, 1]")
        refused(lambda: scene.interact(rays, bad_hit(structs.make_token(structs.TOKEN_TYPE_INSTANCE, 0))), "query 3: hit token is neither")
        nan_rays = rays.copy()
        nan_rays["origin"][5, 1] = np.nan
        refused(lambda: scene.interact(nan_rays, bad_hit(structs.TOKEN_EMPTY)), "query 5: the ray needs a finite origin")
        inf_samples = samples.copy()
        inf_samples[6, 0] = np.inf
        refused(lambda: scene.scatter_sample(rays, bad_hit(structs.TOKEN_EMPTY), inf_samples), "query 6: samples are not finite")
        nan_incident = incident.copy()
        nan_incident[2, 2] = np.nan
        refused(lambda: scene.scatter_evaluate(rays, bad_hit(structs.TOKEN_EMPTY), nan_incident), "query 2: the incident direction")

        layers = np.zeros(8, structs.TOKEN_HIERARCHY)
        layers["instanceCount"][4], layers["instances"][4, 0] = 1, structs.make_token(structs.TOKEN_TYPE_INSTANCE, 0)
        refused(lambda: scene.interact(rays, bad_hit(structs.TOKEN_EMPTY), layers), "query 4: instance layers on a scene without packs")
        refused(lambda: scene.probability_mass(np.full(8, structs.TOKEN_EMPTY, np.uint32), points, layers), "query 4: instance layers on a scene without packs")

        tokens = np.full(8, structs.TOKEN_EMPTY, np.uint32)

        def bad_light(token):
            t = tokens.copy()
            t[1] = token
            return t

        refused(lambda: scene.sample(bad_light(light(structs.LIGHT_TYPE_POINT, len(cornell.point_lights))), points, samples), "query 1: point light index out of range")
        refused(lambda: scene.probability_density(bad_light(light(structs.LIGHT_TYPE_INFINITE, len(cornell.description.infinite_lights))), points, incident),
                "query 1: infinite light index out of range")
        refused(lambda: scene.probability_mass(bad_light(structs.make_token(structs.TOKEN_TYPE_TRIANGLE, len(cornell.triangles))), points), "query 1: triangle emitter index out of range")
        refused(lambda: scene.sample(bad_light(structs.make_token(structs.TOKEN_TYPE_SPHERE, len(cornell.spheres))), points, samples), "query 1: sphere emitter index out of range")
        refused(lambda: scene.probability_mass(bad_light(structs.make_token(structs.TOKEN_TYPE_NODE, 0)), points), "query 1: light token is neither")
        nan_points = points.copy()
        nan_points["normal"][7, 0] = np.inf
        refused(lambda: scene.pick(nan_points, np.full(8, 0.5, np.float32)), "query 7: the surface is not finite")
        refused(lambda: scene.pick(points, np.array([0.5] * 7 + [np.nan], np.float32)), "query 7: the sample is not finite")
        refused(lambda: scene.evaluate_infinite(np.tile(np.float32([0, 2, 0]), (8, 1))), "query 0: the direction is not a finite unit vector")

        lib, handle, p = _native.library(), scene.handle, _native.pointer
        assert lib.echo_b200_interact_batch(handle, p(rays), p(hits), None, 8, None) == _native.ERR_INVALID and b"null buffer" in lib.echo_b200_last_error()
        assert lib.echo_b200_light_pick_batch(handle, None, p(samples), 8, p(tokens), None, p(samples)) == _native.ERR_INVALID
        assert lib.echo_b200_evaluate_infinite_batch(handle, None, 8, 0, p(samples)) == _native.ERR_INVALID
        assert lib.echo_b200_interact_batch(handle, None, None, None, 0, None) == _native.OK  # n == 0 needs no buffers

        # nothing refused reached the device: the scene still answers, and a bounds-check build found no bad index
        contacts = scene.interact(rays, scene.trace(rays))
        assert len(contacts) == 8 and not scene.bounds_violations()

    with PreparedScene(instanced) as scene:
        rays = scenes.random_rays(instanced.bounds, 8, seed=4)
        hits, layers = scene.trace_hierarchy(rays)
        layers[3]["instanceCount"], layers[3]["instances"][0] = 1, structs.make_token(structs.TOKEN_TYPE_TRIANGLE, 0)
        refused(lambda: scene.interact(rays, hits, layers), "query 3: layer 0 is not an instance of its parent pack")
        layers[3]["instanceCount"] = structs.MAX_INSTANCE_LAYERS + 1
        refused(lambda: scene.interact(rays, hits, layers), "query 3: more than ECHO_MAX_INSTANCE_LAYERS")

    lib = _native.library()
    handle = ctypes.c_void_p()
    _native.check(lib.echo_b200_scene_create(ctypes.byref(handle), 0))
    try:
        assert lib.echo_b200_light_mass_batch(handle, _native.pointer(tokens), None, _native.pointer(points), 8, _native.pointer(samples)) == _native.ERR_INVALID
        assert b"not committed" in lib.echo_b200_last_error()
    finally:
        lib.echo_b200_scene_destroy(handle)


def gpu_count():
    try:
        return _native.device_count()
    except _native.EchoNativeError:
        return 0


@pytest.mark.skipif(gpu_count() < 2, reason="needs two GPUs")
def test_multi_device_scene_gives_the_same_bits():
    prepared = host.prepare(scenes.instanced_scene(grid=3, rings=8, segments=10))
    oracle = query_oracle_scene(prepared)
    rays = query_rays(prepared, oracle, seed=6)
    rng = np.random.default_rng(2)
    bounce, picks, radiant = rng.random((len(rays), 2), np.float32), rng.random(len(rays), np.float32), rng.random((len(rays), 2), np.float32)

    def run(scene):
        hits, layers = scene.trace_hierarchy(rays)
        contacts = scene.interact(rays, hits, layers)
        scattered = scene.scatter_sample(rays, hits, bounce, layers)
        points = surfaces(contacts["position"], contacts["normal"])
        tokens, light_layers, pmf = scene.pick(points, picks)
        return [hits, layers, contacts, scattered, tokens, light_layers, pmf, scene.sample(tokens, points, radiant, light_layers),
                scene.probability_mass(tokens, points, light_layers), scene.evaluate_infinite(rays["direction"], True)]

    with PreparedScene(prepared) as single:
        expected = run(single)
    with PreparedScene(prepared, devices=[0, 1]) as multi:
        assert multi.gpu_count == 2
        actual = run(multi)
    for a, b in zip(actual, expected):
        assert same_bits(a, b)
