"""The batched PreparedScene queries of include/echo_b200_query.h without a GPU: the header's PODs against their numpy mirrors,
the exported symbols, the C# block of INTEGRATION.md, clean failure without a device, and the oracle's batch exports against the
single-query exports that already existed."""
import ctypes
import importlib.util
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from echorenderer_b200 import _native, structs
from tests import oracle_lib
from tests.scene_query_oracle import OracleQueries, scene as query_oracle_scene, samples_with_edges, surfaces, unit_vectors
from tests.test_abi import declared_functions, have_gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

QUERY_MIRRORS = {"EchoSurface": "SURFACE", "EchoContact": "CONTACT", "EchoScatter": "SCATTER", "EchoLightSample": "LIGHT_SAMPLE"}


def generator():
    spec = importlib.util.spec_from_file_location("gen_csharp_structs", os.path.join(ROOT, "tools", "gen_csharp_structs.py"))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    return module


def test_query_pod_layouts_match_the_header():
    """sizeof and offsetof of every member of the four query structs, compiled with gcc, equal the numpy mirrors; each struct
    carries its size assertion, and the header declares no other struct."""
    header = open(os.path.join(ROOT, "include", "echo_b200_query.h")).read()
    assert set(re.findall(r"typedef struct (\w+)\s*\{", re.sub(r"/\*.*?\*/", "", header, flags=re.S))) == set(QUERY_MIRRORS)

    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "echo_b200_query.h"', "int main(void) {"]
    for c_name, mirror in QUERY_MIRRORS.items():
        dtype = getattr(structs, mirror)
        assert f"ECHO_B200_ASSERT_SIZE({c_name}, {dtype.itemsize});" in header, c_name
        assert sum(dtype.fields[name][0].itemsize for name in dtype.names) == dtype.itemsize, mirror  # sequential, no padding
        lines.append(f'printf("{c_name} %zu\\n", sizeof({c_name}));')
        for name in dtype.names:
            lines.append(f'printf("{c_name}.{name} %zu %zu\\n", offsetof({c_name}, {name}), sizeof((({c_name}*)0)->{name}));')
    lines.append("return 0; }")

    with tempfile.TemporaryDirectory() as directory:
        source, binary = os.path.join(directory, "layout.c"), os.path.join(directory, "layout")
        open(source, "w").write("\n".join(lines))
        subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), source, "-o", binary], check=True)
        output = subprocess.run([binary], check=True, capture_output=True, text=True).stdout

    checked = 0
    for line in output.splitlines():
        key, *values = line.split()
        c_name, _, member = key.partition(".")
        dtype = getattr(structs, QUERY_MIRRORS[c_name])
        if member:
            assert int(values[0]) == dtype.fields[member][1] and int(values[1]) == dtype.fields[member][0].itemsize, line
        else:
            assert int(values[0]) == dtype.itemsize, line
        checked += 1
    assert checked == len(QUERY_MIRRORS) + sum(len(getattr(structs, m).names) for m in QUERY_MIRRORS.values())
    assert (structs.SURFACE.itemsize, structs.CONTACT.itemsize, structs.SCATTER.itemsize, structs.LIGHT_SAMPLE.itemsize) == (24, 64, 32, 32)


def test_query_symbols_are_declared_bound_and_exported():
    declared = declared_functions("echo_b200_query.h")
    assert declared == set(_native.QUERY_EXPORTS) and len(declared) == 8
    assert not declared & set(_native.EXPORTS)
    lib = _native.library()
    for name in declared:
        assert hasattr(lib, name), name
        assert getattr(lib, name).argtypes is not None, f"{name} has no ctypes signature"


def test_integration_document_holds_the_generated_query_block_and_every_call():
    module = generator()
    assert [pod[0] for pod in module.QUERY_PODS] == list(QUERY_MIRRORS)
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert module.QUERY_BEGIN + "\n" + module.query_block() + "\n" + module.QUERY_END in text
    for name in _native.QUERY_EXPORTS:
        assert re.search(rf"\[DllImport\(Library\)\] public static extern int {name}\(", text), name


@pytest.mark.skipif(have_gpu(), reason="checks the no-device behaviour")
def test_every_query_fails_cleanly_without_a_device():
    """Without a device a host can only hold a NULL scene (echo_b200_scene_create fails): every call refuses it, n = 0 too."""
    lib = _native.library()
    handle = ctypes.c_void_p()
    assert lib.echo_b200_scene_create(ctypes.byref(handle), 0) == _native.ERR_NO_DEVICE and not handle.value

    n = 4
    rays, hits = np.zeros(n, structs.RAY), np.zeros(n, structs.HIT)
    points, tokens, floats = np.zeros(n, structs.SURFACE), np.zeros(n, np.uint32), np.zeros(n * 4, np.float32)
    contacts, scatters, samples = np.zeros(n, structs.CONTACT), np.zeros(n, structs.SCATTER), np.zeros(n, structs.LIGHT_SAMPLE)
    layers = np.zeros(n, structs.TOKEN_HIERARCHY)
    p = _native.pointer
    for count in (n, 0):
        calls = [
            lambda: lib.echo_b200_interact_batch(None, p(rays), p(hits), None, count, p(contacts)),
            lambda: lib.echo_b200_scatter_sample_batch(None, p(rays), p(hits), None, p(floats), count, p(scatters)),
            lambda: lib.echo_b200_scatter_evaluate_batch(None, p(rays), p(hits), None, p(floats), count, p(floats)),
            lambda: lib.echo_b200_light_pick_batch(None, p(points), p(floats), count, p(tokens), p(layers), p(floats)),
            lambda: lib.echo_b200_light_mass_batch(None, p(tokens), None, p(points), count, p(floats)),
            lambda: lib.echo_b200_light_sample_batch(None, p(tokens), None, p(points), p(floats), count, p(samples)),
            lambda: lib.echo_b200_light_pdf_batch(None, p(tokens), None, p(points), p(floats), count, p(floats)),
            lambda: lib.echo_b200_evaluate_infinite_batch(None, p(floats), count, 1, p(floats)),
        ]
        for call in calls:
            assert call() == _native.ERR_INVALID
            assert b"scene is null" in lib.echo_b200_last_error()


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


def light_origins(prepared, count, seed):
    """surfaces spread over the scene's bounds with random unit normals"""
    rng = np.random.default_rng(seed)
    low, high = np.asarray(prepared.bounds[0], np.float64), np.asarray(prepared.bounds[1], np.float64)
    positions = (low + (high - low) * rng.random((count, 3))).astype(np.float32)
    return surfaces(positions, unit_vectors(rng, count)), rng


@pytest.mark.parametrize("fixture", ["cornell", "lights_small"])
def test_oracle_pick_mass_and_geometry_batches_equal_the_single_exports(fixture, request):
    prepared = request.getfixturevalue(fixture)
    queries = OracleQueries(query_oracle_scene(prepared))
    oracle = oracle_lib.OracleScene(prepared)  # liboracle.so's own single-query exports
    points, rng = light_origins(prepared, 600, seed=5)
    picks = samples_with_edges(rng, len(points))

    tokens, layers, pmf = queries.pick(points, picks)
    assert (tokens != structs.TOKEN_EMPTY).mean() > 0.5 and np.all(layers["instanceCount"] == 0)
    for i in range(len(points)):
        token, pdf = oracle.light_pick(points["position"][i], points["normal"][i], picks[i])
        assert token == tokens[i] and bits(pdf) == bits(pmf[i]), i

    mass = queries.probability_mass(tokens, points)
    for i in range(len(points)):
        expected = 0.0 if tokens[i] == structs.TOKEN_EMPTY else oracle.light_mass(tokens[i], points["position"][i], points["normal"][i])
        assert bits(expected) == bits(mass[i]), i

    # emissive geometry: PreparedScene.Sample's pdf is PreparedTriangle / PreparedSphere.Sample's wherever the light sample is possible
    geometry = np.isin(structs.token_type(tokens), [structs.TOKEN_TYPE_TRIANGLE, structs.TOKEN_TYPE_SPHERE])
    assert geometry.sum() > 50
    sample2 = samples_with_edges(rng, (len(points), 2))
    sampled = queries.sample(tokens, points, sample2)
    possible = geometry & (sampled["pdf"] > 0)
    assert possible.sum() > 50
    for i in np.flatnonzero(possible):
        ok, _, _, pdf = oracle.geometry_sample(tokens[i], points["position"][i], sample2[i])
        assert ok and bits(pdf) == bits(sampled["pdf"][i]), i

    # ProbabilityDensity = PreparedTriangle / PreparedSphere.ProbabilityDensity towards directions the normalisation leaves as they are
    incident = sampled["incident"].copy()
    incident[~possible] = unit_vectors(rng, int((~possible).sum()))
    squared = (incident.astype(np.float64) ** 2).sum(axis=1)
    scale = np.float32(1.0) / np.sqrt(squared).astype(np.float32)
    fixed = np.all(incident * scale[:, None] == incident, axis=1)  # oracle/math.hpp normalized(): (1 / (float)sqrt(double)) * v
    pdf = queries.probability_density(tokens, points, incident)
    checked = 0
    for i in np.flatnonzero(geometry & fixed):
        assert bits(oracle.geometry_pdf(tokens[i], points["position"][i], incident[i])) == bits(pdf[i]), i
        checked += 1
    assert checked > 50 and np.count_nonzero(pdf[geometry & fixed]) > 20


@pytest.mark.parametrize("fixture", ["directional_small", "environment_small"])
def test_oracle_infinite_batches_equal_the_single_export(fixture, request):
    prepared = request.getfixturevalue(fixture)
    queries = OracleQueries(query_oracle_scene(prepared))
    oracle = oracle_lib.OracleScene(prepared)  # liboracle.so's own single-query exports
    lights = prepared.description.infinite_lights
    count = 200
    points, rng = light_origins(prepared, count, seed=8)
    directions = unit_vectors(rng, count)
    sample2 = samples_with_edges(rng, (count, 2))

    per_light = []
    for index in range(len(lights)):
        token = structs.make_token(structs.TOKEN_TYPE_LIGHT, (structs.LIGHT_TYPE_INFINITE << structs.LIGHT_INDEX_BITS) | index)
        tokens = np.full(count, token, dtype=np.uint32)
        sampled = queries.sample(tokens, points, sample2)
        pdf = queries.probability_density(tokens, points, directions)
        mass = queries.probability_mass(tokens, points)
        out = np.zeros((count, 11), dtype=np.float32)
        for i in range(count):
            oracle.lib.oracle_infinite_light(oracle.handle, index, oracle_lib.ptr(sample2[i]), oracle_lib.ptr(directions[i]), oracle_lib.ptr(out[i]))
        assert np.array_equal(bits(sampled["radiance"]), bits(out[:, 0:3])) and np.array_equal(bits(sampled["pdf"]), bits(out[:, 3]))
        assert np.array_equal(bits(sampled["incident"]), bits(out[:, 4:7])) and np.all(np.isinf(sampled["travel"]))
        assert np.array_equal(bits(pdf), bits(out[:, 10]))
        assert np.all(bits(mass) == bits(np.float32(prepared.infinite_pdf)))
        per_light.append(out[:, 7:10])

    for direct in (False, True):
        total = np.zeros((count, 3), dtype=np.float32)  # PreparedScene.EvaluateInfinite: the lights summed in order
        for index, value in enumerate(per_light):
            if not direct or lights["directlyVisible"][index]:
                total = total + value
        assert np.array_equal(bits(queries.evaluate_infinite(directions, direct)), bits(total))
    assert np.abs(total).max() > 0
