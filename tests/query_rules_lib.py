"""The validation rules of the batched PreparedScene queries (echorenderer_b200/csrc/echo_query_rules.h) on their own, and a table of
edge inputs for them: tests/c_client/query_rules.cpp is built once per process into a temporary directory with the host library's
floating-point flags. The CPU suite runs the table through the host build of the rules; the GPU suite runs it through the host-buffer
and device-buffer calls. TEST INFRASTRUCTURE ONLY."""
import atexit
import ctypes
import math
import os
import shutil
import subprocess
import tempfile

import numpy as np

from echorenderer_b200 import structs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCE = os.path.join(ROOT, "tests", "c_client", "query_rules.cpp")
FLAGS = ["-std=c++17", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-Wextra", "-shared"]
_lib = None


def library():
    global _lib
    if _lib is not None:
        return _lib
    directory = tempfile.mkdtemp(prefix="query_rules_")
    atexit.register(shutil.rmtree, directory, True)
    path = os.path.join(directory, "libquery_rules.so")
    subprocess.run(["g++"] + FLAGS + ["-o", path, SOURCE], check=True)
    lib = ctypes.CDLL(path)
    p, u32, u64, i32 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int32
    scene = [p, u32, p, p, u32, p, u32, u32, u32, u32]
    lib.rules_contact.argtypes = scene + [p, p, p, p, i32, u64, p]
    lib.rules_light.argtypes = scene + [p, p, p, p, i32, u64, p]
    lib.rules_contact.restype = lib.rules_light.restype = None
    lib.rules_reason.argtypes, lib.rules_reason.restype = [u32], ctypes.c_char_p
    _lib = lib
    return lib


def _pointer(array):
    return None if array is None or len(array) == 0 else ctypes.c_void_p(array.ctypes.data)


def _scene_arguments(prepared):
    packs = None if prepared.packs is None else np.ascontiguousarray(prepared.packs)
    instances = None if prepared.instances is None else np.ascontiguousarray(prepared.instances)
    triangles, spheres = np.ascontiguousarray(prepared.triangles), np.ascontiguousarray(prepared.spheres)
    keep = (packs, instances, triangles, spheres)
    return keep, [_pointer(packs), 0 if packs is None else len(packs), _pointer(instances), _pointer(triangles), len(triangles), _pointer(spheres), len(spheres),
                  len(prepared.point_lights), len(prepared.description.infinite_lights), len(prepared.materials)]


def reason_text(code):
    text = library().rules_reason(code)
    return None if text is None else text.decode()


def run_contact(prepared, table):
    """the reason text each contact row of `table` is refused for by the host build of the rules (None: accepted)"""
    keep, scene = _scene_arguments(prepared)
    codes = np.zeros(len(table["rays"]), np.uint32)
    library().rules_contact(*scene, _pointer(table["rays"]), _pointer(table["hits"]), _pointer(table["layers"]), _pointer(table["values"]), 3, len(codes), _pointer(codes))
    return [reason_text(int(c)) for c in codes]


def run_light(prepared, table):
    keep, scene = _scene_arguments(prepared)
    codes = np.zeros(len(table["tokens"]), np.uint32)
    library().rules_light(*scene, _pointer(table["tokens"]), _pointer(table["layers"]), _pointer(table["points"]), _pointer(table["values"]), 3, len(codes), _pointer(codes))
    return [reason_text(int(c)) for c in codes]


def _unit_length_ok(v):
    """the rule in double precision, in the rules' order: |sqrt(x*x + y*y + z*z) - 1| <= 1e-3"""
    x, y, z = (float(np.float32(c)) for c in v)
    return abs(math.sqrt(x * x + y * y + z * z) - 1.0) <= 1e-3


def _lengths():
    """directions whose length is 1 +- 1e-3 as float32 and the next float on either side, along an axis and along a diagonal"""
    out = []
    for target in (1.0 + 1e-3, 1.0 - 1e-3):
        x = np.float32(target)
        out += [(v, 0.0, 0.0) for v in (np.nextafter(x, np.float32(0)), x, np.nextafter(x, np.float32(2)))]
        a = np.float32(target / math.sqrt(3.0))
        out += [(v, v, v) for v in (np.nextafter(a, np.float32(0)), a, np.nextafter(a, np.float32(2)))]
    return [np.float32(v) for v in out]


def pack_paths(prepared):
    """{pack: instance-layer tokens from the root that reach it} for every pack a hierarchy of at most MAX_INSTANCE_LAYERS reaches"""
    if prepared.packs is None:
        return {0: []}
    paths, frontier = {0: []}, [0]
    while frontier:
        pack = frontier.pop(0)
        if len(paths[pack]) == structs.MAX_INSTANCE_LAYERS:
            continue
        record = prepared.packs[pack]
        for k in range(int(record["instanceCount"])):
            child = int(prepared.instances[int(record["instanceOffset"]) + k]["pack"])
            if child not in paths:
                paths[child] = paths[pack] + [structs.make_token(structs.TOKEN_TYPE_INSTANCE, k)]
                frontier.append(child)
    return paths


def _pack_counts(prepared, pack):
    if prepared.packs is None:
        return len(prepared.triangles), len(prepared.spheres), 0, len(prepared.point_lights)
    record = prepared.packs[pack]
    return int(record["triangleCount"]), int(record["sphereCount"]), int(record["instanceCount"]), int(record["pointLightCount"])


def _hierarchy(tokens, count=None):
    h = np.zeros(1, structs.TOKEN_HIERARCHY)
    h["instanceCount"] = len(tokens) if count is None else count
    h["instances"][0, :len(tokens)] = tokens
    return h[0]


def edge_table(prepared):
    """(contact rows, light rows, expected reason texts of each). Contact rows are scatter_evaluate queries (ray, hit, hit layers,
    incident direction), light rows light_pdf queries (token, layers, surface, incident direction); None is accepted."""
    up = np.float32([0, 1, 0])
    contact, light = [], []  # (ray, hit, layers, incident, expected) / (token, layers, point, incident, expected)

    def ray(direction=up):
        r = np.zeros(1, structs.RAY)[0]
        r["direction"], r["distance"], r["ignore"] = direction, np.inf, structs.TOKEN_EMPTY
        return r

    def hit(token=structs.TOKEN_EMPTY, uv=(0.25, 0.25)):
        h = np.zeros(1, structs.HIT)[0]
        h["token"], h["uv"], h["distance"] = token, uv, 1.0
        return h

    point = np.zeros(1, structs.SURFACE)[0]
    point["normal"] = up
    none = _hierarchy([])

    for v in _lengths():
        ok = _unit_length_ok(v)
        contact.append((ray(v), hit(), none, up, None if ok else "the ray needs a finite origin and a unit direction"))
        contact.append((ray(), hit(), none, v, None if ok else "the incident direction is not a finite unit vector"))
        light.append((structs.TOKEN_EMPTY, none, point, v, None if ok else "the incident direction is not a finite unit vector"))

    below, above = np.nextafter(np.float32(0), np.float32(-1)), np.nextafter(np.float32(1), np.float32(2))
    paths = pack_paths(prepared)
    for pack, path in sorted(paths.items()):
        layers = _hierarchy(path)
        triangles, spheres, instances, point_lights = _pack_counts(prepared, pack)
        triangle, sphere = (lambda i: structs.make_token(structs.TOKEN_TYPE_TRIANGLE, i)), (lambda i: structs.make_token(structs.TOKEN_TYPE_SPHERE, i))
        if triangles:
            for uv in ((0.0, 0.0), (1.0, 1.0), (0.0, 1.0), (-0.0, 0.5)):
                contact.append((ray(), hit(triangle(triangles - 1), uv), layers, up, None))
            for uv in ((above, 0.5), (0.5, below)):
                contact.append((ray(), hit(triangle(0), uv), layers, up, "triangle hit uv outside [0, 1]"))
            light.append((triangle(triangles - 1), layers, point, up, None))
        contact.append((ray(), hit(triangle(triangles)), layers, up, "triangle index out of range for its pack"))
        light.append((triangle(triangles), layers, point, up, "triangle emitter index out of range for its pack"))
        if spheres:
            for uv in ((-1.5, 0.0), (4.5, 0.0), (0.0, -1.0), (0.0, 1.0)):
                contact.append((ray(), hit(sphere(spheres - 1), uv), layers, up, None))
            for uv in ((np.nextafter(np.float32(-1.5), np.float32(-2)), 0.0), (np.nextafter(np.float32(4.5), np.float32(5)), 0.0), (0.0, above)):
                contact.append((ray(), hit(sphere(0), uv), layers, up, "sphere hit uv outside the encoding of SphereEntity"))
            light.append((sphere(spheres - 1), layers, point, up, None))
        contact.append((ray(), hit(sphere(spheres), (0.0, 0.0)), layers, up, "sphere index out of range for its pack"))
        light.append((sphere(spheres), layers, point, up, "sphere emitter index out of range for its pack"))
        if len(path) < structs.MAX_INSTANCE_LAYERS and prepared.packs is not None:
            instance = lambda i: structs.make_token(structs.TOKEN_TYPE_INSTANCE, i)  # noqa: E731
            if instances:
                contact.append((ray(), hit(), _hierarchy(path + [instance(instances - 1)]), up, None))
            contact.append((ray(), hit(), _hierarchy(path + [instance(instances)]), up, "layer is not an instance of its parent pack"))
        point_light = lambda i: structs.make_token(structs.TOKEN_TYPE_LIGHT, (structs.LIGHT_TYPE_POINT << structs.LIGHT_INDEX_BITS) | i)  # noqa: E731
        if point_lights:
            light.append((point_light(point_lights - 1), layers, point, up, None))
        light.append((point_light(point_lights), layers, point, up, "point light index out of range for its pack"))

    infinite = lambda i: structs.make_token(structs.TOKEN_TYPE_LIGHT, (structs.LIGHT_TYPE_INFINITE << structs.LIGHT_INDEX_BITS) | i)  # noqa: E731
    count = len(prepared.description.infinite_lights)
    if count:
        light.append((infinite(count - 1), none, point, up, None))
    light.append((infinite(count), none, point, up, "infinite light index out of range"))

    if prepared.packs is not None:  # layer counts: five pass the count test (the first token then fails), six do not
        bad = [structs.make_token(structs.TOKEN_TYPE_TRIANGLE, 0)] * structs.MAX_INSTANCE_LAYERS
        contact.append((ray(), hit(), _hierarchy(bad, structs.MAX_INSTANCE_LAYERS), up, "layer is not an instance of its parent pack"))
        contact.append((ray(), hit(), _hierarchy(bad, structs.MAX_INSTANCE_LAYERS + 1), up, "more than ECHO_MAX_INSTANCE_LAYERS instance layers"))
        light.append((structs.TOKEN_EMPTY, _hierarchy(bad, structs.MAX_INSTANCE_LAYERS + 1), point, up, "more than ECHO_MAX_INSTANCE_LAYERS instance layers"))

    contact_rows = {"rays": np.array([r[0] for r in contact], structs.RAY), "hits": np.array([r[1] for r in contact], structs.HIT),
                    "layers": np.array([r[2] for r in contact], structs.TOKEN_HIERARCHY), "values": np.array([r[3] for r in contact], np.float32).reshape(-1, 3)}
    light_rows = {"tokens": np.array([r[0] for r in light], np.uint32), "layers": np.array([r[1] for r in light], structs.TOKEN_HIERARCHY),
                  "points": np.array([r[2] for r in light], structs.SURFACE), "values": np.array([r[3] for r in light], np.float32).reshape(-1, 3)}
    return contact_rows, light_rows, [r[4] for r in contact], [r[4] for r in light]


def normalise(message):
    """a host-buffer message without the layer it names, so that it compares with the reason text of its code"""
    import re
    return re.sub(r"layer \d+ is", "layer is", message)
