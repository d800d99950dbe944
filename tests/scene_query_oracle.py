"""The oracle's batch forms of the scene queries of include/echo_b200_query.h (tests/c_client/scene_query_oracle.cpp: oracle/api.cpp
compiled unchanged plus one export per device call, same arguments): built once per process into a temporary directory, with
liboracle.so's compiler flags, and loaded beside it. TEST INFRASTRUCTURE ONLY."""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile
from unittest import mock

import numpy as np

from echorenderer_b200 import structs
from tests import oracle_lib
from tests.oracle_lib import ptr

SOURCE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c_client", "scene_query_oracle.cpp")
FLAGS = ["-std=c++17", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-Wextra", "-pthread", "-shared"]
_lib = None
_oracle_library = oracle_lib.library  # liboracle.so's loader, also while scene() stands this module's in for it


def library():
    global _lib
    if _lib is not None:
        return _lib
    directory = tempfile.mkdtemp(prefix="scene_query_oracle_")
    atexit.register(shutil.rmtree, directory, True)
    path = os.path.join(directory, "libscene_query_oracle.so")
    subprocess.run(["g++"] + FLAGS + ["-o", path, SOURCE], check=True)
    lib = ctypes.CDLL(path)
    # the same prototypes as liboracle.so's (oracle_lib.library() declares them as it loads it)
    for name, function in vars(_oracle_library()).items():
        if isinstance(function, ctypes._CFuncPtr):
            mine = getattr(lib, name)
            mine.argtypes, mine.restype = function.argtypes, function.restype
    p, u64, i32 = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int32
    lib.oracle_interact_batch.argtypes = [p, p, p, p, u64, p]
    lib.oracle_scatter_sample_batch.argtypes = [p, p, p, p, p, u64, p]
    lib.oracle_scatter_evaluate_batch.argtypes = [p, p, p, p, p, u64, p]
    lib.oracle_light_pick_batch.argtypes = [p, p, p, u64, p, p, p]
    lib.oracle_light_mass_batch.argtypes = [p, p, p, p, u64, p]
    lib.oracle_light_sample_batch.argtypes = [p, p, p, p, p, u64, p]
    lib.oracle_light_pdf_batch.argtypes = [p, p, p, p, p, u64, p]
    lib.oracle_evaluate_infinite_batch.argtypes = [p, p, u64, i32, p]
    for name in ("interact", "scatter_sample", "scatter_evaluate", "light_pick", "light_mass", "light_sample", "light_pdf", "evaluate_infinite"):
        getattr(lib, f"oracle_{name}_batch").restype = None
    _lib = lib
    return lib


def scene(prepared):
    """an oracle_lib.OracleScene on this library (its single-query methods work on it as on liboracle.so)"""
    with mock.patch.object(oracle_lib, "library", library):
        return oracle_lib.OracleScene(prepared)


def _layers(layers):
    return None if layers is None else np.ascontiguousarray(layers, dtype=structs.TOKEN_HIERARCHY)


class OracleQueries:
    """The methods of PreparedScene's query interface (echorenderer_b200/scene.py), computed by the oracle on a scene() of this
    module's library."""

    def __init__(self, oracle_scene):
        assert oracle_scene.lib is library(), "the scene must live in the library that has the batch exports"
        self.scene = oracle_scene
        self.lib = oracle_scene.lib

    def interact(self, rays, hits, layers=None):
        out = np.zeros(len(rays), dtype=structs.CONTACT)
        self.lib.oracle_interact_batch(self.scene.handle, ptr(rays), ptr(hits), ptr(_layers(layers)), len(rays), ptr(out))
        return out

    def scatter_sample(self, rays, hits, samples, layers=None):
        samples = np.ascontiguousarray(samples, dtype=np.float32)
        out = np.zeros(len(rays), dtype=structs.SCATTER)
        self.lib.oracle_scatter_sample_batch(self.scene.handle, ptr(rays), ptr(hits), ptr(_layers(layers)), ptr(samples), len(rays), ptr(out))
        return out

    def scatter_evaluate(self, rays, hits, incident, layers=None):
        incident = np.ascontiguousarray(incident, dtype=np.float32)
        out = np.zeros((len(rays), 4), dtype=np.float32)
        self.lib.oracle_scatter_evaluate_batch(self.scene.handle, ptr(rays), ptr(hits), ptr(_layers(layers)), ptr(incident), len(rays), ptr(out))
        return out

    def pick(self, points, samples):
        points, samples = np.ascontiguousarray(points, dtype=structs.SURFACE), np.ascontiguousarray(samples, dtype=np.float32)
        tokens = np.zeros(len(points), dtype=np.uint32)
        layers = np.zeros(len(points), dtype=structs.TOKEN_HIERARCHY)
        pmf = np.zeros(len(points), dtype=np.float32)
        self.lib.oracle_light_pick_batch(self.scene.handle, ptr(points), ptr(samples), len(points), ptr(tokens), ptr(layers), ptr(pmf))
        return tokens, layers, pmf

    def probability_mass(self, tokens, points, layers=None):
        tokens, points = np.ascontiguousarray(tokens, dtype=np.uint32), np.ascontiguousarray(points, dtype=structs.SURFACE)
        out = np.zeros(len(tokens), dtype=np.float32)
        self.lib.oracle_light_mass_batch(self.scene.handle, ptr(tokens), ptr(_layers(layers)), ptr(points), len(tokens), ptr(out))
        return out

    def sample(self, tokens, points, samples, layers=None):
        tokens, points = np.ascontiguousarray(tokens, dtype=np.uint32), np.ascontiguousarray(points, dtype=structs.SURFACE)
        samples = np.ascontiguousarray(samples, dtype=np.float32)
        out = np.zeros(len(tokens), dtype=structs.LIGHT_SAMPLE)
        self.lib.oracle_light_sample_batch(self.scene.handle, ptr(tokens), ptr(_layers(layers)), ptr(points), ptr(samples), len(tokens), ptr(out))
        return out

    def probability_density(self, tokens, points, incident, layers=None):
        tokens, points = np.ascontiguousarray(tokens, dtype=np.uint32), np.ascontiguousarray(points, dtype=structs.SURFACE)
        incident = np.ascontiguousarray(incident, dtype=np.float32)
        out = np.zeros(len(tokens), dtype=np.float32)
        self.lib.oracle_light_pdf_batch(self.scene.handle, ptr(tokens), ptr(_layers(layers)), ptr(points), ptr(incident), len(tokens), ptr(out))
        return out

    def evaluate_infinite(self, directions, direct=False):
        directions = np.ascontiguousarray(directions, dtype=np.float32)
        out = np.zeros((len(directions), 3), dtype=np.float32)
        self.lib.oracle_evaluate_infinite_batch(self.scene.handle, ptr(directions), len(directions), 1 if direct else 0, ptr(out))
        return out


def surfaces(positions, normals):
    out = np.zeros(len(positions), dtype=structs.SURFACE)
    out["position"], out["normal"] = positions, normals
    return out


def unit_vectors(rng, count):
    v = rng.normal(size=(count, 3))
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)


def samples_with_edges(rng, shape):
    """uniform samples with exact 0 and the largest float below 1 mixed in (Sample1D clamps to [0, 1 - ulp])"""
    samples = rng.random(shape, dtype=np.float32)
    flat = samples.reshape(-1)
    flat[::17] = 0.0
    flat[5::19] = np.nextafter(np.float32(1.0), np.float32(0.0))
    flat[9::23] = 1.0
    return samples
