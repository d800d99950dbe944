"""The oracle with the stratified sample sequence (tests/c_client/stratified_oracle.cpp): built once per process into a temporary directory,
with liboracle.so's compiler flags, and loaded beside it. It exports everything liboracle.so does, evaluating with the stratified sequence
when EchoRenderParams.evaluator carries DISTRIBUTION_STRATIFIED (the uniform one otherwise), plus oracle_stratified_value. TEST
INFRASTRUCTURE ONLY."""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile
from unittest import mock

from tests import oracle_lib

SOURCE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c_client", "stratified_oracle.cpp")
FLAGS = ["-std=c++17", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-Wextra", "-pthread", "-shared"]
_lib = None
_oracle_library = oracle_lib.library  # liboracle.so's loader, also while scene() stands this module's in for it


def library():
    global _lib
    if _lib is not None:
        return _lib
    directory = tempfile.mkdtemp(prefix="stratified_oracle_")
    atexit.register(shutil.rmtree, directory, True)
    path = os.path.join(directory, "libstratified_oracle.so")
    subprocess.run(["g++"] + FLAGS + ["-o", path, SOURCE], check=True)
    lib = ctypes.CDLL(path)
    # the same prototypes as liboracle.so's (oracle_lib.library() declares them as it loads it)
    for name, function in vars(_oracle_library()).items():
        if isinstance(function, ctypes._CFuncPtr):
            mine = getattr(lib, name)
            mine.argtypes, mine.restype = function.argtypes, function.restype
    u32 = ctypes.c_uint32
    lib.oracle_stratified_value.argtypes = [u32, u32, u32, u32, u32, ctypes.c_int32, ctypes.c_void_p]
    _lib = lib
    return lib


def scene(prepared):
    """an oracle_lib.OracleScene on this library"""
    with mock.patch.object(oracle_lib, "library", library):
        return oracle_lib.OracleScene(prepared)
