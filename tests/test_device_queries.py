"""The device-buffer queries of include/echo_b200_query_device.h without a GPU: the header on its own, the exported and bound symbols,
the C# declarations of INTEGRATION.md, clean refusal without a device, the refusal texts, and the validation rules they share with the
host-buffer calls (echorenderer_b200/csrc/echo_query_rules.h) compiled for the host against a table of edge inputs."""
import ctypes
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from echorenderer_b200 import _native, host, scenes, structs
from tests import query_rules_lib
from tests.test_abi import declared_functions, have_gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_compiles_as_c99():
    source = '#include "echo_b200_query_device.h"\nint main(void) { unsigned long long clear = ECHO_QUERY_STATUS_CLEAR; return clear == ~0ull ? 0 : 1; }\n'
    with tempfile.TemporaryDirectory() as directory:
        path, binary = os.path.join(directory, "header.c"), os.path.join(directory, "header")
        open(path, "w").write(source)
        subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), path, "-o", binary], check=True)
        subprocess.run([binary], check=True)


def test_device_query_symbols_are_declared_bound_and_exported():
    declared = declared_functions("echo_b200_query_device.h")
    assert declared == set(_native.DEVICE_QUERY_EXPORTS) and len(declared) == 11
    assert not declared & (set(_native.EXPORTS) | set(_native.QUERY_EXPORTS))
    assert {name + "_device" for name in _native.QUERY_EXPORTS} < declared
    lib = _native.library()
    for name in declared:
        assert hasattr(lib, name), name
        assert getattr(lib, name).argtypes is not None, f"{name} has no ctypes signature"


def test_integration_document_declares_every_device_call():
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    for name in _native.DEVICE_QUERY_EXPORTS:
        assert re.search(rf"\[DllImport\(Library\)\] public static extern \w+ {name}\(", text), name


@pytest.mark.skipif(have_gpu(), reason="checks the no-device behaviour")
def test_every_device_call_refuses_a_null_scene():
    """Without a device a host can only hold a NULL scene: every call refuses it, at n = 4 and at n = 0."""
    lib = _native.library()
    handle = ctypes.c_void_p()
    assert lib.echo_b200_scene_create(ctypes.byref(handle), 0) == _native.ERR_NO_DEVICE and not handle.value

    buffer = ctypes.create_string_buffer(4096)  # stands for every device buffer: the calls must refuse before touching one
    b = ctypes.addressof(buffer)
    for n in (4, 0):
        calls = [
            lambda: lib.echo_b200_interact_batch_device(None, b, b, None, n, b, b, None),
            lambda: lib.echo_b200_scatter_sample_batch_device(None, b, b, None, b, n, b, b, None),
            lambda: lib.echo_b200_scatter_evaluate_batch_device(None, b, b, None, b, n, b, b, None),
            lambda: lib.echo_b200_light_pick_batch_device(None, b, b, n, b, b, b, b, None),
            lambda: lib.echo_b200_light_mass_batch_device(None, b, None, b, n, b, b, None),
            lambda: lib.echo_b200_light_sample_batch_device(None, b, None, b, b, n, b, b, None),
            lambda: lib.echo_b200_light_pdf_batch_device(None, b, None, b, b, n, b, b, None),
            lambda: lib.echo_b200_evaluate_infinite_batch_device(None, b, n, 1, b, b, None),
            lambda: lib.echo_b200_trace_batch_hierarchy_device(None, b, None, n, b, b, None),
            lambda: lib.echo_b200_occlude_batch_hierarchy_device(None, b, None, n, b, None),
        ]
        for call in calls:
            assert call() == _native.ERR_INVALID
            assert b"scene is null" in lib.echo_b200_last_error()


def test_every_refusal_code_has_its_own_text():
    known = {}
    for code in range(256):
        text = _native.query_reason(code)
        assert text
        known.setdefault(text, []).append(code)
    fallback = _native.query_reason(255)
    codes = [c for text, cs in known.items() if text != fallback for c in cs]
    assert codes == list(range(1, len(codes) + 1)) and len(codes) >= 23  # one text per code, no gaps
    assert known[fallback] == [0] + list(range(len(codes) + 1, 256))
    # the library's texts are the rules' own
    assert all(_native.query_reason(code) == query_rules_lib.reason_text(code) for code in codes)


def test_query_status_names_the_refused_query():
    _native.query_status(_native.QUERY_STATUS_CLEAR)
    _native.query_status(-1)  # the same word read back as a signed int64
    with pytest.raises(_native.EchoNativeError) as error:
        _native.query_status((41 << 8) | 1)
    assert error.value.status == _native.ERR_INVALID
    assert f"query 41: {_native.query_reason(1)}" in str(error.value)


@pytest.mark.parametrize("name", ["instanced", "cornell_box"])
def test_host_build_of_the_rules_agrees_with_the_edge_table(name):
    prepared = host.prepare(scenes.instanced_scene(grid=3, rings=8, segments=10) if name == "instanced" else scenes.cornell_box())
    contact, light, expected_contact, expected_light = query_rules_lib.edge_table(prepared)
    assert query_rules_lib.run_contact(prepared, contact) == expected_contact
    assert query_rules_lib.run_light(prepared, light) == expected_light

    # the table holds both sides of every edge
    accepted, refused = sum(e is None for e in expected_contact), sum(e is not None for e in expected_contact)
    assert accepted >= 10 and refused >= 10
    lengths = contact["rays"]["direction"][:24:2]
    assert {e for e, d in zip(expected_contact[:24:2], lengths)} == {None, "the ray needs a finite origin and a unit direction"}
    if name == "instanced":
        assert len(query_rules_lib.pack_paths(prepared)) == len(prepared.packs)
        assert "more than ECHO_MAX_INSTANCE_LAYERS instance layers" in expected_contact
        assert any(np.isclose(h["uv"][0], 4.5) for h, e in zip(contact["hits"], expected_contact) if e is None)
