"""Every pack of an instanced scene built in one call (echorenderer_b200/csrc/echo_pack_build.h: rounds of packs of equal height, each
an instance-bounds pass, a QBVH forest and a light forest) on a sequential CPU backend (tests/c_client/pack_emulation.cpp): every pack's
nodes, depth, light nodes, emitter tokens and bit paths must be what the host mirror builds for that pack alone, byte for byte, fed with
the placements' rows of the restatement in pack_build_lib.py. The GPU suite (test_gpu_pack_build.py) asks the same of the CUDA backend."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest

from echorenderer_b200 import host, scene, scenes, structs
from echorenderer_b200.host import InstanceDescription, PackDescription, SceneDescription

from tests import pack_build_lib as lib_expected

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, INVALID, UNSUPPORTED = 0, 1, 4


@pytest.fixture(scope="module")
def emulation(tmp_path_factory):
    library = tmp_path_factory.mktemp("packs") / "libpack_emulation.so"
    subprocess.run(["g++", "-std=c++17", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-Wall", "-Wextra", "-Werror", "-shared", "-fPIC",
                    os.path.join(ROOT, "tests", "c_client", "pack_emulation.cpp"), "-o", str(library)], check=True)
    lib = ctypes.CDLL(str(library))
    p, u32 = ctypes.c_void_p, ctypes.c_uint32
    pu32 = ctypes.POINTER(u32)
    lib.pack_emulation_build.argtypes = [p, u32, p, u32, p, u32, p, u32, p, u32, p, u32, p, u32, pu32, p, u32, pu32, p, p, u32, pu32,
                                         ctypes.POINTER(ctypes.c_float), ctypes.c_int32, u32, p, p]
    lib.pack_emulation_build.restype = ctypes.c_int32
    lib.pack_emulation_message.restype = ctypes.c_char_p

    def build(prepared, reverse=False, depth_limit=63, packs=None, capacity=None):
        (triangles, spheres, materials, points, records, instances), (nodes, light_nodes, tokens, paths) = scene.pack_build_arguments(prepared)
        if packs is not None:
            records = packs
        if capacity is not None:
            nodes, light_nodes, tokens, paths = nodes[:capacity[0]], light_nodes[:capacity[1]], tokens[:capacity[2]], paths[:capacity[2]]
        ptr = lambda a: a.ctypes.data if a.size else None
        rows = np.zeros((max(len(instances), 1), 18), dtype=np.float32)
        stats = np.zeros(4, dtype=np.uint32)
        counts = [u32() for _ in range(3)]
        power = ctypes.c_float()
        status = lib.pack_emulation_build(ptr(triangles), len(triangles), ptr(spheres), len(spheres), ptr(materials), len(materials), ptr(points), len(points),
                                          ptr(records), len(records), ptr(instances), len(instances), ptr(nodes), len(nodes), ctypes.byref(counts[0]),
                                          ptr(light_nodes), len(light_nodes), ctypes.byref(counts[1]), ptr(tokens), ptr(paths), len(tokens), ctypes.byref(counts[2]),
                                          ctypes.byref(power), int(reverse), depth_limit, rows.ctypes.data, stats.ctypes.data)
        return dict(status=status, message=lib.pack_emulation_message().decode(), packs=records, nodes=nodes[:counts[0].value],
                    light_nodes=light_nodes[:counts[1].value], tokens=tokens[:counts[2].value], paths=paths[:counts[2].value],
                    counts=[c.value for c in counts], power=power.value, rows=rows[:len(instances)],
                    rounds=int(stats[0]), sweep_levels=int(stats[1]), light_levels=int(stats[2]), rebuilt=int(stats[3]))

    return build


def check_scene(emulation, description, reverse=False):
    prepared = host.prepare(description)
    expected, rows = lib_expected.expected_packs(prepared)
    result = emulation(prepared, reverse=reverse)
    assert result["status"] == OK, result["message"]
    assert result["rows"].tobytes() == rows.tobytes()
    lib_expected.assert_same_packs(result["packs"], result["nodes"], result["light_nodes"], result["tokens"], result["paths"], result["power"], expected)
    for name in ("triangleOffset", "triangleCount", "sphereOffset", "sphereCount", "instanceOffset", "instanceCount", "materialOffset", "pointLightOffset", "pointLightCount"):
        assert np.array_equal(result["packs"][name], prepared.packs[name])
    return prepared, expected, result


def levels_of(prepared, emulation_levels):
    """Per round the deepest pack's levels, summed; and the sum over all packs (what one build per pack reads back)."""
    height = lib_expected.heights(prepared.packs, prepared.instances)
    forest = sum(max(emulation_levels[p] for p in range(len(height)) if height[p] == h) for h in set(height))
    return forest, sum(emulation_levels)


@pytest.mark.parametrize("reverse", [False, True])
def test_nested_instanced_scene(emulation, reverse):
    """Two layers of placements, swatch overrides, a pack with a point light, emitters inside packs."""
    check_scene(emulation, scenes.instanced_scene(grid=4, rings=12, segments=12), reverse)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_many_packs(emulation, seed):
    prepared, expected, result = check_scene(emulation, scenes.many_packs_scene(pack_count=30, seed=seed, layers=3 if seed != 2 else 2), reverse=seed == 3)
    assert result["rounds"] == (4 if seed != 2 else 3)
    kinds = [(int(r["triangleCount"]) + int(r["sphereCount"]), int(r["emitterCount"]), int(r["pointLightCount"])) for r in result["packs"]]
    assert any(geometry == 0 for geometry, _, _ in kinds[1:])                 # packs of placements only
    assert any(emitters == 0 for _, emitters, _ in kinds[1:])                 # packs without an emitter
    assert any(points > 0 and emitters == points for _, emitters, points in kinds[1:])  # point lights only


def test_instance_rows_agree_with_host_prepare(emulation):
    """The pinned rows agree with what host.prepare computes with numpy matmul (whose rounding belongs to the BLAS kernel) to within
    1e-6 of each box's extent."""
    prepared = host.prepare(scenes.many_packs_scene(pack_count=24, seed=5))
    result = emulation(prepared)
    assert result["status"] == OK, result["message"]
    expected, _ = lib_expected.expected_packs(prepared)
    for i, instance in enumerate(prepared.instances):
        child_nodes, _, child_lights, _, _ = expected[int(instance["pack"])]
        box = host.transformed_bound(host.fill_bounds(child_nodes), instance["inverse"])
        row = result["rows"][i]
        extent = float(np.max(box[3:] - box[:3]))
        assert np.max(np.abs(row[:6] - box)) <= 1e-6 * max(extent, 1.0)
        if len(child_lights):
            root = child_lights[0]
            light_box = host.transformed_bound(np.concatenate([root["boxMin"], root["boxMax"]])[None, :], instance["inverse"])
            assert np.max(np.abs(row[6:12] - light_box)) <= 1e-6 * max(float(np.max(light_box[3:] - light_box[:3])), 1.0)
            axis = instance["inverse"].reshape(3, 4)[:, :3].astype(np.float64) @ root["coneAxis"].astype(np.float64)
            assert np.allclose(row[12:15], axis / np.linalg.norm(axis), atol=1e-6)
            assert row[17] == np.float32(root["power"]) * instance["inverseScale"] * instance["inverseScale"]
        else:
            assert not np.any(row[6:])


def test_read_backs_are_the_deepest_pack_per_round(emulation):
    prepared, _, result = check_scene(emulation, scenes.many_packs_scene(pack_count=40, seed=7))
    sweep_levels, light_levels = [], []
    expected, rows = lib_expected.expected_packs(prepared)
    for p in range(len(prepared.packs)):
        one = emulation_single(prepared, p, rows)
        sweep_levels.append(one["sweep_levels"])
        light_levels.append(one["light_levels"])
    forest, per_pack = levels_of(prepared, sweep_levels)
    assert result["sweep_levels"] == forest and forest < per_pack
    forest, per_pack = levels_of(prepared, light_levels)
    assert result["light_levels"] == forest and forest < per_pack


def emulation_single(prepared, p, rows):
    """The levels pack p reads back when it is built alone (the single-pack emulations of both drivers, fed with the same rows)."""
    record = prepared.packs[p]
    t0, tn = int(record["triangleOffset"]), int(record["triangleCount"])
    s0, sn = int(record["sphereOffset"]), int(record["sphereCount"])
    i0, i_n = int(record["instanceOffset"]), int(record["instanceCount"])
    m0 = int(record["materialOffset"])
    q0, qn = int(record["pointLightOffset"]), int(record["pointLightCount"])
    levels = single_levels(prepared.triangles[t0:t0 + tn], prepared.spheres[s0:s0 + sn], rows[i0:i0 + i_n],
                           prepared.materials[m0:m0 + lib_expected.swatch_size(prepared, m0)], prepared.point_lights[q0:q0 + qn])
    return dict(sweep_levels=levels[0], light_levels=levels[1])


_SINGLE = {}


def single_levels(triangles, spheres, rows, materials, points):
    if "lib" not in _SINGLE:
        sweep = os.path.join(ROOT, "tests", "c_client", "sweep_emulation.cpp")
        light = os.path.join(ROOT, "tests", "c_client", "light_emulation.cpp")
        out = tempfile.mkdtemp(prefix="pack_levels_")
        libs = []
        for source, name in ((sweep, "libsweep_levels.so"), (light, "liblight_levels.so")):
            subprocess.run(["g++", "-std=c++17", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-shared", "-fPIC", source, "-o", os.path.join(out, name)], check=True)
            libs.append(ctypes.CDLL(os.path.join(out, name)))
        _SINGLE["lib"] = libs
    sweep_lib, light_lib = _SINGLE["lib"]
    u32 = ctypes.c_uint32
    ptr = lambda a: a.ctypes.data if a.size else None
    triangles = np.ascontiguousarray(triangles)
    spheres = np.ascontiguousarray(spheres)
    boxes = np.ascontiguousarray(rows[:, :6])
    lights = np.ascontiguousarray(rows[:, 6:])
    total = len(triangles) + len(spheres) + len(boxes)
    nodes = np.zeros(max(total, 1), dtype=structs.QBVH_NODE)
    count, depth, sweep_levels = u32(), u32(), u32()
    assert sweep_lib.sweep_emulation_build(ctypes.c_void_p(ptr(triangles)), u32(len(triangles)), ctypes.c_void_p(ptr(spheres)), u32(len(spheres)), ctypes.c_void_p(ptr(boxes)),
                                           u32(len(boxes)), ctypes.c_int32(0), ctypes.c_void_p(nodes.ctypes.data), ctypes.byref(count), ctypes.byref(depth), ctypes.byref(sweep_levels)) == 0
    candidates = total + len(points)
    light_nodes = np.zeros(max(2 * candidates, 1), dtype=structs.LIGHT_NODE)
    tokens, paths = np.zeros(max(candidates, 1), dtype=np.uint32), np.zeros(max(candidates, 1), dtype=np.uint64)
    materials = np.ascontiguousarray(materials)
    points = np.ascontiguousarray(points)
    node_count, emitter_count, light_levels = u32(), u32(), u32()
    assert light_lib.light_emulation_build(ctypes.c_void_p(ptr(triangles)), u32(len(triangles)), ctypes.c_void_p(ptr(spheres)), u32(len(spheres)), ctypes.c_void_p(ptr(materials)),
                                           u32(len(materials)), ctypes.c_void_p(ptr(points)), u32(len(points)), ctypes.c_void_p(ptr(lights)), u32(len(lights)), ctypes.c_int32(0),
                                           ctypes.c_void_p(light_nodes.ctypes.data), ctypes.byref(node_count), ctypes.c_void_p(tokens.ctypes.data), ctypes.c_void_p(paths.ctypes.data),
                                           ctypes.byref(emitter_count), ctypes.byref(light_levels)) == 0
    return sweep_levels.value, light_levels.value


def chain_scene(layers):
    """`layers` packs, each placing the one below twice (beside a triangle pair), the scene placing the top one."""
    glow = scenes.material(structs.MATERIAL_EMISSIVE, (4.0, 4.0, 4.0))
    packs = [PackDescription(triangles=scenes.plane(0, (1.0, 1.0)), materials=glow)]
    for k in range(1, layers):
        packs.append(PackDescription(triangles=scenes.plane(0, (0.5, 0.5), (0, -1, 0)), materials=scenes.material(structs.MATERIAL_DIFFUSE, (0.5, 0.5, 0.5)),
                                     instances=[InstanceDescription(k - 1, (-1.0, 0.2 * k, 0.0), (0, 15 * k, 0), 0.6),
                                                InstanceDescription(k - 1, (1.0, 0.0, 0.3), (10 * k, 0, 5), 0.5)]))
    return SceneDescription(triangles=scenes.plane(0, (20.0, 20.0)), materials=scenes.material(structs.MATERIAL_DIFFUSE, (0.7, 0.7, 0.7)),
                            instances=[InstanceDescription(layers - 1, (0, 2, 0), (0, 0, 0), 1.0)], packs=packs)


def test_chain_of_five_layers(emulation):
    prepared, _, result = check_scene(emulation, chain_scene(5))
    assert result["rounds"] == 6
    check_scene(emulation, chain_scene(5), reverse=True)


def small_packs_scene():
    """A 2-primitive pack, packs with zero, one and two emitters, a pack of placements only."""
    glow = scenes.material(structs.MATERIAL_EMISSIVE, (3.0, 2.0, 1.0))
    dull = scenes.material(structs.MATERIAL_DIFFUSE, (0.5, 0.5, 0.5))
    two = PackDescription(triangles=scenes.plane(0, (1.0, 1.0)), materials=dull)                            # 2 primitives, no emitter
    one = PackDescription(triangles=scenes.plane(0, (1.0, 1.0)), materials=np.concatenate([dull, glow]))
    one.triangles["material"][1] = 1                                                                      # one emitter
    both = PackDescription(triangles=scenes.plane(0, (1.0, 1.0)), materials=glow)                           # two emitters
    only = PackDescription(instances=[InstanceDescription(0, (0, 0, 0), (0, 0, 0), 1.0), InstanceDescription(1, (2, 0, 0), (0, 90, 0), 0.5),
                                      InstanceDescription(2, (0, 0, 2), (45, 0, 0), 2.0)])                  # placements only
    return SceneDescription(triangles=scenes.plane(0, (20.0, 20.0)), materials=dull,
                            instances=[InstanceDescription(3, (0, 1, 0)), InstanceDescription(0, (5, 1, 0)), InstanceDescription(1, (-5, 1, 0)),
                                       InstanceDescription(2, (0, 1, 5))],
                            packs=[two, one, both, only])


@pytest.mark.parametrize("reverse", [False, True])
def test_small_packs(emulation, reverse):
    prepared, expected, result = check_scene(emulation, small_packs_scene(), reverse)
    emitters = sorted(int(r["emitterCount"]) for r in result["packs"][1:4])
    assert emitters == [0, 1, 2]


def test_refusals(emulation):
    prepared = host.prepare(small_packs_scene())

    small = prepared.packs.copy()
    small[1]["triangleCount"] = 1  # a pack of one primitive
    assert emulation(prepared, packs=small)["status"] == INVALID

    cyclic = prepared.packs.copy()
    instances = prepared.instances.copy()
    instances[int(cyclic[4]["instanceOffset"])]["pack"] = 4  # the placements-only pack places itself
    looped = host.PreparedArrays.__new__(host.PreparedArrays)
    looped.__dict__.update(prepared.__dict__)
    looped.instances = instances
    assert emulation(looped)["status"] == INVALID

    full = emulation(prepared)
    needed = full["counts"]
    short = emulation(prepared, capacity=(needed[0] - 1, needed[1], needed[2]))
    assert short["status"] == INVALID and short["counts"] == needed
    short = emulation(prepared, capacity=(needed[0], needed[1], needed[2] - 1))
    assert short["status"] == INVALID and short["counts"] == needed


def test_six_layers_are_refused(emulation, monkeypatch):
    """Six layers of placements below the scene are deeper than TokenHierarchy.MaxLayer: host.prepare refuses them, and so does the build
    (the arrays come from a host.prepare allowed one more layer)."""
    with pytest.raises(ValueError):
        host.prepare(chain_scene(6))
    monkeypatch.setattr(structs, "MAX_INSTANCE_LAYERS", 6)
    prepared = host.prepare(chain_scene(6))
    result = emulation(prepared)
    assert result["status"] == INVALID and "MaxLayer" in result["message"]


def test_deeper_than_63_light_levels_is_unsupported(emulation):
    """Point lights have boxes without area: every cut costs 0, the first one wins and peels one emitter per level, so 70 of them chain
    70 levels deep — more than a 64-bit path (LightTree.cs:29) holds."""
    points = np.zeros(70, dtype=structs.POINT_LIGHT)
    points["position"][:, 0] = np.arange(70.0)
    points["intensity"] = (1.0, 1.0, 1.0)
    pack = PackDescription(triangles=scenes.plane(0, (1.0, 1.0)), materials=scenes.material(structs.MATERIAL_DIFFUSE, (0.5, 0.5, 0.5)), point_lights=points)
    with pytest.raises(ValueError):
        host.build_light_tree(pack)
    description = SceneDescription(triangles=scenes.plane(0, (20.0, 20.0)), materials=scenes.material(structs.MATERIAL_DIFFUSE, (0.5, 0.5, 0.5)),
                                   instances=[InstanceDescription(0, (0, 1, 0))], packs=[pack])
    refused = lambda *_: (np.zeros(0, dtype=structs.LIGHT_NODE), np.zeros(0, np.uint32), np.zeros(0, np.uint64), 0.0)  # the arrays only
    result = emulation(host.prepare(description, light_tree_builder=refused))
    assert result["status"] == UNSUPPORTED and "63" in result["message"]
