"""What every pack of an instanced scene must come out as, from the host mirror pack by pack: shared by the CPU suite
(test_pack_build.py, the orchestration on a sequential CPU backend) and the GPU suite (test_gpu_pack_build.py, echo_b200_build_packs).

The placements' rows are an explicit numpy scalar restatement of PreparedInstance.BoxBound / LightBound as the pack build pins them:
FillBounds(6) in the mirror's stack order, Float4x4.MultiplyPoint / MultiplyDirection left to right in binary32 without contraction, the
cone axis in binary64 (products summed left to right, divided by sqrt((x^2 + y^2) + z^2), rounded once)."""
import math
from types import SimpleNamespace

import numpy as np

from echorenderer_b200 import host, structs

F = np.float32


def _is_node(token):
    return token != structs.TOKEN_EMPTY and structs.token_type(token) == structs.TOKEN_TYPE_NODE


def fill_bounds_order(nodes):
    """The slots FillBounds(6) reports, as (node, slot) in the order host.fill_bounds lists them."""
    out, first, second = [], [], []
    root = nodes[0]
    for j in range(4):
        token = int(root["token4"][j])
        if token == structs.TOKEN_EMPTY:
            continue
        (first.append(structs.token_index(token)) if _is_node(token) else out.append((0, j)))
    for index in reversed(first):
        for j in range(4):
            token = int(nodes[index]["token4"][j])
            if token == structs.TOKEN_EMPTY:
                continue
            (second.append(structs.token_index(token)) if _is_node(token) else out.append((index, j)))
    for index in reversed(second):
        out.extend((index, j) for j in range(4) if int(nodes[index]["token4"][j]) != structs.TOKEN_EMPTY)
    return out


def transform_box(m, lo, hi):
    """Centre / extent of one box through rows 0..2 of an affine matrix, binary32 scalars left to right."""
    c = [(F(hi[k]) + F(lo[k])) * F(0.5) for k in range(3)]
    e = [(F(hi[k]) - F(lo[k])) * F(0.5) for k in range(3)]
    out_lo, out_hi = [], []
    for r in range(3):
        row = [F(v) for v in m[4 * r:4 * r + 4]]
        centre = ((row[0] * c[0] + row[1] * c[1]) + row[2] * c[2]) + row[3]
        extent = (abs(row[0]) * e[0] + abs(row[1]) * e[1]) + abs(row[2]) * e[2]
        out_lo.append(centre - extent)
        out_hi.append(centre + extent)
    return out_lo, out_hi


def instance_rows(instance, child_nodes, child_light_nodes):
    """(6-float box row, 12-float light row) of one placement."""
    m = [F(v) for v in instance["inverse"]]
    lo, hi = [F(np.inf)] * 3, [F(-np.inf)] * 3
    for index, j in fill_bounds_order(child_nodes):
        node = child_nodes[index]
        box_lo = [node["minX"][j], node["minY"][j], node["minZ"][j]]
        box_hi = [node["maxX"][j], node["maxY"][j], node["maxZ"][j]]
        t_lo, t_hi = transform_box(m, box_lo, box_hi)
        lo = [t_lo[k] if t_lo[k] < lo[k] else lo[k] for k in range(3)]
        hi = [t_hi[k] if t_hi[k] > hi[k] else hi[k] for k in range(3)]
    box = np.array(lo + hi, dtype=np.float32)

    if len(child_light_nodes) == 0:
        return box, np.zeros(12, dtype=np.float32)
    root = child_light_nodes[0]
    l_lo, l_hi = transform_box(m, root["boxMin"], root["boxMax"])
    a = [float(v) for v in root["coneAxis"]]
    axis = [(float(m[4 * r]) * a[0] + float(m[4 * r + 1]) * a[1]) + float(m[4 * r + 2]) * a[2] for r in range(3)]
    norm = max(math.sqrt((axis[0] * axis[0] + axis[1] * axis[1]) + axis[2] * axis[2]), 1e-300)
    power = F(root["power"]) * F(instance["inverseScale"]) * F(instance["inverseScale"])
    light = np.array(l_lo + l_hi + [axis[r] / norm for r in range(3)] + [root["cosOffset"], root["cosExtend"], power], dtype=np.float32)
    return box, light


def swatch_size(prepared, offset):
    """A pack's swatch ends where the next swatch of the material array begins (another pack's or a placement's)."""
    starts = [int(v) for v in prepared.packs["materialOffset"]] + [int(v) for v in prepared.instances["materialOffset"]]
    later = [s for s in starts if s > offset]
    return min(later + [len(prepared.materials)]) - offset


def heights(packs, instances):
    result = {}

    def height(p):
        if p not in result:
            record = packs[p]
            children = instances[int(record["instanceOffset"]):int(record["instanceOffset"] + record["instanceCount"])]["pack"]
            result[p] = 0 if len(children) == 0 else 1 + max(height(int(c)) for c in children)
        return result[p]

    for p in range(len(packs)):
        height(p)
    return [result[p] for p in range(len(packs))]


def expected_packs(prepared):
    """Per pack, children first: (nodes, max depth, light nodes, emitter tokens, bit paths, binary levels, light levels) from the host
    mirror, fed with the restated rows; and the rows of every placement ([n, 18]: box row, light row)."""
    packs, instances = prepared.packs, prepared.instances
    order = sorted(range(len(packs)), key=lambda p: heights(packs, instances)[p])
    built, rows = {}, np.zeros((len(instances), 18), dtype=np.float32)
    for p in order:
        record = packs[p]
        t0, tn = int(record["triangleOffset"]), int(record["triangleCount"])
        s0, sn = int(record["sphereOffset"]), int(record["sphereCount"])
        i0, i_n = int(record["instanceOffset"]), int(record["instanceCount"])
        q0, qn = int(record["pointLightOffset"]), int(record["pointLightCount"])
        m0 = int(record["materialOffset"])
        for i in range(i0, i0 + i_n):
            child = built[int(instances[i]["pack"])]
            box, light = instance_rows(instances[i], child[0], child[2])
            rows[i, :6], rows[i, 6:] = box, light
        triangles, spheres = prepared.triangles[t0:t0 + tn], prepared.spheres[s0:s0 + sn]
        nodes, depth = host.build_qbvh(triangles, spheres, instance_bounds=rows[i0:i0 + i_n, :6] if i_n else None)
        source = SimpleNamespace(triangles=triangles, spheres=spheres, materials=prepared.materials[m0:m0 + swatch_size(prepared, m0)],
                                 point_lights=prepared.point_lights[q0:q0 + qn])
        light_nodes, tokens, paths, _ = host.build_light_tree(source, rows[i0:i0 + i_n, 6:] if i_n else None)
        built[p] = (nodes, depth, light_nodes, tokens, paths)
    return [built[p] for p in range(len(packs))], rows


def assert_same_packs(result_packs, nodes, light_nodes, tokens, paths, power, expected):
    """Every pack's arrays, back to back in pack order, equal the mirror's byte for byte."""
    offsets = dict(node=0, light=0, emitter=0)
    for p, (e_nodes, e_depth, e_light, e_tokens, e_paths) in enumerate(expected):
        record = result_packs[p]
        assert int(record["nodeOffset"]) == offsets["node"] and int(record["nodeCount"]) == len(e_nodes) and int(record["maxDepth"]) == e_depth, p
        assert int(record["lightNodeOffset"]) == offsets["light"] and int(record["lightNodeCount"]) == len(e_light), p
        assert int(record["emitterOffset"]) == offsets["emitter"] and int(record["emitterCount"]) == len(e_tokens), p
        assert nodes[offsets["node"]:offsets["node"] + len(e_nodes)].tobytes() == e_nodes.tobytes(), p
        assert light_nodes[offsets["light"]:offsets["light"] + len(e_light)].tobytes() == e_light.tobytes(), p
        assert tokens[offsets["emitter"]:offsets["emitter"] + len(e_tokens)].tobytes() == e_tokens.tobytes(), p
        assert paths[offsets["emitter"]:offsets["emitter"] + len(e_paths)].tobytes() == e_paths.tobytes(), p
        offsets["node"] += len(e_nodes)
        offsets["light"] += len(e_light)
        offsets["emitter"] += len(e_tokens)
    assert len(nodes) == offsets["node"] and len(light_nodes) == offsets["light"] and len(tokens) == offsets["emitter"]
    e_light = expected[0][2]
    assert np.float32(power).tobytes() == (e_light[0]["power"] if len(e_light) else np.float32(0)).tobytes()
