"""Fixtures and switches for checking every wavefront schedule of the renderer against the oracle: shared by the CPU suite
(test_wavefront_schedules.py, which proves each fixture lands on the stack class it claims and that the hand-built trees are valid)
and the GPU suite (test_gpu_wavefront_schedules.py, which renders them under every schedule).

Which kernels of render.cu run for a call depends on the scene's stack class (48, 96 or 192 traversal-stack entries), on whether it has
packs, on the distribution and on three run-time thresholds (NARROW_LIMIT, TAIL_LIMIT and the counted pass). The fixtures here reach
every stack class with and without packs; `schedule` sets the thresholds so that one render takes the kernels asked for."""
import contextlib
import dataclasses

import numpy as np

from echorenderer_b200 import _native, host, scenes, structs

# echo_b200_debug_set_option's render switches and the values the library starts with when no ECHO_B200_<NAME> is set (render.cu RenderOptions)
DEFAULTS = {"RUN_AHEAD": -1, "BLOCKING_SYNC": -1, "RENDER_WORKERS": 8, "BATCH_PATHS": 1 << 24, "TAIL_LIMIT": 8192, "NARROW_LIMIT": 1 << 20, "GUIDED_BATCHES": 0}

# One pipeline in lock step (RUN_AHEAD 0), so that a render of fewer paths than BATCH_PATHS is one batch whose first bounce has every
# path, and its kernel launches do not depend on how fast the host looks at the counts.
_ONE_BATCH = {"RENDER_WORKERS": 1, "RUN_AHEAD": 0}

SCHEDULES = ("narrow", "persistent", "tail", "mixed", "batched")


def schedule_switches(name, paths=0):
    """The switches of a schedule; `paths` is the number of paths of the render (the `mixed` schedule turns narrow at a quarter of them).
    narrow: the one-thread-per-ray kernels on every bounce, no tail kernel; persistent: the persistent kernels down to the last ray;
    tail: every bounce after the camera rays' extend in tail_kernel; mixed: persistent, then narrow, then tail; batched: several
    batches per call on three pipelines, guided batch sizes, run-ahead and polling waits."""
    if name == "narrow":
        return {**DEFAULTS, **_ONE_BATCH, "NARROW_LIMIT": 1 << 30, "TAIL_LIMIT": 0}
    if name == "persistent":
        return {**DEFAULTS, **_ONE_BATCH, "NARROW_LIMIT": 0, "TAIL_LIMIT": 0}
    if name == "tail":
        return {**DEFAULTS, **_ONE_BATCH, "TAIL_LIMIT": 1 << 30}
    if name == "mixed":
        return {**DEFAULTS, **_ONE_BATCH, "NARROW_LIMIT": max(paths // 4, 1)}
    if name == "batched":
        return {**DEFAULTS, "RENDER_WORKERS": 3, "BATCH_PATHS": 1 << 16, "GUIDED_BATCHES": 1, "RUN_AHEAD": 2, "BLOCKING_SYNC": 2}
    raise ValueError(f"unknown schedule {name!r}")


@contextlib.contextmanager
def schedule(name, paths=0):
    """Sets all seven switches for the schedule `name` and puts every one back to its default afterwards, whatever happens inside."""
    try:
        for option, value in schedule_switches(name, paths).items():
            _native.set_option(option, value)
        yield
    finally:
        for option, value in DEFAULTS.items():
            _native.set_option(option, value)


def stack_entries(prepared):
    """Traversal-stack entries the device sizes a scene's kernels for (api.cu chain_stack and commit_device): 3 * maxDepth + 1 for a
    plain scene; for a scene with packs, each pack's 3 * maxDepth + 1 plus the most any chain of placements below it needs."""
    if prepared.packs is None:
        return 3 * int(prepared.max_depth) + 1
    packs, instances = prepared.packs, prepared.instances
    need = {}

    def walk(index):
        if index not in need:
            pack = packs[index]
            first, count = int(pack["instanceOffset"]), int(pack["instanceCount"])
            below = max((walk(int(instances[i]["pack"])) for i in range(first, first + count)), default=0)
            need[index] = 3 * int(pack["maxDepth"]) + 1 + below
        return need[index]

    return walk(0)


def stack_class(entries):
    """The kernels' stack size for `entries` (trace.cu stack_class, after commit_device rounds a pack chain to the smallest depth with
    3 * depth + 1 >= entries): 48, 96, 192, or None when the device refuses the scene."""
    size = (int(entries) + 1) // 3 * 3 + 1
    for limit in (48, 96, 192):
        if size <= limit:
            return limit
    return None


def _primitive_boxes(prepared):
    triangles, spheres = prepared.triangles, prepared.spheres
    corners = np.stack([triangles["vertex0"], triangles["vertex0"] + triangles["edge1"], triangles["vertex0"] + triangles["edge2"]])
    radius = spheres["radius"][:, None]
    low = np.concatenate([corners.min(axis=0), spheres["position"] - radius]).astype(np.float32)
    high = np.concatenate([corners.max(axis=0), spheres["position"] + radius]).astype(np.float32)
    # one float step outwards: the boxes are only culls and must hold their primitive whatever the vertex sums rounded to
    low, high = np.nextafter(low, np.float32(-np.inf)), np.nextafter(high, np.float32(np.inf))
    tokens = [structs.make_token(structs.TOKEN_TYPE_TRIANGLE, i) for i in range(len(triangles))]
    tokens += [structs.make_token(structs.TOKEN_TYPE_SPHERE, i) for i in range(len(spheres))]
    return low, high, tokens


def chain_qbvh(prepared, per_node):
    """A copy of a plain scene whose QBVH is a left-leaning chain over all of its triangles and spheres (like test_gpu_trace.chain_scene):
    node i holds `per_node` (1 or 2) primitives in slots 0 .. per_node - 1 and node i + 1 in slot 2; the last node holds what is left.
    With two primitives a node orders them along the axis their centres are furthest apart on (axisMinor0), like a built tree would.
    Every other array, bound_radius included, is the scene's own."""
    assert prepared.packs is None and per_node in (1, 2)
    low, high, tokens = _primitive_boxes(prepared)
    centre = (low.astype(np.float64) + high) / 2
    count = len(tokens)
    groups, first = [], 0
    while count - first > per_node + 1:
        groups.append(list(range(first, first + per_node)))
        first += per_node
    groups.append(list(range(first, count)))

    nodes = np.zeros(len(groups), dtype=structs.QBVH_NODE)
    for key in ("minX", "minY", "minZ", "maxX", "maxY", "maxZ"):
        nodes[key] = np.inf
    nodes["token4"] = structs.TOKEN_EMPTY
    nodes["axisMajor"], nodes["axisMinor0"], nodes["axisMinor1"] = 0, 3, 3

    def put(i, slot, lo, hi, token):
        nodes["minX"][i, slot], nodes["minY"][i, slot], nodes["minZ"][i, slot] = lo
        nodes["maxX"][i, slot], nodes["maxY"][i, slot], nodes["maxZ"][i, slot] = hi
        nodes["token4"][i, slot] = token

    for i, group in enumerate(groups):
        last = i == len(groups) - 1
        pair = group if not last else group[:per_node]
        if len(pair) == 2:
            axis = int(np.argmax(np.abs(centre[pair[1]] - centre[pair[0]])))
            pair = sorted(pair, key=lambda p: centre[p][axis])
            nodes["axisMinor0"][i] = axis
        for slot, p in enumerate(pair):
            put(i, slot, low[p], high[p], tokens[p])
        rest = list(range(group[-1] + 1, count)) if not last else group[per_node:]
        if not last:
            put(i, 2, low[rest].min(axis=0), high[rest].max(axis=0), structs.make_token(structs.TOKEN_TYPE_NODE, i + 1))
        elif rest:
            assert len(rest) == 1
            put(i, 2, low[rest[0]], high[rest[0]], tokens[rest[0]])
    # maxDepth counts the leaves' level too, as the builders do (a one-node tree has depth 2)
    return dataclasses.replace(prepared, nodes=nodes, max_depth=len(nodes) + 1, _bound_radius=prepared.bound_radius)


def chain_cornell():
    """The Cornell box with a dielectric (glass) short box and a rough conductor tall box, so that a render of it reaches every material
    class: diffuse, emissive, the one-sided front wall, dielectric and conductor. Both boxes stand 0.05 above the floor: a ray would otherwise
    meet a box's bottom and the floor at the same distance or an ulp apart, where the reference's answer depends on which it tests first,
    and the chain trees would not render like the swept one."""
    description = scenes.cornell_box()
    first = len(description.materials)
    description.materials = np.concatenate([description.materials, scenes.material(structs.MATERIAL_DIELECTRIC, (1, 1, 1), roughness=(0, 0), ior=1.5),
                                            scenes.material(structs.MATERIAL_CONDUCTOR, (1, 1, 1), roughness=(0.3, 0.2), param_a=(0.9, 0.7, 0.4),
                                                            param_b=(1.0, 0.8, 0.6), flags=structs.MATERIAL_FLAG_ARTISTIC)])
    boxes = len(description.triangles) - 24
    description.triangles["material"][boxes:boxes + 12] = first
    description.triangles["vertex0"][boxes:, 1] += np.float32(0.05)
    description.triangles["material"][boxes + 12:] = first + 1
    return host.prepare(description)


def deep_pack_scene(layers, rings=24, segments=26):
    """A chain of packs: instanced_scene's blob (triangles, a conductor sphere and a glowing one) at the bottom, and `layers` - 1 packs
    above it, each a box plus two placements of the pack below; the scene places the top pack twice over a ground plane under a light.
    Hits on the blob carry `layers` instance layers. The boxes cycle through glass, a rough conductor and Oren-Nayar diffuse."""
    from echorenderer_b200.host import InstanceDescription, PackDescription
    blob = scenes.instanced_scene(grid=1, rings=rings, segments=segments, nested=False).packs[0]
    box_materials = [scenes.material(structs.MATERIAL_DIELECTRIC, (1, 1, 1), roughness=(0.05, 0.05), ior=1.5),
                     scenes.material(structs.MATERIAL_CONDUCTOR, (1, 1, 1), roughness=(0.3, 0.2), param_a=(0.9, 0.7, 0.4), param_b=(1.0, 0.8, 0.6),
                                     flags=structs.MATERIAL_FLAG_ARTISTIC),
                     scenes.material(structs.MATERIAL_DIFFUSE, (0.4, 0.6, 0.8), roughness=(0.5, 0.5))]
    packs = [blob]
    for level in range(1, layers):
        below = len(packs) - 1
        packs.append(PackDescription(triangles=scenes.box(0, (1.0, 0.3, 1.0), (0, -1.2, 0)), materials=box_materials[level % 3],
                                     instances=[InstanceDescription(below, (-1.1, 0.2, 0.0), (0, 25 * level, 0), 0.55),
                                                InstanceDescription(below, (1.1, 0.3, 0.3), (15, 40 * level, 10), 0.5)]))
    top = len(packs) - 1
    materials = np.concatenate([scenes.material(structs.MATERIAL_DIFFUSE, (0.7, 0.7, 0.7)), scenes.material(structs.MATERIAL_EMISSIVE, (10.0, 9.0, 8.0))])
    triangles = np.concatenate([scenes.plane(0, (16, 16), (0, -2.5, 0)), scenes.plane(1, (4, 4), (0, 6, 0), (180, 0, 0))])
    position = (0.0, 3.0, -7.0)
    camera = scenes.perspective_camera(position, scenes.look_rotation(position, (0, -0.5, 0)), field_of_view=50.0)
    description = host.SceneDescription(triangles=triangles, materials=materials, packs=packs, infinite_lights=scenes.ambient_light((0.2, 0.22, 0.25)),
                                        instances=[InstanceDescription(top, (-1.6, 0, 0), (0, 10, 0), 1.6), InstanceDescription(top, (1.8, 0.2, 0.5), (0, -35, 5), 1.4)],
                                        camera=camera, name=f"deep_packs_{layers}")
    return host.prepare(description)
