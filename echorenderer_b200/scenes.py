"""Seeded synthetic scenes and ray batches for the configurations BASELINE.json names (SURVEY.md §8d).

C1 `cornell_box`      Echo's CornellBox (Scenic/CornellBox.cs:18-60 == ext/Scenes/Simple/cornell.echo)
C2 `terrain_scene`    1 M-triangle fbm terrain + 10 k hovering spheres, with `random_rays` / `secondary_rays`
C3 `mixed_material_scene`  Oren-Nayar ground, blobs cycling Dielectric / specular Dielectric / Conductor / Diffuse
C4 `many_lights_scene`     diffuse geometry + 10 k small emissive triangles (light-tree NEE)
C5 `large_scene`      ~10 M-triangle terrain with the C3 material mix

Everything is authoring-side (what Echo's Scene/Entity classes do on the host); only the flattened arrays cross the C ABI.
All randomness is a counter-based integer hash so C++/CUDA/Python agree on the inputs.
"""
import math

import numpy as np

from . import structs
from .host import SceneDescription

F32 = np.float32


# ---------------------------------------------------------------- hashing
def hash32(x):
    """The 32-bit mixer shared with the device sample sequence (csrc/echo_device_math.cuh)."""
    x = np.asarray(x, dtype=np.uint64) & 0xFFFFFFFF
    x ^= x >> 16
    x = (x * 0x7FEB352D) & 0xFFFFFFFF
    x ^= x >> 15
    x = (x * 0x846CA68B) & 0xFFFFFFFF
    x ^= x >> 16
    return x.astype(np.uint32)


def uniform(seed, index, dimension=0):
    """float32 in [0, 1) for (seed, index, dimension)."""
    index = np.asarray(index, dtype=np.uint64)
    h = hash32((index * 0x9E3779B1 + np.uint64(seed) * 0x85EBCA6B + np.uint64(dimension) * 0xC2B2AE35 + 0x165667B1) & 0xFFFFFFFF)
    h = hash32(h.astype(np.uint64) ^ 0x68E31DA4)
    return ((h >> 8).astype(np.float32) * F32(2.0 ** -24)).astype(np.float32)


# ---------------------------------------------------------------- authoring helpers
def rotation_matrix(angle_x, angle_y, angle_z):
    """Versor(x, y, z) in degrees -> 3x3 (Common/Mathematics/Primitives/Versor.cs:16-35,179-199; ZXY order)."""
    hx, hy, hz = (math.radians(a) * 0.5 for a in (angle_x, angle_y, angle_z))
    sx, cx, sy, cy, sz, cz = math.sin(hx), math.cos(hx), math.sin(hy), math.cos(hy), math.sin(hz), math.cos(hz)
    x = sx * cy * cz + cx * sy * sz
    y = cx * sy * cz - sx * cy * sz
    z = cx * cy * sz - sx * sy * cz
    w = cx * cy * cz + sx * sy * sz
    return np.array([
        [1 - 2 * y * y - 2 * z * z, 2 * x * y - 2 * z * w, 2 * x * z + 2 * y * w],
        [2 * x * y + 2 * z * w, 1 - 2 * x * x - 2 * z * z, 2 * y * z - 2 * x * w],
        [2 * x * z - 2 * y * w, 2 * y * z + 2 * x * w, 1 - 2 * x * x - 2 * y * y],
    ])


def make_triangles(v0, v1, v2, material, n0=None, n1=None, n2=None):
    """PreparedTriangle constructor (TriangleEntity.cs:59-116): flat normal unless shading normals are given."""
    v0, v1, v2 = (np.asarray(v, dtype=np.float32).reshape(-1, 3) for v in (v0, v1, v2))
    count = len(v0)
    triangles = np.zeros(count, dtype=structs.TRIANGLE)
    triangles["vertex0"] = v0
    triangles["edge1"] = v1 - v0
    triangles["edge2"] = v2 - v0

    if n0 is None:
        normal = np.cross(triangles["edge1"].astype(np.float64), triangles["edge2"].astype(np.float64))
        length = np.linalg.norm(normal, axis=1, keepdims=True)
        normal = np.where(length > 0, normal / np.maximum(length, 1e-300), np.array([0.0, 1.0, 0.0]))
        n0 = n1 = n2 = normal

    for key, n in (("normal0", n0), ("normal1", n1), ("normal2", n2)):
        n = np.asarray(n, dtype=np.float64).reshape(-1, 3)
        n = n / np.maximum(np.linalg.norm(n, axis=1, keepdims=True), 1e-300)
        triangles[key] = n.astype(np.float32)

    triangles["texcoord0"] = (0, 0)
    triangles["texcoord1"] = (0, 1)
    triangles["texcoord2"] = (1, 1)
    triangles["material"] = material
    return triangles


def plane(material, size, position=(0, 0, 0), rotation=(0, 0, 0)):
    """PlaneEntity.Extract (Scenic/Geometries/PlaneEntity.cs:46-59)."""
    ex, ez = size[0] / 2, size[1] / 2
    matrix = rotation_matrix(*rotation)
    local = np.array([[-ex, 0, -ez], [ex, 0, -ez], [-ex, 0, ez], [ex, 0, ez]], dtype=np.float64)
    p00, p01, p10, p11 = (local @ matrix.T + np.asarray(position, dtype=np.float64)).astype(np.float32)
    return make_triangles([p00, p00], [p10, p11], [p11, p01], material)


def box(material, size, position=(0, 0, 0), rotation=(0, 0, 0)):
    """BoxEntity.Extract (Scenic/Geometries/BoxEntity.cs:46-84), same triangle order."""
    extend = np.asarray(size, dtype=np.float64) / 2
    matrix = rotation_matrix(*rotation)

    def vertex(x, y, z):
        return (matrix @ (np.array([x, y, z]) * extend) + np.asarray(position, dtype=np.float64)).astype(np.float32)

    nnn, nnp, npn, npp = vertex(-1, -1, -1), vertex(-1, -1, 1), vertex(-1, 1, -1), vertex(-1, 1, 1)
    pnn, pnp, ppn, ppp = vertex(1, -1, -1), vertex(1, -1, 1), vertex(1, 1, -1), vertex(1, 1, 1)
    faces = [(pnn, ppp, pnp), (pnn, ppn, ppp), (nnp, npn, nnn), (nnp, npp, npn),
             (npn, ppp, ppn), (npn, npp, ppp), (pnn, nnp, nnn), (pnn, pnp, nnp),
             (pnp, npp, nnp), (pnp, ppp, npp), (nnn, ppn, pnn), (nnn, npn, ppn)]
    v0, v1, v2 = (np.array([f[i] for f in faces]) for i in range(3))
    return make_triangles(v0, v1, v2, material)


def material(kind, albedo=(1, 1, 1), alpha=1.0, roughness=(0, 0), ior=1.5, param_a=(1, 1, 1), param_b=(1, 1, 1), flags=0, base=0):
    m = np.zeros(1, dtype=structs.MATERIAL)
    m["type"], m["flags"], m["base"] = kind, flags, base
    m["albedo"] = (*albedo, alpha)
    m["roughness"], m["ior"] = roughness, ior
    m["paramA"], m["paramB"] = param_a, param_b
    return m


def coated_diffuse(albedo=(1, 1, 1), roughness=(0, 0), ior=1.5):
    """CoatedDiffuse (Evaluation/Materials/CoatedDiffuse.cs:13-55) with the reflectance its Prepare() caches."""
    from .host import fresnel_diffuse_reflectance
    reflectance = fresnel_diffuse_reflectance(np.float32(1.0) / np.float32(ior))
    return material(structs.MATERIAL_COATED_DIFFUSE, albedo, roughness=roughness, ior=ior, param_a=(reflectance, 0, 0))


def hex_color(value):
    """RGBA128.Parse("0xRRGGBB"): byte / 255, linear, no sRGB decode (Textures/Colors/RGBA128.Parser.cs:293-316)."""
    return tuple(np.float32(((value >> shift) & 0xFF) / 255.0) for shift in (16, 8, 0))


def perspective_camera(position, rotation=(0, 0, 0), field_of_view=65.0, lens_radius=0.01, focal_distance=0.0):
    """PerspectiveCamera (Scenic/Cameras/PerspectiveCamera.cs:25-48): forwardLength = 0.5 / tan(fov / 2)."""
    camera = np.zeros(1, dtype=structs.CAMERA)
    matrix = np.zeros((3, 4))
    matrix[:, :3] = rotation_matrix(*rotation)
    matrix[:, 3] = position
    camera["transform"] = matrix.reshape(-1).astype(np.float32)
    camera["forwardLength"] = F32(0.5) / F32(math.tan(math.radians(field_of_view) / 2))
    camera["lensRadius"] = lens_radius
    camera["focalDistance"] = focal_distance
    return camera


def orthographic_camera(position, rotation=(0, 0, 0), width=8.0):
    """OrthographicCamera (Scenic/Cameras/OrthographicCamera.cs:15-39): parallel rays along the camera's forward axis from a
    `width`-wide window."""
    camera = perspective_camera(position, rotation)
    matrix = rotation_matrix(*rotation)
    camera["type"], camera["width"] = structs.CAMERA_ORTHOGRAPHIC, width
    camera["direction"] = (matrix @ np.array([0.0, 0.0, 1.0])).astype(np.float32)  # RootedRotation * Float3.Forward
    return camera


def cylindrical_camera(position, rotation=(0, 0, 0)):
    """CylindricalCamera (Scenic/Cameras/CylindricalCamera.cs:12-34): a full latitude-longitude panorama around `position`."""
    camera = perspective_camera(position, rotation)
    camera["type"] = structs.CAMERA_CYLINDRICAL
    return camera


def look_rotation(position, target):
    """Euler angles (x, y) in degrees so the camera's +Z looks from position to target."""
    d = np.asarray(target, dtype=np.float64) - np.asarray(position, dtype=np.float64)
    yaw = math.degrees(math.atan2(d[0], d[2]))
    pitch = -math.degrees(math.atan2(d[1], math.hypot(d[0], d[2])))
    return (pitch, yaw, 0.0)


def ambient_light(radiance, directly_visible=True):
    light = np.zeros(1, dtype=structs.INFINITE_LIGHT)
    light["radiance"] = radiance
    light["directlyVisible"] = 1 if directly_visible else 0
    return light


# ---------------------------------------------------------------- C1
def environment_light(texture, intensity=(1, 1, 1), rotation=(0, 0, 0), directly_visible=True):
    """AmbientLight over a CylindricalTexture (Scenic/Lights/AmbientLight.cs, Textures/Directional/CylindricalTexture.cs):
    `texture` indexes SceneDescription.textures (a latitude-longitude map, v = 0 at the bottom)."""
    light = np.zeros(1, dtype=structs.INFINITE_LIGHT)
    matrix = rotation_matrix(*rotation)
    light["radiance"], light["directlyVisible"], light["type"] = intensity, 1 if directly_visible else 0, structs.INFINITE_ENVIRONMENT
    light["texture"] = texture
    light["rotation"] = matrix.astype(np.float32).reshape(-1)            # LocalToWorldRotation
    light["inverseRotation"] = matrix.T.astype(np.float32).reshape(-1)   # WorldToLocalRotation = (Float3x3)RootedRotation.Inverse
    return light


def cubemap_light(first_texture, intensity=(1, 1, 1), rotation=(0, 0, 0), directly_visible=True):
    """AmbientLight over a Cubemap (Textures/Directional/Cubemap.cs): SceneDescription.textures[first_texture : first_texture + 6]
    are its px, nx, py, ny, pz, nz faces."""
    light = environment_light(first_texture, intensity, rotation, directly_visible)
    light["type"] = structs.INFINITE_CUBEMAP
    return light


def directional_light(intensity, rotation=(0, 0, 0), angle=0.6, directly_visible=False):
    """DirectionalLight (Scenic/Lights/DirectionalLight.cs:12-75) with what its Prepare() computes: the light shines along its
    local backward axis, `angle` (degrees, default 0.6) is the half opening of the cone it is visible in; 0 makes it a delta light."""
    light = np.zeros(1, dtype=structs.INFINITE_LIGHT)
    matrix = rotation_matrix(*rotation).astype(np.float32)
    direction = matrix.astype(np.float64) @ np.array([0.0, 0.0, -1.0])  # Float3.Backward
    direction = direction / np.linalg.norm(direction)
    radians = np.float32(math.radians(angle))
    cos_angle = np.float32(math.cos(radians))                           # MathF.Cos
    is_delta = not (np.float32(1) - cos_angle >= np.float32(8e-7))      # !FastMath.Positive(1f - cosAngle)
    intensity = np.asarray(intensity, dtype=np.float32)

    if not is_delta:
        scale = np.float32(0.5) - np.float32(0.5) * np.float32(math.cos(radians * np.float32(2)))
        scaled = intensity / scale * np.float32(1 / math.pi)            # Intensity / scale * Scalars.PiR
    else:
        scaled = np.zeros(3, dtype=np.float32)

    light["radiance"], light["directlyVisible"] = scaled, 1 if directly_visible else 0
    light["type"], light["isDelta"], light["cosAngle"] = structs.INFINITE_DIRECTIONAL, 1 if is_delta else 0, cos_angle
    light["intensity"], light["direction"], light["rotation"] = intensity, direction.astype(np.float32), matrix.reshape(-1)
    return light


def cornell_box():
    """Scenic/CornellBox.cs:18-60 with the camera of ext/Scenes/Simple/cornell.echo:43 (FOV 42 at z = -18.025444)."""
    green, red, blue, white = (hex_color(v) for v in (0x00CB21, 0xCB0021, 0x0021CB, 0xEEEEF2))
    materials = np.concatenate([
        material(structs.MATERIAL_DIFFUSE, white),                                      # 0 white
        material(structs.MATERIAL_DIFFUSE, blue),                                       # 1 blue
        material(structs.MATERIAL_ONESIDED, flags=structs.MATERIAL_FLAG_BACKFACE, base=0),  # 2 cullable
        material(structs.MATERIAL_DIFFUSE, green),                                      # 3 green
        material(structs.MATERIAL_DIFFUSE, red),                                        # 4 red
        material(structs.MATERIAL_EMISSIVE, hex_color(0xFFFAF4)),                        # 5 light
    ])
    wall, wall5 = (10, 10), (5, 5)
    triangles = np.concatenate([
        plane(0, wall),                                        # floor
        plane(0, wall, (0, 10, 0), (180, 0, 0)),               # roof
        plane(1, wall, (0, 5, 5), (-90, 0, 0)),                # back
        plane(2, wall, (0, 5, -5), (90, 0, 0)),                # front
        plane(3, wall, (5, 5, 0), (0, 0, 90)),                 # right
        plane(4, wall, (-5, 5, 0), (0, 0, -90)),               # left
        plane(5, wall5, (0, 9.99, 0), (180, 0, 0)),            # light
        box(0, (3, 3, 3), (2, 1.5, -2), (0, 21, 0)),
        box(0, (3, 6, 3), (-2, 3, 2), (0, -21, 0)),
    ])
    camera = perspective_camera((0, 5, -18.025444), field_of_view=42.0)
    return SceneDescription(triangles=triangles, materials=materials, camera=camera, name="cornell")


# ---------------------------------------------------------------- terrain (C2 / C5)
def _value_noise(x, z, seed):
    xi, zi = np.floor(x).astype(np.int64), np.floor(z).astype(np.int64)
    fx, fz = x - xi, z - zi
    fx, fz = fx * fx * (3 - 2 * fx), fz * fz * (3 - 2 * fz)

    def lattice(ix, iz):
        return uniform(seed, (ix & 0xFFFF) * 65536 + (iz & 0xFFFF)).astype(np.float64)

    a, b = lattice(xi, zi), lattice(xi + 1, zi)
    c, d = lattice(xi, zi + 1), lattice(xi + 1, zi + 1)
    return (a + (b - a) * fx) * (1 - fz) + (c + (d - c) * fx) * fz


def fbm(x, z, seed=7, octaves=5):
    total, amplitude, frequency = np.zeros_like(x, dtype=np.float64), 0.5, 0.08
    for octave in range(octaves):
        total += amplitude * _value_noise(x * frequency + 100.0, z * frequency + 100.0, seed + octave)
        amplitude *= 0.5
        frequency *= 2.0
    return total


def terrain_triangles(quads_x, quads_z, material_index=0, extent=50.0, height=8.0, seed=7, smooth=False):
    """quads_x x quads_z quads (2 triangles each) over [-extent, extent]^2 with height * fbm(x, z)."""
    xs = np.linspace(-extent, extent, quads_x + 1)
    zs = np.linspace(-extent, extent, quads_z + 1)
    gx, gz = np.meshgrid(xs, zs, indexing="ij")
    gy = height * fbm(gx, gz, seed)
    points = np.stack([gx, gy, gz], axis=-1).astype(np.float32)

    p00 = points[:-1, :-1].reshape(-1, 3)
    p10 = points[1:, :-1].reshape(-1, 3)
    p01 = points[:-1, 1:].reshape(-1, 3)
    p11 = points[1:, 1:].reshape(-1, 3)

    normals = [None] * 6
    if smooth:
        dx = np.gradient(gy, xs, axis=0)
        dz = np.gradient(gy, zs, axis=1)
        n = np.stack([-dx, np.ones_like(dx), -dz], axis=-1)
        n00, n10 = n[:-1, :-1].reshape(-1, 3), n[1:, :-1].reshape(-1, 3)
        n01, n11 = n[:-1, 1:].reshape(-1, 3), n[1:, 1:].reshape(-1, 3)
        normals = [n00, n01, n11, n00, n11, n10]

    # winding so that the geometric normal points up (+Y): (p00, p01, p11) and (p00, p11, p10)
    first = make_triangles(p00, p01, p11, material_index, *normals[:3])
    second = make_triangles(p00, p11, p10, material_index, *normals[3:])
    triangles = np.empty(len(first) * 2, dtype=structs.TRIANGLE)
    triangles[0::2], triangles[1::2] = first, second
    return triangles


def terrain_scene(quads_x=1000, quads_z=500, sphere_count=10000, seed=7):
    """C2: 1 000 000 terrain triangles + 10 000 spheres r in [0.05, 0.5] hovering above (SURVEY.md §8d)."""
    materials = np.concatenate([material(structs.MATERIAL_DIFFUSE, (0.7, 0.7, 0.7)),
                                material(structs.MATERIAL_DIFFUSE, (0.8, 0.3, 0.2))])
    triangles = terrain_triangles(quads_x, quads_z, 0, seed=seed)

    index = np.arange(sphere_count)
    spheres = np.zeros(sphere_count, dtype=structs.SPHERE)
    x = (uniform(seed + 101, index, 0) * 2 - 1) * F32(48.0)
    z = (uniform(seed + 101, index, 1) * 2 - 1) * F32(48.0)
    y = (8.0 * fbm(x.astype(np.float64), z.astype(np.float64), seed)).astype(np.float32) + F32(0.6) + uniform(seed + 101, index, 2) * F32(6.0)
    spheres["position"] = np.stack([x, y, z], axis=-1)
    spheres["radius"] = F32(0.05) + uniform(seed + 101, index, 3) * F32(0.45)
    spheres["material"] = 1

    camera = perspective_camera((0, 30, -70), look_rotation((0, 30, -70), (0, 2, 0)), field_of_view=50.0)
    lights = ambient_light((0.8, 0.9, 1.0))
    return SceneDescription(triangles=triangles, spheres=spheres, materials=materials, infinite_lights=lights, camera=camera, name="terrain")


def uniform_sphere_directions(u, v):
    """Sample2D.UniformSphere (Evaluation/Sampling/Sample2D.cs:35,153-158) in float64, normalised in float32."""
    z = 1.0 - 2.0 * u.astype(np.float64)
    r = np.sqrt(np.maximum(0.0, 1.0 - z * z))
    phi = 2.0 * np.pi * v.astype(np.float64)
    d = np.stack([r * np.cos(phi), r * np.sin(phi), z], axis=-1)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d = d.astype(np.float32)
    # one float32 renormalisation pass keeps |d|^2 within 1 ulp of 1 (Ray's constructor asserts unit length, Ray.cs:21)
    d64 = d.astype(np.float64)
    return (d64 / np.linalg.norm(d64, axis=1, keepdims=True)).astype(np.float32)


def random_rays(bounds, count, seed=11, occlusion=False, start=0):
    """Fully incoherent batch: origin uniform in the scene AABB inflated 1.5x, direction uniform on the sphere.

    Closest-hit rays get distance = +inf; occlusion rays get travel uniform in [0, AABB diagonal] (SURVEY.md §8d, C2).
    """
    low, high = (np.asarray(b, dtype=np.float64) for b in bounds)
    center, half = (low + high) / 2, (high - low) / 2 * 1.5
    index = np.arange(start, start + count, dtype=np.uint64)
    rays = np.zeros(count, dtype=structs.RAY)
    jitter = np.stack([uniform(seed, index, k) for k in range(3)], axis=-1).astype(np.float64) * 2 - 1
    rays["origin"] = (center + jitter * half).astype(np.float32)
    rays["direction"] = uniform_sphere_directions(uniform(seed + 2, index, 0), uniform(seed + 2, index, 1))
    rays["ignore"] = structs.TOKEN_EMPTY
    if occlusion:
        diagonal = float(np.linalg.norm(high - low))
        rays["distance"] = uniform(seed + 6, index, 0) * F32(diagonal)
    else:
        rays["distance"] = np.inf
    return rays


def secondary_rays(prepared, primary, hits, seed=19):
    """Rays leaving the surfaces hit by `primary`: origin = hit position, cosine-hemisphere direction about the
    geometric normal, ignore = hit token — the self-intersection rule of TraceQuery.SpawnTrace (TraceQuery.cs:76-88)."""
    hit = hits["token"] != structs.TOKEN_EMPTY
    primary, hits = primary[hit], hits[hit]
    count = len(primary)
    distance = np.maximum(hits["distance"], F32(8e-7))
    origin = primary["direction"] * distance[:, None] + primary["origin"]

    kind = structs.token_type(hits["token"])
    index = structs.token_index(hits["token"])
    normal = np.zeros((count, 3), dtype=np.float64)
    tri = kind == structs.TOKEN_TYPE_TRIANGLE
    t = prepared.triangles[index[tri]]
    normal[tri] = np.cross(t["edge1"].astype(np.float64), t["edge2"].astype(np.float64))
    sph = kind == structs.TOKEN_TYPE_SPHERE
    s = prepared.spheres[index[sph]]
    normal[sph] = origin[sph].astype(np.float64) - s["position"].astype(np.float64)
    normal /= np.maximum(np.linalg.norm(normal, axis=1, keepdims=True), 1e-300)
    facing = np.sum(normal * primary["direction"].astype(np.float64), axis=1) > 0
    normal[facing] *= -1

    i = np.arange(count, dtype=np.uint64)
    u, v = uniform(seed, i, 0).astype(np.float64), uniform(seed, i, 1).astype(np.float64)
    r, phi = np.sqrt(u), 2 * np.pi * v
    local = np.stack([r * np.cos(phi), r * np.sin(phi), np.sqrt(np.maximum(0.0, 1 - u))], axis=-1)
    helper = np.where(np.abs(normal[:, :1]) > 0.9, np.array([[0.0, 1.0, 0.0]]), np.array([[1.0, 0.0, 0.0]]))
    tangent = np.cross(helper, normal)
    tangent /= np.linalg.norm(tangent, axis=1, keepdims=True)
    bitangent = np.cross(normal, tangent)
    d = local[:, :1] * tangent + local[:, 1:2] * bitangent + local[:, 2:] * normal
    d /= np.linalg.norm(d, axis=1, keepdims=True)

    rays = np.zeros(count, dtype=structs.RAY)
    rays["origin"] = origin
    rays["direction"] = d.astype(np.float32)
    rays["distance"] = np.inf
    rays["ignore"] = hits["token"]
    return rays


# ---------------------------------------------------------------- C3 / C4 / C5
def blob_triangles(center, radius, material_index, rings=128, segments=128, seed=3):
    """A tessellated, smoothly displaced sphere with per-vertex shading normals (2 * rings * segments triangles)."""
    theta = np.linspace(0, np.pi, rings + 1)
    phi = np.linspace(0, 2 * np.pi, segments + 1)
    t, p = np.meshgrid(theta, phi, indexing="ij")
    direction = np.stack([np.sin(t) * np.cos(p), np.cos(t), np.sin(t) * np.sin(p)], axis=-1)
    bump = 1.0 + 0.12 * np.sin(3 * t + seed) * np.cos(4 * p) + 0.06 * np.cos(7 * t) * np.sin(5 * p + seed)
    points = direction * (radius * bump)[..., None]

    # shading normals from the displaced surface's tangents (analytic enough for a smooth blob)
    dt = np.gradient(points, theta, axis=0)
    dp = np.gradient(points, phi, axis=1)
    normals = np.cross(dp, dt)
    length = np.linalg.norm(normals, axis=-1, keepdims=True)
    normals = np.where(length > 1e-9, normals / np.maximum(length, 1e-300), direction)
    normals = np.where(np.sum(normals * direction, axis=-1, keepdims=True) < 0, -normals, normals)
    points = points + np.asarray(center, dtype=np.float64)

    def grid(a, i0, i1, j0, j1):
        return a[i0:i1, j0:j1].reshape(-1, 3)

    r, s = rings, segments
    p00, p10, p01, p11 = grid(points, 0, r, 0, s), grid(points, 1, r + 1, 0, s), grid(points, 0, r, 1, s + 1), grid(points, 1, r + 1, 1, s + 1)
    n00, n10, n01, n11 = grid(normals, 0, r, 0, s), grid(normals, 1, r + 1, 0, s), grid(normals, 0, r, 1, s + 1), grid(normals, 1, r + 1, 1, s + 1)

    first = make_triangles(p00, p01, p11, material_index, n00, n01, n11)
    second = make_triangles(p00, p11, p10, material_index, n00, n11, n10)
    triangles = np.concatenate([first, second])

    # drop the degenerate triangles at the poles
    area = np.linalg.norm(np.cross(triangles["edge1"].astype(np.float64), triangles["edge2"].astype(np.float64)), axis=1)
    return triangles[area > 1e-12]


def mixed_materials():
    """The C3 swatch: Oren-Nayar ground (bunny.echo:6), rough and specular Dielectric, artistic Conductor (bunny.echo:12-23), Diffuse, Emissive."""
    return np.concatenate([
        material(structs.MATERIAL_DIFFUSE, (0.75, 0.75, 0.75), roughness=(0.7, 0.7)),                        # 0 Oren-Nayar ground
        material(structs.MATERIAL_DIELECTRIC, (1, 1, 1), roughness=(0.1, 0.1), ior=1.5),                     # 1 rough glass
        material(structs.MATERIAL_DIELECTRIC, (1, 1, 1), roughness=(0, 0), ior=1.5),                         # 2 specular glass
        material(structs.MATERIAL_CONDUCTOR, (1, 1, 1), roughness=(0.05, 0.25), param_a=(0.6, 0.7, 0.9),
                 param_b=(0.0, 1.0, 0.5), flags=structs.MATERIAL_FLAG_ARTISTIC),                              # 3 conductor
        material(structs.MATERIAL_DIFFUSE, (0.8, 0.25, 0.2)),                                                # 4 Lambertian
        material(structs.MATERIAL_EMISSIVE, (12.0, 11.0, 9.5)),                                              # 5 emissive quad
        material(structs.MATERIAL_EMISSIVE, (6.0, 7.0, 9.0)),                                                # 6 emissive sphere
    ])


def mixed_material_scene(rings=128, segments=130):
    """C3: ground + 3x3 blobs (~300 k triangles) cycling four materials, one emissive quad + one emissive sphere, ambient 0.05."""
    materials = mixed_materials()
    parts = [plane(0, (60, 60))]
    cycle = [1, 2, 3, 4]
    k = 0
    for ix in range(3):
        for iz in range(3):
            center = ((ix - 1) * 6.0, 2.2, (iz - 1) * 6.0)
            parts.append(blob_triangles(center, 2.0, cycle[k % 4], rings, segments, seed=k))
            k += 1
    parts.append(plane(5, (6, 6), (0, 14, 0), (180, 0, 0)))
    triangles = np.concatenate(parts)

    spheres = np.zeros(1, dtype=structs.SPHERE)
    spheres["position"], spheres["radius"], spheres["material"] = (-11, 5, -4), 1.5, 6

    position = (0.0, 9.0, -22.0)
    camera = perspective_camera(position, look_rotation(position, (0, 2, 0)), field_of_view=45.0)
    return SceneDescription(triangles=triangles, spheres=spheres, materials=materials, infinite_lights=ambient_light((0.05, 0.05, 0.05)),
                            camera=camera, name="mixed")


def instanced_scene(grid=6, rings=24, segments=26, nested=True):
    """SURVEY.md 8f rank 2: a ground plane plus `grid` x `grid` placements of two packs with different rotations and uniform
    scales. Pack 0 is a blob with two spheres; pack 1 ("cluster") holds a box and three placements of pack 0, so hits inside it
    carry two instance layers. Every third placement overrides the pack's swatch (PackInstance materials)."""
    from .host import InstanceDescription, PackDescription
    blob_materials = np.concatenate([material(structs.MATERIAL_DIFFUSE, (0.8, 0.3, 0.25)), material(structs.MATERIAL_CONDUCTOR, (1, 1, 1), roughness=(0.1, 0.1),
                                    param_a=(0.9, 0.8, 0.5), param_b=(1.0, 0.9, 0.7), flags=structs.MATERIAL_FLAG_ARTISTIC),
                                    material(structs.MATERIAL_EMISSIVE, (6.0, 4.0, 2.0))])
    blob_spheres = np.zeros(2, dtype=structs.SPHERE)
    blob_spheres["position"], blob_spheres["radius"], blob_spheres["material"] = [(1.4, 0.3, 0.0), (-0.4, 1.5, 0.6)], [0.35, 0.25], [1, 2]  # the second one glows
    blob = PackDescription(triangles=blob_triangles((0, 0, 0), 1.0, 0, rings, segments, seed=5), spheres=blob_spheres, materials=blob_materials)

    cluster_materials = material(structs.MATERIAL_DIFFUSE, (0.3, 0.6, 0.8), roughness=(0.5, 0.5))
    cluster_light = np.zeros(1, dtype=structs.POINT_LIGHT)
    cluster_light["intensity"], cluster_light["position"] = (3.0, 3.0, 4.0), (0.0, 1.8, 0.0)
    cluster = PackDescription(triangles=box(0, (1.2, 0.4, 1.2), (0, -0.9, 0)), materials=cluster_materials, point_lights=cluster_light,
                              instances=[InstanceDescription(0, (-1.3, 0.4, 0.0), (0, 30, 0), 0.5), InstanceDescription(0, (1.3, 0.4, 0.2), (20, 0, 45), 0.45),
                                         InstanceDescription(0, (0.0, 0.6, 1.4), (0, 200, 10), 0.4)])
    override = np.concatenate([material(structs.MATERIAL_DIELECTRIC, (1, 1, 1), roughness=(0.05, 0.05), ior=1.5), material(structs.MATERIAL_DIFFUSE, (0.2, 0.8, 0.3)),
                               material(structs.MATERIAL_EMISSIVE, (6.0, 4.0, 2.0))])

    instances = []
    k = 0
    for ix in range(grid):
        for iz in range(grid):
            position = ((ix - (grid - 1) / 2) * 4.0, 1.4 + 0.3 * ((ix * 7 + iz * 3) % 5), (iz - (grid - 1) / 2) * 4.0)
            rotation = ((ix * 37) % 360, (iz * 53 + ix * 11) % 360, (k * 29) % 360)
            scale = 0.6 + 0.15 * ((ix + 2 * iz) % 5)
            pack = 1 if nested and k % 2 == 1 else 0
            instances.append(InstanceDescription(pack, position, rotation, scale, override if k % 3 == 0 and pack == 0 else None))
            k += 1

    materials = np.concatenate([material(structs.MATERIAL_DIFFUSE, (0.7, 0.7, 0.7)), material(structs.MATERIAL_EMISSIVE, (10.0, 9.0, 8.0))])
    extent = grid * 4.0 + 8.0
    triangles = np.concatenate([plane(0, (extent, extent)), plane(1, (extent / 3, extent / 3), (0, 9, 0), (180, 0, 0))])
    spheres = np.zeros(1, dtype=structs.SPHERE)
    spheres["position"], spheres["radius"], spheres["material"] = (0, 3.5, 0), 0.8, 0

    position = (0.0, 9.0, -extent * 0.75)
    camera = perspective_camera(position, look_rotation(position, (0, 1, 0)), field_of_view=50.0)
    return SceneDescription(triangles=triangles, spheres=spheres, materials=materials, instances=instances, packs=[blob, cluster],
                            infinite_lights=ambient_light((0.3, 0.35, 0.4)), camera=camera, name="instanced")


def many_packs_scene(pack_count=40, seed=1, layers=3):
    """Many distinct packs placed in `layers` (2 or 3) layers: the input of a build that serves all packs of one height together
    (echo_b200_build_packs). Packs of the bottom layer are small blobs, some with glowing triangles or spheres, some without any
    emitter, some lit by point lights only; packs of the layers above hold two to four placements of the layer below, some of them
    nothing else. The scene places every top-layer pack, so host.prepare keeps them all."""
    from .host import InstanceDescription, PackDescription
    rng = np.random.default_rng(seed)
    layers = max(2, min(3, int(layers)))
    sizes = [pack_count // 2 + pack_count % 2] + [pack_count // (2 * (layers - 1))] * (layers - 1)
    sizes[-1] += pack_count - sum(sizes)
    glow = material(structs.MATERIAL_EMISSIVE, (5.0, 4.0, 3.0))
    packs, previous = [], []

    def placement(candidates):
        position = tuple(rng.uniform(-3.0, 3.0, 3))
        rotation = tuple(float(v) for v in rng.integers(0, 360, 3))
        return InstanceDescription(int(rng.choice(candidates)), position, rotation, float(rng.uniform(0.3, 0.8)))

    for k in range(sizes[0]):
        kind = k % 4  # 0: glowing triangles, 1: glowing sphere, 2: no emitter, 3: point lights only
        materials = np.concatenate([material(structs.MATERIAL_DIFFUSE, tuple(rng.uniform(0.2, 0.9, 3))), glow])
        triangles = blob_triangles(tuple(rng.uniform(-1, 1, 3)), float(rng.uniform(0.5, 1.5)), 0, 4 + k % 5, 5 + k % 4, seed=seed * 1000 + k)
        if kind == 0:
            triangles["material"][::7] = 1
        spheres = np.zeros(1 + k % 3, dtype=structs.SPHERE)
        spheres["position"] = rng.uniform(-1.5, 1.5, (len(spheres), 3))
        spheres["radius"] = rng.uniform(0.1, 0.4, len(spheres))
        spheres["material"] = 1 if kind == 1 else 0
        points = np.zeros(1 + k % 2 if kind == 3 else 0, dtype=structs.POINT_LIGHT)
        points["position"], points["intensity"] = rng.uniform(-2, 2, (len(points), 3)), (2.0, 2.0, 2.5)
        packs.append(PackDescription(triangles=triangles, spheres=spheres, materials=materials, point_lights=points))
        previous.append(len(packs) - 1)

    for layer in range(1, layers):
        current = []
        for k in range(sizes[layer]):
            instances = [placement(previous) for _ in range(2 + k % 3)]
            if k % 2 == 0:  # placements only
                packs.append(PackDescription(instances=instances))
            else:
                packs.append(PackDescription(triangles=box(0, tuple(rng.uniform(0.3, 1.0, 3)), tuple(rng.uniform(-1, 1, 3))),
                                             materials=material(structs.MATERIAL_DIFFUSE, (0.6, 0.6, 0.6)), instances=instances))
            current.append(len(packs) - 1)
        previous = current

    used = set()
    for pack in packs:
        used.update(instance.pack for instance in pack.instances)
    roots = [index for index in range(len(packs)) if index not in used]
    instances = []
    for k, index in enumerate(roots):
        position = ((k % 8 - 3.5) * 8.0, 2.0, (k // 8 - 3.0) * 8.0)
        instances.append(InstanceDescription(index, position, (0.0, float((k * 37) % 360), 0.0), 1.0))

    materials = np.concatenate([material(structs.MATERIAL_DIFFUSE, (0.7, 0.7, 0.7)), material(structs.MATERIAL_EMISSIVE, (8.0, 8.0, 7.0))])
    extent = 80.0
    triangles = np.concatenate([plane(0, (extent, extent)), plane(1, (10.0, 10.0), (0, 20, 0), (180, 0, 0))])
    position = (0.0, 30.0, -60.0)
    camera = perspective_camera(position, look_rotation(position, (0, 0, 0)), field_of_view=60.0)
    return SceneDescription(triangles=triangles, materials=materials, instances=instances, packs=packs,
                            infinite_lights=ambient_light((0.2, 0.2, 0.25)), camera=camera, name="many_packs")


def _planar_texcoords(triangles, scale, axes=(0, 2)):
    """Texture coordinates from two position axes (a planar projection), `scale` repeats per unit."""
    v0 = triangles["vertex0"].astype(np.float64)
    v1, v2 = v0 + triangles["edge1"], v0 + triangles["edge2"]
    for key, v in (("texcoord0", v0), ("texcoord1", v1), ("texcoord2", v2)):
        triangles[key] = (v[:, list(axes)] * scale).astype(np.float32)
    return triangles


def textured_scene(rings=24, segments=26):
    """SURVEY.md 8f rank 3: image textures in every material slot — a point-filtered repeating checker on the ground, bilinear
    albedo + tangent-space normal map on a diffuse blob, roughness and main-colour maps on a conductor, a roughness map on
    rough glass, a mirrored albedo map on a sphere (sphere texture coordinates) and an alpha cut-out quad."""
    from .host import TextureDescription
    rng = np.random.default_rng(17)

    def grid(height, width):
        y, x = np.meshgrid((np.arange(height) + 0.5) / height, (np.arange(width) + 0.5) / width, indexing="ij")
        return x, y

    x, y = grid(8, 8)
    checker = np.where(((np.floor(x * 8) + np.floor(y * 8)) % 2 == 0)[..., None], [0.85, 0.85, 0.8, 1.0], [0.15, 0.2, 0.3, 1.0])
    x, y = grid(48, 64)
    marble = np.stack([0.5 + 0.4 * np.sin(9 * x + 4 * np.sin(7 * y)), 0.45 + 0.3 * np.cos(5 * y + 2 * x), 0.4 + 0.35 * np.sin(6 * (x + y)), np.ones_like(x)], axis=-1)
    bumps = np.stack([0.5 + 0.35 * np.sin(25 * x), 0.5 + 0.35 * np.cos(19 * y), 0.9 + 0.1 * np.sin(7 * x * y), np.ones_like(x)], axis=-1)
    x, y = grid(32, 32)
    rough = np.stack([0.05 + 0.5 * x, 0.05 + 0.5 * y, np.zeros_like(x), np.ones_like(x)], axis=-1)
    tint = np.stack([0.55 + 0.4 * x, 0.6 + 0.3 * y, 0.95 - 0.5 * x * y, np.ones_like(x)], axis=-1)
    stripes = np.stack([0.9 * np.ones_like(x), 0.5 + 0.4 * np.sin(12 * y), 0.2 + 0.2 * x, np.ones_like(x)], axis=-1)
    cutout = np.concatenate([rng.uniform(0.2, 0.9, (16, 16, 3)), (rng.uniform(0, 1, (16, 16, 1)) > 0.45).astype(np.float64)], axis=-1)

    textures = [TextureDescription(checker, structs.FILTER_POINT, structs.WRAPPER_REPEAT),     # 0
                TextureDescription(marble, structs.FILTER_BILINEAR, structs.WRAPPER_MIRROR),   # 1
                TextureDescription(bumps, structs.FILTER_BILINEAR, structs.WRAPPER_REPEAT),    # 2
                TextureDescription(rough, structs.FILTER_BILINEAR, structs.WRAPPER_CLAMP),     # 3
                TextureDescription(tint, structs.FILTER_BILINEAR, structs.WRAPPER_REPEAT),     # 4
                TextureDescription(stripes, structs.FILTER_BILINEAR, structs.WRAPPER_MIRROR),  # 5
                TextureDescription(cutout, structs.FILTER_POINT, structs.WRAPPER_CLAMP)]       # 6

    materials = np.concatenate([
        material(structs.MATERIAL_DIFFUSE, (1, 1, 1), roughness=(0.4, 0.4)),                                  # 0 ground: checker albedo
        material(structs.MATERIAL_DIFFUSE, (1, 1, 1)),                                                        # 1 marble albedo + normal map
        material(structs.MATERIAL_CONDUCTOR, (1, 1, 1), roughness=(0.2, 0.2), param_a=(0.9, 0.8, 0.6), param_b=(1.0, 0.9, 0.8),
                 flags=structs.MATERIAL_FLAG_ARTISTIC),                                                       # 2 roughness + main colour maps
        material(structs.MATERIAL_DIELECTRIC, (1, 1, 1), roughness=(0.1, 0.1), ior=1.5),                      # 3 roughness map
        material(structs.MATERIAL_DIFFUSE, (1, 1, 1)),                                                        # 4 sphere: striped albedo
        material(structs.MATERIAL_DIFFUSE, (1, 1, 1)),                                                        # 5 alpha cut-out quad
        material(structs.MATERIAL_EMISSIVE, (14.0, 13.0, 11.0)),                                              # 6 light
        material(structs.MATERIAL_COATED_DIFFUSE, (1, 1, 1), roughness=(0.1, 0.3), ior=1.5,
                 param_a=(coated_diffuse()["paramA"][0][0], 0, 0)),                                           # 7 coated: marble albedo + roughness map
    ])
    slots = structs.material_textures(len(materials))
    slots["albedo"][[0, 1, 4, 5, 7]] = [0, 1, 5, 6, 1]
    slots["normal"][1], slots["normalIntensity"][1] = 2, 0.6
    slots["roughness"][[2, 3, 7]] = 3
    slots["paramA"][2] = 4

    parts = [_planar_texcoords(plane(0, (40, 40)), 0.5),
             _planar_texcoords(blob_triangles((-4.5, 2.0, 0.0), 1.8, 1, rings, segments, seed=1), 0.3, (0, 1)),
             _planar_texcoords(blob_triangles((0.0, 2.0, 2.0), 1.8, 2, rings, segments, seed=2), 0.25, (0, 1)),
             _planar_texcoords(blob_triangles((4.5, 2.0, 0.0), 1.8, 3, rings, segments, seed=3), 0.25, (1, 2)),
             _planar_texcoords(blob_triangles((0.0, 1.4, -4.0), 1.2, 7, rings, segments, seed=4), 0.4, (0, 1)),
             _planar_texcoords(plane(5, (3, 3), (2.4, 1.6, -5.0), (90, 0, 0)), 0.33, (0, 1)),
             plane(6, (5, 5), (0, 11, 0), (180, 0, 0))]
    triangles = np.concatenate(parts)

    spheres = np.zeros(2, dtype=structs.SPHERE)
    spheres["position"], spheres["radius"], spheres["material"] = [(-2.4, 0.9, -5.5), (-6.0, 0.8, -4.5)], [0.9, 0.8], [4, 4]

    position = (0.0, 6.5, -15.0)
    camera = perspective_camera(position, look_rotation(position, (0, 1.5, 0)), field_of_view=50.0)
    return SceneDescription(triangles=triangles, spheres=spheres, materials=materials, infinite_lights=ambient_light((0.25, 0.28, 0.35)),
                            camera=camera, textures=textures, material_textures=slots, name="textured")


def many_lights_scene(light_count=10000, rings=128, segments=130, seed=23):
    """C4: the C3 geometry, diffuse only, plus `light_count` small emissive triangles in a 60 x 20 x 60 volume."""
    base_materials = np.concatenate([
        material(structs.MATERIAL_DIFFUSE, (0.75, 0.75, 0.75), roughness=(0.7, 0.7)),
        material(structs.MATERIAL_DIFFUSE, (0.7, 0.7, 0.72)),
    ])
    palette = 16
    i = np.arange(palette)
    emissive = np.concatenate([
        material(structs.MATERIAL_EMISSIVE, tuple(float(F32(5.0) + uniform(seed + 1, k, c) * F32(45.0)) for c in range(3))) for k in i
    ])
    materials = np.concatenate([base_materials, emissive])

    parts = [plane(0, (60, 60))]
    k = 0
    for ix in range(3):
        for iz in range(3):
            parts.append(blob_triangles(((ix - 1) * 6.0, 2.2, (iz - 1) * 6.0), 2.0, 1, rings, segments, seed=k))
            k += 1

    j = np.arange(light_count, dtype=np.uint64)
    center = np.stack([(uniform(seed, j, 0) * 2 - 1) * F32(30.0), F32(1.0) + uniform(seed, j, 1) * F32(19.0), (uniform(seed, j, 2) * 2 - 1) * F32(30.0)], axis=-1)
    axis_a = uniform_sphere_directions(uniform(seed, j, 3), uniform(seed, j, 4)).astype(np.float64)
    helper = uniform_sphere_directions(uniform(seed, j, 5), uniform(seed, j, 6)).astype(np.float64)
    axis_b = np.cross(axis_a, helper)
    axis_b /= np.maximum(np.linalg.norm(axis_b, axis=1, keepdims=True), 1e-12)
    area = 0.01 + uniform(seed, j, 7).astype(np.float64) * 0.03
    side = np.sqrt(2 * area)[:, None]
    v0 = center.astype(np.float64)
    lights = make_triangles(v0, v0 + axis_a * side, v0 + axis_b * side, 2 + (hash32(j + 77) % palette))
    parts.append(lights)
    triangles = np.concatenate(parts)

    position = (0.0, 9.0, -22.0)
    camera = perspective_camera(position, look_rotation(position, (0, 2, 0)), field_of_view=45.0)
    return SceneDescription(triangles=triangles, materials=materials, camera=camera, name="many_lights")


def large_scene(quads_x=3162, quads_z=1581):
    """C5: the C2 terrain refined to ~10 M triangles with the C3 material mix in bands, one sun-like emissive quad, ambient sky."""
    materials = mixed_materials()
    triangles = terrain_triangles(quads_x, quads_z, 0, smooth=True)
    band = (np.arange(len(triangles)) // (2 * quads_z * 64)) % 5
    triangles["material"] = np.array([0, 4, 3, 1, 0], dtype=np.uint32)[band]
    light = plane(5, (40, 40), (0, 60, 0), (180, 0, 0))
    triangles = np.concatenate([triangles, light])

    index = np.arange(2000)
    spheres = np.zeros(len(index), dtype=structs.SPHERE)
    x = (uniform(301, index, 0) * 2 - 1) * F32(48.0)
    z = (uniform(301, index, 1) * 2 - 1) * F32(48.0)
    y = (8.0 * fbm(x.astype(np.float64), z.astype(np.float64), 7)).astype(np.float32) + F32(1.2)
    spheres["position"] = np.stack([x, y, z], axis=-1)
    spheres["radius"] = F32(0.3) + uniform(301, index, 3) * F32(0.7)
    spheres["material"] = np.array([2, 3, 1, 4], dtype=np.uint32)[index % 4]

    position = (0.0, 28.0, -66.0)
    camera = perspective_camera(position, look_rotation(position, (0, 2, 0)), field_of_view=50.0)
    return SceneDescription(triangles=triangles, spheres=spheres, materials=materials, infinite_lights=ambient_light((0.35, 0.4, 0.5)),
                            camera=camera, name="large")


def tile_grid(width, height, tile_size):
    """All tile positions of a RenderTexture, row-major (RenderTexture tiles, Textures/Evaluation/RenderTexture.cs)."""
    tiles_x = (width + tile_size - 1) // tile_size
    tiles_y = (height + tile_size - 1) // tile_size
    ty, tx = np.meshgrid(np.arange(tiles_y), np.arange(tiles_x), indexing="ij")
    return np.stack([tx.reshape(-1), ty.reshape(-1)], axis=-1).astype(np.int32)


def assemble_tiles(tiles_rgba, tile_xy, width, height, tile_size):
    """Tile-major Float4 output of render_tiles -> (height, width, 4) image, row 0 at the bottom like Echo's textures."""
    image = np.zeros((height, width, 4), dtype=np.float32)
    tiles = np.asarray(tiles_rgba, dtype=np.float32).reshape(-1, tile_size, tile_size, 4)
    for tile, (tx, ty) in zip(tiles, tile_xy):
        x0, y0 = tx * tile_size, ty * tile_size
        w, h = min(tile_size, width - x0), min(tile_size, height - y0)
        image[y0:y0 + h, x0:x0 + w] = tile[:h, :w]
    return image
