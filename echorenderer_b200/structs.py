"""numpy mirrors of the POD structs in include/echo_b200.h (byte-identical layouts; sizes asserted below).

The C# originals these follow are cited in the header: QuadBoundingVolumeHierarchy.Node (128 B), PreparedTriangle
(100 B), PreparedSphere (20 B), Ray + TraceQuery inputs (32 B) and TraceQuery outputs (16 B).
"""
import numpy as np

TOKEN_TYPE_NODE = 0
TOKEN_TYPE_TRIANGLE = 1
TOKEN_TYPE_SPHERE = 2
TOKEN_TYPE_INSTANCE = 3
TOKEN_TYPE_LIGHT = 4
TOKEN_EMPTY = 0xFFFFFFFF
TOKEN_INDEX_BITS = 28
LIGHT_TYPE_INFINITE = 0
LIGHT_TYPE_INFINITE_DELTA = 1
LIGHT_TYPE_POINT = 2
LIGHT_INDEX_BITS = 22

MATERIAL_DIFFUSE = 0
MATERIAL_DIELECTRIC = 1
MATERIAL_CONDUCTOR = 2
MATERIAL_EMISSIVE = 3
MATERIAL_ONESIDED = 4
MATERIAL_INVISIBLE = 5
MATERIAL_COATED_DIFFUSE = 6
MATERIAL_FLAG_TRANSMISSIVE = 1
MATERIAL_FLAG_ARTISTIC = 2
MATERIAL_FLAG_BACKFACE = 4


def make_token(token_type, index):
    return np.uint32((int(token_type) << TOKEN_INDEX_BITS) | int(index))


def token_type(token):
    return np.asarray(token, dtype=np.uint32) >> TOKEN_INDEX_BITS


def token_index(token):
    return np.asarray(token, dtype=np.uint32) & np.uint32((1 << TOKEN_INDEX_BITS) - 1)


QBVH_NODE = np.dtype([
    ("minX", "<f4", 4), ("minY", "<f4", 4), ("minZ", "<f4", 4),
    ("maxX", "<f4", 4), ("maxY", "<f4", 4), ("maxZ", "<f4", 4),
    ("axisMajor", "<i4"), ("axisMinor0", "<i4"), ("axisMinor1", "<i4"),
    ("token4", "<u4", 4), ("pad", "<u4"),
])

TRIANGLE = np.dtype([
    ("vertex0", "<f4", 3), ("edge1", "<f4", 3), ("edge2", "<f4", 3),
    ("normal0", "<f4", 3), ("normal1", "<f4", 3), ("normal2", "<f4", 3),
    ("texcoord0", "<f4", 2), ("texcoord1", "<f4", 2), ("texcoord2", "<f4", 2),
    ("material", "<u4"),
])

SPHERE = np.dtype([("position", "<f4", 3), ("radius", "<f4"), ("material", "<u4")])

RAY = np.dtype([("origin", "<f4", 3), ("direction", "<f4", 3), ("distance", "<f4"), ("ignore", "<u4")])

HIT = np.dtype([("token", "<u4"), ("distance", "<f4"), ("uv", "<f4", 2)])

MAX_INSTANCE_LAYERS = 5  # TokenHierarchy.MaxLayer
PACK = np.dtype([("nodeOffset", "<u4"), ("nodeCount", "<u4"), ("maxDepth", "<u4"), ("triangleOffset", "<u4"), ("triangleCount", "<u4"),
                 ("sphereOffset", "<u4"), ("sphereCount", "<u4"), ("instanceOffset", "<u4"), ("instanceCount", "<u4"), ("materialOffset", "<u4"),
                 ("lightNodeOffset", "<u4"), ("lightNodeCount", "<u4"), ("emitterOffset", "<u4"), ("emitterCount", "<u4"),
                 ("pointLightOffset", "<u4"), ("pointLightCount", "<u4")])
INSTANCE = np.dtype([("forward", "<f4", 12), ("inverse", "<f4", 12), ("forwardScale", "<f4"), ("inverseScale", "<f4"), ("pack", "<u4"),
                     ("materialOffset", "<u4"), ("reserved", "<u4", 4)])
TOKEN_HIERARCHY = np.dtype([("instanceCount", "<u4"), ("instances", "<u4", MAX_INSTANCE_LAYERS)])

MATERIAL = np.dtype([
    ("type", "<u4"), ("flags", "<u4"), ("albedo", "<f4", 4), ("roughness", "<f4", 2), ("ior", "<f4"),
    ("paramA", "<f4", 3), ("paramB", "<f4", 3), ("base", "<u4"),
])

TEXTURE_NONE = 0xFFFFFFFF
FILTER_POINT, FILTER_BILINEAR = 0, 1
WRAPPER_CLAMP, WRAPPER_REPEAT, WRAPPER_MIRROR = 0, 1, 2
TEXTURE = np.dtype([("width", "<u4"), ("height", "<u4"), ("texelOffset", "<u4"), ("filter", "<u4"), ("wrapper", "<u4"), ("reserved", "<u4", 3)])
MATERIAL_TEXTURES = np.dtype([("albedo", "<u4"), ("normal", "<u4"), ("roughness", "<u4"), ("paramA", "<u4"), ("paramB", "<u4"), ("normalIntensity", "<f4"),
                              ("reserved", "<u4", 2)])


def material_textures(count, **slots):
    """`count` EchoMaterialTextures records with every slot empty (NormalIntensity 0.25, Material.cs:54)."""
    records = np.zeros(count, dtype=MATERIAL_TEXTURES)
    for name in ("albedo", "normal", "roughness", "paramA", "paramB"):
        records[name] = TEXTURE_NONE
    records["normalIntensity"] = 0.25
    return records


LIGHT_NODE = np.dtype([
    ("boxMin", "<f4", 3), ("boxMax", "<f4", 3), ("coneAxis", "<f4", 3), ("cosOffset", "<f4"), ("cosExtend", "<f4"),
    ("power", "<f4"), ("child0", "<u4"), ("child1", "<u4"), ("pad", "<u4", 2),
])

POINT_LIGHT = np.dtype([("intensity", "<f4", 3), ("position", "<f4", 3)])

INFINITE_AMBIENT, INFINITE_DIRECTIONAL, INFINITE_ENVIRONMENT, INFINITE_CUBEMAP = 0, 1, 2, 3
INFINITE_LIGHT = np.dtype([("radiance", "<f4", 3), ("directlyVisible", "<u4"), ("type", "<u4"), ("isDelta", "<u4"), ("cosAngle", "<f4"), ("pad0", "<f4"),
                           ("intensity", "<f4", 3), ("pad1", "<f4"), ("direction", "<f4", 3), ("pad2", "<f4"), ("rotation", "<f4", 9), ("texture", "<u4"), ("distribution", "<u4"), ("pad3", "<f4"),
                           ("inverseRotation", "<f4", 9), ("pad4", "<f4", 3)])

CAMERA_PERSPECTIVE, CAMERA_ORTHOGRAPHIC, CAMERA_CYLINDRICAL = 0, 1, 2
CAMERA = np.dtype([("transform", "<f4", 12), ("forwardLength", "<f4"), ("lensRadius", "<f4"), ("focalDistance", "<f4"), ("type", "<u4"),
                   ("direction", "<f4", 3), ("width", "<f4")])

RENDER_PARAMS = np.dtype([
    ("width", "<i4"), ("height", "<i4"), ("tileSize", "<i4"), ("extend", "<i4"), ("minEpoch", "<i4"), ("maxEpoch", "<i4"),
    ("noiseThreshold", "<f4"), ("bounceLimit", "<i4"), ("survivability", "<f4"), ("seed", "<u4"), ("epochOffset", "<i4"),
    ("evaluator", "<i4"),
])

EVALUATOR_PATH_TRACED, EVALUATOR_ALBEDO, EVALUATOR_NORMAL_DEPTH, EVALUATOR_NAIVE = 0, 1, 2, 3
EVALUATOR_DIVERGE_ONCE = 0x100
EVALUATOR_COUNT_VISITS = 0x200  # counted pass: EchoStats reports node / triangle / sphere / light-node visits (bench roofline)
DISTRIBUTION_STRATIFIED = 0x400  # StratifiedDistribution: jittered, shuffled strata per epoch and dimension (any evaluator)
DISTRIBUTION_STRATIFIED_EXTEND_MAX = 1 << 23

STATS_FIELDS = [
    "sampleEvaluated", "sampleRejected", "pixelEvaluated", "bounceCreated", "bounceSpecular", "bounceMis",
    "lightSampled", "lightOcclusionChecked", "lightOcclusionPassed", "lightEvaluatedInfinite",
    "traceQueries", "occludeQueries", "kernelLaunches",
]
# labels as the reference reports them (EvaluationOperation.cs:130-140, PathTracedEvaluator.cs:50-199)
STATS_LABELS = [
    "Sample/Evaluated", "Sample/Rejected", "Pixel/Evaluated", "Bounce/Created", "Bounce/Specular",
    "Bounce/Multiple Importance", "Light/Sampled", "Light/Occlusion Checked", "Light/Occlusion Passed",
    "Light/Evaluated Infinite",
]
# filled only by a counted pass (EVALUATOR_COUNT_VISITS): the inputs of the algorithmic bytes per sample (SURVEY.md 8d)
STATS_VISIT_FIELDS = ["nodeVisits", "triangleVisits", "sphereVisits", "lightNodeVisits"]
STATS = np.dtype([(name, "<u8") for name in STATS_FIELDS + STATS_VISIT_FIELDS] + [("reserved", "<u8", 7)])

assert QBVH_NODE.itemsize == 128
assert TRIANGLE.itemsize == 100
assert SPHERE.itemsize == 20
assert RAY.itemsize == 32
assert HIT.itemsize == 16
assert MATERIAL.itemsize == 64
assert LIGHT_NODE.itemsize == 64
assert POINT_LIGHT.itemsize == 24
assert INFINITE_LIGHT.itemsize == 160
assert CAMERA.itemsize == 80
assert RENDER_PARAMS.itemsize == 48
assert STATS.itemsize == 192


def render_params(width, height, tile_size=16, extend=16, min_epoch=1, max_epoch=1, noise_threshold=0.045,
                  bounce_limit=128, survivability=2.5, seed=1, epoch_offset=0, evaluator=EVALUATOR_PATH_TRACED):
    """EvaluationProfile + PathTracedEvaluator defaults (EvaluationProfile.cs:42-60, PathTracedEvaluator.cs:33,40).
    evaluator: EVALUATOR_* [| EVALUATOR_DIVERGE_ONCE] [| DISTRIBUTION_STRATIFIED] (AlbedoEvaluator.cs, NormalDepthEvaluator.cs,
    StratifiedDistribution.cs)."""
    params = np.zeros(1, dtype=RENDER_PARAMS)
    params["width"], params["height"], params["tileSize"] = width, height, tile_size
    params["extend"], params["minEpoch"], params["maxEpoch"] = extend, min_epoch, max_epoch
    params["noiseThreshold"], params["bounceLimit"], params["survivability"] = noise_threshold, bounce_limit, survivability
    params["seed"], params["epochOffset"], params["evaluator"] = seed, epoch_offset, evaluator
    return params
