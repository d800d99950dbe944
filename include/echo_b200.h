/*
 * echo_b200.h — C ABI of libecho_b200.so, the B200-native path-tracing core behind Echo's
 * evaluator/aggregator interface.
 *
 * Echo (GaryHuan9/EchoRenderer) has no FFI on this path: it is in-process C# virtual calls. The seams this
 * library sits behind (all paths relative to the reference's src/Echo.Core/):
 *   - Accelerator.Trace(ref TraceQuery) / Accelerator.Occlude(ref OccludeQuery)
 *       Aggregation/Acceleration/Accelerator.cs:90,96   -> echo_b200_trace_batch / echo_b200_occlude_batch
 *   - EvaluationOperation.Execute (pixel -> epoch -> sample loop, Accumulator, tile write)
 *       Processes/Evaluation/EvaluationOperation.cs:83-148 -> echo_b200_render_tiles
 *   - the prepared, flattened scene those calls read:
 *       QuadBoundingVolumeHierarchy.Node  Aggregation/Acceleration/QuadBoundingVolumeHierarchy.cs:406-469
 *       PreparedTriangle                  Scenic/Geometries/TriangleEntity.cs:57-129
 *       PreparedSphere                    Scenic/Geometries/SphereEntity.cs:48-63
 *       PreparedSwatch materials          Scenic/Preparation/PreparedSwatch.cs:20
 *       LightTree                         Aggregation/Selection/LightTree.cs:19-171
 *       PreparedScene infinite lights     Aggregation/Preparation/PreparedScene.cs:34-39
 *       PerspectiveCamera                 Scenic/Cameras/PerspectiveCamera.cs:41-98
 * P/Invoke conventions follow Echo's one native precedent, Processes/Composition/OidnDenoise.cs:48-300:
 * opaque handle, raw pinned pointers that the library never retains, errors pulled with a *_last_error call.
 *
 * Every function returns 0 on success and a non-zero ECHO_B200_ERR_* code otherwise. The library copies host
 * data on upload and owns device memory until echo_b200_scene_destroy. There is no CPU fallback: without a
 * CUDA device every compute entry point fails with ECHO_B200_ERR_NO_DEVICE.
 */
#ifndef ECHO_B200_H
#define ECHO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#define ECHO_B200_STATIC_ASSERT(condition, message) static_assert(condition, message)
#else
#define ECHO_B200_STATIC_ASSERT(condition, message) _Static_assert(condition, message)
#endif
/* every POD below is followed by its size: a binding (C#, ctypes ...) that disagrees with one of them corrupts memory silently */
#define ECHO_B200_ASSERT_SIZE(type, bytes) ECHO_B200_STATIC_ASSERT(sizeof(type) == (bytes), #type " must be " #bytes " bytes")

#define ECHO_B200_OK 0
#define ECHO_B200_ERR_INVALID 1     /* bad argument / scene not committed */
#define ECHO_B200_ERR_NO_DEVICE 2   /* no usable CUDA device */
#define ECHO_B200_ERR_CUDA 3        /* CUDA runtime failure; see echo_b200_last_error() */
#define ECHO_B200_ERR_UNSUPPORTED 4 /* feature outside the hot path (e.g. instanced tokens) */

/* ---- tokens: Aggregation/Primitives/EntityToken.cs:22-73, TokenType.cs:12-38 ---- */
#define ECHO_TOKEN_TYPE_NODE 0u
#define ECHO_TOKEN_TYPE_TRIANGLE 1u
#define ECHO_TOKEN_TYPE_SPHERE 2u
#define ECHO_TOKEN_TYPE_INSTANCE 3u
#define ECHO_TOKEN_TYPE_LIGHT 4u
#define ECHO_TOKEN_EMPTY 0xFFFFFFFFu
#define ECHO_TOKEN_INDEX_BITS 28
#define ECHO_TOKEN_MAKE(type, index) ((((uint32_t)(type)) << ECHO_TOKEN_INDEX_BITS) | (uint32_t)(index))
/* light tokens: 6-bit LightType above a 22-bit index (EntityToken.cs:29,68-71; Scenic/Lights/LightType.cs) */
#define ECHO_LIGHT_TYPE_INFINITE 0u
#define ECHO_LIGHT_TYPE_INFINITE_DELTA 1u
#define ECHO_LIGHT_TYPE_POINT 2u
#define ECHO_LIGHT_INDEX_BITS 22
#define ECHO_LIGHT_TOKEN_MAKE(ltype, index) \
	ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_LIGHT, (((uint32_t)(ltype)) << ECHO_LIGHT_INDEX_BITS) | (uint32_t)(index))

/* ---- QuadBoundingVolumeHierarchy.Node, 128 B explicit layout (QuadBoundingVolumeHierarchy.cs:406-469) ---- */
typedef struct EchoQbvhNode
{
	float minX[4], minY[4], minZ[4]; /* BoxBound4 @0 (Aggregation/Bounds/BoxBound4.cs:32-38) */
	float maxX[4], maxY[4], maxZ[4];
	int32_t axisMajor;  /* @96  0..2 */
	int32_t axisMinor0; /* @100 0..2, or 3 = [leaf, empty] pair */
	int32_t axisMinor1; /* @104 */
	uint32_t token4[4]; /* @108 child tokens; ECHO_TOKEN_EMPTY for none */
	uint32_t pad;       /* @124 */
} EchoQbvhNode;
ECHO_B200_ASSERT_SIZE(EchoQbvhNode, 128);

/* ---- PreparedTriangle, 100 B sequential layout (TriangleEntity.cs:118-139) ---- */
typedef struct EchoTriangle
{
	float vertex0[3], edge1[3], edge2[3];
	float normal0[3], normal1[3], normal2[3]; /* unit shading normals */
	float texcoord0[2], texcoord1[2], texcoord2[2];
	uint32_t material; /* MaterialIndex */
} EchoTriangle;
ECHO_B200_ASSERT_SIZE(EchoTriangle, 100);

/* ---- PreparedSphere, 20 B (SphereEntity.cs:59-63) ---- */
typedef struct EchoSphere
{
	float position[3];
	float radius;
	uint32_t material;
} EchoSphere;
ECHO_B200_ASSERT_SIZE(EchoSphere, 20);

/* ---- one query: Ray + TraceQuery/OccludeQuery inputs (Ray.cs:17-28, TraceQuery.cs:16-40, OccludeQuery.cs:10-30).
 * `direction` must be unit length; `distance` is TraceQuery.distance / OccludeQuery.travel (may be +inf);
 * `ignore` is the top token of the TokenHierarchy to skip (ECHO_TOKEN_EMPTY for none). ---- */
typedef struct EchoRay
{
	float origin[3];
	float direction[3];
	float distance;
	uint32_t ignore;
} EchoRay;
ECHO_B200_ASSERT_SIZE(EchoRay, 32);

/* ---- TraceQuery outputs (TraceQuery.cs:42-58). token == ECHO_TOKEN_EMPTY and distance == input distance on a miss. ---- */
typedef struct EchoHit
{
	uint32_t token;
	float distance;
	float uv[2];
} EchoHit;
ECHO_B200_ASSERT_SIZE(EchoHit, 16);

/* ---- materials with constant (Pure) textures flattened (Evaluation/Materials/) ---- */
#define ECHO_MATERIAL_DIFFUSE 0u    /* Diffuse.cs:33-47 */
#define ECHO_MATERIAL_DIELECTRIC 1u /* Dielectric.cs:29-47 */
#define ECHO_MATERIAL_CONDUCTOR 2u  /* Conductor.cs:72-124 */
#define ECHO_MATERIAL_EMISSIVE 3u   /* Emissive.cs:30-64 */
#define ECHO_MATERIAL_ONESIDED 4u   /* OneSided.cs:50-58 */
#define ECHO_MATERIAL_INVISIBLE 5u  /* Invisible.cs:22-26 */
#define ECHO_MATERIAL_COATED_DIFFUSE 6u /* CoatedDiffuse.cs:37-55 (SURVEY.md §8f rank 2) */
#define ECHO_MATERIAL_FLAG_TRANSMISSIVE 1u /* Diffuse.Transmissive */
#define ECHO_MATERIAL_FLAG_ARTISTIC 2u     /* Conductor.Artistic */
#define ECHO_MATERIAL_FLAG_BACKFACE 4u     /* OneSided.Backface */

typedef struct EchoMaterial
{
	uint32_t type;
	uint32_t flags;
	float albedo[4];    /* RGBA; alpha < 0.5 makes the surface Invisible (Material.cs:63-75). Emissive: emission RGB */
	float roughness[2]; /* R and G of the Roughness texture */
	float ior;          /* Dielectric.RefractiveIndex / CoatedDiffuse.RefractiveIndex */
	float paramA[3];    /* Conductor: MainColor (artistic) or RefractiveIndex (physical); CoatedDiffuse: [0] = the reflectance cached by
	                       CoatedDiffuse.Prepare = FresnelDiffuseReflectance(1 / RefractiveIndex) (echo_host_fresnel_diffuse_reflectance) */
	float paramB[3];    /* Conductor: EdgeColor (artistic) or Extinction (physical) */
	uint32_t base;      /* OneSided.Base material index */
} EchoMaterial; /* 64 B */
ECHO_B200_ASSERT_SIZE(EchoMaterial, 64);

/* ---- image textures (SURVEY.md 8f rank 3): TextureGrid (Textures/Grids/TextureGrid.cs) flattened to RGBA128 texels, with its
 * IFilter (Textures/Grids/IFilter.cs) and IWrapper (Textures/Grids/IWrapper.cs). Texel (x, y) of texture t is
 * texels[t.texelOffset + y * t.width + x], rows growing upward like every Echo texture. ---- */
#define ECHO_TEXTURE_NONE 0xFFFFFFFFu /* the slot keeps the constant of EchoMaterial (a Pure texture) */
#define ECHO_FILTER_POINT 0u
#define ECHO_FILTER_BILINEAR 1u
#define ECHO_WRAPPER_CLAMP 0u
#define ECHO_WRAPPER_REPEAT 1u
#define ECHO_WRAPPER_MIRROR 2u

typedef struct EchoTexture
{
	uint32_t width, height;
	uint32_t texelOffset; /* in texels */
	uint32_t filter;      /* ECHO_FILTER_* */
	uint32_t wrapper;     /* ECHO_WRAPPER_* */
	uint32_t reserved[3];
} EchoTexture; /* 32 bytes */
ECHO_B200_ASSERT_SIZE(EchoTexture, 32);

/* the texture slots of one material, parallel to the material array; a slot holding a texture index replaces the constant
 * of the same name in EchoMaterial with `(RGB128)texture[contact.shade.Texcoord]` (Material.Sample, Material.cs:102) */
typedef struct EchoMaterialTextures
{
	uint32_t albedo;       /* Material.Albedo, RGBA (Material.cs:63-75,100) */
	uint32_t normal;       /* Material.Normal: tangent-space normal map (Material.ApplyNormalMapping, Material.cs:77-98) */
	uint32_t roughness;    /* R and G of the Roughness texture */
	uint32_t paramA;       /* Conductor.MainColor / RefractiveIndex */
	uint32_t paramB;       /* Conductor.EdgeColor / Extinction */
	float normalIntensity; /* Material.NormalIntensity (default 0.25); ~0 switches normal mapping off (Material.cs:58) */
	uint32_t reserved[2];
} EchoMaterialTextures; /* 32 bytes */
ECHO_B200_ASSERT_SIZE(EchoMaterialTextures, 32);

/* ---- flattened LightTree node (LightTree.cs:156-171, LightBound.cs:10-20, ConeBound.cs:20-24). Node 0 = root.
 * Branch: child0/child1 are node indices. Leaf: child0 == ECHO_TOKEN_EMPTY and child1 holds the light's token. ---- */
typedef struct EchoLightNode
{
	float boxMin[3], boxMax[3];
	float coneAxis[3];
	float cosOffset, cosExtend;
	float power;
	uint32_t child0, child1;
	uint32_t pad[2];
} EchoLightNode; /* 64 B */
ECHO_B200_ASSERT_SIZE(EchoLightNode, 64);

/* ---- PreparedPointLight (Scenic/Lights/PointLight.cs:20-33) ---- */
typedef struct EchoPointLight
{
	float intensity[3];
	float position[3];
} EchoPointLight;
ECHO_B200_ASSERT_SIZE(EchoPointLight, 24);

/* ---- infinite lights (Scenic/Lights/InfiniteLight.cs): AmbientLight over a constant (Pure) texture (AmbientLight.cs) and
 * DirectionalLight (DirectionalLight.cs:12-108), with everything DirectionalLight.Prepare computes on the host (:52-75). ---- */
#define ECHO_INFINITE_AMBIENT 0u
#define ECHO_INFINITE_DIRECTIONAL 1u
#define ECHO_INFINITE_ENVIRONMENT 2u /* AmbientLight over a CylindricalTexture (Textures/Directional/CylindricalTexture.cs) */
#define ECHO_INFINITE_CUBEMAP 3u     /* AmbientLight over a Cubemap (Textures/Directional/Cubemap.cs): `texture` is the first of six
                                        consecutive EchoTexture records in px, nx, py, ny, pz, nz order (Cubemap.cs:49); sampled
                                        uniformly over the sphere (IDirectionalTexture's defaults), no distribution */

typedef struct EchoInfiniteLight
{
	float radiance[3];        /* Ambient: Intensity * texture colour. Directional: scaledIntensity (black when delta), :63-69 */
	uint32_t directlyVisible; /* InfiniteLight.DirectlyVisible (DirectionalLight defaults to false, :15) */
	uint32_t type;            /* ECHO_INFINITE_* */
	uint32_t isDelta;         /* DirectionalLight.IsDelta: !Positive(1 - cosAngle), :50 */
	float cosAngle;           /* cos(Angle), :61 */
	float pad0;
	float intensity[3];       /* DirectionalLight.Intensity: what a delta light's Sample returns, :101 */
	float pad1;
	float direction[3];       /* incidentDirection = (LocalToWorldRotation * Float3.Backward).Normalized, :58 */
	float pad2;
	float rotation[9];        /* LocalToWorldRotation, row-major (InfiniteLight.cs:31-37): orients the sampled cone / the environment */
	uint32_t texture;         /* Environment: the CylindricalTexture's grid (EchoTexture index); radiance then holds Intensity */
	uint32_t distribution;    /* Environment: offset of its DiscreteDistribution2D in the array of set_distributions */
	float pad3;
	float inverseRotation[9]; /* WorldToLocalRotation (InfiniteLight.cs:37), Environment only */
	float pad4[3];
} EchoInfiniteLight; /* 160 bytes; an ambient light only needs the first 16, the rest zero */
ECHO_B200_ASSERT_SIZE(EchoInfiniteLight, 160);

/* ---- instancing (SURVEY.md 8f rank 2): PreparedPack / PreparedInstance / TokenHierarchy ----
 * A scene with instances is a set of packs (PreparedPack.cs:13-24): pack 0 is the PreparedScene itself, the others are the
 * packs its instances refer to (packs may be instanced many times and may hold instances themselves, at most
 * ECHO_MAX_INSTANCE_LAYERS deep). The arrays handed to set_qbvh / set_triangles / set_spheres / set_materials hold all
 * packs back to back; every token inside a pack (node children, triangle / sphere / instance indices) is relative to
 * the pack's own offsets, exactly as each C# pack sees its own arrays. The root of a pack's accelerator is its node 0. */
#define ECHO_MAX_INSTANCE_LAYERS 5u /* TokenHierarchy.MaxLayer, TokenHierarchy.cs:41 */

typedef struct EchoPack
{
	uint32_t nodeOffset, nodeCount; /* into the node array; maxDepth as for set_qbvh */
	uint32_t maxDepth;
	uint32_t triangleOffset, triangleCount;
	uint32_t sphereOffset, sphereCount;
	uint32_t instanceOffset, instanceCount; /* into the instance array: GeometryCollection.instances of this pack */
	uint32_t materialOffset;                /* the pack's own swatch (LightCollection reads it, LightCollection.cs:145,151) */
	/* the pack's LightTree / LightCollection (PreparedPack.cs:21-23): ranges of the arrays handed to set_light_tree, child
	 * indices and emitter tokens pack-relative; a placement with light inside appears as a TokenType.Instance leaf of its
	 * parent's light tree (LightCollection.cs:123-135) */
	uint32_t lightNodeOffset, lightNodeCount;
	uint32_t emitterOffset, emitterCount;
	uint32_t pointLightOffset, pointLightCount;
} EchoPack; /* 64 bytes */
ECHO_B200_ASSERT_SIZE(EchoPack, 64);

typedef struct EchoInstance
{
	float forward[12];   /* rows 0..2 of PreparedInstance.forwardTransform (parent -> local), PreparedInstance.cs:22 */
	float inverse[12];   /* rows 0..2 of PreparedInstance.inverseTransform (local -> parent), :23 */
	float forwardScale;  /* parent -> local scale multiplier, :26 */
	float inverseScale;  /* local -> parent scale multiplier, :27 */
	uint32_t pack;       /* index of the instanced pack */
	uint32_t materialOffset; /* PreparedInstance.swatch: material index of a hit = this + the geometry's own index */
	uint32_t reserved[4];
} EchoInstance; /* 128 bytes */
ECHO_B200_ASSERT_SIZE(EchoInstance, 128);

/* the instance layers of a TokenHierarchy (TokenHierarchy.cs:19-60); its TopToken travels in EchoRay.ignore / EchoHit.token */
typedef struct EchoTokenHierarchy
{
	uint32_t instanceCount;
	uint32_t instances[ECHO_MAX_INSTANCE_LAYERS]; /* TokenType.Instance tokens, outermost first */
} EchoTokenHierarchy; /* 24 bytes */
ECHO_B200_ASSERT_SIZE(EchoTokenHierarchy, 24);

/* ---- Camera.SpawnRay inputs (Scenic/Cameras/{Perspective,Orthographic,Cylindrical}Camera.cs, RaySpawner.cs:11-64) ---- */
#define ECHO_CAMERA_PERSPECTIVE 0u  /* PerspectiveCamera.cs:41-98 (thin lens when lensRadius and focalDistance are both >= 8e-7) */
#define ECHO_CAMERA_ORTHOGRAPHIC 1u /* OrthographicCamera.cs:15-39: origin = InverseTransform * (SpawnX(shift) * Width, 0), fixed direction */
#define ECHO_CAMERA_CYLINDRICAL 2u  /* CylindricalCamera.cs:12-34: direction = rotation * CylindricalTexture.ToDirection((pixel + shift) / size) */

typedef struct EchoCamera
{
	float transform[12]; /* rows 0..2 of Entity.InverseTransform (entity -> world), row-major f00..f23 */
	float forwardLength; /* Perspective: 0.5 / tan(fov / 2) */
	float lensRadius;
	float focalDistance; /* depth of field is on iff lensRadius and focalDistance are both >= 8e-7 */
	uint32_t type;       /* ECHO_CAMERA_* */
	float direction[3];  /* Orthographic: RootedRotation * Float3.Forward (OrthographicCamera.cs:22-26) */
	float width;         /* Orthographic: Width (:18) */
} EchoCamera; /* 80 bytes */
ECHO_B200_ASSERT_SIZE(EchoCamera, 80);

/* ---- EvaluationProfile + PathTracedEvaluator knobs (EvaluationProfile.cs:42-60, PathTracedEvaluator.cs:33,40) ---- */
typedef struct EchoRenderParams
{
	int32_t width, height;  /* RenderTexture size */
	int32_t tileSize;       /* square tiles (RenderProfile.cs:45) */
	int32_t extend;         /* samples per epoch (ContinuousDistribution.Extend) */
	int32_t minEpoch, maxEpoch;
	float noiseThreshold;
	int32_t bounceLimit;    /* PathTracedEvaluator.BounceLimit */
	float survivability;    /* PathTracedEvaluator.Survivability */
	uint32_t seed;          /* counter-based sample sequence seed */
	int32_t epochOffset;    /* first epoch index this call renders (sample sharding across devices) */
	int32_t evaluator;      /* ECHO_EVALUATOR_* [| ECHO_EVALUATOR_DIVERGE_ONCE] [| ECHO_DISTRIBUTION_STRATIFIED]; 0 = PathTracedEvaluator */
} EchoRenderParams;
ECHO_B200_ASSERT_SIZE(EchoRenderParams, 48);

/* EvaluationProfile.Evaluator (EvaluationProfile.cs:23): the path tracer, or one of the two auxiliary evaluators the
 * StandardPathTracedProfile runs for its denoiser (Processes/StandardPathTracedProfile.cs:27-45). The auxiliary ones
 * follow purely specular bounces from the camera and report the first other surface: its albedo, W = 0
 * (Evaluation/Evaluators/AlbedoEvaluator.cs:18-55) or NormalDepth128.ToFloat4() = shading normal, W = depth travelled
 * (Evaluation/Evaluators/NormalDepthEvaluator.cs:20-60). bounceLimit / survivability are not read by them. */
#define ECHO_EVALUATOR_PATH_TRACED 0
#define ECHO_EVALUATOR_ALBEDO 1
#define ECHO_EVALUATOR_NORMAL_DEPTH 2
#define ECHO_EVALUATOR_NAIVE 3 /* StandardNaiveEvaluator (Evaluation/Evaluators/StandardNaiveEvaluator.cs:16-55): no light sampling, no
                                 roulette; reads bounceLimit (<= 128 here: the device unrolls the recursion into two arrays) */
#define ECHO_EVALUATOR_KIND_MASK 0xFF
#define ECHO_EVALUATOR_DIVERGE_ONCE 0x100 /* the evaluator's DivergeOnce property (default: true for Albedo, false for NormalDepth) */
#define ECHO_EVALUATOR_COUNT_VISITS 0x200 /* PathTracedEvaluator only: a counted pass. Same samples, same results, but the traversal runs
                                             on the one-thread-per-query kernels with visit counters and EchoStats reports node / triangle /
                                             sphere / light-node visits. A measurement aid (bench.py's roofline), several times slower. */
#define ECHO_DISTRIBUTION_STRATIFIED 0x400 /* EvaluationProfile.Distribution is a StratifiedDistribution (StratifiedDistribution.cs:34-50):
                                              each pixel's epoch of `extend` samples is one jittered, shuffled stratified set per dimension
                                              (2D draws correlated multi-jittered) instead of independent uniform numbers. Any evaluator,
                                              counted passes too; extend at most 2^23 (ECHO_B200_ERR_INVALID above). */
#define ECHO_DISTRIBUTION_STRATIFIED_EXTEND_MAX (1 << 23)

/* ---- EvaluatorStatistics rows on the hot path, same labels/order as the reference reports them
 * (EvaluationOperation.cs:130-140; PathTracedEvaluator.cs:50-199) ---- */
typedef struct EchoStats
{
	uint64_t sampleEvaluated;        /* "Sample/Evaluated" */
	uint64_t sampleRejected;         /* "Sample/Rejected" */
	uint64_t pixelEvaluated;         /* "Pixel/Evaluated" */
	uint64_t bounceCreated;          /* "Bounce/Created" */
	uint64_t bounceSpecular;         /* "Bounce/Specular" */
	uint64_t bounceMis;              /* "Bounce/Multiple Importance" */
	uint64_t lightSampled;           /* "Light/Sampled" */
	uint64_t lightOcclusionChecked;  /* "Light/Occlusion Checked" */
	uint64_t lightOcclusionPassed;   /* "Light/Occlusion Passed" */
	uint64_t lightEvaluatedInfinite; /* "Light/Evaluated Infinite" */
	uint64_t traceQueries;           /* closest-hit queries issued */
	uint64_t occludeQueries;         /* occlusion queries issued */
	uint64_t kernelLaunches;         /* CUDA kernels launched by this call */
	/* visit counters, filled only by a call with ECHO_EVALUATOR_COUNT_VISITS (zero otherwise): the inputs of the algorithmic
	 * bytes per sample of SURVEY.md 8(d), counted on the reference's own visit order */
	uint64_t nodeVisits;             /* BoxBound4.Intersect calls of the closest-hit and occlusion queries (128 B each) */
	uint64_t triangleVisits;         /* PreparedTriangle.Intersect calls (36 B each) */
	uint64_t sphereVisits;           /* PreparedSphere.Intersect calls (16 B each) */
	uint64_t lightNodeVisits;        /* LightBound.Importance evaluations of LightTree.Pick / ProbabilityMass (64 B each) */
	uint64_t reserved[7];
} EchoStats; /* 192 bytes */
ECHO_B200_ASSERT_SIZE(EchoStats, 192);

typedef struct EchoScene EchoScene;

int32_t echo_b200_device_count(int32_t* out);
int32_t echo_b200_scene_create(EchoScene** out, int32_t device);

/* One scene on SEVERAL devices of this process — the reference is one process whose Device drives N workers
 * (Common/Compute/Device.cs:20-24), so its host makes one call and the library fans out. Bit d of device_mask = CUDA device d.
 * The set_* calls stage on the host as usual; commit uploads a replica to every device of the mask (SURVEY.md 8e: the scene is
 * replicated). echo_b200_trace_batch / occlude_batch (and the _hierarchy forms) cut a batch into one contiguous range per device;
 * echo_b200_render_tiles deals blocks of 64 consecutive tiles of the caller's sequence round-robin to the devices
 * (Common/Compute/Operation.cs:164-177's procedure claiming, made static) and gathers the accumulated tiles into the caller's
 * tile-major buffer — every tile is rendered by exactly one device, so results equal the single-device ones bit for bit and no
 * reduction is needed. One host thread per device, inside the call. The *_device entry points (caller-owned device memory on
 * one device) need a single-device scene and fail with ECHO_B200_ERR_INVALID on a multi-device one. */
int32_t echo_b200_scene_create_multi(EchoScene** out, uint64_t device_mask);
int32_t echo_b200_scene_gpu_count(EchoScene*, int32_t* out); /* devices the scene is replicated on (1 for echo_b200_scene_create) */

/* scene upload; pointers are only read during the call */
int32_t echo_b200_scene_set_qbvh(EchoScene*, const EchoQbvhNode* nodes, uint32_t node_count, uint32_t max_depth);
int32_t echo_b200_scene_set_triangles(EchoScene*, const EchoTriangle* triangles, uint32_t count);
int32_t echo_b200_scene_set_spheres(EchoScene*, const EchoSphere* spheres, uint32_t count);
int32_t echo_b200_scene_set_materials(EchoScene*, const EchoMaterial* materials, uint32_t count);
/* optional: image textures and the texture slots of every material (material_textures: one record per material set with
 * set_materials, or NULL when texture_count is 0). texels_rgba holds texel_count RGBA128 texels. */
int32_t echo_b200_scene_set_textures(EchoScene*, const EchoTexture* textures, uint32_t texture_count, const float* texels_rgba, uint64_t texel_count,
                                     const EchoMaterialTextures* material_textures, uint32_t material_count);
int32_t echo_b200_scene_set_light_tree(EchoScene*, const EchoLightNode* nodes, uint32_t node_count,
                                       const uint32_t* emitter_tokens, const uint64_t* emitter_bitpaths, uint32_t emitter_count,
                                       const EchoPointLight* points, uint32_t point_count);
int32_t echo_b200_scene_set_infinite(EchoScene*, const EchoInfiniteLight* lights, uint32_t count, float threshold, float pdf);
/* The DiscreteDistribution2D of every environment light (Evaluation/Sampling/DiscreteDistribution2D.cs, built by
 * CylindricalTexture.Prepare, CylindricalTexture.cs:33-96): for a width x height grid, `height` cdfValues of the vertical
 * DiscreteDistribution1D followed by height rows of `width` cdfValues of the slices (DiscreteDistribution1D.cs:12-56). */
int32_t echo_b200_scene_set_distributions(EchoScene*, const float* values, uint64_t count);
int32_t echo_b200_scene_set_camera(EchoScene*, const EchoCamera* camera);
/* Accelerator.SphereBound.radius of the scene (Accelerator.cs:43-63): the NormalDepthEvaluator reports twice this as the
 * depth of rays that escape (NormalDepthEvaluator.cs:57). Optional; 0 when never set. May be called after commit. */
int32_t echo_b200_scene_set_bound_radius(EchoScene*, float radius);
/* optional: declares the scene instanced (see EchoPack). Without it the scene is the single pack the arrays describe. */
int32_t echo_b200_scene_set_packs(EchoScene*, const EchoPack* packs, uint32_t pack_count, const EchoInstance* instances, uint32_t instance_count);
int32_t echo_b200_scene_commit(EchoScene*);
int32_t echo_b200_scene_destroy(EchoScene*);

/* batched Accelerator.Trace / Accelerator.Occlude through PreparedScene's guards (PreparedScene.cs:66-86). Host buffers. */
int32_t echo_b200_trace_batch(EchoScene*, const EchoRay* rays, uint64_t n, EchoHit* hits);
int32_t echo_b200_occlude_batch(EchoScene*, const EchoRay* rays, uint64_t n, uint8_t* occluded);

/* the same queries with full TokenHierarchy in and out, for instanced scenes (GeometryCollection.cs:123-131,160-168,
 * PreparedInstance.cs:47-83). `ignore` (nullable) holds the instance layers of each query's ignore hierarchy;
 * `hit_layers` (nullable) receives the instance layers of each hit. Plain trace_batch / occlude_batch on an instanced
 * scene behave as if `ignore` held empty hierarchies and drop the hit layers. Host buffers. */
int32_t echo_b200_trace_batch_hierarchy(EchoScene*, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n,
                                        EchoHit* hits, EchoTokenHierarchy* hit_layers);
int32_t echo_b200_occlude_batch_hierarchy(EchoScene*, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, uint8_t* occluded);

/* same, device-resident buffers on `stream` (a cudaStream_t passed as void*; NULL = default stream). Asynchronous. */
int32_t echo_b200_trace_batch_device(EchoScene*, const EchoRay* d_rays, uint64_t n, EchoHit* d_hits, void* stream);
int32_t echo_b200_occlude_batch_device(EchoScene*, const EchoRay* d_rays, uint64_t n, uint8_t* d_occluded, void* stream);

/* one EvaluationOperation worth of tiles. tile_xy holds tile_count (x, y) tile positions (in tiles, not pixels).
 * out_rgba is tile-major: tile i occupies tileSize*tileSize Float4s, row-major inside the tile, rows growing upward
 * like Echo's textures; pixels of a partial tile outside the image are left zero. Host buffer. */
int32_t echo_b200_render_tiles(EchoScene*, const EchoRenderParams*, const int32_t* tile_xy, uint32_t tile_count,
                               float* out_rgba, EchoStats* stats);

/* device-resident accumulation into a full-frame buffer (width*height Float4): every rendered pixel ADDS (mean * n, n), n = the
 * samples it accumulated. Used for multi-GPU sharding: each device renders its tiles (tile sharding) or its epochs of every
 * tile (sample sharding, epochOffset) into its own zeroed frame, the frames are summed with one NCCL all-reduce, then
 * echo_b200_frame_resolve_device divides RGB by W. Exact for a pixel rendered by one device whenever n is a power of two.
 * Asynchronous on `stream`. */
int32_t echo_b200_render_frame_device(EchoScene*, const EchoRenderParams*, const int32_t* tile_xy, uint32_t tile_count,
                                      float* d_frame_rgba, EchoStats* stats, void* stream);
int32_t echo_b200_frame_resolve_device(EchoScene*, float* d_frame_rgba, int32_t width, int32_t height, void* stream);

/* Optional device-side tree build (SURVEY.md 8f rank 4) in the reference's QBVH node format. By default the tree is the reference's
 * own: SweepBuilder.Build (Aggregation/Acceleration/SweepBuilder.cs:24-160 — stable sort by min + max along the major axis of the
 * node's volume, one-axis sweep for the first cut of lowest cost, larger-area child first) and the QuadBoundingVolumeHierarchy collapse
 * (QuadBoundingVolumeHierarchy.cs:363-565, nodes in pre-order), run level by level on the device; the emitted array equals what the
 * recursive build emits byte for byte (echo_host.h's mirror; tests/test_gpu_build.py, tests/test_sweep_build.py). 1 010 000 primitives:
 * 10-12 ms of device work against 430 ms for the host mirror on 16 cores. Inputs whose tree chains deeper than the traversal stacks allow
 * (thousands of coincident primitives) — and ECHO_B200_BUILD_ALGORITHM=1 / 0 — get a clustered (PLOC) or Morton-ordered (Karras 2012)
 * binary tree collapsed the same way instead: valid, lower quality, not the reference's. Tokens: triangles, then spheres, as
 * GeometryCollection.CreateBounds numbers them. `out_nodes` (host) needs room for triangle_count + sphere_count - 1 nodes;
 * out_max_depth is the depth CreateNode reports (what set_qbvh takes). */
int32_t echo_b200_build_qbvh(int32_t device, const EchoTriangle* triangles, uint32_t triangle_count, const EchoSphere* spheres, uint32_t sphere_count,
                             EchoQbvhNode* out_nodes, uint32_t* out_node_count, uint32_t* out_max_depth);
/* The same for a pack that holds placements (GeometryCollection.CreateBounds, GeometryCollection.cs:52-81: triangles, spheres, then
 * instances): `instance_bounds` = 6 floats per placement, PreparedInstance.BoxBound as min xyz, max xyz; their tokens are
 * TokenType.Instance in the order given. Mirrors echo_host_build_qbvh_instanced (echo_host.h). */
int32_t echo_b200_build_qbvh_instanced(int32_t device, const EchoTriangle* triangles, uint32_t triangle_count, const EchoSphere* spheres, uint32_t sphere_count,
                                       const float* instance_bounds, uint32_t instance_count, EchoQbvhNode* out_nodes, uint32_t* out_node_count, uint32_t* out_max_depth);
/* The same build for a scene handle: builds the accelerator of the triangles and spheres already uploaded with set_triangles /
 * set_spheres on the scene's device and installs it as if set_qbvh had been called with the SweepBuilder's nodes — a host that
 * does not want to run Accelerator construction (AcceleratorCreator.cs) on its CPU calls this instead of set_qbvh, before commit.
 * out_node_count / out_max_depth are optional. Scenes with packs: ECHO_B200_ERR_UNSUPPORTED (build each pack, set_qbvh + set_packs). */
int32_t echo_b200_scene_build_qbvh(EchoScene*, uint32_t* out_node_count, uint32_t* out_max_depth);

/* Optional device-side LIGHT TREE build (SURVEY.md 8f rank 4): LightCollection.CreateBounds (Aggregation/Preparation/LightCollection.cs:91-137
 * — point lights, emissive triangles, emissive spheres, then the placements' PreparedInstance.LightBound rows, those below FastMath.Epsilon
 * of power dropped), LightTree.Build (Aggregation/Selection/LightTree.cs:62-113 — sort by box centre along the major axis, one sweep from
 * each end over LightBound.Encapsulate / RelativeArea, first cut of lowest cost, tail subtree first) and AddToMap (:26-37), run level by
 * level on the device. The shape of this tree IS the light-sampling distribution (LightTree.Pick, :115-154), so the build emits the
 * reference's own tree: nodes in pre-order, emitter tokens and bit paths equal to echo_host_build_light_tree's byte for byte
 * (tests/test_light_build.py, tests/test_gpu_build.py). MathF.Acos / Cos, Math.Acos and the Versor's Math.Sin / Cos are pinned (csrc/echo_light_build.h) so
 * that host and device agree; the sort is stable (the reference's Span.Sort leaves the order of equal centres to the runtime).
 * Mirrors echo_host_build_light_tree_instanced (echo_host.h), with caller-owned output: out_nodes needs room for node_capacity nodes,
 * out_emitter_tokens / out_emitter_bitpaths for emitter_capacity entries; 2 e - 1 nodes for e emitters, and e <= point_count + the
 * primitives with an Emissive material + instance_count. Too little room: ECHO_B200_ERR_INVALID with the needed counts in out_node_count /
 * out_emitter_count. A tree deeper than 63 levels (LightTree.cs:29: a path is 64 bits): ECHO_B200_ERR_UNSUPPORTED. No emitters: both counts 0.
 * out_power receives the root's LightBound.power (what PreparedScene.CalculateThreshold takes, echo_host_infinite_threshold).
 * instance_lights: 12 floats per placement (box min xyz, max xyz, cone axis xyz, cosOffset, cosExtend, power), or NULL. */
int32_t echo_b200_build_light_tree(int32_t device, const EchoTriangle* triangles, uint32_t triangle_count, const EchoSphere* spheres, uint32_t sphere_count,
                                   const EchoMaterial* materials, uint32_t material_count, const EchoPointLight* points, uint32_t point_count,
                                   const float* instance_lights, uint32_t instance_count,
                                   EchoLightNode* out_nodes, uint32_t node_capacity, uint32_t* out_node_count,
                                   uint32_t* out_emitter_tokens, uint64_t* out_emitter_bitpaths, uint32_t emitter_capacity, uint32_t* out_emitter_count,
                                   float* out_power);
/* The same build for a scene handle: the light tree of the triangles, spheres and materials already uploaded (set_triangles / set_spheres /
 * set_materials) and of `points`, built on the scene's device and installed as if set_light_tree had been called with it — a host that
 * does not want to run LightCollection / LightTree construction on its CPU calls this instead of set_light_tree, before commit.
 * out_* are optional. Scenes with packs: ECHO_B200_ERR_UNSUPPORTED (build each pack's tree with echo_b200_build_light_tree). */
int32_t echo_b200_scene_build_light_tree(EchoScene*, const EchoPointLight* points, uint32_t point_count,
                                         uint32_t* out_node_count, uint32_t* out_emitter_count, float* out_power);

/* Optional device-side build of EVERY PACK of an instanced scene in one call: each pack's QBVH and light tree as echo_b200_build_qbvh_instanced
 * and echo_b200_build_light_tree build them (byte for byte the host mirror's, pack by pack), and the rows those calls take for the placements
 * — PreparedInstance.BoxBound (FillBounds(6) of the child's accelerator, centre / extent through EchoInstance.inverse) and LightBound (the
 * child's light-tree root moved the same way; a zero row without emitters) — computed on the device from the finished child trees. Packs of
 * equal height (0 without placements, else 1 + the tallest pack placed) are built together, as one forest per driver, so a call reads back
 * as many levels per height as its deepest pack has (csrc/echo_pack_build.h). Inputs: the arrays of all packs back to back, `packs` with
 * each pack's triangle / sphere / instance / point-light ranges and materialOffset (a pack's swatch ends where the next swatch of the
 * array begins, another pack's or a placement's), `instances` with forward / inverse / scales / pack. On return every pack record also
 * holds nodeOffset / nodeCount / maxDepth / lightNodeOffset / lightNodeCount / emitterOffset / emitterCount, and the outputs hold every
 * pack's nodes, light nodes, emitter tokens and bit paths back to back in pack order (host.prepare's layout), ready for set_qbvh /
 * set_light_tree / set_packs. out_power = pack 0's light-tree root power (what echo_host_infinite_threshold takes). Room: nodes <= the
 * primitives (placements included), light nodes <= 2 x emitters, emitters <= point lights + primitives. Refusals: a pack of fewer than 2
 * primitives, a cycle, nesting deeper than ECHO_MAX_INSTANCE_LAYERS, too little room (with the needed counts): ECHO_B200_ERR_INVALID; a light
 * tree deeper than 63 levels: ECHO_B200_ERR_UNSUPPORTED. Trees of a height the forest cannot build as the reference's (see build_qbvh) are
 * built pack by pack, falling back as echo_b200_build_qbvh does. */
int32_t echo_b200_build_packs(int32_t device, const EchoTriangle* triangles, uint32_t triangle_count, const EchoSphere* spheres, uint32_t sphere_count,
                              const EchoMaterial* materials, uint32_t material_count, const EchoPointLight* points, uint32_t point_count,
                              EchoPack* packs, uint32_t pack_count, const EchoInstance* instances, uint32_t instance_count,
                              EchoQbvhNode* out_nodes, uint32_t node_capacity, uint32_t* out_node_count,
                              EchoLightNode* out_light_nodes, uint32_t light_node_capacity, uint32_t* out_light_node_count,
                              uint32_t* out_emitter_tokens, uint64_t* out_emitter_bitpaths, uint32_t emitter_capacity, uint32_t* out_emitter_count,
                              float* out_power);
/* The same build for a scene handle: call it after set_triangles / set_spheres / set_materials / set_packs instead of set_qbvh and
 * set_light_tree. It builds on the scene's (first) device, installs the nodes, light trees and emitter maps with `points`, and completes the
 * staged pack records; commit uploads them (to every device of a multi-device handle). out_* are optional. */
int32_t echo_b200_scene_build_packs(EchoScene*, const EchoPointLight* points, uint32_t point_count,
                                    uint32_t* out_node_count, uint32_t* out_light_node_count, uint32_t* out_emitter_count, float* out_power);

/* Page-locked host memory for the host-buffer entry points. A P/Invoke caller pins managed arrays with `fixed`
 * (Processes/Composition/OidnDenoise.cs:109-110): that stops the GC from moving them but leaves them PAGEABLE for CUDA, so every
 * copy is staged through the driver's bounce buffer and cannot overlap the kernels (measured: bench.py `e2e_pageable`). Either
 * allocate the batch buffers here (use them as the backing store of the managed view) or register the caller's own memory once.
 * Registered memory stays owned by the caller; it must be unregistered before it is released. */
int32_t echo_b200_host_alloc(void** out, uint64_t bytes);
int32_t echo_b200_host_free(void* pointer);
int32_t echo_b200_host_register(void* pointer, uint64_t bytes);
int32_t echo_b200_host_unregister(void* pointer);

const char* echo_b200_last_error(void);
const char* echo_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif
