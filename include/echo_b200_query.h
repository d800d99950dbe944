/*
 * echo_b200_query.h — the rest of the reference's scene interface as batched device queries: everything a custom
 * Evaluator (Evaluation/Evaluators/Evaluator.cs: `Float4 Evaluate(PreparedScene, in Ray, ...)`) calls on a PreparedScene
 * besides Trace / Occlude (echo_b200.h), and the BSDF that Material.Scatter leaves on a Contact:
 *
 *   PreparedScene.Interact + Material.Scatter  Aggregation/Preparation/PreparedScene.cs:95-105 -> echo_b200_interact_batch
 *   BSDF.Sample                                Evaluation/Scattering/BSDF.cs:150-208           -> echo_b200_scatter_sample_batch
 *   BSDF.Evaluate / BSDF.ProbabilityDensity    BSDF.cs:97-143                                   -> echo_b200_scatter_evaluate_batch
 *   PreparedScene.Pick                         PreparedScene.cs:113-150                         -> echo_b200_light_pick_batch
 *   PreparedScene.ProbabilityMass              PreparedScene.cs:158-179                         -> echo_b200_light_mass_batch
 *   PreparedScene.Sample                       PreparedScene.cs:182-204                         -> echo_b200_light_sample_batch
 *   PreparedScene.ProbabilityDensity           PreparedScene.cs:207-225                         -> echo_b200_light_pdf_batch
 *   PreparedScene.EvaluateInfinite             PreparedScene.cs:233-253                         -> echo_b200_evaluate_infinite_batch
 *
 * Every call runs the device functions the path kernels of echo_b200_render_tiles run, in the instantiation the renderer picks
 * for the scene, so a query answers bit for bit what a rendered path computes for the same inputs.
 *
 * Conventions. Host buffers, read or written only during the call; n == 0 is accepted and does nothing. A `layers` argument
 * (EchoTokenHierarchy, one per query) may be NULL, meaning empty hierarchies; it is the only way to pass instance layers. The calls
 * are stateless: the two scatter calls run Interact again from (ray, hit, hit_layers) instead of taking a contact back, so no BSDF
 * crosses the ABI and a host may batch the three contact calls in any order. Caller samples are clamped to [0, 1 - ulp] like
 * Sample1D / Sample2D (Evaluation/Sampling/Sample1D.cs). A miss (hit.token == ECHO_TOKEN_EMPTY) or an ECHO_TOKEN_EMPTY light token
 * gives zeroed outputs with pdf 0 (and material == ECHO_TOKEN_EMPTY from interact). A multi-device scene cuts a batch into one
 * contiguous range per device, like echo_b200_trace_batch.
 *
 * Validation. Tokens and layers come from outside the library here, so every element is checked on the host before anything is
 * uploaded; the first bad one fails the call with ECHO_B200_ERR_INVALID and a message naming its index. Accepted:
 *   - layers: instanceCount <= ECHO_MAX_INSTANCE_LAYERS and every token an Instance of its parent pack (the first of pack 0), with
 *     the material swatch each one selects inside the material array; on a scene without packs, NULL or empty hierarchies only;
 *   - hit tokens: ECHO_TOKEN_EMPTY, or a Triangle / Sphere of the pack the layers end in, whose material index is in range;
 *   - hit values (hits only, a miss is not read): finite distance and uv; uv of a triangle hit in [0, 1] x [0, 1] (barycentrics);
 *     uv of a sphere hit as SphereEntity.cs:112-122 encodes it: y = sin(phi) in [-1, 1], x = sin(theta), or sin(theta) + 3 behind the
 *     sphere, in [-1.5, 4.5] (x above 1.5 decodes as sin(theta) + 3; rounding lets sin(theta) pass 1 slightly near the poles);
 *   - rays: finite origin and a finite direction of unit length within 1e-3 (`distance` and `ignore` are not read);
 *   - light tokens: ECHO_TOKEN_EMPTY; an infinite light (ECHO_LIGHT_TYPE_INFINITE or _DELTA) below the scene's infinite count; a point
 *     light below its pack's point-light count; a Triangle / Sphere emitter of the pack the layers end in, its pack-swatch material in
 *     range. Other token types are refused;
 *   - surfaces: finite position and normal; samples: finite (then clamped); incident3 / directions3: finite, unit length within 1e-3.
 * Also refused with ECHO_B200_ERR_INVALID: a NULL scene (all a host without a device holds, since echo_b200_scene_create fails there),
 * an uncommitted scene, a scene without materials (interact and scatter calls), and a NULL required buffer with n > 0.
 */
#ifndef ECHO_B200_QUERY_H
#define ECHO_B200_QUERY_H

#include "echo_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- GeometryPoint (Aggregation/Primitives/GeometryPoint.cs:10-26): the origin of the light queries ---- */
typedef struct EchoSurface
{
	float position[3];
	float normal[3];
} EchoSurface;
ECHO_B200_ASSERT_SIZE(EchoSurface, 24);

/* ---- Contact (Aggregation/Primitives/Contact.cs:16-40) with GeometryShade (GeometryShade.cs) and its material ---- */
typedef struct EchoContact
{
	float position[3];    /* Contact.point.position: TraceQuery.Position (TraceQuery.cs:76-82) */
	float normal[3];      /* Contact.point.normal: geometric normal, world space */
	float shadeNormal[3]; /* GeometryShade.Normal after normal mapping (Material.ApplyNormalMapping, Material.cs:77-98), world space */
	float texcoord[2];    /* GeometryShade.Texcoord ((0, 0) on a scene without textures, as the renderer keeps it) */
	uint32_t material;    /* swatch index after the placement's offset (PreparedInstance.swatch); ECHO_TOKEN_EMPTY on a miss */
	float emission[3];    /* Emissive.Emit (Emissive.cs:64): what a path adds at this hit; 0 unless Emissive with positive power, facing the ray */
	uint32_t lobes;       /* BSDF.count, the functions Material.Scatter added; 0 = empty BSDF (Emissive), where a path ends */
} EchoContact;
ECHO_B200_ASSERT_SIZE(EchoContact, 64);

/* ---- BSDF.Sample's Probable<RGB128> and out values (BSDF.cs:150-208) ---- */
typedef struct EchoScatter
{
	float incident[3]; /* out Float3 incident, world space; 0 when impossible */
	float pdf;
	float value[3];    /* tint * sum of the matching functions' values, without the cosine */
	uint32_t specular; /* 1 when the sampled function (out BxDF function) is FunctionType.Specular */
} EchoScatter;
ECHO_B200_ASSERT_SIZE(EchoScatter, 32);

/* ---- PreparedScene.Sample (PreparedScene.cs:182-204): Probable<RGB128> and its out values ---- */
typedef struct EchoLightSample
{
	float radiance[3];
	float pdf;
	float incident[3]; /* out Float3 incident, world space */
	float travel;      /* out float travel: the occlusion distance (+inf for infinite lights) */
} EchoLightSample;
ECHO_B200_ASSERT_SIZE(EchoLightSample, 32);

/* PreparedScene.Interact + Material.Scatter for each (ray, hit, hit_layers) of a trace: what the path kernels make of a hit */
int32_t echo_b200_interact_batch(EchoScene*, const EchoRay* rays, const EchoHit* hits, const EchoTokenHierarchy* hit_layers, uint64_t n, EchoContact* out);
/* BSDF.Sample at the contact of each hit, with samples2[2 i .. 2 i + 1] (Sample2D) */
int32_t echo_b200_scatter_sample_batch(EchoScene*, const EchoRay* rays, const EchoHit* hits, const EchoTokenHierarchy* hit_layers, const float* samples2,
                                       uint64_t n, EchoScatter* out);
/* BSDF.Evaluate (RGB) and BSDF.ProbabilityDensity (W) at the contact of each hit towards incident3[3 i ..] */
int32_t echo_b200_scatter_evaluate_batch(EchoScene*, const EchoRay* rays, const EchoHit* hits, const EchoTokenHierarchy* hit_layers, const float* incident3,
                                         uint64_t n, float* out_rgba);
/* PreparedScene.Pick from each surface with samples1[i] (Sample1D): the light token, its hierarchy's layers (nullable) and pmf */
int32_t echo_b200_light_pick_batch(EchoScene*, const EchoSurface* points, const float* samples1, uint64_t n, uint32_t* tokens, EchoTokenHierarchy* layers,
                                   float* pmf);
/* PreparedScene.ProbabilityMass of each light token (with its hierarchy's layers) seen from each surface */
int32_t echo_b200_light_mass_batch(EchoScene*, const uint32_t* tokens, const EchoTokenHierarchy* layers, const EchoSurface* points, uint64_t n, float* pmf);
/* PreparedScene.Sample of each light token from each surface with samples2[2 i ..] (Sample2D) */
int32_t echo_b200_light_sample_batch(EchoScene*, const uint32_t* tokens, const EchoTokenHierarchy* layers, const EchoSurface* points, const float* samples2,
                                     uint64_t n, EchoLightSample* out);
/* PreparedScene.ProbabilityDensity of each light token from each surface towards incident3[3 i ..] */
int32_t echo_b200_light_pdf_batch(EchoScene*, const uint32_t* tokens, const EchoTokenHierarchy* layers, const EchoSurface* points, const float* incident3,
                                  uint64_t n, float* pdf);
/* PreparedScene.EvaluateInfinite along directions3[3 i ..]; direct != 0 sums only the DirectlyVisible lights (out_rgb3: 3 floats each) */
int32_t echo_b200_evaluate_infinite_batch(EchoScene*, const float* directions3, uint64_t n, int32_t direct, float* out_rgb3);

#ifdef __cplusplus
}
#endif
#endif
