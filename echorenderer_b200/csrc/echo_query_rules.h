// echo_query_rules.h — which inputs the batched PreparedScene queries accept (include/echo_b200_query.h,
// include/echo_b200_query_device.h), defined once for both sides: the host-buffer calls of api.cu run these rules on the host
// before anything is uploaded, the checked query kernels of render.cu run them on the device, one thread per query. Both must
// reach the same decision for the same input, so everything here is exact: bit tests for finiteness, and a unit length computed
// in double precision, where the products of floats are exact and contraction cannot change the sum (compile the host side with
// -ffp-contract=off all the same; the device build is -fmad=false).
//
// The rules are templated over how they reach the scene. `Scene` provides:
//   uint32_t packCount(), EchoPack pack(uint32_t), void instance(uint32_t, uint32_t& pack, uint32_t& materialOffset),
//   uint32_t triangleCount(), sphereCount(), pointLightCount(), infiniteLightCount(), materialCount(),
//   uint32_t triangleMaterial(uint32_t), sphereMaterial(uint32_t)
// over the whole arrays of the scene. Nothing is read with an index the rules have not accepted first; pack ranges and the pack of
// every placement are validated by echo_b200_scene_commit.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "../../include/echo_b200_query.h"

#if defined(__CUDACC__)
#define ECHO_RULE __host__ __device__ __forceinline__
// the templates below are host and device code; each instantiation only runs on the side its `Scene` lives on
#define ECHO_RULE_TEMPLATE _Pragma("nv_exec_check_disable") template<class Scene>
#else
#define ECHO_RULE inline
#define ECHO_RULE_TEMPLATE template<class Scene>
#endif

namespace echo
{
namespace rules
{

// why a query is refused: the low 8 bits of a device status word (echo_b200_query_device.h), and the message of a host-buffer call
enum Reason : uint32_t
{
	ACCEPTED = 0,
	LAYERS_WITHOUT_PACKS,
	TOO_MANY_LAYERS,
	LAYER_NOT_INSTANCE, // the host message names the layer: "layer k is not ..."
	RAY,
	HIT_NOT_FINITE,
	TRIANGLE_RANGE,
	TRIANGLE_UV,
	SPHERE_RANGE,
	SPHERE_UV,
	HIT_TOKEN,
	HIT_MATERIAL,
	INFINITE_RANGE,
	POINT_RANGE,
	LIGHT_TYPE,
	EMITTER_TRIANGLE_RANGE,
	EMITTER_SPHERE_RANGE,
	LIGHT_TOKEN,
	EMITTER_MATERIAL,
	SURFACE,
	SAMPLES,
	SAMPLE,
	INCIDENT,
	DIRECTION,
	REASON_COUNT
};

// the text of each reason; null for ACCEPTED and unknown codes
inline const char* reason_text(uint32_t code)
{
	static const char* const texts[REASON_COUNT] = {
		nullptr,
		"instance layers on a scene without packs",
		"more than ECHO_MAX_INSTANCE_LAYERS instance layers",
		"layer is not an instance of its parent pack",
		"the ray needs a finite origin and a unit direction",
		"hit distance or uv is not finite",
		"triangle index out of range for its pack",
		"triangle hit uv outside [0, 1]",
		"sphere index out of range for its pack",
		"sphere hit uv outside the encoding of SphereEntity",
		"hit token is neither a triangle, a sphere nor ECHO_TOKEN_EMPTY",
		"the hit's material index is out of range",
		"infinite light index out of range",
		"point light index out of range for its pack",
		"unknown light type",
		"triangle emitter index out of range for its pack",
		"sphere emitter index out of range for its pack",
		"light token is neither a light, a triangle, a sphere nor ECHO_TOKEN_EMPTY",
		"the emitter's material index is out of range",
		"the surface is not finite",
		"samples are not finite",
		"the sample is not finite",
		"the incident direction is not a finite unit vector",
		"the direction is not a finite unit vector",
	};
	return code < REASON_COUNT ? texts[code] : nullptr;
}

ECHO_RULE bool finite(float x)
{
#if defined(__CUDA_ARCH__)
	uint32_t bits = __float_as_uint(x);
#else
	uint32_t bits;
	memcpy(&bits, &x, sizeof bits);
#endif
	return (bits & 0x7F800000u) != 0x7F800000u;
}

ECHO_RULE bool all_finite(const float* values, int count)
{
	for (int i = 0; i < count; i++)
		if (!finite(values[i])) return false;
	return true;
}

ECHO_RULE bool unit_direction(const float* v)
{
	if (!all_finite(v, 3)) return false;
	double length = sqrt((double)v[0] * v[0] + (double)v[1] * v[1] + (double)v[2] * v[2]);
	return fabs(length - 1.0) <= 1e-3;
}

ECHO_RULE uint32_t token_kind(uint32_t token) { return token >> ECHO_TOKEN_INDEX_BITS; }
ECHO_RULE uint32_t token_number(uint32_t token) { return token & ((1u << ECHO_TOKEN_INDEX_BITS) - 1u); }

// FindLayer over the packs and placements: the pack hierarchy `layers` (null: empty) ends in and the swatch offset it selects.
// `failedLayer` is the layer a LAYER_NOT_INSTANCE refusal names.
ECHO_RULE_TEMPLATE
ECHO_RULE uint32_t check_layers(const Scene& scene, const EchoTokenHierarchy* layers, EchoPack& pack, uint32_t& materialOffset, uint32_t& failedLayer)
{
	if (scene.packCount() == 0u)
	{
		pack = EchoPack{};
		pack.triangleCount = scene.triangleCount();
		pack.sphereCount = scene.sphereCount();
		pack.pointLightCount = scene.pointLightCount();
	}
	else pack = scene.pack(0u);

	materialOffset = pack.materialOffset;
	const uint32_t count = layers ? layers->instanceCount : 0u;
	if (count == 0u) return ACCEPTED;
	if (scene.packCount() == 0u) return LAYERS_WITHOUT_PACKS;
	if (count > ECHO_MAX_INSTANCE_LAYERS) return TOO_MANY_LAYERS;

	for (uint32_t k = 0; k < count; k++)
	{
		const uint32_t token = layers->instances[k];
		if (token_kind(token) != ECHO_TOKEN_TYPE_INSTANCE || token_number(token) >= pack.instanceCount)
		{
			failedLayer = k;
			return LAYER_NOT_INSTANCE;
		}
		uint32_t next;
		scene.instance(pack.instanceOffset + token_number(token), next, materialOffset);
		pack = scene.pack(next);
	}

	return ACCEPTED;
}

ECHO_RULE_TEMPLATE
ECHO_RULE uint32_t check_hit(const Scene& scene, const EchoRay& ray, const EchoHit& hit, const EchoPack& pack, uint32_t materialOffset)
{
	if (!all_finite(ray.origin, 3) || !unit_direction(ray.direction)) return RAY;
	if (hit.token == ECHO_TOKEN_EMPTY) return ACCEPTED;
	if (!finite(hit.distance) || !all_finite(hit.uv, 2)) return HIT_NOT_FINITE;

	const uint32_t index = token_number(hit.token);
	const float x = hit.uv[0], y = hit.uv[1];
	uint32_t material;

	if (token_kind(hit.token) == ECHO_TOKEN_TYPE_TRIANGLE)
	{
		if (index >= pack.triangleCount) return TRIANGLE_RANGE;
		if (!(x >= 0.0f && x <= 1.0f && y >= 0.0f && y <= 1.0f)) return TRIANGLE_UV;
		material = scene.triangleMaterial(pack.triangleOffset + index);
	}
	else if (token_kind(hit.token) == ECHO_TOKEN_TYPE_SPHERE)
	{
		if (index >= pack.sphereCount) return SPHERE_RANGE;
		// x = sin(theta), plus 3 behind the sphere; sin(theta) = point.x / sqrt(r^2 - y^2) may pass 1 by rounding near the poles
		if (!(y >= -1.0f && y <= 1.0f && x >= -1.5f && x <= 4.5f)) return SPHERE_UV;
		material = scene.sphereMaterial(pack.sphereOffset + index);
	}
	else return HIT_TOKEN;

	return (uint64_t)materialOffset + material >= scene.materialCount() ? HIT_MATERIAL : ACCEPTED;
}

ECHO_RULE_TEMPLATE
ECHO_RULE uint32_t check_light(const Scene& scene, uint32_t token, const EchoPack& pack)
{
	if (token == ECHO_TOKEN_EMPTY) return ACCEPTED;
	const uint32_t index = token_number(token);

	if (token_kind(token) == ECHO_TOKEN_TYPE_LIGHT)
	{
		const uint32_t lightType = index >> ECHO_LIGHT_INDEX_BITS, lightIndex = index & ((1u << ECHO_LIGHT_INDEX_BITS) - 1u);
		if (lightType == ECHO_LIGHT_TYPE_INFINITE || lightType == ECHO_LIGHT_TYPE_INFINITE_DELTA) return lightIndex < scene.infiniteLightCount() ? ACCEPTED : INFINITE_RANGE;
		if (lightType == ECHO_LIGHT_TYPE_POINT) return lightIndex < pack.pointLightCount ? ACCEPTED : POINT_RANGE;
		return LIGHT_TYPE;
	}

	uint32_t material;

	if (token_kind(token) == ECHO_TOKEN_TYPE_TRIANGLE)
	{
		if (index >= pack.triangleCount) return EMITTER_TRIANGLE_RANGE;
		material = scene.triangleMaterial(pack.triangleOffset + index);
	}
	else if (token_kind(token) == ECHO_TOKEN_TYPE_SPHERE)
	{
		if (index >= pack.sphereCount) return EMITTER_SPHERE_RANGE;
		material = scene.sphereMaterial(pack.sphereOffset + index);
	}
	else return LIGHT_TOKEN;

	return (uint64_t)pack.materialOffset + material >= scene.materialCount() ? EMITTER_MATERIAL : ACCEPTED;
}

// interact / scatter_sample / scatter_evaluate: `values` holds `valueCount` floats of this query (2: samples, 3: an incident direction)
ECHO_RULE_TEMPLATE
ECHO_RULE uint32_t check_contact(const Scene& scene, const EchoTokenHierarchy* layers, const EchoRay& ray, const EchoHit& hit, const float* values, int valueCount,
                                 uint32_t& failedLayer)
{
	EchoPack pack;
	uint32_t materialOffset;
	uint32_t code = check_layers(scene, layers, pack, materialOffset, failedLayer);
	if (code == ACCEPTED) code = check_hit(scene, ray, hit, pack, materialOffset);
	if (code == ACCEPTED && valueCount == 2 && !all_finite(values, 2)) code = SAMPLES;
	if (code == ACCEPTED && valueCount == 3 && !unit_direction(values)) code = INCIDENT;
	return code;
}

// mass / sample / pdf of a light token seen from a surface; `values` as above
ECHO_RULE_TEMPLATE
ECHO_RULE uint32_t check_light_query(const Scene& scene, const EchoTokenHierarchy* layers, uint32_t token, const EchoSurface& point, const float* values, int valueCount,
                                     uint32_t& failedLayer)
{
	EchoPack pack;
	uint32_t materialOffset;
	uint32_t code = check_layers(scene, layers, pack, materialOffset, failedLayer);
	if (code == ACCEPTED) code = check_light(scene, token, pack);
	if (code == ACCEPTED && (!all_finite(point.position, 3) || !all_finite(point.normal, 3))) code = SURFACE;
	if (code == ACCEPTED && valueCount == 2 && !all_finite(values, 2)) code = SAMPLES;
	if (code == ACCEPTED && valueCount == 3 && !unit_direction(values)) code = INCIDENT;
	return code;
}

ECHO_RULE uint32_t check_pick(const EchoSurface& point, float sample)
{
	if (!all_finite(point.position, 3) || !all_finite(point.normal, 3)) return SURFACE;
	return finite(sample) ? ACCEPTED : SAMPLE;
}

ECHO_RULE uint32_t check_infinite(const float* direction) { return unit_direction(direction) ? ACCEPTED : DIRECTION; }

} // namespace rules
} // namespace echo
