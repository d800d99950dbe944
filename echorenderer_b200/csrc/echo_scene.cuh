// echo_scene.cuh — device-resident scene layout (HBM) and the QBVH closest-hit / occlusion traversal.
//
// Layout (see DESIGN.md "Data layout in HBM"):
//   nodes       8 x float4 per node — the reference's 128-byte QuadBoundingVolumeHierarchy.Node verbatim
//               (QuadBoundingVolumeHierarchy.cs:406-469): 6 x float4 SoA bounds, then {axisMajor, axisMinor0,
//               axisMinor1, token0}, {token1, token2, token3, pad}. One node = one 128-byte line = 8 LDG.128.
//   triHot      3 x float4 per triangle: vertex0, edge1, edge2 (the 36 bytes Möller–Trumbore reads, padded to 48)
//   triShade    3 x float4 per triangle: shading normals, .w of the first = material index bits
//   spheres     float4 {position, radius}; sphereMaterial u32
// Traversal order, culling tests and leaf acceptance follow the reference exactly (QuadBoundingVolumeHierarchy.cs:123-315,
// GeometryCollection.cs:85-171) so that hit tokens agree bit for bit, ties and near-ties included.
#pragma once
#include "../../include/echo_b200.h"
#include "echo_device_math.cuh"

namespace echo
{

struct DeviceScene
{
	const float4* nodes;
	const float4* triHot;
	const float4* triShade;
	const float4* spheres;
	const uint32_t* sphereMaterial;
	const float4* materials;       // 4 x float4 per EchoMaterial
	const float4* lightNodes;      // 4 x float4 per EchoLightNode
	const uint32_t* emitterTokens; // sorted ascending
	const uint64_t* emitterPaths;  // LightTree.map values, parallel to emitterTokens
	const float4* pointLights;     // 2 x float4: {intensity, 0}, {position, 0}
	const float4* infiniteLights;  // 10 x float4 per EchoInfiniteLight
	const float* distributions;    // DiscreteDistribution2D cdf values of the environment lights
	const uint4* textures;         // 2 x uint4 per EchoTexture; null without image textures
	const float4* texels;          // RGBA128 texels of every texture back to back
	const uint4* materialTextures; // 2 x uint4 per EchoMaterialTextures, parallel to materials
	const float4* triTexcoord;     // 2 x float4 per triangle: texcoord0.xy texcoord1.xy | texcoord2.xy - - (only with textures)
	const uint4* packs;            // 4 x uint4 per EchoPack; null when the scene is a single pack
	const float4* instances;       // 8 x float4 per EchoInstance

	unsigned int* violations;      // ECHO_BOUNDS_CHECK builds: bit k set = check k failed somewhere (see ECHO_CHECK); null otherwise
	unsigned long long* lightVisits; // counted passes only (ECHO_EVALUATOR_COUNT_VISITS): LightBound.Importance evaluations; null otherwise

	uint32_t nodeCount, triangleCount, sphereCount, materialCount;
	uint32_t lightNodeCount, emitterCount, pointLightCount, infiniteLightCount;
	uint32_t maxDepth;             // quad depth whose 3 * maxDepth + 1 stack entries serve the deepest chain of packs
	uint32_t packCount, instanceCount, textureCount;
	uint32_t texelCount, distributionCount; // extents of `texels` and `distributions`, for the bounds-check build
	float infiniteThreshold, infinitePdf;
	float boundRadius; // Accelerator.SphereBound.radius, read by the NormalDepth evaluator

	EchoCamera camera;
};

// compute-sanitizer is not available on the GPU pool, so the library can be built with -DECHO_BOUNDS_CHECK (variants/bounds.sh):
// every index the kernels derive from scene data or from a stack pointer is then checked before use and a failure sets a bit
// that tests read back through echo_b200_debug_bounds_violations. Release builds compile the checks out.
enum : int
{
	CHECK_NODE = 0, CHECK_TRIANGLE, CHECK_SPHERE, CHECK_STACK, CHECK_INSTANCE, CHECK_PACK, CHECK_MATERIAL, CHECK_LIGHT_NODE, CHECK_EMITTER,
	CHECK_POINT_LIGHT, CHECK_INFINITE_LIGHT, CHECK_TEXTURE, CHECK_TEXEL, CHECK_DISTRIBUTION, CHECK_LAYER
};

#ifdef ECHO_BOUNDS_CHECK
#define ECHO_CHECK(scene, condition, code) do { if (!(condition) && (scene).violations) atomicOr((scene).violations, 1u << (code)); } while (0)
#else
#define ECHO_CHECK(scene, condition, code) do {} while (0)
#endif

struct VisitCounts
{
	uint32_t nodes, triangles, spheres;
};

// a per-thread counter summed over the warp and added to stats[slot] by lane 0, one atomic per warp and none for a zero sum;
// every lane of the warp must call it
ECHO_DEVICE void warp_add(unsigned long long* stats, int slot, uint32_t value)
{
	for (int offset = 16; offset > 0; offset >>= 1) value += __shfl_down_sync(0xFFFFFFFFu, value, offset);
	if ((threadIdx.x & 31u) == 0u && value) atomicAdd(stats + slot, (unsigned long long)value);
}

// the visit counters of one thread's queries into stats[firstSlot], [firstSlot + 1], [firstSlot + 2]
ECHO_DEVICE void visit_flush(unsigned long long* stats, int firstSlot, VisitCounts local)
{
	warp_add(stats, firstSlot + 0, local.nodes);
	warp_add(stats, firstSlot + 1, local.triangles);
	warp_add(stats, firstSlot + 2, local.spheres);
}

ECHO_DEVICE uint32_t token_type(uint32_t token) { return token >> ECHO_TOKEN_INDEX_BITS; }
ECHO_DEVICE uint32_t token_index(uint32_t token) { return token & ((1u << ECHO_TOKEN_INDEX_BITS) - 1u); }
ECHO_DEVICE bool token_is_geometry(uint32_t token) { return (token_type(token) - 1u) <= 2u; } // Triangle, Sphere, Instance

// ---- PreparedTriangle.IntersectImpl(out uv), TriangleEntity.cs:204-235 ----
ECHO_DEVICE float triangle_intersect(vec3 vertex0, vec3 edge1, vec3 edge2, vec3 origin, vec3 direction, vec2& uv)
{
	vec3 cross2 = cross(direction, edge2);
	float determinant = dot(edge1, cross2);

	if (determinant == 0.0f) return kInfinity;
	float determinantR = rcp(determinant);

	vec3 offset = origin - vertex0;
	float u = dot(offset, cross2) * determinantR;
	uv.x = u;

	if ((u < 0.0f) | (u > 1.0f)) return kInfinity;

	vec3 cross1 = cross(offset, edge1);
	float v = dot(direction, cross1) * determinantR;
	uv.y = v;

	if ((v < 0.0f) | (u + v > 1.0f)) return kInfinity;

	float distance = dot(edge2, cross1) * determinantR;
	return distance < 0.0f ? kInfinity : distance;
}

// ---- PreparedTriangle.IntersectImpl(travel), TriangleEntity.cs:237-263 ----
ECHO_DEVICE bool triangle_occlude(vec3 vertex0, vec3 edge1, vec3 edge2, vec3 origin, vec3 direction, float travel)
{
	vec3 cross2 = cross(direction, edge2);
	float determinant = dot(edge1, cross2);

	if (determinant == 0.0f) return false;
	float sign = determinant < 0.0f ? -1.0f : 1.0f;
	determinant *= sign;

	vec3 offset = origin - vertex0;
	float u = dot(offset, cross2) * sign;

	if ((u < 0.0f) | (u > determinant)) return false;

	vec3 cross1 = cross(offset, edge1);
	float v = dot(direction, cross1) * sign;

	if ((v < 0.0f) | (u + v > determinant)) return false;

	float distance = dot(edge2, cross1) * sign;
	return (distance >= 0.0f) & (distance < travel * determinant);
}

constexpr float kSphereDistanceThreshold = 6E-4f; // SphereEntity.cs:79

// ---- PreparedSphere.Intersect(out uv), SphereEntity.cs:88-126 ----
ECHO_DEVICE float sphere_intersect(float4 sphere, vec3 origin, vec3 direction, vec2& uv, bool findFar)
{
	float radius = sphere.w;
	vec3 offset = origin - vec3{ sphere.x, sphere.y, sphere.z };
	float radius2 = radius * radius;
	float center = -dot(offset, direction);

	float extend2 = fma_f(center, center, radius2 - squared_magnitude(offset));
	if (extend2 < 0.0f) return kInfinity;

	float extend = sqrt0(extend2);
	float distance = center - extend;

	float threshold = findFar ? kSphereDistanceThreshold : 0.0f;

	if (distance < threshold) distance = center + extend;
	if (distance < threshold) return kInfinity;

	vec3 point = offset + direction * distance;
	float sinP = clamp11(div(point.y, radius));
	float sinT = 0.0f;

	float smallRadius = fma_f(-point.y, point.y, radius2);
	if (smallRadius > 0.0f) sinT = point.x * sqrt_r0(smallRadius);
	if (point.z < 0.0f) sinT += 3.0f;

	uv = { sinT, sinP };
	return distance;
}

// ---- PreparedSphere.Intersect(travel), SphereEntity.cs:129-148 ----
ECHO_DEVICE bool sphere_occlude(float4 sphere, vec3 origin, vec3 direction, float travel, bool findFar)
{
	float radius = sphere.w;
	vec3 offset = origin - vec3{ sphere.x, sphere.y, sphere.z };
	float center = -dot(offset, direction);

	float squared = fma_f(radius, radius, -squared_magnitude(offset));
	float extend2 = fma_f(center, center, squared);
	if (extend2 < 0.0f) return false;

	float extend = sqrt0(extend2);
	float distance = center - extend;

	float threshold = findFar ? kSphereDistanceThreshold : 0.0f;

	if (distance < threshold) distance = center + extend;
	return distance >= threshold && distance < travel;
}

// ---- BoxBound4.Intersect, BoxBound4.cs:64-112, one lane ----
ECHO_DEVICE float slab(float minX, float minY, float minZ, float maxX, float maxY, float maxZ, vec3 origin, vec3 directionR)
{
	float length0 = (minX - origin.x) * directionR.x;
	float length1 = (maxX - origin.x) * directionR.x;

	float far = max_sse(length0, length1);
	float near = min_sse(length0, length1);

	length0 = (minY - origin.y) * directionR.y;
	length1 = (maxY - origin.y) * directionR.y;

	far = min_sse(far, max_sse(length0, length1));
	near = max_sse(near, min_sse(length0, length1));

	length0 = (minZ - origin.z) * directionR.z;
	length1 = (maxZ - origin.z) * directionR.z;

	far = min_sse(far, max_sse(length0, length1));
	near = max_sse(near, min_sse(length0, length1));

	far *= 1.00000024f; // BoxBound.FarMultiplier, BoxBound.cs:67

	return ((far >= near) & (far >= 0.0f)) ? near : kInfinity;
}

ECHO_DEVICE float select4(int slot, float v0, float v1, float v2, float v3) { return (slot & 2) ? ((slot & 1) ? v3 : v2) : ((slot & 1) ? v1 : v0); }
ECHO_DEVICE uint32_t select4(int slot, uint32_t v0, uint32_t v1, uint32_t v2, uint32_t v3) { return (slot & 2) ? ((slot & 1) ? v3 : v2) : ((slot & 1) ? v1 : v0); }

// The four Push calls of one node visit, in the reference's order, as 2-bit slot fields (first push in bits 0-1).
// orders: bit a = directionR[a] > 0 for a in 0..2, bit 3 = 1 (QuadBoundingVolumeHierarchy.cs:132-138,151-198).
ECHO_DEVICE uint32_t visit_order(uint32_t orders, int axisMajor, int axisMinor0, int axisMinor1)
{
	uint32_t oMajor = (orders >> axisMajor) & 1u;
	uint32_t o0 = (orders >> axisMinor0) & 1u;
	uint32_t o1 = (orders >> axisMinor1) & 1u;

	uint32_t pair0 = o0 ? (1u | (0u << 2)) : (0u | (1u << 2)); // slots of the first pair: {1,0} or {0,1}
	uint32_t pair1 = o1 ? (3u | (2u << 2)) : (2u | (3u << 2)); // slots of the second pair: {3,2} or {2,3}

	return oMajor ? (pair1 | (pair0 << 4)) : (pair0 | (pair1 << 4));
}

struct NodeData
{
	float4 minX, minY, minZ, maxX, maxY, maxZ;
	uint32_t token0, token1, token2, token3;
	uint32_t order;
};

ECHO_DEVICE void load_node(const DeviceScene& scene, uint32_t index, uint32_t orders, NodeData& node)
{
	ECHO_CHECK(scene, index < scene.nodeCount, CHECK_NODE);
	const float4* base = scene.nodes + (size_t)index * 8;
	node.minX = __ldg(base + 0);
	node.minY = __ldg(base + 1);
	node.minZ = __ldg(base + 2);
	node.maxX = __ldg(base + 3);
	node.maxY = __ldg(base + 4);
	node.maxZ = __ldg(base + 5);
	float4 a = __ldg(base + 6);
	float4 b = __ldg(base + 7);
	node.token0 = __float_as_uint(a.w);
	node.token1 = __float_as_uint(b.x);
	node.token2 = __float_as_uint(b.y);
	node.token3 = __float_as_uint(b.z);
	node.order = visit_order(orders, __float_as_int(a.x), __float_as_int(a.y), __float_as_int(a.z));
}

// ---- QuadBoundingVolumeHierarchy.TraceImpl (:123-219) + GeometryCollection.Trace (:85-134) ----
// `distance` is TraceQuery.distance (in: limit, out: closest hit); token/uv are written only when a hit is accepted.
template<int STACK, bool COUNT>
ECHO_DEVICE void trace_closest(const DeviceScene& scene, vec3 origin, vec3 direction, uint32_t ignore,
                               float& distance, uint32_t& token, vec2& uv, VisitCounts* counts)
{
	vec3 directionR = { rcp(direction.x), rcp(direction.y), rcp(direction.z) }; // Ray.cs:23
	uint32_t orders = (directionR.x > 0.0f ? 1u : 0u) | (directionR.y > 0.0f ? 2u : 0u) | (directionR.z > 0.0f ? 4u : 0u) | 8u;

	uint2 stack[STACK];
	int next = 0;
	stack[next++] = make_uint2(0u, __float_as_uint(0.0f)); // NewNodeToken(0), hit 0

	do
	{
		uint2 entry = stack[--next];
		if (__uint_as_float(entry.y) >= distance) continue;

		NodeData node;
		load_node(scene, token_index(entry.x), orders, node);
		if (COUNT) ++counts->nodes;

		float t0 = slab(node.minX.x, node.minY.x, node.minZ.x, node.maxX.x, node.maxY.x, node.maxZ.x, origin, directionR);
		float t1 = slab(node.minX.y, node.minY.y, node.minZ.y, node.maxX.y, node.maxY.y, node.maxZ.y, origin, directionR);
		float t2 = slab(node.minX.z, node.minY.z, node.minZ.z, node.maxX.z, node.maxY.z, node.maxZ.z, origin, directionR);
		float t3 = slab(node.minX.w, node.minY.w, node.minZ.w, node.maxX.w, node.maxY.w, node.maxZ.w, origin, directionR);

		uint32_t order = node.order;

#pragma unroll 1
		for (int k = 0; k < 4; k++, order >>= 2)
		{
			int slot = order & 3;
			float hit = select4(slot, t0, t1, t2, t3);
			if (hit >= distance) continue; // Push: :203-205

			uint32_t child = select4(slot, node.token0, node.token1, node.token2, node.token3);
			uint32_t type = token_type(child);

			if (type == ECHO_TOKEN_TYPE_NODE)
			{
				ECHO_CHECK(scene, next < STACK, CHECK_STACK);
				stack[next++] = make_uint2(child, __float_as_uint(hit));
			}
			else if (type == ECHO_TOKEN_TYPE_TRIANGLE)
			{
				if (child == ignore) continue; // GeometryCollection.cs:93-94
				if (COUNT) ++counts->triangles;
				ECHO_CHECK(scene, token_index(child) < scene.triangleCount, CHECK_TRIANGLE);

				const float4* data = scene.triHot + (size_t)token_index(child) * 3;
				float4 a = __ldg(data), b = __ldg(data + 1), c = __ldg(data + 2);

				vec2 hitUV;
				float d = triangle_intersect({ a.x, a.y, a.z }, { b.x, b.y, b.z }, { c.x, c.y, c.z }, origin, direction, hitUV);

				if (!(d >= distance)) // "if (distance >= query.distance) return", :99 (a NaN distance is accepted, like the reference)
				{
					distance = d;
					token = child;
					uv = hitUV;
				}
			}
			else if (type == ECHO_TOKEN_TYPE_SPHERE)
			{
				if (COUNT) ++counts->spheres;
				ECHO_CHECK(scene, token_index(child) < scene.sphereCount, CHECK_SPHERE);

				vec2 hitUV;
				float d = sphere_intersect(__ldg(scene.spheres + token_index(child)), origin, direction, hitUV, child == ignore);

				if (!(d >= distance))
				{
					distance = d;
					token = child;
					uv = hitUV;
				}
			}
		}
	}
	while (next != 0);
}

// ---- QuadBoundingVolumeHierarchy.OccludeImpl (:223-315) + GeometryCollection.Occlude (:140-171) ----
template<int STACK, bool COUNT>
ECHO_DEVICE bool trace_any(const DeviceScene& scene, vec3 origin, vec3 direction, uint32_t ignore, float travel, VisitCounts* counts)
{
	vec3 directionR = { rcp(direction.x), rcp(direction.y), rcp(direction.z) };
	uint32_t orders = (directionR.x > 0.0f ? 1u : 0u) | (directionR.y > 0.0f ? 2u : 0u) | (directionR.z > 0.0f ? 4u : 0u) | 8u;

	uint32_t stack[STACK];
	int next = 0;
	stack[next++] = 0u;

	do
	{
		NodeData node;
		load_node(scene, token_index(stack[--next]), orders, node);
		if (COUNT) ++counts->nodes;

		float t0 = slab(node.minX.x, node.minY.x, node.minZ.x, node.maxX.x, node.maxY.x, node.maxZ.x, origin, directionR);
		float t1 = slab(node.minX.y, node.minY.y, node.minZ.y, node.maxX.y, node.maxY.y, node.maxZ.y, origin, directionR);
		float t2 = slab(node.minX.z, node.minY.z, node.minZ.z, node.maxX.z, node.maxY.z, node.maxZ.z, origin, directionR);
		float t3 = slab(node.minX.w, node.minY.w, node.minZ.w, node.maxX.w, node.maxY.w, node.maxZ.w, origin, directionR);

		uint32_t order = node.order;

#pragma unroll 1
		for (int k = 0; k < 4; k++, order >>= 2)
		{
			int slot = order & 3;
			float hit = select4(slot, t0, t1, t2, t3);
			if (hit >= travel) continue;

			uint32_t child = select4(slot, node.token0, node.token1, node.token2, node.token3);
			uint32_t type = token_type(child);

			if (type == ECHO_TOKEN_TYPE_NODE)
			{
				ECHO_CHECK(scene, next < STACK, CHECK_STACK);
				stack[next++] = child;
			}
			else if (type == ECHO_TOKEN_TYPE_TRIANGLE)
			{
				if (child == ignore) continue;
				if (COUNT) ++counts->triangles;
				ECHO_CHECK(scene, token_index(child) < scene.triangleCount, CHECK_TRIANGLE);

				const float4* data = scene.triHot + (size_t)token_index(child) * 3;
				float4 a = __ldg(data), b = __ldg(data + 1), c = __ldg(data + 2);
				if (triangle_occlude({ a.x, a.y, a.z }, { b.x, b.y, b.z }, { c.x, c.y, c.z }, origin, direction, travel)) return true;
			}
			else if (type == ECHO_TOKEN_TYPE_SPHERE)
			{
				if (COUNT) ++counts->spheres;
				ECHO_CHECK(scene, token_index(child) < scene.sphereCount, CHECK_SPHERE);
				if (sphere_occlude(__ldg(scene.spheres + token_index(child)), origin, direction, travel, child == ignore)) return true;
			}
		}
	}
	while (next != 0);

	return false;
}

// ---- PreparedScene.Trace / Occlude guards, PreparedScene.cs:66-86 ----
template<int STACK, bool COUNT>
ECHO_DEVICE bool scene_trace(const DeviceScene& scene, vec3 origin, vec3 direction, uint32_t ignore,
                             float& distance, uint32_t& token, vec2& uv, VisitCounts* counts)
{
	if (!positive(distance)) return false;
	float original = distance;
	trace_closest<STACK, COUNT>(scene, origin, direction, ignore, distance, token, uv, counts);
	return distance < original;
}

template<int STACK, bool COUNT>
ECHO_DEVICE bool scene_occlude(const DeviceScene& scene, vec3 origin, vec3 direction, uint32_t ignore, float travel, VisitCounts* counts)
{
	if (!positive(travel)) return false;
	return trace_any<STACK, COUNT>(scene, origin, direction, ignore, travel, counts);
}

} // namespace echo
