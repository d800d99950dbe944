// echo_instanced.cuh — closest-hit / occlusion traversal through instanced packs (SURVEY.md §8f rank 2).
//
// Reference: GeometryCollection.Trace / Occlude on a TokenType.Instance leaf push the token on the query's TokenHierarchy
// and call PreparedInstance.Trace / Occlude (GeometryCollection.cs:123-131,160-168), which transforms the ray into the
// pack's local space, scales the distance, runs the pack's own accelerator and restores the ray
// (PreparedInstance.cs:47-83,105-111). The recursion happens in the middle of a node visit of the parent accelerator
// (leaves are intersected at push time), so it is restated here as an explicit frame stack: entering an instance saves
// the parent's ray, node and slot position; when the child's part of the traversal stack runs empty the frame is popped,
// `distance *= inverseScale` (or the old travel is restored) and the parent's node visit resumes at the next slot. The
// slab distances of the resumed node are recomputed — they depend only on the parent ray, so they are the same bits.
// One traversal stack serves all layers (the reference stackallocs one per recursion): commit checks that the deepest
// chain of packs fits.
#pragma once
#include "echo_scene.cuh"

namespace echo
{

struct InstanceFrame
{
	vec3 origin, direction;
	float travel;      // OccludeQuery.travel before the instance was entered (PreparedInstance.cs:66,79)
	uint32_t node;     // parent node token whose visit is suspended
	uint32_t position; // next slot (0..4) of that visit
	uint32_t base;     // parent's stack base
	uint32_t pack;     // parent pack
	uint32_t instance; // global instance index (for inverseScale)
};

struct PackView
{
	uint32_t nodeOffset, triangleOffset, sphereOffset, instanceOffset;
};

// EchoInstance, 128 bytes = 8 float4: forward rows 0..2, inverse rows 3..5, {forwardScale, inverseScale, pack, materialOffset}, reserved
ECHO_DEVICE const float4* instance_data(const DeviceScene& scene, uint32_t instance) { return scene.instances + (size_t)instance * 8; }

// everything shading needs to know about a pack (EchoPack): geometry offsets, its own swatch, its light tree ranges
struct PackInfo
{
	uint32_t triangleOffset, sphereOffset, instanceOffset, materialOffset;
	uint32_t lightNodeOffset, lightNodeCount, emitterOffset, emitterCount, pointLightOffset;
};

ECHO_DEVICE PackInfo whole_scene_pack(const DeviceScene& scene) // a scene without packs is one pack
{
	return { 0u, 0u, 0u, 0u, 0u, scene.lightNodeCount, 0u, scene.emitterCount, 0u };
}

ECHO_DEVICE PackInfo load_pack_info(const DeviceScene& scene, uint32_t pack)
{
	if (scene.packCount == 0u) return whole_scene_pack(scene);
	ECHO_CHECK(scene, pack < scene.packCount, CHECK_PACK);
	const uint4* data = scene.packs + (size_t)pack * 4;
	uint4 a = __ldg(data), b = __ldg(data + 1), c = __ldg(data + 2), d = __ldg(data + 3);
	// a = nodeOffset nodeCount maxDepth triangleOffset | b = triangleCount sphereOffset sphereCount instanceOffset
	// c = instanceCount materialOffset lightNodeOffset lightNodeCount | d = emitterOffset emitterCount pointLightOffset pointLightCount
	return { a.w, b.y, b.w, c.y, c.z, c.w, d.x, d.y, d.z };
}

// rows 0..2 of an affine Float4x4 (the bottom row is 0 0 0 1)
struct Transform
{
	float m[12];
};

ECHO_DEVICE Transform identity_transform() { return { { 1.0f, 0.0f, 0.0f, 0.0f, 0.0f, 1.0f, 0.0f, 0.0f, 0.0f, 0.0f, 1.0f, 0.0f } }; }

ECHO_DEVICE vec3 transform_point(const Transform& t, vec3 p) // Float4x4.MultiplyPoint, Float4x4.cs:260-265
{
	const float* m = t.m;
	return { m[0] * p.x + m[1] * p.y + m[2] * p.z + m[3], m[4] * p.x + m[5] * p.y + m[6] * p.z + m[7], m[8] * p.x + m[9] * p.y + m[10] * p.z + m[11] };
}

ECHO_DEVICE vec3 transform_direction(const Transform& t, vec3 d) // Float4x4.MultiplyDirection, Float4x4.cs:267-272
{
	const float* m = t.m;
	return { m[0] * d.x + m[1] * d.y + m[2] * d.z, m[4] * d.x + m[5] * d.y + m[6] * d.z, m[8] * d.x + m[9] * d.y + m[10] * d.z };
}

// Utility.GetScale (Utility.cs:82): Float4 Magnitude of row 0 with W = 0 = SqrtScalar((x*x + y*y) + (z*z + 0)), Float4.cs:51-61,73-81
ECHO_DEVICE float transform_scale(const Transform& t) { return __fsqrt_rn((t.m[0] * t.m[0] + t.m[1] * t.m[1]) + (t.m[2] * t.m[2] + 0.0f)); }

// Float4x4 operator * (Float4x4.cs:352-358) of two affine matrices: `first` straight from an EchoInstance's rows
ECHO_DEVICE Transform multiply_rows(const float4* first, const Transform& second)
{
	Transform result;

#pragma unroll
	for (int i = 0; i < 3; i++)
	{
		float4 a = __ldg(first + i);

#pragma unroll
		for (int j = 0; j < 4; j++)
		{
			float bottom = j == 3 ? 1.0f : 0.0f; // second.f3j
			result.m[i * 4 + j] = a.x * second.m[j] + a.y * second.m[4 + j] + a.z * second.m[8 + j] + a.w * bottom;
		}
	}

	return result;
}

// the instance layers of a TokenHierarchy as the wavefront stores them: 8 words {count, 5 tokens, 2 pad}
struct PathLayers
{
	uint32_t count;
	uint32_t tokens[ECHO_MAX_INSTANCE_LAYERS];
};

ECHO_DEVICE PathLayers no_layers() { return { 0u, { 0u, 0u, 0u, 0u, 0u } }; }

ECHO_DEVICE PathLayers load_layers(const uint4* buffer, uint32_t slot)
{
	uint4 a = buffer[(size_t)slot * 2], b = buffer[(size_t)slot * 2 + 1];
	return { a.x, { a.y, a.z, a.w, b.x, b.y } };
}

ECHO_DEVICE void store_layers(uint4* buffer, uint32_t slot, const PathLayers& layers)
{
	buffer[(size_t)slot * 2] = make_uint4(layers.count, layers.tokens[0], layers.tokens[1], layers.tokens[2]);
	buffer[(size_t)slot * 2 + 1] = make_uint4(layers.tokens[3], layers.tokens[4], 0u, 0u);
}

// PreparedScene.FindLayer (PreparedScene.cs:255-277). Both products put the new placement on the LEFT, as the reference
// does (:272-273): for the inverse transform of nested placements that is not the geometric order, and it is kept.
struct Layer
{
	Transform forward, inverse;
	uint32_t pack;           // the pack the hierarchy ends in
	uint32_t materialOffset; // its placement's swatch (PreparedInstance.swatch); the scene's own without layers
	PackInfo info;
};

template<bool INST>
ECHO_DEVICE Layer find_layer(const DeviceScene& scene, const PathLayers& layers)
{
	Layer layer;
	layer.forward = identity_transform();
	layer.inverse = identity_transform();
	layer.pack = 0u;
	layer.materialOffset = 0u;

	if (!INST)
	{
		layer.info = whole_scene_pack(scene);
		return layer;
	}

	layer.info = load_pack_info(scene, 0u);
	layer.materialOffset = layer.info.materialOffset;

	for (uint32_t k = 0; k < layers.count; k++)
	{
		ECHO_CHECK(scene, layers.count <= ECHO_MAX_INSTANCE_LAYERS, CHECK_LAYER);
		ECHO_CHECK(scene, layer.info.instanceOffset + token_index(layers.tokens[k]) < scene.instanceCount, CHECK_INSTANCE);
		const float4* data = instance_data(scene, layer.info.instanceOffset + token_index(layers.tokens[k]));
		layer.forward = multiply_rows(data, layer.forward);
		layer.inverse = multiply_rows(data + 3, layer.inverse);
		float4 tail = __ldg(data + 6);
		layer.pack = __float_as_uint(tail.z);
		layer.materialOffset = __float_as_uint(tail.w);
		layer.info = load_pack_info(scene, layer.pack);
	}

	return layer;
}

ECHO_DEVICE PackView load_pack(const DeviceScene& scene, uint32_t pack)
{
	ECHO_CHECK(scene, pack < scene.packCount, CHECK_PACK);
	const uint4* data = scene.packs + (size_t)pack * 4; // EchoPack, 64 bytes
	uint4 a = __ldg(data), b = __ldg(data + 1), c = __ldg(data + 2);
	// a = nodeOffset nodeCount maxDepth triangleOffset | b = triangleCount sphereOffset sphereCount instanceOffset | c = instanceCount materialOffset ..
	(void)c;
	return { a.x, a.w, b.y, b.w };
}

ECHO_DEVICE vec3 multiply_point(const float4* rows, vec3 p) // Float4x4.MultiplyPoint, Float4x4.cs:260-265
{
	float4 r0 = __ldg(rows), r1 = __ldg(rows + 1), r2 = __ldg(rows + 2);
	return { r0.x * p.x + r0.y * p.y + r0.z * p.z + r0.w, r1.x * p.x + r1.y * p.y + r1.z * p.z + r1.w, r2.x * p.x + r2.y * p.y + r2.z * p.z + r2.w };
}

ECHO_DEVICE vec3 multiply_direction(const float4* rows, vec3 d) // Float4x4.MultiplyDirection, Float4x4.cs:267-272
{
	float4 r0 = __ldg(rows), r1 = __ldg(rows + 1), r2 = __ldg(rows + 2);
	return { r0.x * d.x + r0.y * d.y + r0.z * d.z, r1.x * d.x + r1.y * d.y + r1.z * d.z, r2.x * d.x + r2.y * d.y + r2.z * d.z };
}


// TokenHierarchy equality of the query's `ignore` and `current` instance layers (TokenHierarchy.cs:117-129)
ECHO_DEVICE bool layers_match(const uint32_t* ignoreLayers, uint32_t ignoreCount, const uint32_t* current, uint32_t level)
{
	if (ignoreCount != level) return false;
	for (uint32_t k = 0; k < level; k++) if (ignoreLayers[k] != current[k]) return false;
	return true;
}

// ANY = false: QuadBoundingVolumeHierarchy.TraceImpl (:123-219); `distance` in: TraceQuery.distance, out: closest hit;
//              token / uv / hitLayers[0..hitCount) are written when a hit is accepted.
// ANY = true:  OccludeImpl (:223-315); `distance` is OccludeQuery.travel; returns true on the first hit.
template<int STACK, bool ANY, bool COUNT>
ECHO_DEVICE bool traverse_instanced(const DeviceScene& scene, vec3 origin, vec3 direction, uint32_t ignore, const uint32_t* ignoreLayers, uint32_t ignoreCount,
                                    float& distance, uint32_t& token, vec2& uv, uint32_t* hitLayers, uint32_t& hitCount, VisitCounts* counts)
{
	vec3 directionR = { rcp(direction.x), rcp(direction.y), rcp(direction.z) }; // Ray.cs:23
	uint32_t orders = (directionR.x > 0.0f ? 1u : 0u) | (directionR.y > 0.0f ? 2u : 0u) | (directionR.z > 0.0f ? 4u : 0u) | 8u;

	InstanceFrame frames[ECHO_MAX_INSTANCE_LAYERS];
	uint32_t current[ECHO_MAX_INSTANCE_LAYERS];
	uint32_t level = 0u, packIndex = 0u, base = 0u;
	PackView pack = load_pack(scene, 0u);
	bool ignoreHere = ignoreCount == 0u; // query.ignore's layers == query.current's layers

	uint2 stack[STACK];
	uint32_t next = 0u;
	stack[next++] = make_uint2(0u, __float_as_uint(0.0f)); // NewNodeToken(0), hit 0

	while (true)
	{
		uint32_t nodeToken, position = 0u;

		if (next == base)
		{
			if (level == 0u) break;

			// the instanced pack's accelerator returned: back to parent space (PreparedInstance.cs:58-60 / :78-80)
			const InstanceFrame& frame = frames[--level];
			origin = frame.origin;
			direction = frame.direction;
			directionR = { rcp(direction.x), rcp(direction.y), rcp(direction.z) };
			orders = (directionR.x > 0.0f ? 1u : 0u) | (directionR.y > 0.0f ? 2u : 0u) | (directionR.z > 0.0f ? 4u : 0u) | 8u;

			if (ANY) distance = frame.travel;
			else distance *= __ldg(instance_data(scene, frame.instance) + 6).y;

			packIndex = frame.pack;
			pack = load_pack(scene, packIndex);
			base = frame.base;
			nodeToken = frame.node;
			position = frame.position;
			ignoreHere = layers_match(ignoreLayers, ignoreCount, current, level);
		}
		else
		{
			uint2 entry = stack[--next];
			if (!ANY && __uint_as_float(entry.y) >= distance) continue; // :144-146
			nodeToken = entry.x;
		}

		NodeData node;
		{
			ECHO_CHECK(scene, pack.nodeOffset + token_index(nodeToken) < scene.nodeCount, CHECK_NODE);
			DeviceScene view = scene; // node array of the current pack
			view.nodes = scene.nodes + (size_t)pack.nodeOffset * 8;
			view.nodeCount = scene.nodeCount - pack.nodeOffset;
			load_node(view, token_index(nodeToken), orders, node);
		}

		if (COUNT && position == 0u) ++counts->nodes;

		float t0 = slab(node.minX.x, node.minY.x, node.minZ.x, node.maxX.x, node.maxY.x, node.maxZ.x, origin, directionR);
		float t1 = slab(node.minX.y, node.minY.y, node.minZ.y, node.maxX.y, node.maxY.y, node.maxZ.y, origin, directionR);
		float t2 = slab(node.minX.z, node.minY.z, node.minZ.z, node.maxX.z, node.maxY.z, node.maxZ.z, origin, directionR);
		float t3 = slab(node.minX.w, node.minY.w, node.minZ.w, node.maxX.w, node.maxY.w, node.maxZ.w, origin, directionR);

		uint32_t order = node.order >> (2u * position);

#pragma unroll 1
		for (uint32_t k = position; k < 4u; k++, order >>= 2)
		{
			int slot = order & 3;
			float hit = select4(slot, t0, t1, t2, t3);
			if (hit >= distance) continue; // Push: :203-205 / :299-301

			uint32_t child = select4(slot, node.token0, node.token1, node.token2, node.token3);
			uint32_t type = token_type(child);

			if (type == ECHO_TOKEN_TYPE_NODE)
			{
				ECHO_CHECK(scene, next < (uint32_t)STACK, CHECK_STACK);
				stack[next++] = make_uint2(child, __float_as_uint(hit));
			}
			else if (type == ECHO_TOKEN_TYPE_TRIANGLE)
			{
				if (ignoreHere && child == ignore) continue; // query.ignore == query.current, GeometryCollection.cs:93-94
				if (COUNT) ++counts->triangles;

				ECHO_CHECK(scene, pack.triangleOffset + token_index(child) < scene.triangleCount, CHECK_TRIANGLE);
				const float4* data = scene.triHot + ((size_t)pack.triangleOffset + token_index(child)) * 3;
				float4 a = __ldg(data), b = __ldg(data + 1), c = __ldg(data + 2);

				if (ANY)
				{
					if (triangle_occlude({ a.x, a.y, a.z }, { b.x, b.y, b.z }, { c.x, c.y, c.z }, origin, direction, distance)) return true;
				}
				else
				{
					vec2 hitUV;
					float d = triangle_intersect({ a.x, a.y, a.z }, { b.x, b.y, b.z }, { c.x, c.y, c.z }, origin, direction, hitUV);

					if (!(d >= distance))
					{
						distance = d;
						token = child;
						uv = hitUV;
						hitCount = level;
						for (uint32_t i = 0; i < level; i++) hitLayers[i] = current[i];
					}
				}
			}
			else if (type == ECHO_TOKEN_TYPE_SPHERE)
			{
				if (COUNT) ++counts->spheres;
				ECHO_CHECK(scene, pack.sphereOffset + token_index(child) < scene.sphereCount, CHECK_SPHERE);
				float4 sphere = __ldg(scene.spheres + pack.sphereOffset + token_index(child));
				bool findFar = ignoreHere && child == ignore;

				if (ANY)
				{
					if (sphere_occlude(sphere, origin, direction, distance, findFar)) return true;
				}
				else
				{
					vec2 hitUV;
					float d = sphere_intersect(sphere, origin, direction, hitUV, findFar);

					if (!(d >= distance))
					{
						distance = d;
						token = child;
						uv = hitUV;
						hitCount = level;
						for (uint32_t i = 0; i < level; i++) hitLayers[i] = current[i];
					}
				}
			}
			else if (type == ECHO_TOKEN_TYPE_INSTANCE && level < ECHO_MAX_INSTANCE_LAYERS)
			{
				// query.current.Push(token); instances[token.Index].Trace(ref query)
				uint32_t instance = pack.instanceOffset + token_index(child);
				ECHO_CHECK(scene, instance < scene.instanceCount, CHECK_INSTANCE);
				ECHO_CHECK(scene, next < (uint32_t)STACK, CHECK_STACK);
				const float4* data = instance_data(scene, instance);
				float4 scales = __ldg(data + 6);

				InstanceFrame& frame = frames[level];
				frame.origin = origin;
				frame.direction = direction;
				frame.travel = distance;
				frame.node = nodeToken;
				frame.position = k + 1u;
				frame.base = base;
				frame.pack = packIndex;
				frame.instance = instance;
				current[level++] = child;

				// TransformForward, PreparedInstance.cs:105-111
				vec3 localOrigin = multiply_point(data, origin);
				vec3 localDirection = multiply_direction(data, direction) * scales.y;
				origin = localOrigin;
				direction = localDirection;
				directionR = { rcp(direction.x), rcp(direction.y), rcp(direction.z) };
				orders = (directionR.x > 0.0f ? 1u : 0u) | (directionR.y > 0.0f ? 2u : 0u) | (directionR.z > 0.0f ? 4u : 0u) | 8u;
				distance *= scales.x;

				packIndex = __float_as_uint(scales.z);
				pack = load_pack(scene, packIndex);
				base = next;
				stack[next++] = make_uint2(0u, __float_as_uint(0.0f));
				ignoreHere = layers_match(ignoreLayers, ignoreCount, current, level);
				break; // the suspended visit resumes at frame.position once the pack is done
			}
		}
	}

	return false;
}

// ---- PreparedScene.Trace / Occlude through the packs: the guards of scene_trace / scene_occlude (PreparedScene.cs:66-86) ----
// `hitLayers` receives the hit's instance layers when a hit is accepted.
template<int STACK, bool COUNT>
ECHO_DEVICE bool scene_trace_layers(const DeviceScene& scene, vec3 origin, vec3 direction, uint32_t ignore, const PathLayers& ignoreLayers,
                                    float& distance, uint32_t& token, vec2& uv, PathLayers& hitLayers, VisitCounts* counts)
{
	if (!positive(distance)) return false;
	float original = distance;
	traverse_instanced<STACK, false, COUNT>(scene, origin, direction, ignore, ignoreLayers.tokens, ignoreLayers.count, distance, token, uv, hitLayers.tokens, hitLayers.count, counts);
	return distance < original;
}

template<int STACK, bool COUNT>
ECHO_DEVICE bool scene_occlude_layers(const DeviceScene& scene, vec3 origin, vec3 direction, uint32_t ignore, const PathLayers& ignoreLayers, float travel, VisitCounts* counts)
{
	if (!positive(travel)) return false;
	uint32_t token = ECHO_TOKEN_EMPTY, hitCount = 0u; // an occlusion query records no hit
	vec2 uv = { 0.0f, 0.0f };
	return traverse_instanced<STACK, true, COUNT>(scene, origin, direction, ignore, ignoreLayers.tokens, ignoreLayers.count, travel, token, uv, nullptr, hitCount, counts);
}

} // namespace echo
