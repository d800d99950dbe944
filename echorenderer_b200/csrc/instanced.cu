// instanced.cu — batched Accelerator.Trace / Occlude for scenes with instanced packs (SURVEY.md §8f rank 2): the kernels
// behind echo_b200_trace_batch_hierarchy / echo_b200_occlude_batch_hierarchy, and behind the plain batch calls when the
// committed scene has packs. One thread per query; the traversal itself is echo_instanced.cuh.
#include "echo_instanced.cuh"
#include "echo_internal.h"

namespace echo
{

constexpr int kInstancedBlock = 128;

template<int STACK, bool ANY, bool COUNT>
__global__ void __launch_bounds__(kInstancedBlock) instanced_batch_kernel(DeviceScene scene, const float4* __restrict__ rays, const uint32_t* __restrict__ ignoreLayers,
                                                                          uint64_t n, float4* __restrict__ hits, uint32_t* __restrict__ hitLayers,
                                                                          uint8_t* __restrict__ occluded, unsigned long long* __restrict__ counts)
{
	uint64_t i = (uint64_t)blockIdx.x * kInstancedBlock + threadIdx.x;
	VisitCounts local = { 0u, 0u, 0u };

	if (i < n)
	{
		float4 a = __ldg(rays + i * 2);     // origin.xyz, direction.x
		float4 b = __ldg(rays + i * 2 + 1); // direction.yz, distance, ignore

		vec3 origin = { a.x, a.y, a.z };
		vec3 direction = { a.w, b.x, b.y };
		float limit = b.z;
		uint32_t ignore = __float_as_uint(b.w);

		uint32_t ignoreStack[ECHO_MAX_INSTANCE_LAYERS] = {};
		uint32_t ignoreCount = 0u;

		if (ignoreLayers)
		{
			const uint32_t* in = ignoreLayers + i * 6; // EchoTokenHierarchy
			ignoreCount = min(__ldg(in), ECHO_MAX_INSTANCE_LAYERS);
			for (uint32_t k = 0; k < ignoreCount; k++) ignoreStack[k] = __ldg(in + 1 + k);
		}

		float distance = limit;
		uint32_t token = ECHO_TOKEN_EMPTY;
		vec2 uv = { 0.0f, 0.0f };
		uint32_t layers[ECHO_MAX_INSTANCE_LAYERS] = {};
		uint32_t layerCount = 0u;
		bool result = false;

		if (positive(limit)) // PreparedScene.Trace / Occlude guards, PreparedScene.cs:69,84
		{
			bool any = traverse_instanced<STACK, ANY, COUNT>(scene, origin, direction, ignore, ignoreStack, ignoreCount, distance, token, uv, layers, layerCount, &local);
			result = ANY ? any : distance < limit;
		}

		if (ANY) occluded[i] = result ? 1 : 0;
		else
		{
			hits[i] = make_float4(__uint_as_float(result ? token : ECHO_TOKEN_EMPTY), result ? distance : limit, result ? uv.x : 0.0f, result ? uv.y : 0.0f);

			if (hitLayers)
			{
				uint32_t* out = hitLayers + i * 6;
				out[0] = result ? layerCount : 0u;
				for (uint32_t k = 0; k < ECHO_MAX_INSTANCE_LAYERS; k++) out[1 + k] = result && k < layerCount ? layers[k] : 0u;
			}
		}
	}

	if (COUNT) visit_flush(counts, 0, local);
}

template<bool ANY, bool COUNT>
static bool launch_instanced(const DeviceScene& scene, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, EchoHit* hits,
                             EchoTokenHierarchy* hitLayers, uint8_t* occluded, unsigned long long* counts, cudaStream_t stream)
{
	if (n == 0) return true;
	if (scene.packCount == 0u) { set_error("the scene has no packs: use the plain batch calls"); return false; }

	unsigned int blocks = (unsigned int)((n + kInstancedBlock - 1) / kInstancedBlock);
	const float4* in = reinterpret_cast<const float4*>(rays);
	const uint32_t* layersIn = reinterpret_cast<const uint32_t*>(ignore);
	float4* out = reinterpret_cast<float4*>(hits);
	uint32_t* layersOut = reinterpret_cast<uint32_t*>(hitLayers);

	switch (stack_class(scene.maxDepth))
	{
		case 0: instanced_batch_kernel<48, ANY, COUNT><<<blocks, kInstancedBlock, 0, stream>>>(scene, in, layersIn, n, out, layersOut, occluded, counts); break;
		case 1: instanced_batch_kernel<96, ANY, COUNT><<<blocks, kInstancedBlock, 0, stream>>>(scene, in, layersIn, n, out, layersOut, occluded, counts); break;
		case 2: instanced_batch_kernel<192, ANY, COUNT><<<blocks, kInstancedBlock, 0, stream>>>(scene, in, layersIn, n, out, layersOut, occluded, counts); break;
		default: set_error("the deepest chain of instanced packs needs more than 192 stack entries"); return false;
	}

	return check_cuda(cudaGetLastError(), "instanced_batch_kernel launch");
}

bool launch_trace_instanced(const DeviceScene& scene, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, EchoHit* hits,
                            EchoTokenHierarchy* hitLayers, unsigned long long* counts, cudaStream_t stream)
{
	if (n == 0) return true;

	if (!counts && scene.packCount != 0u)
	{
		bool launched = false;
		bool ok = launch_persistent_instanced(scene, rays, ignore, n, hits, hitLayers, nullptr, stream, launched);
		if (launched || !ok) return ok;
	}

	return counts ? launch_instanced<false, true>(scene, rays, ignore, n, hits, hitLayers, nullptr, counts, stream)
	              : launch_instanced<false, false>(scene, rays, ignore, n, hits, hitLayers, nullptr, nullptr, stream);
}

bool launch_occlude_instanced(const DeviceScene& scene, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, uint8_t* occluded,
                              unsigned long long* counts, cudaStream_t stream)
{
	if (n == 0) return true;

	if (!counts && scene.packCount != 0u)
	{
		bool launched = false;
		bool ok = launch_persistent_instanced(scene, rays, ignore, n, nullptr, nullptr, occluded, stream, launched);
		if (launched || !ok) return ok;
	}

	return counts ? launch_instanced<true, true>(scene, rays, ignore, n, nullptr, nullptr, occluded, counts, stream)
	              : launch_instanced<true, false>(scene, rays, ignore, n, nullptr, nullptr, occluded, nullptr, stream);
}

} // namespace echo
