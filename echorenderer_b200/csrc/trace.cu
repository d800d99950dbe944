// trace.cu — batched Accelerator.Trace / Accelerator.Occlude: one thread per query over AoS EchoRay input read with
// two 128-bit loads, EchoHit output written with one 128-bit store. These are the kernels behind
// echo_b200_trace_batch / echo_b200_occlude_batch (BASELINE config C2) and the batched analogue of the benchmark loops in
// the reference's src/Echo.Experimental/Benchmarks/Accelerators.cs:131-157.
#include <algorithm>
#include <cstdlib>
#include <map>
#include <mutex>
#include <utility>

#include "echo_internal.h"
#include "echo_traverse.cuh"

namespace echo
{

constexpr int kTraceBlock = 128;

template<int STACK, bool COUNT>
__global__ void __launch_bounds__(kTraceBlock) trace_batch_kernel(DeviceScene scene, const float4* __restrict__ rays, uint64_t n,
                                                                  float4* __restrict__ hits, unsigned long long* __restrict__ counts)
{
	uint64_t i = (uint64_t)blockIdx.x * kTraceBlock + threadIdx.x;
	VisitCounts local = { 0u, 0u, 0u };

	if (i < n)
	{
		float4 a = __ldg(rays + i * 2);     // origin.xyz, direction.x
		float4 b = __ldg(rays + i * 2 + 1); // direction.yz, distance, ignore

		vec3 origin = { a.x, a.y, a.z };
		vec3 direction = { a.w, b.x, b.y };
		float limit = b.z;
		uint32_t ignore = __float_as_uint(b.w);

		float distance = limit;
		uint32_t token = ECHO_TOKEN_EMPTY;
		vec2 uv = { 0.0f, 0.0f };

		bool hit = scene_trace<STACK, COUNT>(scene, origin, direction, ignore, distance, token, uv, &local);

		float4 out;
		out.x = __uint_as_float(hit ? token : ECHO_TOKEN_EMPTY);
		out.y = hit ? distance : limit;
		out.z = hit ? uv.x : 0.0f;
		out.w = hit ? uv.y : 0.0f;
		hits[i] = out;
	}

	if (COUNT) visit_flush(counts, 0, local);
}

template<int STACK, bool COUNT>
__global__ void __launch_bounds__(kTraceBlock) occlude_batch_kernel(DeviceScene scene, const float4* __restrict__ rays, uint64_t n,
                                                                    uint8_t* __restrict__ occluded, unsigned long long* __restrict__ counts)
{
	uint64_t i = (uint64_t)blockIdx.x * kTraceBlock + threadIdx.x;
	VisitCounts local = { 0u, 0u, 0u };

	if (i < n)
	{
		float4 a = __ldg(rays + i * 2);
		float4 b = __ldg(rays + i * 2 + 1);

		vec3 origin = { a.x, a.y, a.z };
		vec3 direction = { a.w, b.x, b.y };

		bool result = scene_occlude<STACK, COUNT>(scene, origin, direction, __float_as_uint(b.w), b.z, &local);
		occluded[i] = result ? 1 : 0;
	}

	if (COUNT) visit_flush(counts, 0, local);
}

// AoS EchoRay in (two 128-bit loads), EchoHit out (one 128-bit store) / one byte per occlusion query
struct BatchIO
{
	const float4* __restrict__ rays;
	float4* __restrict__ hits;
	uint8_t* __restrict__ occluded;
	const uint32_t* __restrict__ ignoreLayers; // instanced scenes: EchoTokenHierarchy per query (6 words), nullable
	uint32_t* __restrict__ hitLayers;          // EchoTokenHierarchy per hit, nullable

	ECHO_DEVICE uint32_t load_ignore_layers(uint32_t index, uint32_t* tokens) const
	{
		if (!ignoreLayers) return 0u;
		const uint32_t* in = ignoreLayers + (size_t)index * 6;
		uint32_t count = min(__ldg(in), ECHO_MAX_INSTANCE_LAYERS);
		for (uint32_t k = 0; k < count; k++) tokens[k] = __ldg(in + 1 + k);
		return count;
	}

	ECHO_DEVICE void store_hit_layers(uint32_t index, bool hit, const uint32_t* tokens, uint32_t count) const
	{
		if (!hitLayers) return;
		uint32_t* out = hitLayers + (size_t)index * 6;
		out[0] = hit ? count : 0u;
		for (uint32_t k = 0; k < ECHO_MAX_INSTANCE_LAYERS; k++) out[1 + k] = hit && k < count ? tokens[k] : 0u;
	}

	ECHO_DEVICE const float4* ray_pointer(uint32_t index) const { return rays + (size_t)index * 2; }
	ECHO_DEVICE float4* prepared_pointer(uint32_t index) const { return hits + index; }

	ECHO_DEVICE void store_closest(uint32_t index, bool hit, uint32_t token, float distance, vec2 uv, float limit) const
	{
		__stcs(hits + index, make_float4(__uint_as_float(hit ? token : ECHO_TOKEN_EMPTY), hit ? distance : limit, hit ? uv.x : 0.0f, hit ? uv.y : 0.0f));
	}

	ECHO_DEVICE void store_any(uint32_t index, bool result) const { occluded[index] = result ? 1 : 0; }
};

template<int STACK, bool ANY>
__global__ void __launch_bounds__(kTraverseBlock, ECHO_MIN_BLOCKS) persistent_batch_kernel(DeviceScene scene, BatchIO io, uint32_t n, unsigned long long* __restrict__ nextRay)
{
	__shared__ float4 stagedRays[kTraverseBlock * kStagedFloat4];
	persistent_traverse<STACK, ANY>(scene, io, n, nextRay, stagedRays);
	persistent_finish(nextRay);
}

// the same through instanced packs (echo_traverse.cuh INST); more per-lane state than the plain kernel: 95 registers when
// left alone. A/B on the instanced bench scene (variants/ab6.sh): 6 CTAs per SM (80 registers) 3691 / 6692 Mrays/s closest
// hit / occlusion, unconstrained 3507 / 6233, 7 CTAs (72 registers, spills) 3430 / 6773.
template<int STACK, bool ANY>
__global__ void __launch_bounds__(kTraverseBlock, ECHO_INST_MIN_BLOCKS) persistent_instanced_kernel(DeviceScene scene, BatchIO io, uint32_t n, unsigned long long* __restrict__ nextRay)
{
	__shared__ float4 stagedRays[kTraverseBlock * kStagedFloat4];
	persistent_traverse<STACK, ANY, true>(scene, io, n, nextRay, stagedRays);
	persistent_finish(nextRay);
}

// The work counter pair of persistent launches on `stream` of the current device (echo_traverse.cuh persistent_finish). Launches
// on one stream run in order and every kernel leaves its pair zeroed, so one pair per (device, stream) is enough however
// many launches are outstanding and whoever issued them — there is nothing to hand out, recycle or memset. The pairs of
// destroyed streams stay allocated (16 bytes each); a recycled stream handle simply finds its old, zeroed pair.
unsigned long long* ray_counters(cudaStream_t stream)
{
	static std::mutex guard;
	static std::map<std::pair<int, cudaStream_t>, unsigned long long*> pairs;

	int device = 0;
	cudaGetDevice(&device);

	std::lock_guard<std::mutex> lock(guard);
	unsigned long long*& pair = pairs[{ device, stream }];

	if (!pair)
	{
		// synchronous on purpose: the pair is zero before any launch on any stream can see it
		if (!check_cuda(cudaMalloc((void**)&pair, sizeof(unsigned long long) * 2), "cudaMalloc(ray counters)")) { pair = nullptr; return nullptr; }
		if (!check_cuda(cudaMemset(pair, 0, sizeof(unsigned long long) * 2), "cudaMemset(ray counters)")) return nullptr;
	}

	return pair;
}

// one resident wave of a persistent kernel on the current device: 148 SMs x resident CTAs per SM; remembered per device and kernel
int persistent_grid(const void* kernel)
{
	static std::mutex guard;
	static std::map<std::pair<int, const void*>, int> grids;

	int device = 0;
	cudaGetDevice(&device);

	std::lock_guard<std::mutex> lock(guard);
	int& grid = grids[{ device, kernel }];

	if (grid == 0)
	{
		int sms = 0, perSM = 0;
		cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
		cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, kernel, kTraverseBlock, 0);
		grid = std::max(sms, 1) * (perSM > 0 ? perSM : 1);
	}

	return grid;
}

template<int STACK, bool ANY>
static bool launch_persistent(const DeviceScene& scene, const EchoRay* rays, uint64_t n, EchoHit* hits, uint8_t* occluded, cudaStream_t stream)
{
	const int grid = persistent_grid((const void*)persistent_batch_kernel<STACK, ANY>);
	constexpr uint64_t kLaunchLimit = 1ull << 31; // ray indices are 32-bit inside the kernel

	for (uint64_t first = 0; first < n; first += kLaunchLimit)
	{
		uint64_t count = n - first < kLaunchLimit ? n - first : kLaunchLimit;
		unsigned long long* counter = ray_counters(stream);
		if (!counter) return false;

		BatchIO io = { reinterpret_cast<const float4*>(rays + first), hits ? reinterpret_cast<float4*>(hits + first) : nullptr, occluded ? occluded + first : nullptr, nullptr, nullptr };
		uint64_t needed = (count + kTraverseBlock - 1) / kTraverseBlock;
		unsigned int blocks = (unsigned int)(needed < (uint64_t)grid ? needed : (uint64_t)grid);
		persistent_batch_kernel<STACK, ANY><<<blocks, kTraverseBlock, 0, stream>>>(scene, io, (uint32_t)count, counter);
		if (!check_cuda(cudaGetLastError(), "persistent_batch_kernel launch")) return false;
	}

	return true;
}

template<int STACK, bool ANY>
static bool launch_persistent_instanced_impl(const DeviceScene& scene, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, EchoHit* hits,
                                             EchoTokenHierarchy* hitLayers, uint8_t* occluded, cudaStream_t stream)
{
	const int grid = persistent_grid((const void*)persistent_instanced_kernel<STACK, ANY>);
	constexpr uint64_t kLaunchLimit = 1ull << 31;

	for (uint64_t first = 0; first < n; first += kLaunchLimit)
	{
		uint64_t count = n - first < kLaunchLimit ? n - first : kLaunchLimit;
		unsigned long long* counter = ray_counters(stream);
		if (!counter) return false;

		BatchIO io = { reinterpret_cast<const float4*>(rays + first), hits ? reinterpret_cast<float4*>(hits + first) : nullptr, occluded ? occluded + first : nullptr,
		               ignore ? reinterpret_cast<const uint32_t*>(ignore + first) : nullptr, hitLayers ? reinterpret_cast<uint32_t*>(hitLayers + first) : nullptr };
		uint64_t needed = (count + kTraverseBlock - 1) / kTraverseBlock;
		unsigned int blocks = (unsigned int)(needed < (uint64_t)grid ? needed : (uint64_t)grid);
		persistent_instanced_kernel<STACK, ANY><<<blocks, kTraverseBlock, 0, stream>>>(scene, io, (uint32_t)count, counter);
		if (!check_cuda(cudaGetLastError(), "persistent_instanced_kernel launch")) return false;
	}

	return true;
}

static bool use_simple_kernels();

// persistent, work-replacing kernels for instanced scenes; false + no error when the simple kernels should be used instead
bool launch_persistent_instanced(const DeviceScene& scene, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, EchoHit* hits,
                                 EchoTokenHierarchy* hitLayers, uint8_t* occluded, cudaStream_t stream, bool& launched)
{
	launched = false;
	if (use_simple_kernels()) return true;
	launched = true;
	bool any = occluded != nullptr;

	switch (stack_class(scene.maxDepth))
	{
		case 0: return any ? launch_persistent_instanced_impl<48, true>(scene, rays, ignore, n, hits, hitLayers, occluded, stream)
		                   : launch_persistent_instanced_impl<48, false>(scene, rays, ignore, n, hits, hitLayers, occluded, stream);
		case 1: return any ? launch_persistent_instanced_impl<96, true>(scene, rays, ignore, n, hits, hitLayers, occluded, stream)
		                   : launch_persistent_instanced_impl<96, false>(scene, rays, ignore, n, hits, hitLayers, occluded, stream);
		case 2: return any ? launch_persistent_instanced_impl<192, true>(scene, rays, ignore, n, hits, hitLayers, occluded, stream)
		                   : launch_persistent_instanced_impl<192, false>(scene, rays, ignore, n, hits, hitLayers, occluded, stream);
		default: set_error("the deepest chain of instanced packs needs more than 192 stack entries"); return false;
	}
}

static bool use_simple_kernels()
{
	static int cached = -1;
	if (cached < 0)
	{
		const char* value = std::getenv("ECHO_B200_SIMPLE_TRACE"); // A/B switch: one thread per ray, no work replacement
		cached = value && value[0] == '1' ? 1 : 0;
	}
	return cached == 1;
}

int stack_class(uint32_t maxDepth)
{
	uint32_t size = maxDepth * 3 + 1;
	if (size <= 48) return 0;
	if (size <= 96) return 1;
	if (size <= 192) return 2;
	return -1;
}

template<bool COUNT>
static bool launch_trace_impl(const DeviceScene& scene, const EchoRay* rays, uint64_t n, EchoHit* hits, unsigned long long* counts, cudaStream_t stream)
{
	if (n == 0) return true;
	unsigned int blocks = (unsigned int)((n + kTraceBlock - 1) / kTraceBlock);
	const float4* in = reinterpret_cast<const float4*>(rays);
	float4* out = reinterpret_cast<float4*>(hits);

	switch (stack_class(scene.maxDepth))
	{
		case 0: trace_batch_kernel<48, COUNT><<<blocks, kTraceBlock, 0, stream>>>(scene, in, n, out, counts); break;
		case 1: trace_batch_kernel<96, COUNT><<<blocks, kTraceBlock, 0, stream>>>(scene, in, n, out, counts); break;
		case 2: trace_batch_kernel<192, COUNT><<<blocks, kTraceBlock, 0, stream>>>(scene, in, n, out, counts); break;
		default: set_error("QBVH deeper than 63 quad levels is not supported"); return false;
	}

	return check_cuda(cudaGetLastError(), "trace_batch_kernel launch");
}

template<bool COUNT>
static bool launch_occlude_impl(const DeviceScene& scene, const EchoRay* rays, uint64_t n, uint8_t* occluded, unsigned long long* counts, cudaStream_t stream)
{
	if (n == 0) return true;
	unsigned int blocks = (unsigned int)((n + kTraceBlock - 1) / kTraceBlock);
	const float4* in = reinterpret_cast<const float4*>(rays);

	switch (stack_class(scene.maxDepth))
	{
		case 0: occlude_batch_kernel<48, COUNT><<<blocks, kTraceBlock, 0, stream>>>(scene, in, n, occluded, counts); break;
		case 1: occlude_batch_kernel<96, COUNT><<<blocks, kTraceBlock, 0, stream>>>(scene, in, n, occluded, counts); break;
		case 2: occlude_batch_kernel<192, COUNT><<<blocks, kTraceBlock, 0, stream>>>(scene, in, n, occluded, counts); break;
		default: set_error("QBVH deeper than 63 quad levels is not supported"); return false;
	}

	return check_cuda(cudaGetLastError(), "occlude_batch_kernel launch");
}

bool launch_trace(const DeviceScene& scene, const EchoRay* rays, uint64_t n, EchoHit* hits, unsigned long long* counts, cudaStream_t stream)
{
	if (n == 0) return true;
	if (scene.packCount != 0u) return launch_trace_instanced(scene, rays, nullptr, n, hits, nullptr, counts, stream);

	if (!counts && !use_simple_kernels())
	{
		switch (stack_class(scene.maxDepth))
		{
			case 0: return launch_persistent<48, false>(scene, rays, n, hits, nullptr, stream);
			case 1: return launch_persistent<96, false>(scene, rays, n, hits, nullptr, stream);
			case 2: return launch_persistent<192, false>(scene, rays, n, hits, nullptr, stream);
			default: set_error("QBVH deeper than 63 quad levels is not supported"); return false;
		}
	}

	return counts ? launch_trace_impl<true>(scene, rays, n, hits, counts, stream) : launch_trace_impl<false>(scene, rays, n, hits, nullptr, stream);
}

bool launch_occlude(const DeviceScene& scene, const EchoRay* rays, uint64_t n, uint8_t* occluded, unsigned long long* counts, cudaStream_t stream)
{
	if (n == 0) return true;
	if (scene.packCount != 0u) return launch_occlude_instanced(scene, rays, nullptr, n, occluded, counts, stream);

	if (!counts && !use_simple_kernels())
	{
		switch (stack_class(scene.maxDepth))
		{
			case 0: return launch_persistent<48, true>(scene, rays, n, nullptr, occluded, stream);
			case 1: return launch_persistent<96, true>(scene, rays, n, nullptr, occluded, stream);
			case 2: return launch_persistent<192, true>(scene, rays, n, nullptr, occluded, stream);
			default: set_error("QBVH deeper than 63 quad levels is not supported"); return false;
		}
	}

	return counts ? launch_occlude_impl<true>(scene, rays, n, occluded, counts, stream) : launch_occlude_impl<false>(scene, rays, n, occluded, nullptr, stream);
}

} // namespace echo
