// lightbuild.cu — the CUDA backend of echo_light_build.h: the reference's light tree (LightCollection.CreateBounds + LightTree.Build +
// AddToMap, Aggregation/Preparation/LightCollection.cs:91-137, Aggregation/Selection/LightTree.cs:21-113) built on the device level by
// level and emitted byte for byte as the host mirror's recursive build emits it. The passes and the driver live in echo_light_build.h,
// shared with the host mirror's arithmetic and with the CPU emulation the -m "not gpu" suite checks against it; this file only supplies
// the generic kernel, the CUB sort / sums, memory and the copies.
//
// What the device can and cannot buy here: the two sweeps of a node are chains of non-associative cone unions (echo_light_build.h), one
// thread each; the root's two chains ARE the first level, so the build time is a few chain lengths however wide the machine is — but only
// the longest chain of every level is waited for (2-3 n steps in all against the recursion's n log n) and everything around the chains is
// parallel: 3-5x the host recursion on 10 k - 100 k emitters (profiles/README.md), and a scene whose geometry already lives on the device gets
// the reference's own light tree without the emitter scan crossing the host.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <chrono>
#include <cstdio>
#include <cstdlib>

#include "echo_internal.h"
#include "echo_light_build.h"

namespace echo
{

namespace
{

constexpr int kLightBlock = 128;

template<class F>
__global__ void __launch_bounds__(kLightBlock) light_for_each_kernel(uint32_t n, F f)
{
	uint32_t i = blockIdx.x * kLightBlock + threadIdx.x;
	if (i < n) f(i);
}

struct CudaBackend
{
	cudaStream_t stream = nullptr;
	std::vector<void*> blocks;
	void* scratch = nullptr;
	size_t scratchBytes = 0;
	uint32_t launches = 0, syncs = 0;

	~CudaBackend()
	{
		for (void* block : blocks) cudaFree(block);
		cudaFree(scratch);
	}

	// CUB's temporary storage, grown to what the call at hand asks for: the sums over the candidates come first (10 M triangles of which three
	// emit light must not reserve the sort's storage for 10 M keys), the sorts over the emitters after; cudaFree orders itself behind the stream
	bool ensure(size_t bytes)
	{
		if (bytes <= scratchBytes) return true;
		if (scratch && !check_cuda(cudaFree(scratch), "cudaFree(light build scratch)")) return false;
		scratch = nullptr;
		scratchBytes = (bytes + 255) & ~size_t(255);
		return check_cuda(cudaMalloc(&scratch, scratchBytes), "cudaMalloc(light build scratch)");
	}

	char* allocate(size_t bytes)
	{
		void* block = nullptr;
		if (!check_cuda(cudaMalloc(&block, bytes), "cudaMalloc(light build)")) return nullptr;
		blocks.push_back(block);
		return (char*)block;
	}

	template<class F>
	bool for_each(uint32_t n, const F& f)
	{
		if (n == 0u) return true;
		light_for_each_kernel<<<(n + kLightBlock - 1) / kLightBlock, kLightBlock, 0, stream>>>(n, f);
		++launches;
		return check_cuda(cudaGetLastError(), "light build launch");
	}

	bool sort_pairs(const unsigned long long* keysIn, unsigned long long* keysOut, const uint32_t* valuesIn, uint32_t* valuesOut, uint32_t n, int endBit)
	{
		size_t bytes = 0; // cub's radix sort is stable
		if (!check_cuda(cub::DeviceRadixSort::SortPairs(nullptr, bytes, keysIn, keysOut, valuesIn, valuesOut, (int)n, 0, endBit, stream), "cub sort (size)") || !ensure(bytes)) return false;
		++launches;
		return check_cuda(cub::DeviceRadixSort::SortPairs(scratch, bytes, keysIn, keysOut, valuesIn, valuesOut, (int)n, 0, endBit, stream), "cub sort");
	}

	bool exclusive_sum(const uint32_t* in, uint32_t* out, uint32_t n)
	{
		size_t bytes = 0;
		if (!check_cuda(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, (int)n, stream), "cub sum (size)") || !ensure(bytes)) return false;
		++launches;
		return check_cuda(cub::DeviceScan::ExclusiveSum(scratch, bytes, in, out, (int)n, stream), "cub sum");
	}

	template<class T>
	bool read(const T* source, T* destination, uint32_t n)
	{
		++syncs;
		return check_cuda(cudaMemcpyAsync(destination, source, sizeof(T) * n, cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(light read)")
			&& check_cuda(cudaStreamSynchronize(stream), "light build level");
	}

	template<class T>
	bool write(T* destination, const T* source, uint32_t n) // from pageable host memory: the copy has left `source` on return
	{
		return check_cuda(cudaMemcpyAsync(destination, source, sizeof(T) * n, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(light write)");
	}

	bool fill_zero(void* pointer, size_t bytes) { return check_cuda(cudaMemsetAsync(pointer, 0, bytes, stream), "cudaMemsetAsync(light)"); }
};

struct LastBuild { float uploadMs, buildMs, downloadMs, levels; };
thread_local LastBuild gLastLightBuild = { 0.0f, 0.0f, 0.0f, 0.0f };

template<class T>
bool upload(const T* host, uint32_t count, const T*& device, CudaBackend& backend)
{
	device = nullptr;
	if (count == 0u) return true;
	char* block = backend.allocate(sizeof(T) * count);
	if (!block) return false;
	device = (const T*)block;
	return check_cuda(cudaMemcpyAsync(block, host, sizeof(T) * count, cudaMemcpyHostToDevice, backend.stream), "cudaMemcpyAsync(light sources)");
}

} // namespace

// the calling thread's last build_light_tree_device: {upload, device build, download} in ms of host wall time around synchronised phases, levels
void last_light_build(float* out4)
{
	out4[0] = gLastLightBuild.uploadMs; out4[1] = gLastLightBuild.buildMs; out4[2] = gLastLightBuild.downloadMs; out4[3] = gLastLightBuild.levels;
}

// Host buffers in, host vectors out. false: a CUDA call failed. `refused`: the tree is deeper than a 64-bit path (LightTree.cs:29).
bool build_light_tree_device(const lightbuild::Sources& host, std::vector<EchoLightNode>& nodes, std::vector<uint32_t>& tokens, std::vector<uint64_t>& paths, bool* refused)
{
	*refused = false;
	nodes.clear();
	tokens.clear();
	paths.clear();

	const uint32_t candidates = host.candidates();
	if (candidates == 0u) return true;
	if (candidates >= (1u << ECHO_TOKEN_INDEX_BITS)) { set_error("a light tree holds fewer than 2^28 emitters"); return false; }

	const bool profile = std::getenv("ECHO_B200_PROFILE") != nullptr;
	auto clock = [] { return std::chrono::steady_clock::now(); };
	auto since = [&](std::chrono::steady_clock::time_point from) { return std::chrono::duration<double, std::milli>(clock() - from).count(); };
	auto started = clock();

	CudaBackend backend;

	lightbuild::Sources device = host;
	if (!upload(host.triangles, host.triangleCount, device.triangles, backend) || !upload(host.spheres, host.sphereCount, device.spheres, backend)
		|| !upload(host.materials, host.materialCount, device.materials, backend) || !upload(host.points, host.pointCount, device.points, backend)
		|| !upload(host.instanceLights, host.instanceCount * 12u, device.instanceLights, backend)) return false;
	if (!check_cuda(cudaStreamSynchronize(backend.stream), "light upload")) return false; // the phases are reported separately (last_light_build)
	double uploadMs = since(started);
	auto phase = clock();

	lightbuild::Result result = lightbuild::build(backend, device);
	if (!result.ok) return false;
	if (result.unsupported) { *refused = true; return true; }
	if (!check_cuda(cudaStreamSynchronize(backend.stream), "light build")) return false;

	double buildMs = since(phase);
	phase = clock();

	nodes.resize(result.nodeCount);
	tokens.resize(result.emitterCount);
	paths.resize(result.emitterCount);

	if (result.emitterCount != 0u)
	{
		static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "bit paths are 64 bits");
		if (!check_cuda(cudaMemcpy(nodes.data(), result.nodes, sizeof(EchoLightNode) * result.nodeCount, cudaMemcpyDeviceToHost), "cudaMemcpy(light nodes)")
			|| !check_cuda(cudaMemcpy(tokens.data(), result.emitterTokens, sizeof(uint32_t) * result.emitterCount, cudaMemcpyDeviceToHost), "cudaMemcpy(emitter tokens)")
			|| !check_cuda(cudaMemcpy(paths.data(), result.emitterPaths, sizeof(uint64_t) * result.emitterCount, cudaMemcpyDeviceToHost), "cudaMemcpy(emitter paths)")) return false;
	}

	double downloadMs = since(phase);
	gLastLightBuild = { (float)uploadMs, (float)buildMs, (float)downloadMs, (float)result.levels };

	if (profile)
		std::fprintf(stderr, "[echo_b200 build] light tree: %u candidates -> %u emitters, %u nodes, %u levels: upload %.2f ms, build %.2f ms (%u launches, %u syncs), download %.2f ms\n",
		             candidates, result.emitterCount, result.nodeCount, result.levels, uploadMs, buildMs, backend.launches, backend.syncs, downloadMs);
	return true;
}

} // namespace echo
