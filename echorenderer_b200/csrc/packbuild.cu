// packbuild.cu — the CUDA backend of echo_pack_build.h: every pack of an instanced scene, QBVH and light tree, built on the device in
// rounds of packs of equal height (a QBVH forest and a light forest per round, the placements' rows computed from the finished child trees
// between rounds). The passes, the forests and the orchestration live in the headers, shared with the CPU emulation the -m "not gpu" suite
// checks against the host mirror; this file only supplies the generic kernel, CUB, memory, the copies, and the per-pack fallback.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <chrono>
#include <cstdio>
#include <cstdlib>

#include "echo_internal.h"
#include "echo_pack_build.h"

namespace echo
{

namespace
{

constexpr int kPackBlock = 128; // the light passes' block (lightbuild.cu); the sweep passes run as well at 128

template<class F>
__global__ void __launch_bounds__(kPackBlock) pack_for_each_kernel(uint32_t n, F f)
{
	uint32_t i = blockIdx.x * kPackBlock + threadIdx.x;
	if (i < n) f(i);
}

struct CudaBackend // both drivers' backend concept: blocks that live as long as the call, CUB storage grown on demand
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

	bool ensure(size_t bytes)
	{
		if (bytes <= scratchBytes) return true;
		if (scratch && !check_cuda(cudaFree(scratch), "cudaFree(pack build scratch)")) return false;
		scratch = nullptr;
		scratchBytes = (bytes + 255) & ~size_t(255);
		return check_cuda(cudaMalloc(&scratch, scratchBytes), "cudaMalloc(pack build scratch)");
	}

	char* allocate(size_t bytes)
	{
		void* block = nullptr;
		if (!check_cuda(cudaMalloc(&block, bytes), "cudaMalloc(pack build)")) return nullptr;
		blocks.push_back(block);
		return (char*)block;
	}

	template<class F>
	bool for_each(uint32_t n, const F& f)
	{
		if (n == 0u) return true;
		pack_for_each_kernel<<<(n + kPackBlock - 1) / kPackBlock, kPackBlock, 0, stream>>>(n, f);
		++launches;
		return check_cuda(cudaGetLastError(), "pack build launch");
	}

	bool sort_pairs(const unsigned long long* keysIn, unsigned long long* keysOut, const uint32_t* valuesIn, uint32_t* valuesOut, uint32_t n, int endBit)
	{
		size_t bytes = 0; // cub's radix sort is stable
		if (!check_cuda(cub::DeviceRadixSort::SortPairs(nullptr, bytes, keysIn, keysOut, valuesIn, valuesOut, (int)n, 0, endBit, stream), "cub sort (size)") || !ensure(bytes)) return false;
		++launches;
		return check_cuda(cub::DeviceRadixSort::SortPairs(scratch, bytes, keysIn, keysOut, valuesIn, valuesOut, (int)n, 0, endBit, stream), "cub sort");
	}

	bool scan_items(const sweep::ScanItem* in, sweep::ScanItem* out, uint32_t n)
	{
		size_t bytes = 0;
		if (!check_cuda(cub::DeviceScan::InclusiveScan(nullptr, bytes, in, out, sweep::ScanOp(), (int)n, stream), "cub scan (size)") || !ensure(bytes)) return false;
		++launches;
		return check_cuda(cub::DeviceScan::InclusiveScan(scratch, bytes, in, out, sweep::ScanOp(), (int)n, stream), "cub scan");
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
		return check_cuda(cudaMemcpyAsync((void*)destination, (const void*)source, sizeof(T) * n, cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(pack build read)")
			&& check_cuda(cudaStreamSynchronize(stream), "pack build");
	}

	template<class T>
	bool write(T* destination, const T* source, uint32_t n) // from pageable host memory: the copy has left `source` on return
	{
		return check_cuda(cudaMemcpyAsync((void*)destination, (const void*)source, sizeof(T) * n, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(pack build write)");
	}

	bool fill_zero(void* pointer, size_t bytes) { return check_cuda(cudaMemsetAsync(pointer, 0, bytes, stream), "cudaMemsetAsync(pack build)"); }
};

struct Rebuild // the packs of a round the forest gives up on: the per-pack device build, with its clustered fallback (build.cu)
{
	bool fits(uint32_t maxDepth) const { return stack_class(maxDepth) >= 0; }

	bool build(const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount, const float* boxes, uint32_t boxCount,
	           std::vector<EchoQbvhNode>& nodes, uint32_t& maxDepth)
	{
		nodes.resize((size_t)triangleCount + sphereCount + boxCount);
		uint32_t count = 0;
		if (!build_qbvh_device(triangles, triangleCount, spheres, sphereCount, boxes, boxCount, nodes.data(), &count, &maxDepth)) return false;
		nodes.resize(count);
		return true;
	}
};

struct LastBuild { float rounds, sweepLevels, lightLevels, syncs, launches, buildMs, rebuilt, pad; };
thread_local LastBuild gLastPackBuild = {};

} // namespace

// the calling thread's last build_packs_device: {rounds, QBVH levels read back, light levels read back, synchronising read-backs in all,
// launches, ms of host wall time for the whole build (synchronised), packs rebuilt one by one, 0}
void last_pack_build(float* out8)
{
	const LastBuild& b = gLastPackBuild;
	const float values[8] = { b.rounds, b.sweepLevels, b.lightLevels, b.syncs, b.launches, b.buildMs, b.rebuilt, 0.0f };
	for (int k = 0; k < 8; k++) out8[k] = values[k];
}

int32_t build_packs_device(const packbuild::Inputs& inputs, packbuild::Output& output)
{
	const bool profile = std::getenv("ECHO_B200_PROFILE") != nullptr;
	auto started = std::chrono::steady_clock::now();

	int32_t status;
	uint32_t syncs = 0, launches = 0;
	{
		CudaBackend backend;
		Rebuild rebuild;
		std::string message;
		status = packbuild::build_packs(backend, inputs, rebuild, output, message);
		if (status == ECHO_B200_OK && !check_cuda(cudaStreamSynchronize(backend.stream), "pack build")) status = ECHO_B200_ERR_CUDA;
		if (status != ECHO_B200_OK && !message.empty()) set_error(message);
		syncs = backend.syncs;
		launches = backend.launches;
	}
	if (status != ECHO_B200_OK) return status;

	double buildMs = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - started).count();
	gLastPackBuild = { (float)output.rounds, (float)output.sweepLevels, (float)output.lightLevels, (float)syncs, (float)launches, (float)buildMs, (float)output.rebuilt.size(), 0.0f };
	if (profile)
		std::fprintf(stderr, "[echo_b200 build] packs: %u packs, %u rounds, %u + %u levels, %u syncs, %u launches, %.2f ms\n", inputs.packCount, output.rounds,
		             output.sweepLevels, output.lightLevels, syncs, launches, buildMs);
	return ECHO_B200_OK;
}

} // namespace echo
