// sweep.cu — the CUDA backend of echo_sweep.h: the reference's SweepBuilder tree (SweepBuilder.cs + the QuadBoundingVolumeHierarchy
// collapse), built on the device level by level and emitted byte for byte as the reference's recursive build emits it. The passes and
// the driver live in echo_sweep.h, shared with the CPU emulation the -m "not gpu" suite checks against the host mirror; this file only
// supplies the generic kernel, the CUB sort / scans, memory and the copies. BUILD_ALGORITHM = 2 (the default of echo_b200_build_qbvh).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <chrono>
#include <cstdio>
#include <cstdlib>

#include "echo_internal.h"
#include "echo_sweep.h"

namespace echo
{

namespace
{

constexpr int kSweepBlock = 256;

template<class F>
__global__ void __launch_bounds__(kSweepBlock) sweep_for_each_kernel(uint32_t n, F f)
{
	uint32_t i = blockIdx.x * kSweepBlock + threadIdx.x;
	if (i < n) f(i);
}

struct CudaBackend
{
	cudaStream_t stream = nullptr;
	char* block = nullptr;
	void* scratch = nullptr;
	size_t scratchBytes = 0;
	uint32_t launches = 0, syncs = 0;

	~CudaBackend() { cudaFree(block); }

	bool prepare(uint32_t total) // the largest temporary storage any CUB call of the build can ask for
	{
		size_t sortBytes = 0, scanBytes = 0, sumBytes = 0;
		if (!check_cuda(cub::DeviceRadixSort::SortPairs(nullptr, sortBytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (const uint32_t*)nullptr, (uint32_t*)nullptr,
		                                                 (int)total, 0, 64, stream), "cub sort (size)")) return false;
		if (!check_cuda(cub::DeviceScan::InclusiveScan(nullptr, scanBytes, (const sweep::ScanItem*)nullptr, (sweep::ScanItem*)nullptr, sweep::ScanOp(), (int)total, stream), "cub scan (size)")) return false;
		if (!check_cuda(cub::DeviceScan::ExclusiveSum(nullptr, sumBytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)total + 2, stream), "cub sum (size)")) return false;
		scratchBytes = std::max(sortBytes, std::max(scanBytes, sumBytes));
		scratchBytes = (scratchBytes + 255) & ~size_t(255);
		return true;
	}

	char* allocate(size_t bytes)
	{
		if (!check_cuda(cudaMalloc((void**)&block, bytes + scratchBytes), "cudaMalloc(sweep build)")) return nullptr;
		scratch = block + bytes;
		return block;
	}

	template<class F>
	bool for_each(uint32_t n, const F& f)
	{
		if (n == 0u) return true;
		sweep_for_each_kernel<<<(n + kSweepBlock - 1) / kSweepBlock, kSweepBlock, 0, stream>>>(n, f);
		++launches;
		return check_cuda(cudaGetLastError(), "sweep build launch");
	}

	bool sort_pairs(const unsigned long long* keysIn, unsigned long long* keysOut, const uint32_t* valuesIn, uint32_t* valuesOut, uint32_t n, int endBit)
	{
		size_t bytes = scratchBytes; // cub's radix sort is stable
		++launches;
		return check_cuda(cub::DeviceRadixSort::SortPairs(scratch, bytes, keysIn, keysOut, valuesIn, valuesOut, (int)n, 0, endBit, stream), "cub sort");
	}

	bool scan_items(const sweep::ScanItem* in, sweep::ScanItem* out, uint32_t n)
	{
		size_t bytes = scratchBytes;
		++launches;
		return check_cuda(cub::DeviceScan::InclusiveScan(scratch, bytes, in, out, sweep::ScanOp(), (int)n, stream), "cub scan");
	}

	bool exclusive_sum(const uint32_t* in, uint32_t* out, uint32_t n)
	{
		size_t bytes = scratchBytes;
		++launches;
		return check_cuda(cub::DeviceScan::ExclusiveSum(scratch, bytes, in, out, (int)n, stream), "cub sum");
	}

	template<class T>
	bool read(const T* source, T* destination, uint32_t n)
	{
		++syncs;
		return check_cuda(cudaMemcpyAsync(destination, source, sizeof(T) * n, cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(sweep read)")
			&& check_cuda(cudaStreamSynchronize(stream), "sweep build level");
	}

	template<class T>
	bool write(T* destination, const T* source, uint32_t n)
	{
		// the source is a local of the driver: the copy must have left it before the driver moves on (pageable memory: it has, on return)
		return check_cuda(cudaMemcpyAsync(destination, source, sizeof(T) * n, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(sweep write)");
	}

	bool fill_zero(void* pointer, size_t bytes) { return check_cuda(cudaMemsetAsync(pointer, 0, bytes, stream), "cudaMemsetAsync(sweep)"); }
};

struct LastBuild { float uploadMs, buildMs, downloadMs, levels; };
thread_local LastBuild gLastBuild = { 0.0f, 0.0f, 0.0f, 0.0f };

} // namespace

// the calling thread's last build_qbvh_sweep: {upload, device build, download} in ms of host wall time around synchronised phases, binary levels
void last_sweep_build(float* out4)
{
	out4[0] = gLastBuild.uploadMs; out4[1] = gLastBuild.buildMs; out4[2] = gLastBuild.downloadMs; out4[3] = gLastBuild.levels;
}

// false: a CUDA call failed. `gaveUp`: the tree chains deeper than sweep::kMaxLevels (thousands of coincident primitives) or the device
// lacks the working memory; nothing was written.
bool build_qbvh_sweep(const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
                      const float* instanceBounds, uint32_t instanceCount, EchoQbvhNode* outNodes, uint32_t* outNodeCount, uint32_t* outMaxDepth, bool* gaveUp)
{
	*gaveUp = false;
	uint64_t total64 = (uint64_t)triangleCount + sphereCount + instanceCount;
	if (total64 < 2 || total64 >= (1ull << ECHO_TOKEN_INDEX_BITS)) { set_error("a tree needs 2..2^28-1 primitives"); return false; }

	const bool profile = std::getenv("ECHO_B200_PROFILE") != nullptr;
	auto clock = [] { return std::chrono::steady_clock::now(); };
	auto since = [&](std::chrono::steady_clock::time_point from) { return std::chrono::duration<double, std::milli>(clock() - from).count(); };
	auto started = clock();

	CudaBackend backend;
	if (!backend.prepare((uint32_t)total64)) return false;

	// ~450 bytes of working memory per primitive: when the device cannot spare them the caller's clustered build (~150) takes over
	{
		sweep::Buffers probe;
		sweep::Arena measure;
		probe.carve(measure, total64, 1u);
		size_t freeBytes = 0, totalBytes = 0;
		if (!check_cuda(cudaMemGetInfo(&freeBytes, &totalBytes), "cudaMemGetInfo")) return false;
		size_t needed = measure.used + backend.scratchBytes + sizeof(EchoTriangle) * triangleCount + sizeof(EchoSphere) * sphereCount + sizeof(float) * 6 * instanceCount + (1u << 20);
		if (needed > freeBytes - freeBytes / 16) { *gaveUp = true; return true; }
	}

	struct Inputs
	{
		char* base = nullptr;
		~Inputs() { cudaFree(base); }
	} inputs;

	size_t triangleBytes = (sizeof(EchoTriangle) * triangleCount + 255) & ~size_t(255), sphereBytes = (sizeof(EchoSphere) * sphereCount + 255) & ~size_t(255);
	size_t instanceBytes = sizeof(float) * 6 * instanceCount;
	if (!check_cuda(cudaMalloc((void**)&inputs.base, triangleBytes + sphereBytes + instanceBytes + 256), "cudaMalloc(sweep inputs)")) return false;
	EchoTriangle* dTriangles = (EchoTriangle*)inputs.base;
	EchoSphere* dSpheres = (EchoSphere*)(inputs.base + triangleBytes);
	float* dInstanceBounds = (float*)(inputs.base + triangleBytes + sphereBytes);

	if (!check_cuda(cudaMemcpyAsync(dTriangles, triangles, sizeof(EchoTriangle) * triangleCount, cudaMemcpyHostToDevice, backend.stream), "cudaMemcpyAsync(triangles)")
		|| !check_cuda(cudaMemcpyAsync(dSpheres, spheres, sizeof(EchoSphere) * sphereCount, cudaMemcpyHostToDevice, backend.stream), "cudaMemcpyAsync(spheres)")
		|| (instanceCount != 0u && !check_cuda(cudaMemcpyAsync(dInstanceBounds, instanceBounds, instanceBytes, cudaMemcpyHostToDevice, backend.stream), "cudaMemcpyAsync(instance bounds)"))) return false;
	if (!check_cuda(cudaStreamSynchronize(backend.stream), "sweep upload")) return false; // the phases are reported separately (last_sweep_build)
	double uploadMs = since(started);
	auto phase = clock();

	sweep::Result result = sweep::build(backend, dTriangles, triangleCount, dSpheres, sphereCount, dInstanceBounds, instanceCount);
	if (!result.ok) return false;
	if (result.gaveUp) { *gaveUp = true; return true; }

	double buildMs = since(phase);
	phase = clock();

	if (!check_cuda(cudaMemcpy(outNodes, result.quads, sizeof(EchoQbvhNode) * result.nodeCount, cudaMemcpyDeviceToHost), "cudaMemcpy(nodes)")) return false;
	double downloadMs = since(phase);

	*outNodeCount = result.nodeCount;
	*outMaxDepth = result.maxDepth;
	gLastBuild = { (float)uploadMs, (float)buildMs, (float)downloadMs, (float)result.levels };

	if (profile)
		std::fprintf(stderr, "[echo_b200 build] sweep: %llu primitives -> %u nodes, quad depth %u, %u binary levels: upload %.2f ms, build %.2f ms (%u launches, %u syncs), download %.2f ms\n",
		             (unsigned long long)total64, result.nodeCount, result.maxDepth, result.levels, uploadMs, buildMs, backend.launches, backend.syncs, downloadMs);
	return true;
}

} // namespace echo
