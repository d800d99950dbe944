// pack_emulation.cpp — test infrastructure: a sequential CPU backend for echorenderer_b200/csrc/echo_pack_build.h, so that the CPU suite
// (-m "not gpu") runs the very orchestration, forests and instance-bounds pass echo_b200_build_packs runs (packbuild.cu) and compares every
// pack's trees with the host mirror's byte for byte. Not part of the product: libecho_b200.so never links this file, and nothing here is timed.
//
//   g++ -std=c++17 -O2 -ffp-contract=off -shared -fPIC tests/c_client/pack_emulation.cpp -o libpack_emulation.so
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

#include "../../echorenderer_b200/csrc/echo_pack_build.h"

namespace
{

using namespace echo;

struct CpuBackend // both drivers' backend concept, memory in the host's address space
{
	std::vector<char*> blocks;
	bool reverse = false; // run every pass over descending indices: no pass may depend on the order of its indices

	~CpuBackend() { for (char* block : blocks) std::free(block); }

	char* allocate(size_t bytes)
	{
		blocks.push_back((char*)std::calloc(bytes ? bytes : 1, 1));
		return blocks.back();
	}

	template<class F>
	bool for_each(uint32_t n, const F& f)
	{
		if (reverse) for (uint32_t i = n; i-- > 0u;) f(i);
		else for (uint32_t i = 0; i < n; i++) f(i);
		return true;
	}

	bool sort_pairs(const unsigned long long* keysIn, unsigned long long* keysOut, const uint32_t* valuesIn, uint32_t* valuesOut, uint32_t n, int endBit)
	{
		const unsigned long long mask = endBit >= 64 ? ~0ull : (1ull << endBit) - 1ull;
		std::vector<uint32_t> order(n);
		std::iota(order.begin(), order.end(), 0u);
		std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return (keysIn[a] & mask) < (keysIn[b] & mask); });
		for (uint32_t i = 0; i < n; i++) { keysOut[i] = keysIn[order[i]]; valuesOut[i] = valuesIn[order[i]]; }
		return true;
	}

	bool scan_items(const sweep::ScanItem* in, sweep::ScanItem* out, uint32_t n)
	{
		sweep::ScanOp op;
		for (uint32_t i = 0; i < n; i++) out[i] = i == 0u ? in[0] : op(out[i - 1u], in[i]);
		return true;
	}

	bool exclusive_sum(const uint32_t* in, uint32_t* out, uint32_t n)
	{
		uint32_t sum = 0u;
		for (uint32_t i = 0; i < n; i++) { uint32_t value = in[i]; out[i] = sum; sum += value; }
		return true;
	}

	template<class T> bool read(const T* source, T* destination, uint32_t n) { std::memcpy((void*)destination, (const void*)source, sizeof(T) * n); return true; }
	template<class T> bool write(T* destination, const T* source, uint32_t n) { std::memcpy((void*)destination, (const void*)source, sizeof(T) * n); return true; }
	bool fill_zero(void* pointer, size_t bytes) { std::memset(pointer, 0, bytes); return true; }
};

struct Rebuild // the per-pack path: the single-pack sweep build (the CUDA library falls back further, to a clustered build)
{
	uint32_t depthLimit;
	bool reverse;

	bool fits(uint32_t maxDepth) const { return maxDepth <= depthLimit; }

	bool build(const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount, const float* boxes, uint32_t boxCount,
	           std::vector<EchoQbvhNode>& nodes, uint32_t& maxDepth)
	{
		CpuBackend backend;
		backend.reverse = reverse;
		sweep::Result result = sweep::build(backend, triangles, triangleCount, spheres, sphereCount, boxes, boxCount);
		if (!result.ok || result.gaveUp) return false;
		nodes.assign(result.quads, result.quads + result.nodeCount);
		maxDepth = result.maxDepth;
		return true;
	}
};

thread_local std::string gMessage;

} // namespace

// echo_b200_build_packs' arguments (without the device) and status, on the CPU backend; plus `reverse`, a depth above which a forest tree is
// rebuilt by the per-pack path, `outRows` (18 floats per placement: its box row, then its light row) and `outStats` {rounds, QBVH levels read
// back, light levels read back, packs rebuilt}.
extern "C" int32_t pack_emulation_build(const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
                                        const EchoMaterial* materials, uint32_t materialCount, const EchoPointLight* points, uint32_t pointCount,
                                        EchoPack* packs, uint32_t packCount, const EchoInstance* instances, uint32_t instanceCount,
                                        EchoQbvhNode* outNodes, uint32_t nodeCapacity, uint32_t* outNodeCount,
                                        EchoLightNode* outLightNodes, uint32_t lightNodeCapacity, uint32_t* outLightNodeCount,
                                        uint32_t* outTokens, uint64_t* outPaths, uint32_t emitterCapacity, uint32_t* outEmitterCount, float* outPower,
                                        int32_t reverse, uint32_t depthLimit, float* outRows, uint32_t* outStats)
{
	CpuBackend backend;
	backend.reverse = reverse != 0;
	Rebuild rebuild = { depthLimit, reverse != 0 };
	const packbuild::Inputs inputs = { triangles, triangleCount, spheres, sphereCount, materials, materialCount, points, pointCount, packs, packCount, instances, instanceCount };
	packbuild::Output output;
	int32_t status = packbuild::build_packs(backend, inputs, rebuild, output, gMessage);
	if (status != ECHO_B200_OK) return status;

	if (outRows && !output.instanceRows.empty()) std::memcpy(outRows, output.instanceRows.data(), sizeof(float) * output.instanceRows.size());
	outStats[0] = output.rounds;
	outStats[1] = output.sweepLevels;
	outStats[2] = output.lightLevels;
	outStats[3] = (uint32_t)output.rebuilt.size();
	return packbuild::deliver(output, packs, outNodes, nodeCapacity, outNodeCount, outLightNodes, lightNodeCapacity, outLightNodeCount, outTokens, outPaths, emitterCapacity,
	                          outEmitterCount, outPower, gMessage);
}

extern "C" const char* pack_emulation_message() { return gMessage.c_str(); }
