// echo_pack_build.h — every pack of an instanced scene built in one call: the reference's QBVH (echo_sweep.h) and light tree
// (echo_light_build.h) of each pack, with PreparedInstance.BoxBound / LightBound of every placement computed where the child trees are.
//
// ScenePreparer builds pack by pack, children before parents: a placement's box is FillBounds(6) of its child's accelerator moved to the
// parent's space, its light row the child's light-tree root moved the same way. A pack therefore waits for nothing but its children, and
// all packs of one HEIGHT (0 for a pack without placements, otherwise 1 + the largest height of the packs it places) can be built together.
// Both level-synchronous drivers take a forest — one root segment per pack — so a call runs at most ECHO_MAX_INSTANCE_LAYERS + 1 rounds of
//   instance bounds   one thread per placement of the round's packs (InstanceBoundsPass)
//   QBVH forest       sweep::build_forest over the round's packs
//   light forest      lightbuild::build_forest over the same packs
// and reads back, per round, as many levels as the deepest tree of the round has instead of every pack's levels one build after another.
// At the end every pack's nodes, light nodes and emitters are laid back to back in pack order, the layout host.prepare gives them.
//
// Everything here is backend-generic: the CUDA backend (packbuild.cu) and the sequential CPU backend of the -m "not gpu" suite
// (tests/c_client/pack_emulation.cpp) run the same passes and the same orchestration.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <string>
#include <vector>

#include "echo_light_build.h"
#include "echo_sweep.h"

namespace echo
{
namespace packbuild
{

// ---- PreparedInstance.BoxBound / LightBound (PreparedInstance.cs:31-40, BoxBound.cs:39-57) ----
// Float4x4.MultiplyPoint / MultiplyDirection left to right without contraction (oracle/math.hpp multiply_point / multiply_direction); the
// cone axis in binary64 as ConeBound's operator * does it (ConeBound.cs:68-72): products summed left to right, divided by
// sqrt((x^2 + y^2) + z^2), rounded once to binary32.

struct Extent
{
	float lo[3], hi[3];
};

SWEEP_HD void transform_box(const float* m, const float* lo, const float* hi, float* outLo, float* outHi) // one box: centre / extent through the matrix
{
	using sweep::f_add;
	using sweep::f_mul;
	using sweep::f_sub;
	float c[3], e[3];
	for (int k = 0; k < 3; k++) { c[k] = f_mul(f_add(hi[k], lo[k]), 0.5f); e[k] = f_mul(f_sub(hi[k], lo[k]), 0.5f); }

	for (int r = 0; r < 3; r++)
	{
		const float* row = m + 4 * r;
		float centre = f_add(f_add(f_add(f_mul(row[0], c[0]), f_mul(row[1], c[1])), f_mul(row[2], c[2])), row[3]);
		float extent = f_add(f_add(f_mul(fabsf(row[0]), e[0]), f_mul(fabsf(row[1]), e[1])), f_mul(fabsf(row[2]), e[2]));
		outLo[r] = f_sub(centre, extent);
		outHi[r] = f_add(centre, extent);
	}
}

SWEEP_HD void unite_box(Extent& into, const float* lo, const float* hi)
{
	for (int k = 0; k < 3; k++)
	{
		into.lo[k] = lo[k] < into.lo[k] ? lo[k] : into.lo[k];
		into.hi[k] = hi[k] > into.hi[k] ? hi[k] : into.hi[k];
	}
}

SWEEP_HD void add_slot(Extent& into, const float* m, const EchoQbvhNode& node, int j)
{
	const float lo[3] = { node.minX[j], node.minY[j], node.minZ[j] }, hi[3] = { node.maxX[j], node.maxY[j], node.maxZ[j] };
	float tlo[3], thi[3];
	transform_box(m, lo, hi, tlo, thi);
	unite_box(into, tlo, thi);
}

SWEEP_HD bool is_node(uint32_t token) { return token != ECHO_TOKEN_EMPTY && (token >> ECHO_TOKEN_INDEX_BITS) == ECHO_TOKEN_TYPE_NODE; }
SWEEP_HD uint32_t token_index(uint32_t token) { return token & ((1u << ECHO_TOKEN_INDEX_BITS) - 1u); }

SWEEP_HD double d_add(double a, double b)
{
#if defined(__CUDA_ARCH__)
	return __dadd_rn(a, b);
#else
	return a + b;
#endif
}

SWEEP_HD double d_mul(double a, double b)
{
#if defined(__CUDA_ARCH__)
	return __dmul_rn(a, b);
#else
	return a * b;
#endif
}

// one thread per placement of the round's packs: the 6-float box row BoundsPass reads for TokenType.Instance and the 12-float row the
// light candidates read. The boxes are united in FillBounds' order (QuadBoundingVolumeHierarchy.cs:62-118, host.fill_bounds): the root's
// leaf slots, then — the mirror pops a stack — its node slots from the last to the first with their leaf slots, then the nodes found there,
// again from the last to the first, with all their slots.
struct InstanceBoundsPass
{
	uint32_t round;
	const uint32_t* instanceRound; // the height of the pack that holds the placement
	const EchoInstance* instances;
	const EchoQbvhNode* const* packNodes;  // every finished pack's quad nodes (root first)
	const EchoLightNode* const* packLights; // every finished pack's light-tree root, null for a pack without emitters
	float* boxes;
	float* lights;

	SWEEP_HD void operator()(uint32_t i) const
	{
		if (instanceRound[i] != round) return;
		const EchoInstance& instance = instances[i];
		const float* m = instance.inverse;
		const EchoQbvhNode* nodes = packNodes[instance.pack];

		const float infinity = sweep::bits_float(0x7F800000u);
		Extent box = { { infinity, infinity, infinity }, { -infinity, -infinity, -infinity } };
		uint32_t first[4], second[16];
		uint32_t firstCount = 0u, secondCount = 0u;

		const EchoQbvhNode& root = nodes[0];
		for (int j = 0; j < 4; j++)
		{
			uint32_t token = root.token4[j];
			if (token == ECHO_TOKEN_EMPTY) continue;
			if (is_node(token)) first[firstCount++] = token_index(token);
			else add_slot(box, m, root, j);
		}

		for (uint32_t f = firstCount; f-- > 0u;)
		{
			const EchoQbvhNode& node = nodes[first[f]];
			for (int j = 0; j < 4; j++)
			{
				uint32_t token = node.token4[j];
				if (token == ECHO_TOKEN_EMPTY) continue;
				if (is_node(token)) second[secondCount++] = token_index(token);
				else add_slot(box, m, node, j);
			}
		}

		for (uint32_t f = secondCount; f-- > 0u;)
		{
			const EchoQbvhNode& node = nodes[second[f]];
			for (int j = 0; j < 4; j++)
				if (node.token4[j] != ECHO_TOKEN_EMPTY) add_slot(box, m, node, j);
		}

		float* out = boxes + (size_t)i * 6;
		for (int k = 0; k < 3; k++) { out[k] = box.lo[k]; out[3 + k] = box.hi[k]; }

		float* row = lights + (size_t)i * 12;
		const EchoLightNode* light = packLights[instance.pack];
		if (!light)
		{
			for (int k = 0; k < 12; k++) row[k] = 0.0f;
			return;
		}

		transform_box(m, light->boxMin, light->boxMax, row, row + 3);
		double axis[3];
		for (int r = 0; r < 3; r++)
		{
			const float* mr = m + 4 * r;
			axis[r] = d_add(d_add(d_mul((double)mr[0], (double)light->coneAxis[0]), d_mul((double)mr[1], (double)light->coneAxis[1])), d_mul((double)mr[2], (double)light->coneAxis[2]));
		}
		double norm = sqrt(d_add(d_add(d_mul(axis[0], axis[0]), d_mul(axis[1], axis[1])), d_mul(axis[2], axis[2])));
		if (!(norm > 1e-300)) norm = 1e-300; // host.prepare's max(norm, 1e-300)
		for (int r = 0; r < 3; r++) row[6 + r] = (float)(axis[r] / norm);
		row[9] = light->cosOffset;
		row[10] = light->cosExtend;
		row[11] = sweep::f_mul(sweep::f_mul(light->power, instance.inverseScale), instance.inverseScale);
	}
};

// ---- the orchestration ----

struct Inputs // host memory
{
	const EchoTriangle* triangles;
	uint32_t triangleCount;
	const EchoSphere* spheres;
	uint32_t sphereCount;
	const EchoMaterial* materials;
	uint32_t materialCount;
	const EchoPointLight* points;
	uint32_t pointCount;
	const EchoPack* packs;
	uint32_t packCount;
	const EchoInstance* instances;
	uint32_t instanceCount;
};

struct Output
{
	std::vector<EchoPack> packs; // the inputs' records with nodeOffset / nodeCount / maxDepth / lightNode* / emitter* filled in
	std::vector<EchoQbvhNode> nodes;
	std::vector<EchoLightNode> lightNodes;
	std::vector<uint32_t> emitterTokens;
	std::vector<uint64_t> emitterPaths;
	std::vector<float> instanceRows; // per placement: the 6-float box row, then the 12-float light row
	float power = 0.0f;              // pack 0's light-tree root power (0 without emitters)
	uint32_t rounds = 0, sweepLevels = 0, lightLevels = 0; // levels read back, summed over the rounds
	std::vector<uint32_t> rebuilt;   // packs the forest gave up on, built one by one instead
};

// Heights of all packs (memoised walk), false on a cycle or nesting deeper than ECHO_MAX_INSTANCE_LAYERS
inline bool pack_heights(const Inputs& in, std::vector<uint32_t>& height)
{
	std::vector<uint8_t> mark(in.packCount, 0); // 1 on the walk, 2 done
	height.assign(in.packCount, 0u);
	std::vector<std::pair<uint32_t, uint32_t>> stack; // (pack, next placement)

	for (uint32_t start = 0; start < in.packCount; start++)
	{
		if (mark[start] == 2) continue;
		stack.push_back({ start, 0u });
		mark[start] = 1;

		while (!stack.empty())
		{
			uint32_t pack = stack.back().first, next = stack.back().second;
			const EchoPack& p = in.packs[pack];

			if (next == p.instanceCount)
			{
				uint32_t layers = 0u;
				for (uint32_t i = 0; i < p.instanceCount; i++)
				{
					uint32_t child = in.instances[p.instanceOffset + i].pack;
					if (height[child] + 1u > layers) layers = height[child] + 1u;
				}
				if (layers > ECHO_MAX_INSTANCE_LAYERS) return false;
				height[pack] = layers;
				mark[pack] = 2;
				stack.pop_back();
				continue;
			}

			stack.back().second = next + 1u;
			uint32_t child = in.instances[p.instanceOffset + next].pack;
			if (mark[child] == 1) return false; // the pack contains itself
			if (mark[child] == 0) { mark[child] = 1; stack.push_back({ child, 0u }); }
		}
	}
	return true;
}

// A pack's swatch ends where the next swatch of the material array begins (another pack's or a placement's), or at the array's end.
inline uint32_t swatch_size(const Inputs& in, uint32_t offset)
{
	uint32_t end = in.materialCount;
	for (uint32_t p = 0; p < in.packCount; p++) if (in.packs[p].materialOffset > offset && in.packs[p].materialOffset < end) end = in.packs[p].materialOffset;
	for (uint32_t i = 0; i < in.instanceCount; i++) if (in.instances[i].materialOffset > offset && in.instances[i].materialOffset < end) end = in.instances[i].materialOffset;
	return end > offset ? end - offset : 0u;
}

template<class Backend, class T>
T* upload(Backend& backend, const T* source, uint64_t count)
{
	T* destination = (T*)backend.allocate(sizeof(T) * count + 256);
	if (destination && count != 0u && !backend.write(destination, source, (uint32_t)count)) return nullptr;
	return destination;
}

// Backend: both drivers' concept (allocate: a block that lives as long as the backend; write). Rebuild: the per-pack path for the packs of a
// round the forest gives up on —
//   bool fits(uint32_t maxDepth)                                        a forest tree of this depth can be used as it is
//   bool build(triangles, n, spheres, n, boxes, n, std::vector<EchoQbvhNode>& nodes, uint32_t& maxDepth)   host memory in and out
// Returns an ECHO_B200_* status; `message` says why when it is not OK.
template<class Backend, class Rebuild>
int32_t build_packs(Backend& backend, const Inputs& in, Rebuild& rebuild, Output& out, std::string& message)
{
	const uint32_t P = in.packCount, I = in.instanceCount;
	if (P == 0u) { message = "a scene has at least one pack"; return ECHO_B200_ERR_INVALID; }

	for (uint32_t p = 0; p < P; p++)
	{
		const EchoPack& pack = in.packs[p];
		if ((uint64_t)pack.triangleOffset + pack.triangleCount > in.triangleCount || (uint64_t)pack.sphereOffset + pack.sphereCount > in.sphereCount
			|| (uint64_t)pack.instanceOffset + pack.instanceCount > I || (uint64_t)pack.pointLightOffset + pack.pointLightCount > in.pointCount
			|| pack.materialOffset > in.materialCount) { message = "pack range out of bounds"; return ECHO_B200_ERR_INVALID; }
		uint64_t primitives = (uint64_t)pack.triangleCount + pack.sphereCount + pack.instanceCount;
		if (primitives < 2u) { message = "every pack needs at least 2 primitives (placements included)"; return ECHO_B200_ERR_INVALID; }
		if (primitives >= (1ull << ECHO_TOKEN_INDEX_BITS)) { message = "a pack holds fewer than 2^28 primitives"; return ECHO_B200_ERR_INVALID; }
	}
	for (uint32_t i = 0; i < I; i++)
		if (in.instances[i].pack >= P || in.instances[i].pack == 0u) { message = "instance refers to a pack that does not exist (pack 0 is the scene)"; return ECHO_B200_ERR_INVALID; }

	std::vector<uint32_t> height;
	if (!pack_heights(in, height)) { message = "instancing deeper than TokenHierarchy.MaxLayer (5) or cyclic"; return ECHO_B200_ERR_INVALID; }
	uint32_t tallest = 0u;
	for (uint32_t h : height) tallest = h > tallest ? h : tallest;

	std::vector<uint32_t> instanceRound(I, 0u);
	for (uint32_t p = 0; p < P; p++)
		for (uint32_t i = 0; i < in.packs[p].instanceCount; i++) instanceRound[in.packs[p].instanceOffset + i] = height[p];

	// the shared arrays in backend memory; the placements' rows and the finished packs' trees fill in round by round
	const EchoTriangle* triangles = upload(backend, in.triangles, in.triangleCount);
	const EchoSphere* spheres = upload(backend, in.spheres, in.sphereCount);
	const EchoMaterial* materials = upload(backend, in.materials, in.materialCount);
	const EchoPointLight* points = upload(backend, in.points, in.pointCount);
	const EchoInstance* instances = upload(backend, in.instances, I);
	const uint32_t* rounds = upload(backend, instanceRound.data(), I);
	float* boxes = (float*)backend.allocate(sizeof(float) * 6 * I + 256);
	float* lights = (float*)backend.allocate(sizeof(float) * 12 * I + 256);
	const EchoQbvhNode** packNodes = (const EchoQbvhNode**)backend.allocate(sizeof(void*) * P + 256);
	const EchoLightNode** packLights = (const EchoLightNode**)backend.allocate(sizeof(void*) * P + 256);
	if (!triangles || !spheres || !materials || !points || !instances || !rounds || !boxes || !lights || !packNodes || !packLights) return ECHO_B200_ERR_CUDA;

	std::vector<const EchoQbvhNode*> nodeTable(P, nullptr);
	std::vector<const EchoLightNode*> lightTable(P, nullptr);
	std::vector<std::vector<EchoQbvhNode>> packNodeArrays(P);
	std::vector<uint32_t> packDepth(P, 0u);
	std::vector<std::vector<EchoLightNode>> packLightNodes(P);
	std::vector<std::vector<uint32_t>> packTokens(P);
	std::vector<std::vector<uint64_t>> packPaths(P);

	for (uint32_t round = 0; round <= tallest; round++)
	{
		std::vector<uint32_t> members;
		for (uint32_t p = 0; p < P; p++) if (height[p] == round) members.push_back(p);
		if (members.empty()) continue;
		++out.rounds;

		if (round > 0u && !backend.for_each(I, InstanceBoundsPass{ round, rounds, instances, packNodes, packLights, boxes, lights })) return ECHO_B200_ERR_CUDA;

		// the QBVH forest
		std::vector<sweep::PackRange> ranges(members.size());
		uint32_t begin = 0u;
		for (size_t k = 0; k < members.size(); k++)
		{
			const EchoPack& pack = in.packs[members[k]];
			ranges[k] = { pack.triangleOffset, pack.triangleCount, pack.sphereOffset, pack.sphereCount, pack.instanceOffset, pack.instanceCount, begin };
			begin += sweep::range_size(ranges[k]);
		}

		sweep::Result trees = sweep::build_forest(backend, ranges.data(), (uint32_t)members.size(), triangles, spheres, boxes);
		if (!trees.ok) return ECHO_B200_ERR_CUDA;
		out.sweepLevels += trees.levels;

		std::vector<EchoQbvhNode> all;
		if (!trees.gaveUp)
		{
			all.resize(trees.nodeCount);
			if (!backend.read(trees.quads, all.data(), trees.nodeCount)) return ECHO_B200_ERR_CUDA;
		}

		for (size_t k = 0; k < members.size(); k++)
		{
			const uint32_t p = members[k];
			if (!trees.gaveUp && rebuild.fits(trees.packMaxDepth[k]))
			{
				const EchoQbvhNode* first = all.data() + trees.packNodeBase[k];
				packNodeArrays[p].assign(first, first + trees.packNodeCount[k]);
				packDepth[p] = trees.packMaxDepth[k];
				nodeTable[p] = trees.quads + trees.packNodeBase[k];
				continue;
			}

			// the existing per-pack path (which falls back to another builder where the reference's tree cannot be used)
			const EchoPack& pack = in.packs[p];
			std::vector<float> packBoxes(6 * (size_t)pack.instanceCount);
			if (pack.instanceCount != 0u && !backend.read(boxes + (size_t)6 * pack.instanceOffset, packBoxes.data(), 6u * pack.instanceCount)) return ECHO_B200_ERR_CUDA;
			if (!rebuild.build(in.triangles + pack.triangleOffset, pack.triangleCount, in.spheres + pack.sphereOffset, pack.sphereCount, packBoxes.data(), pack.instanceCount,
			                   packNodeArrays[p], packDepth[p])) { message = "the per-pack build of a pack the forest gave up on failed"; return ECHO_B200_ERR_CUDA; }
			const EchoQbvhNode* nodes = upload(backend, packNodeArrays[p].data(), packNodeArrays[p].size());
			if (!nodes) return ECHO_B200_ERR_CUDA;
			nodeTable[p] = nodes;
			out.rebuilt.push_back(p);
		}

		// the light forest
		std::vector<lightbuild::LightPack> lightPacks(members.size());
		for (size_t k = 0; k < members.size(); k++)
		{
			const EchoPack& pack = in.packs[members[k]];
			lightbuild::LightPack& light = lightPacks[k];
			light = {};
			light.triangleOffset = pack.triangleOffset; light.triangleCount = pack.triangleCount;
			light.sphereOffset = pack.sphereOffset; light.sphereCount = pack.sphereCount;
			light.instanceOffset = pack.instanceOffset; light.instanceCount = pack.instanceCount;
			light.materialOffset = pack.materialOffset; light.materialCount = swatch_size(in, pack.materialOffset);
			light.pointOffset = pack.pointLightOffset; light.pointCount = pack.pointLightCount;
		}

		const lightbuild::Forest forest = { triangles, spheres, materials, points, lights, lightPacks.data(), (uint32_t)members.size() };
		lightbuild::Result trees2 = lightbuild::build_forest(backend, forest);
		if (!trees2.ok) return ECHO_B200_ERR_CUDA;
		if (trees2.unsupported) { message = "light tree deeper than 63 levels (LightTree.cs:29)"; return ECHO_B200_ERR_UNSUPPORTED; }
		out.lightLevels += trees2.levels;

		std::vector<EchoLightNode> lightNodes(trees2.nodeCount);
		std::vector<uint32_t> tokens(trees2.emitterCount);
		std::vector<unsigned long long> paths(trees2.emitterCount);
		if (trees2.emitterCount != 0u
			&& (!backend.read(trees2.nodes, lightNodes.data(), trees2.nodeCount) || !backend.read(trees2.emitterTokens, tokens.data(), trees2.emitterCount)
				|| !backend.read(trees2.emitterPaths, paths.data(), trees2.emitterCount))) return ECHO_B200_ERR_CUDA;

		for (size_t k = 0; k < members.size(); k++)
		{
			const uint32_t p = members[k];
			const lightbuild::LightPack& light = trees2.packs[k];
			if (light.emitterCount == 0u) continue;
			uint32_t nodeCount = 2u * light.emitterCount - 1u;
			packLightNodes[p].assign(lightNodes.begin() + light.nodeBase, lightNodes.begin() + light.nodeBase + nodeCount);
			packTokens[p].assign(tokens.begin() + light.emitterBase, tokens.begin() + light.emitterBase + light.emitterCount);
			packPaths[p].assign(paths.begin() + light.emitterBase, paths.begin() + light.emitterBase + light.emitterCount);
			lightTable[p] = trees2.nodes + light.nodeBase;
		}

		if (!backend.write(packNodes, nodeTable.data(), P) || !backend.write(packLights, lightTable.data(), P)) return ECHO_B200_ERR_CUDA;
	}

	// every pack's arrays back to back in pack order (host.prepare's layout)
	out.packs.assign(in.packs, in.packs + P);
	for (uint32_t p = 0; p < P; p++)
	{
		EchoPack& pack = out.packs[p];
		pack.nodeOffset = (uint32_t)out.nodes.size();
		pack.nodeCount = (uint32_t)packNodeArrays[p].size();
		pack.maxDepth = packDepth[p];
		pack.lightNodeOffset = (uint32_t)out.lightNodes.size();
		pack.lightNodeCount = (uint32_t)packLightNodes[p].size();
		pack.emitterOffset = (uint32_t)out.emitterTokens.size();
		pack.emitterCount = (uint32_t)packTokens[p].size();
		out.nodes.insert(out.nodes.end(), packNodeArrays[p].begin(), packNodeArrays[p].end());
		out.lightNodes.insert(out.lightNodes.end(), packLightNodes[p].begin(), packLightNodes[p].end());
		out.emitterTokens.insert(out.emitterTokens.end(), packTokens[p].begin(), packTokens[p].end());
		out.emitterPaths.insert(out.emitterPaths.end(), packPaths[p].begin(), packPaths[p].end());
	}
	out.power = packLightNodes[0].empty() ? 0.0f : packLightNodes[0][0].power;

	out.instanceRows.resize((size_t)18 * I);
	std::vector<float> rows(12 * (size_t)I);
	if (I != 0u && (!backend.read(boxes, rows.data(), 6u * I))) return ECHO_B200_ERR_CUDA;
	for (uint32_t i = 0; i < I; i++) memcpy(&out.instanceRows[18 * (size_t)i], &rows[6 * (size_t)i], sizeof(float) * 6);
	if (I != 0u && (!backend.read(lights, rows.data(), 12u * I))) return ECHO_B200_ERR_CUDA;
	for (uint32_t i = 0; i < I; i++) memcpy(&out.instanceRows[18 * (size_t)i + 6], &rows[12 * (size_t)i], sizeof(float) * 12);
	return ECHO_B200_OK;
}

// The caller-owned outputs of echo_b200_build_packs: too little room is ECHO_B200_ERR_INVALID with the needed counts.
inline int32_t deliver(const Output& out, EchoPack* packs, EchoQbvhNode* nodes, uint32_t nodeCapacity, uint32_t* nodeCount, EchoLightNode* lightNodes, uint32_t lightNodeCapacity,
                       uint32_t* lightNodeCount, uint32_t* emitterTokens, uint64_t* emitterPaths, uint32_t emitterCapacity, uint32_t* emitterCount, float* power, std::string& message)
{
	*nodeCount = (uint32_t)out.nodes.size();
	*lightNodeCount = (uint32_t)out.lightNodes.size();
	*emitterCount = (uint32_t)out.emitterTokens.size();
	*power = out.power;
	if (out.nodes.size() > nodeCapacity || out.lightNodes.size() > lightNodeCapacity || out.emitterTokens.size() > emitterCapacity)
	{
		message = "pack build output buffers too small (needed counts returned)";
		return ECHO_B200_ERR_INVALID;
	}

	memcpy(packs, out.packs.data(), sizeof(EchoPack) * out.packs.size());
	if (!out.nodes.empty()) memcpy(nodes, out.nodes.data(), sizeof(EchoQbvhNode) * out.nodes.size());
	if (!out.lightNodes.empty()) memcpy(lightNodes, out.lightNodes.data(), sizeof(EchoLightNode) * out.lightNodes.size());
	if (!out.emitterTokens.empty())
	{
		memcpy(emitterTokens, out.emitterTokens.data(), sizeof(uint32_t) * out.emitterTokens.size());
		memcpy(emitterPaths, out.emitterPaths.data(), sizeof(uint64_t) * out.emitterPaths.size());
	}
	return ECHO_B200_OK;
}

} // namespace packbuild
} // namespace echo
