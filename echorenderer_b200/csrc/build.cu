// build.cu — optional device-side tree build (SURVEY.md §8f rank 4): a binary BVH built on the device and collapsed into the
// reference's QBVH node format (QuadBoundingVolumeHierarchy.cs:363-565: every other binary level becomes a quad node, children
// sorted by the lower bound along the split axis, a leaf child becomes a [leaf, empty] pair with axis 3, empty slots at +infinity).
// Two ways to get the binary tree, both over the primitives sorted by 63-bit Morton code:
//   PLOC (default)  parallel locally-ordered clustering (Meister & Bittner 2018): bottom-up agglomeration — every cluster looks
//                   for the neighbour within +-16 positions whose union with it has the smallest surface area, mutual
//                   nearest neighbours merge, the survivors are compacted, repeat until one cluster is left. The surface-area
//                   criterion is the SAH's, applied locally; it closes most of the gap to the reference's full-sweep SAH tree.
//   LBVH            the linear BVH of Karras 2012 ("Maximizing Parallelism in the Construction of BVHs, Octrees, and k-d Trees"):
//                   splits at the highest differing Morton bit. Fastest to build, lowest quality (ECHO_B200_BUILD_ALGORITHM=0).
//
// Neither is the reference's SweepBuilder tree (full-sweep SAH; echo_host_build_qbvh is its host-side mirror and the default of
// the tests and the bench). Hit results do not depend on the tree except for the order in which exact ties are found, and both
// the device and the oracle walk whichever tree they are given.
// Sorting and the prefix sums are CUB (a CUDA toolkit library); the other passes are written here.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "echo_internal.h"

namespace echo
{

namespace
{

constexpr int kBuildBlock = 256;
constexpr uint32_t kLeafFlag = 0x80000000u; // child reference: leaf (sorted position) or internal node index

struct BuildBox
{
	float minX, minY, minZ, maxX, maxY, maxZ;
};

__device__ __forceinline__ int float_to_ordered(float value)
{
	int bits = __float_as_int(value);
	return bits >= 0 ? bits : bits ^ 0x7FFFFFFF;
}

__device__ __forceinline__ float ordered_to_float(int value) { return __int_as_float(value >= 0 ? value : value ^ 0x7FFFFFFF); }

// PreparedTriangle.BoxBound (TriangleEntity.cs:142) / PreparedSphere.BoxBound (SphereEntity.cs:66) + the scene bound of the centres
__global__ void primitive_bounds_kernel(const EchoTriangle* __restrict__ triangles, uint32_t triangleCount, const EchoSphere* __restrict__ spheres, uint32_t sphereCount,
                                        const float* __restrict__ instanceBounds, uint32_t instanceCount, BuildBox* __restrict__ boxes, uint32_t* __restrict__ tokens, int* __restrict__ sceneBound)
{
	uint32_t i = blockIdx.x * kBuildBlock + threadIdx.x;
	uint32_t total = triangleCount + sphereCount + instanceCount;
	if (i >= total) return;

	BuildBox box;

	if (i < triangleCount)
	{
		const EchoTriangle& t = triangles[i];
		float v1x = t.vertex0[0] + t.edge1[0], v1y = t.vertex0[1] + t.edge1[1], v1z = t.vertex0[2] + t.edge1[2];
		float v2x = t.vertex0[0] + t.edge2[0], v2y = t.vertex0[1] + t.edge2[1], v2z = t.vertex0[2] + t.edge2[2];
		box = { fminf(t.vertex0[0], fminf(v1x, v2x)), fminf(t.vertex0[1], fminf(v1y, v2y)), fminf(t.vertex0[2], fminf(v1z, v2z)),
		        fmaxf(t.vertex0[0], fmaxf(v1x, v2x)), fmaxf(t.vertex0[1], fmaxf(v1y, v2y)), fmaxf(t.vertex0[2], fmaxf(v1z, v2z)) };
		tokens[i] = ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_TRIANGLE, i);
	}
	else if (i >= triangleCount + sphereCount) // PreparedInstance.BoxBound of a placement: min xyz, max xyz
	{
		const float* b = instanceBounds + (size_t)(i - triangleCount - sphereCount) * 6;
		box = { b[0], b[1], b[2], b[3], b[4], b[5] };
		tokens[i] = ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_INSTANCE, i - triangleCount - sphereCount);
	}
	else
	{
		const EchoSphere& s = spheres[i - triangleCount];
		box = { s.position[0] - s.radius, s.position[1] - s.radius, s.position[2] - s.radius, s.position[0] + s.radius, s.position[1] + s.radius, s.position[2] + s.radius };
		tokens[i] = ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_SPHERE, i - triangleCount);
	}

	boxes[i] = box;

	float cx = (box.minX + box.maxX) * 0.5f, cy = (box.minY + box.maxY) * 0.5f, cz = (box.minZ + box.maxZ) * 0.5f;
	atomicMin(sceneBound + 0, float_to_ordered(cx));
	atomicMin(sceneBound + 1, float_to_ordered(cy));
	atomicMin(sceneBound + 2, float_to_ordered(cz));
	atomicMax(sceneBound + 3, float_to_ordered(cx));
	atomicMax(sceneBound + 4, float_to_ordered(cy));
	atomicMax(sceneBound + 5, float_to_ordered(cz));
}

__device__ __forceinline__ unsigned long long spread21(unsigned long long v) // 21 bits -> every third bit
{
	v &= 0x1FFFFFull;
	v = (v | v << 32) & 0x1F00000000FFFFull;
	v = (v | v << 16) & 0x1F0000FF0000FFull;
	v = (v | v << 8) & 0x100F00F00F00F00Full;
	v = (v | v << 4) & 0x10C30C30C30C30C3ull;
	v = (v | v << 2) & 0x1249249249249249ull;
	return v;
}

__global__ void morton_kernel(const BuildBox* __restrict__ boxes, uint32_t total, const int* __restrict__ sceneBound, unsigned long long* __restrict__ keys, uint32_t* __restrict__ order)
{
	uint32_t i = blockIdx.x * kBuildBlock + threadIdx.x;
	if (i >= total) return;

	float lowX = ordered_to_float(sceneBound[0]), lowY = ordered_to_float(sceneBound[1]), lowZ = ordered_to_float(sceneBound[2]);
	float highX = ordered_to_float(sceneBound[3]), highY = ordered_to_float(sceneBound[4]), highZ = ordered_to_float(sceneBound[5]);
	BuildBox box = boxes[i];

	auto quantise = [](float centre, float low, float high) -> unsigned long long
	{
		float extent = high - low;
		float unit = extent > 0.0f ? (centre - low) / extent : 0.0f;
		unit = fminf(fmaxf(unit, 0.0f), 1.0f);
		return (unsigned long long)fminf(unit * 2097152.0f, 2097151.0f);
	};

	unsigned long long x = quantise((box.minX + box.maxX) * 0.5f, lowX, highX);
	unsigned long long y = quantise((box.minY + box.maxY) * 0.5f, lowY, highY);
	unsigned long long z = quantise((box.minZ + box.maxZ) * 0.5f, lowZ, highZ);
	keys[i] = spread21(x) << 2 | spread21(y) << 1 | spread21(z);
	order[i] = i;
}

// length of the common prefix of sorted keys i and j; equal keys fall back to the positions so that every pair differs
__device__ __forceinline__ int common_prefix(const unsigned long long* __restrict__ keys, int total, int i, int j)
{
	if (j < 0 || j >= total) return -1;
	unsigned long long a = keys[i], b = keys[j];
	if (a != b) return __clzll((long long)(a ^ b));
	return 64 + __clz(i ^ j);
}

// Karras 2012, section 4: internal node i of the binary radix tree over `total` sorted keys
__global__ void radix_tree_kernel(const unsigned long long* __restrict__ keys, int total, uint32_t* __restrict__ left, uint32_t* __restrict__ right,
                                  uint32_t* __restrict__ parentOfInternal, uint32_t* __restrict__ parentOfLeaf)
{
	int i = blockIdx.x * kBuildBlock + threadIdx.x;
	if (i >= total - 1) return;

	int direction = common_prefix(keys, total, i, i + 1) - common_prefix(keys, total, i, i - 1) >= 0 ? 1 : -1;
	int minimum = common_prefix(keys, total, i, i - direction);

	int limit = 2;
	while (common_prefix(keys, total, i, i + limit * direction) > minimum) limit *= 2;

	int length = 0;
	for (int step = limit / 2; step >= 1; step /= 2)
		if (common_prefix(keys, total, i, i + (length + step) * direction) > minimum) length += step;

	int last = i + length * direction;
	int node = common_prefix(keys, total, i, last);

	int split = 0;
	for (int divisor = 2, step = (length + 1) / 2;; divisor *= 2, step = (length + divisor - 1) / divisor)
	{
		if (common_prefix(keys, total, i, i + (split + step) * direction) > node) split += step;
		if (step <= 1) break;
	}

	int gamma = i + split * direction + min(direction, 0);
	int low = min(i, last), high = max(i, last);

	uint32_t leftChild = low == gamma ? ((uint32_t)gamma | kLeafFlag) : (uint32_t)gamma;
	uint32_t rightChild = high == gamma + 1 ? ((uint32_t)(gamma + 1) | kLeafFlag) : (uint32_t)(gamma + 1);
	left[i] = leftChild;
	right[i] = rightChild;

	if (leftChild & kLeafFlag) parentOfLeaf[gamma] = (uint32_t)i;
	else parentOfInternal[gamma] = (uint32_t)i;
	if (rightChild & kLeafFlag) parentOfLeaf[gamma + 1] = (uint32_t)i;
	else parentOfInternal[gamma + 1] = (uint32_t)i;
	if (i == 0) parentOfInternal[0] = 0xFFFFFFFFu;
}

// bottom-up boxes: the second thread to reach a node merges its children (Karras 2012, section 5)
__global__ void fit_kernel(const BuildBox* __restrict__ boxes, const uint32_t* __restrict__ order, int total, const uint32_t* __restrict__ left, const uint32_t* __restrict__ right,
                           const uint32_t* __restrict__ parentOfInternal, const uint32_t* __restrict__ parentOfLeaf, BuildBox* __restrict__ nodeBoxes, uint32_t* __restrict__ visits)
{
	int i = blockIdx.x * kBuildBlock + threadIdx.x;
	if (i >= total) return;

	uint32_t node = parentOfLeaf[i];

	while (node != 0xFFFFFFFFu)
	{
		if (atomicAdd(visits + node, 1u) == 0u) return; // the sibling subtree is not finished yet
		__threadfence();

		uint32_t a = left[node], b = right[node];
		BuildBox boxA = (a & kLeafFlag) ? boxes[order[a & ~kLeafFlag]] : nodeBoxes[a];
		BuildBox boxB = (b & kLeafFlag) ? boxes[order[b & ~kLeafFlag]] : nodeBoxes[b];
		nodeBoxes[node] = { fminf(boxA.minX, boxB.minX), fminf(boxA.minY, boxB.minY), fminf(boxA.minZ, boxB.minZ),
		                    fmaxf(boxA.maxX, boxB.maxX), fmaxf(boxA.maxY, boxB.maxY), fmaxf(boxA.maxZ, boxB.maxZ) };
		__threadfence();
		node = parentOfInternal[node];
	}
}

// binary depth of every internal node; nodes at even depth become quad nodes (QuadBoundingVolumeHierarchy.cs:363-404)
__global__ void depth_kernel(const uint32_t* __restrict__ parentOfInternal, int internalCount, uint32_t* __restrict__ isQuad)
{
	int i = blockIdx.x * kBuildBlock + threadIdx.x;
	if (i >= internalCount) return;

	uint32_t depth = 0u;
	for (uint32_t node = parentOfInternal[i]; node != 0xFFFFFFFFu; node = parentOfInternal[node]) ++depth;
	isQuad[i] = (depth & 1u) == 0u ? 1u : 0u;
}

// ---- PLOC ----
// A/B on the C2 geometry (r2i): radius 4 / 8 / 16 / 32 / 64 -> 8.01 / 8.13 / 7.71 / 7.75 / 7.84 node visits per query, 4562 / 4574 / 4670 / 4665 / 4657 Mrays/s
constexpr int kPlocRadius = 16; // neighbours examined on each side by default (ECHO_B200_BUILD_PLOC_RADIUS / set_option("BUILD_PLOC_RADIUS"))

std::atomic<int>& ploc_radius()
{
	static std::atomic<int> value{ [] { const char* text = std::getenv("ECHO_B200_BUILD_PLOC_RADIUS"); return text ? std::atoi(text) : kPlocRadius; }() };
	return value;
}

__device__ __forceinline__ float union_half_area(const BuildBox& a, const BuildBox& b)
{
	float dx = fmaxf(a.maxX, b.maxX) - fminf(a.minX, b.minX), dy = fmaxf(a.maxY, b.maxY) - fminf(a.minY, b.minY), dz = fmaxf(a.maxZ, b.maxZ) - fminf(a.minZ, b.minZ);
	return dx * dy + dy * dz + dz * dx;
}

__global__ void ploc_init_kernel(const BuildBox* __restrict__ boxes, const uint32_t* __restrict__ order, int total, uint32_t* __restrict__ clusterRef, BuildBox* __restrict__ clusterBox)
{
	int i = blockIdx.x * kBuildBlock + threadIdx.x;
	if (i >= total) return;
	clusterRef[i] = (uint32_t)i | kLeafFlag;
	clusterBox[i] = boxes[order[i]];
}

// the neighbour within the window whose union with cluster i has the smallest surface area (ties: the lower position)
__global__ void ploc_nearest_kernel(const BuildBox* __restrict__ clusterBox, int count, int radius, uint32_t* __restrict__ nearest)
{
	int i = blockIdx.x * kBuildBlock + threadIdx.x;
	if (i >= count) return;

	BuildBox box = clusterBox[i];
	float best = __int_as_float(0x7F800000);
	int bestIndex = i == 0 ? 1 : i - 1;
	int first = max(i - radius, 0), last = min(i + radius, count - 1);

	for (int j = first; j <= last; j++)
	{
		if (j == i) continue;
		float area = union_half_area(box, clusterBox[j]);
		if (area < best) { best = area; bestIndex = j; }
	}

	nearest[i] = (uint32_t)bestIndex;
}

// mutual nearest neighbours merge into a new internal node (the lower position keeps the merged cluster, the higher one is dropped).
// Node ids are handed out downwards from total - 2, so the last merge — the root — is node 0, where the collapse expects it.
__global__ void ploc_merge_kernel(uint32_t* __restrict__ clusterRef, BuildBox* __restrict__ clusterBox, const uint32_t* __restrict__ nearest, int count, int* __restrict__ nextNode,
                                  uint32_t* __restrict__ left, uint32_t* __restrict__ right, uint32_t* __restrict__ parentOfInternal, uint32_t* __restrict__ parentOfLeaf,
                                  BuildBox* __restrict__ nodeBoxes, uint32_t* __restrict__ keep)
{
	int i = blockIdx.x * kBuildBlock + threadIdx.x;
	if (i >= count) return;

	int j = (int)nearest[i];
	bool mutual = (int)nearest[j] == i;

	if (!mutual) { keep[i] = 1u; return; }
	if (i > j) { keep[i] = 0u; return; }

	uint32_t a = clusterRef[i], b = clusterRef[j];
	BuildBox boxA = clusterBox[i], boxB = clusterBox[j];
	BuildBox merged = { fminf(boxA.minX, boxB.minX), fminf(boxA.minY, boxB.minY), fminf(boxA.minZ, boxB.minZ),
	                    fmaxf(boxA.maxX, boxB.maxX), fmaxf(boxA.maxY, boxB.maxY), fmaxf(boxA.maxZ, boxB.maxZ) };

	uint32_t node = (uint32_t)(atomicSub(nextNode, 1) - 1);
	left[node] = a;
	right[node] = b;
	nodeBoxes[node] = merged;
	if (a & kLeafFlag) parentOfLeaf[a & ~kLeafFlag] = node; else parentOfInternal[a] = node;
	if (b & kLeafFlag) parentOfLeaf[b & ~kLeafFlag] = node; else parentOfInternal[b] = node;

	clusterRef[i] = node; // only this thread touches clusters i and j in this pass
	clusterBox[i] = merged;
	keep[i] = 1u;
}

__global__ void ploc_compact_kernel(const uint32_t* __restrict__ clusterRef, const BuildBox* __restrict__ clusterBox, const uint32_t* __restrict__ keep, const uint32_t* __restrict__ position,
                                    int count, uint32_t* __restrict__ outRef, BuildBox* __restrict__ outBox, int* __restrict__ outCount)
{
	int i = blockIdx.x * kBuildBlock + threadIdx.x;
	if (i >= count) return;

	if (keep[i])
	{
		outRef[position[i]] = clusterRef[i];
		outBox[position[i]] = clusterBox[i];
	}

	if (i == count - 1) *outCount = (int)(position[i] + keep[i]);
}

struct ChildRef
{
	uint32_t reference; // kLeafFlag | sorted position, or internal node index; 0xFFFFFFFF = none
};

__device__ __forceinline__ BuildBox reference_box(uint32_t reference, const BuildBox* boxes, const uint32_t* order, const BuildBox* nodeBoxes)
{
	return (reference & kLeafFlag) ? boxes[order[reference & ~kLeafFlag]] : nodeBoxes[reference];
}

// GetChildrenSorted (:551-563): the split axis (here: the axis along which the two children's centres are furthest apart)
// and the two children ordered by their lower bound on it
__device__ int sorted_children(uint32_t node, const uint32_t* left, const uint32_t* right, const BuildBox* boxes, const uint32_t* order, const BuildBox* nodeBoxes,
                               uint32_t& child0, uint32_t& child1)
{
	child0 = left[node];
	child1 = right[node];
	BuildBox a = reference_box(child0, boxes, order, nodeBoxes), b = reference_box(child1, boxes, order, nodeBoxes);

	float dx = fabsf((a.minX + a.maxX) - (b.minX + b.maxX)), dy = fabsf((a.minY + a.maxY) - (b.minY + b.maxY)), dz = fabsf((a.minZ + a.maxZ) - (b.minZ + b.maxZ));
	int axis = dx >= dy ? (dx >= dz ? 0 : 2) : (dy >= dz ? 1 : 2);
	float lowA = axis == 0 ? a.minX : (axis == 1 ? a.minY : a.minZ), lowB = axis == 0 ? b.minX : (axis == 1 ? b.minY : b.minZ);

	if (lowA > lowB)
	{
		uint32_t swap = child0;
		child0 = child1;
		child1 = swap;
	}

	return axis;
}

__global__ void emit_kernel(int internalCount, const uint32_t* __restrict__ isQuad, const uint32_t* __restrict__ quadIndex, const uint32_t* __restrict__ left,
                            const uint32_t* __restrict__ right, const BuildBox* __restrict__ boxes, const uint32_t* __restrict__ order, const uint32_t* __restrict__ tokens,
                            const BuildBox* __restrict__ nodeBoxes, EchoQbvhNode* __restrict__ out)
{
	int i = blockIdx.x * kBuildBlock + threadIdx.x;
	if (i >= internalCount || isQuad[i] == 0u) return;

	uint32_t child0, child1;
	int axisMajor = sorted_children((uint32_t)i, left, right, boxes, order, nodeBoxes, child0, child1);

	uint32_t slots[4];
	int axisMinor[2];
	const uint32_t children[2] = { child0, child1 };

	for (int k = 0; k < 2; k++) // AddChildren (:517-543): a leaf becomes [leaf, empty] with axis 3
	{
		if (children[k] & kLeafFlag)
		{
			slots[k * 2] = children[k];
			slots[k * 2 + 1] = 0xFFFFFFFFu;
			axisMinor[k] = 3;
		}
		else axisMinor[k] = sorted_children(children[k], left, right, boxes, order, nodeBoxes, slots[k * 2], slots[k * 2 + 1]);
	}

	EchoQbvhNode node;
	node.axisMajor = axisMajor;
	node.axisMinor0 = axisMinor[0];
	node.axisMinor1 = axisMinor[1];
	node.pad = 0u;

	const float infinity = __int_as_float(0x7F800000);

	for (int k = 0; k < 4; k++)
	{
		BuildBox box = { infinity, infinity, infinity, infinity, infinity, infinity }; // BoxBound.None, BoxBound.cs:94
		uint32_t token = ECHO_TOKEN_EMPTY;

		if (slots[k] != 0xFFFFFFFFu)
		{
			box = reference_box(slots[k], boxes, order, nodeBoxes);
			token = (slots[k] & kLeafFlag) ? tokens[order[slots[k] & ~kLeafFlag]] : ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_NODE, quadIndex[slots[k]]);
		}

		node.minX[k] = box.minX; node.minY[k] = box.minY; node.minZ[k] = box.minZ;
		node.maxX[k] = box.maxX; node.maxY[k] = box.maxY; node.maxZ[k] = box.maxZ;
		node.token4[k] = token;
	}

	out[quadIndex[i]] = node;
}

// 2 = the reference's SweepBuilder tree (sweep.cu, default), 1 = PLOC, 0 = LBVH; ECHO_B200_BUILD_ALGORITHM / echo_b200_debug_set_option("BUILD_ALGORITHM", ...)
std::atomic<int>& build_algorithm()
{
	static std::atomic<int> value{ [] { const char* text = std::getenv("ECHO_B200_BUILD_ALGORITHM"); return text ? std::atoi(text) : 2; }() };
	return value;
}

unsigned int build_blocks(uint64_t count) { return (unsigned int)((count + kBuildBlock - 1) / kBuildBlock); }

// one cudaMalloc for every build buffer (eighteen separate ones cost ~60 ms, far more than the build itself)
struct DeviceArena
{
	char* base = nullptr;
	size_t bytes = 0;
	std::vector<std::pair<void**, size_t>> slots;

	template<class T>
	void reserve(T*& pointer, uint64_t count)
	{
		slots.push_back({ (void**)&pointer, bytes });
		bytes += (sizeof(T) * (count ? count : 1) + 255) & ~size_t(255);
	}

	bool commit()
	{
		if (!check_cuda(cudaMalloc((void**)&base, bytes), "cudaMalloc(build)")) return false;
		for (auto& [pointer, offset] : slots) *pointer = base + offset;
		return true;
	}

	~DeviceArena() { cudaFree(base); }
};

} // namespace

bool set_build_option(const char* name, long long value)
{
	const std::string key = name ? name : "";
	if (key == "BUILD_ALGORITHM") build_algorithm() = (int)value;
	else if (key == "BUILD_PLOC_RADIUS") ploc_radius() = (int)value;
	else return false;
	return true;
}

bool get_build_option(const char* name, long long& value)
{
	const std::string key = name ? name : "";
	if (key == "BUILD_ALGORITHM") value = build_algorithm();
	else if (key == "BUILD_PLOC_RADIUS") value = ploc_radius();
	else return false;
	return true;
}

static bool build_qbvh_with(bool ploc, const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
                            const float* instanceBounds, uint32_t instanceCount, EchoQbvhNode* outNodes, uint32_t* outNodeCount, uint32_t* outMaxDepth, bool* stalled);

bool build_qbvh_device(const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
                       const float* instanceBounds, uint32_t instanceCount, EchoQbvhNode* outNodes, uint32_t* outNodeCount, uint32_t* outMaxDepth)
{
	const int algorithm = build_algorithm();

	if (algorithm >= 2)
	{
		// The reference's own tree. Its depth is unbounded for degenerate inputs (coincident primitives peel off one per level, in the
		// recursive original as well); then, or when the tree would not fit the deepest compiled traversal stack, the clustering takes over.
		bool gaveUp = false;
		if (!build_qbvh_sweep(triangles, triangleCount, spheres, sphereCount, instanceBounds, instanceCount, outNodes, outNodeCount, outMaxDepth, &gaveUp)) return false;
		if (!gaveUp && stack_class(*outMaxDepth) >= 0) return true;
	}

	const bool ploc = algorithm != 0;
	bool stalled = false;
	if (!build_qbvh_with(ploc, triangles, triangleCount, spheres, sphereCount, instanceBounds, instanceCount, outNodes, outNodeCount, outMaxDepth, &stalled)) return false;

	// Agglomeration has neither a depth bound nor a bound on its passes: thousands of coincident primitives merge one pair per pass
	// and chain. The Morton tree has both (63 key bits). Fall back to it when the clustering stalls or when the clustered tree would
	// not fit the deepest compiled traversal stack (192 entries = 63 quad levels).
	if (ploc && (stalled || stack_class(*outMaxDepth) < 0)) return build_qbvh_with(false, triangles, triangleCount, spheres, sphereCount, instanceBounds, instanceCount, outNodes, outNodeCount, outMaxDepth, &stalled);
	return true;
}

static bool build_qbvh_with(bool ploc, const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
                            const float* instanceBounds, uint32_t instanceCount, EchoQbvhNode* outNodes, uint32_t* outNodeCount, uint32_t* outMaxDepth, bool* stalled)
{
	*stalled = false;
	uint64_t total64 = (uint64_t)triangleCount + sphereCount + instanceCount;
	if (total64 < 2 || total64 >= (1ull << ECHO_TOKEN_INDEX_BITS)) { set_error("a tree needs 2..2^28-1 primitives"); return false; }
	int total = (int)total64, internal = total - 1;

	const bool profile = std::getenv("ECHO_B200_PROFILE") != nullptr;
	auto clock = [] { return std::chrono::steady_clock::now(); };
	auto since = [&](std::chrono::steady_clock::time_point from) { return std::chrono::duration<double, std::milli>(clock() - from).count(); };
	auto started = clock();

	DeviceArena arena;
	EchoTriangle* dTriangles;
	EchoSphere* dSpheres;
	float* dInstanceBounds;
	BuildBox *boxes, *nodeBoxes;
	uint32_t *tokens, *order, *orderSorted, *left, *right, *parentOfInternal, *parentOfLeaf, *visits, *isQuad, *quadIndex;
	unsigned long long *keys, *keysSorted;
	int* sceneBound;
	EchoQbvhNode* nodes;
	char* scratch;
	uint32_t *clusterRef[2], *nearest, *keep, *keepPosition;
	BuildBox* clusterBox[2];
	int* plocCounters; // [0] the next node id + 1, [1] clusters left

	size_t sortBytes = 0, scanBytes = 0;
	cub::DeviceRadixSort::SortPairs(nullptr, sortBytes, (unsigned long long*)nullptr, (unsigned long long*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, total, 0, 63);
	cub::DeviceScan::ExclusiveSum(nullptr, scanBytes, (uint32_t*)nullptr, (uint32_t*)nullptr, internal);

	arena.reserve(dTriangles, triangleCount); arena.reserve(dSpheres, sphereCount); arena.reserve(dInstanceBounds, (uint64_t)instanceCount * 6); arena.reserve(boxes, total); arena.reserve(nodeBoxes, internal);
	arena.reserve(tokens, total); arena.reserve(order, total); arena.reserve(orderSorted, total); arena.reserve(left, internal); arena.reserve(right, internal);
	arena.reserve(parentOfInternal, internal); arena.reserve(parentOfLeaf, total); arena.reserve(visits, internal); arena.reserve(isQuad, internal);
	arena.reserve(quadIndex, internal); arena.reserve(keys, total); arena.reserve(keysSorted, total); arena.reserve(sceneBound, 6); arena.reserve(nodes, internal);
	arena.reserve(scratch, std::max(sortBytes, scanBytes));
	if (ploc)
	{
		for (int side = 0; side < 2; side++) { arena.reserve(clusterRef[side], total); arena.reserve(clusterBox[side], total); }
		arena.reserve(nearest, total); arena.reserve(keep, total); arena.reserve(keepPosition, total); arena.reserve(plocCounters, 2);
	}
	if (!arena.commit()) return false;
	bool ok = true;

	double allocateMs = since(started);
	auto phase = clock();
	cudaStream_t stream = nullptr;
	ok = check_cuda(cudaMemcpyAsync(dTriangles, triangles, sizeof(EchoTriangle) * triangleCount, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(triangles)")
		&& check_cuda(cudaMemcpyAsync(dSpheres, spheres, sizeof(EchoSphere) * sphereCount, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(spheres)")
		&& (instanceCount == 0u || check_cuda(cudaMemcpyAsync(dInstanceBounds, instanceBounds, sizeof(float) * 6 * instanceCount, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(instance bounds)"));
	if (!ok) return false;

	const int initial[6] = { 0x7FFFFFFF, 0x7FFFFFFF, 0x7FFFFFFF, (int)0x80000000, (int)0x80000000, (int)0x80000000 };
	ok = check_cuda(cudaMemcpyAsync(sceneBound, initial, sizeof(initial), cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(bound)")
		&& check_cuda(cudaMemsetAsync(visits, 0, sizeof(uint32_t) * internal, stream), "cudaMemsetAsync(visits)");
	if (!ok) return false;

	if (profile) cudaStreamSynchronize(stream);
	double uploadMs = since(phase);
	phase = clock();

	primitive_bounds_kernel<<<build_blocks(total), kBuildBlock, 0, stream>>>(dTriangles, triangleCount, dSpheres, sphereCount, dInstanceBounds, instanceCount, boxes, tokens, sceneBound);
	morton_kernel<<<build_blocks(total), kBuildBlock, 0, stream>>>(boxes, (uint32_t)total, sceneBound, keys, order);

	cub::DeviceRadixSort::SortPairs(scratch, sortBytes, keys, keysSorted, order, orderSorted, total, 0, 63, stream);

	if (ploc)
	{
		ploc_init_kernel<<<build_blocks(total), kBuildBlock, 0, stream>>>(boxes, orderSorted, total, clusterRef[0], clusterBox[0]);
		const int firstCounters[2] = { internal, total };
		if (!check_cuda(cudaMemcpyAsync(plocCounters, firstCounters, sizeof(firstCounters), cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(ploc)")) return false;
		const uint32_t noParent = 0xFFFFFFFFu;
		if (!check_cuda(cudaMemcpyAsync(parentOfInternal, &noParent, sizeof(uint32_t), cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(root)")) return false; // node 0 is the root

		int count = total, side = 0;
		const int radius = std::min(std::max(ploc_radius().load(), 1), 256);

		for (int iteration = 0; count > 1; iteration++)
		{
			if (iteration >= 384) { *stalled = true; return true; } // ordinary inputs need 25-40 passes
			ploc_nearest_kernel<<<build_blocks(count), kBuildBlock, 0, stream>>>(clusterBox[side], count, radius, nearest);
			ploc_merge_kernel<<<build_blocks(count), kBuildBlock, 0, stream>>>(clusterRef[side], clusterBox[side], nearest, count, plocCounters, left, right, parentOfInternal, parentOfLeaf, nodeBoxes, keep);
			cub::DeviceScan::ExclusiveSum(scratch, scanBytes, keep, keepPosition, count, stream);
			ploc_compact_kernel<<<build_blocks(count), kBuildBlock, 0, stream>>>(clusterRef[side], clusterBox[side], keep, keepPosition, count, clusterRef[side ^ 1], clusterBox[side ^ 1], plocCounters + 1);
			if (!check_cuda(cudaMemcpyAsync(&count, plocCounters + 1, sizeof(int), cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(ploc count)")
				|| !check_cuda(cudaStreamSynchronize(stream), "ploc iteration")) return false;
			side ^= 1;
		}
	}
	else
	{
		radix_tree_kernel<<<build_blocks(internal), kBuildBlock, 0, stream>>>(keysSorted, total, left, right, parentOfInternal, parentOfLeaf);
		fit_kernel<<<build_blocks(total), kBuildBlock, 0, stream>>>(boxes, orderSorted, total, left, right, parentOfInternal, parentOfLeaf, nodeBoxes, visits);
	}

	depth_kernel<<<build_blocks(internal), kBuildBlock, 0, stream>>>(parentOfInternal, internal, isQuad);
	cub::DeviceScan::ExclusiveSum(scratch, scanBytes, isQuad, quadIndex, internal, stream);
	emit_kernel<<<build_blocks(internal), kBuildBlock, 0, stream>>>(internal, isQuad, quadIndex, left, right, boxes, orderSorted, tokens, nodeBoxes, nodes);
	if (!check_cuda(cudaGetLastError(), "tree build launch")) return false;

	uint32_t lastFlag = 0, lastIndex = 0;
	ok = check_cuda(cudaMemcpyAsync(&lastFlag, isQuad + internal - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(count)")
		&& check_cuda(cudaMemcpyAsync(&lastIndex, quadIndex + internal - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(count)")
		&& check_cuda(cudaStreamSynchronize(stream), "tree build");
	if (!ok) return false;

	double kernelsMs = since(phase);
	phase = clock();
	uint32_t nodeCount = lastIndex + lastFlag;
	if (!check_cuda(cudaMemcpy(outNodes, nodes, sizeof(EchoQbvhNode) * nodeCount, cudaMemcpyDeviceToHost), "cudaMemcpy(nodes)")) return false;

	double downloadMs = since(phase);
	phase = clock();

	// depth as CreateNode counts it (:375-414): an empty slot 0, a leaf 1, a node 1 + the deepest of its slots
	std::vector<uint32_t> depth(nodeCount, 0u);
	std::vector<std::pair<uint32_t, int>> stack = { { 0u, 0 } };

	while (!stack.empty())
	{
		auto& [index, slot] = stack.back();

		if (slot == 4)
		{
			uint32_t deepest = 0u;
			for (uint32_t token : outNodes[index].token4)
			{
				if (token == ECHO_TOKEN_EMPTY) continue;
				bool isNode = (token >> ECHO_TOKEN_INDEX_BITS) == ECHO_TOKEN_TYPE_NODE;
				deepest = std::max(deepest, isNode ? depth[token & ((1u << ECHO_TOKEN_INDEX_BITS) - 1u)] : 1u);
			}
			depth[index] = deepest + 1u;
			stack.pop_back();
			continue;
		}

		uint32_t token = outNodes[index].token4[slot++];
		if (token != ECHO_TOKEN_EMPTY && (token >> ECHO_TOKEN_INDEX_BITS) == ECHO_TOKEN_TYPE_NODE) stack.push_back({ token & ((1u << ECHO_TOKEN_INDEX_BITS) - 1u), 0 });
	}

	if (profile)
		std::fprintf(stderr, "[echo_b200 build] %d primitives -> %u nodes: allocate %.2f ms, upload %.2f ms, kernels + sort %.2f ms, download %.2f ms, depth pass %.2f ms\n",
		             total, nodeCount, allocateMs, uploadMs, kernelsMs, downloadMs, since(phase));

	*outNodeCount = nodeCount;
	*outMaxDepth = depth[0];
	return true;
}

} // namespace echo
