// echo_sweep.h — the reference's SweepBuilder (Aggregation/Acceleration/SweepBuilder.cs) and the binary -> quad collapse of
// QuadBoundingVolumeHierarchy (QuadBoundingVolumeHierarchy.cs:363-565) restated as a LEVEL-SYNCHRONOUS data-parallel build that
// produces the reference's tree itself — the same nodes, in the same order, byte for byte — instead of some other valid tree.
//
// The reference recurses: a node sorts its primitives (stably) by `min[axis] + max[axis]` when the major axis of its volume
// differs from its parent's, sweeps ONE axis for the cut with the lowest `area(head) * i + area(tail) * (n - i)` (first minimum),
// and recurses into both halves. Nothing in that couples two nodes of the same depth, so here all nodes ("segments") of one
// binary depth are processed together, over one array of primitive positions in which every segment is a contiguous range:
//   keys      per position: (segment << 32) | Sorter.Transform(min[axis] + max[axis]), or (segment << 32) for segments that keep
//             their order — one stable radix sort of the whole level re-sorts exactly the segments the reference re-sorts
//   gather    the boxes in position order as order-preserving integer images, once forwards and once backwards
//   scans     two segmented inclusive scans (box union): head volumes (PrepareCutTailVolumes, :115-127, runs the other way round,
//             but min / max are exact and associative, so the order of the unions cannot change a bit) and tail volumes
//   cost      per cut position the reference's float expression (:148), reduced per segment by a 64-bit atomic min over
//             (monotone image of the cost, cut index): the lowest cost, the FIRST cut among equals — `cost < minCost`, :150
//   split     per segment: volumes of the two halves, the node (bound, axis = MajorAxis, larger-area child first, :38-88), the two child
//             ranges; a range of one primitive becomes a leaf node and drops out, the others are the next level's segments
//   compact   positions and segments that live on move to the front (two exclusive prefix sums)
// followed by the collapse: quad nodes are the internal binary nodes at even depth; the reference emits them in pre-order
// (CreateNode claims a child's index before it descends), so subtree sizes are summed bottom-up level by level and the indices
// handed out top-down — then the emitted array equals the host mirror's (libecho_host.so, echo_host_build_qbvh) byte for byte.
//
// Every pass is a functor over an index; a Backend supplies `for_each`, the stable pair sort, the scans and memory. The CUDA backend
// (sweep.cu: one generic kernel, CUB for sort and scans) and a sequential CPU backend (tests/c_client/sweep_emulation.cpp: the -m "not gpu"
// suite runs the very same passes and driver against the host mirror) share everything in this file.
#pragma once
#include <stdint.h>
#include <string.h>

#include <utility>
#include <vector>

#include "../../include/echo_b200.h"

#if defined(__CUDACC__)
#define SWEEP_HD __host__ __device__ __forceinline__
#else
#define SWEEP_HD inline
#endif

namespace echo
{
namespace sweep
{

constexpr uint32_t kNeedSort = 4u;           // Segment.flags: bits 0-1 = the axis the segment is (to be) sorted by, bit 2 = sort it at this level
constexpr uint32_t kNone = 0xFFFFFFFFu;
constexpr unsigned long long kNoCut = ~0ull;
constexpr int kMaxLevels = 3072;             // binary depth beyond which the build gives up (degenerate inputs chain; the caller falls back)

struct Box
{
	float lo[3], hi[3];
};

struct ScanItem // a box as order-preserving integers (int order == float order, -0 < +0) + the segmented-scan head flag
{
	int32_t lo[3], hi[3];
	uint32_t flag;
};

struct Segment // a node under construction: positions [begin, begin + length) of the level's position array
{
	uint32_t begin, length, node, flags;
};

struct BinNode // HierarchyBuilder.Node (HierarchyBuilder.cs:17-94)
{
	Box box;
	uint32_t child0, child1; // kNone: leaf
	uint32_t axis, token;
};

// ---- scalar helpers (the float expressions are the reference's, evaluated without contraction on both backends) ----

SWEEP_HD uint32_t float_bits(float value)
{
#if defined(__CUDA_ARCH__)
	return __float_as_uint(value);
#else
	uint32_t bits;
	memcpy(&bits, &value, 4);
	return bits;
#endif
}

SWEEP_HD float bits_float(uint32_t bits)
{
#if defined(__CUDA_ARCH__)
	return __uint_as_float(bits);
#else
	float value;
	memcpy(&value, &bits, 4);
	return value;
#endif
}

SWEEP_HD float f_add(float a, float b)
{
#if defined(__CUDA_ARCH__)
	return __fadd_rn(a, b);
#else
	return a + b;
#endif
}

SWEEP_HD float f_sub(float a, float b)
{
#if defined(__CUDA_ARCH__)
	return __fsub_rn(a, b);
#else
	return a - b;
#endif
}

SWEEP_HD float f_mul(float a, float b)
{
#if defined(__CUDA_ARCH__)
	return __fmul_rn(a, b);
#else
	return a * b;
#endif
}

SWEEP_HD int32_t to_ordered(float value)
{
	int32_t bits = (int32_t)float_bits(value);
	return bits >= 0 ? bits : bits ^ 0x7FFFFFFF;
}

SWEEP_HD float from_ordered(int32_t value) { return bits_float((uint32_t)(value >= 0 ? value : value ^ 0x7FFFFFFF)); }

SWEEP_HD uint32_t sort_key(float value) // Sorter.Transform, SweepBuilder.cs:241-251
{
	uint32_t converted = float_bits(value);
	uint32_t flip = (converted >> 31) * (0xFFFFFFFFu - 0x80000000u);
	return converted ^ (flip + 0x80000000u);
}

SWEEP_HD float select_min(float a, float b) { return a < b ? a : b; } // Sse.Min: the second operand unless a < b
SWEEP_HD float select_max(float a, float b) { return a > b ? a : b; }

SWEEP_HD float half_area(const Box& box) // BoxBound.HalfArea, BoxBound.cs:80-87
{
	float x = f_sub(box.hi[0], box.lo[0]), y = f_sub(box.hi[1], box.lo[1]), z = f_sub(box.hi[2], box.lo[2]);
	return f_add(f_mul(x, f_add(y, z)), f_mul(y, z));
}

SWEEP_HD uint32_t major_axis(const Box& box) // BoxBound.MajorAxis (:92) + Float3.MaxIndex (Float3.cs:130-138)
{
	float x = f_sub(box.hi[0], box.lo[0]), y = f_sub(box.hi[1], box.lo[1]), z = f_sub(box.hi[2], box.lo[2]);
	if (x > y) return x > z ? 0u : 2u;
	return y > z ? 1u : 2u;
}

SWEEP_HD ScanItem to_item(const Box& box, uint32_t flag)
{
	ScanItem item;
	for (int k = 0; k < 3; k++) { item.lo[k] = to_ordered(box.lo[k]); item.hi[k] = to_ordered(box.hi[k]); }
	item.flag = flag;
	return item;
}

SWEEP_HD Box to_box(const ScanItem& item)
{
	Box box;
	for (int k = 0; k < 3; k++) { box.lo[k] = from_ordered(item.lo[k]); box.hi[k] = from_ordered(item.hi[k]); }
	return box;
}

SWEEP_HD ScanItem unite(const ScanItem& a, const ScanItem& b) // BoxBound.Encapsulate (:128-132) on the integer images
{
	ScanItem r;
	for (int k = 0; k < 3; k++) { r.lo[k] = a.lo[k] < b.lo[k] ? a.lo[k] : b.lo[k]; r.hi[k] = a.hi[k] > b.hi[k] ? a.hi[k] : b.hi[k]; }
	r.flag = a.flag;
	return r;
}

struct ScanOp // segmented inclusive scan: an item that starts a segment forgets everything before it
{
	SWEEP_HD ScanItem operator()(const ScanItem& a, const ScanItem& b) const
	{
		if (b.flag) return b;
		return unite(a, b);
	}
};

SWEEP_HD void atomic_min_u64(unsigned long long* address, unsigned long long value)
{
#if defined(__CUDA_ARCH__)
	atomicMin(address, value);
#else
	if (value < *address) *address = value;
#endif
}

SWEEP_HD void atomic_or_u32(uint32_t* address, uint32_t value)
{
#if defined(__CUDA_ARCH__)
	atomicOr(address, value);
#else
	*address |= value;
#endif
}

// ---- passes ----

struct PackRange // one tree of a forest: the pack's primitives (offsets into the shared arrays) and its first position
{
	uint32_t triangleOffset, triangleCount, sphereOffset, sphereCount, instanceOffset, instanceCount;
	uint32_t begin; // positions [begin, begin + triangleCount + sphereCount + instanceCount) of the build
};

SWEEP_HD uint32_t range_size(const PackRange& pack) { return pack.triangleCount + pack.sphereCount + pack.instanceCount; }

SWEEP_HD uint32_t pack_of(const PackRange* packs, uint32_t packCount, uint32_t position) // the last pack that begins at or before `position`
{
	uint32_t low = 0u, high = packCount;
	while (high - low > 1u)
	{
		uint32_t middle = (low + high) / 2u;
		if (packs[middle].begin <= position) low = middle;
		else high = middle;
	}
	return low;
}

// GeometryCollection.CreateBounds (GeometryCollection.cs:52-81) of every pack: triangles, spheres, then instances, tokens relative to the
// pack's own arrays; position i starts as primitive i, in the segment of its pack (segment p = the root of pack p)
struct BoundsPass
{
	const PackRange* packs;
	uint32_t packCount;
	const EchoTriangle* triangles;
	const EchoSphere* spheres;
	const float* instanceBounds; // PreparedInstance.BoxBound of the placements: min xyz, max xyz
	Box* boxes;
	uint32_t* tokens;
	uint32_t* perm;
	uint32_t* segmentOf;

	SWEEP_HD void operator()(uint32_t i) const
	{
		uint32_t p = pack_of(packs, packCount, i);
		const PackRange pack = packs[p];
		uint32_t local = i - pack.begin;
		Box box;

		if (local < pack.triangleCount) // PreparedTriangle.BoxBound, TriangleEntity.cs:142 (Float4 min / max = Sse.Min / Max)
		{
			const EchoTriangle& t = triangles[pack.triangleOffset + local];
			for (int k = 0; k < 3; k++)
			{
				float v0 = t.vertex0[k], v1 = f_add(v0, t.edge1[k]), v2 = f_add(v0, t.edge2[k]);
				box.lo[k] = select_min(select_min(v0, v1), v2);
				box.hi[k] = select_max(select_max(v0, v1), v2);
			}
			tokens[i] = ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_TRIANGLE, local);
		}
		else if (local >= pack.triangleCount + pack.sphereCount)
		{
			uint32_t instance = local - pack.triangleCount - pack.sphereCount;
			const float* bound = instanceBounds + (size_t)(pack.instanceOffset + instance) * 6;
			for (int k = 0; k < 3; k++) { box.lo[k] = bound[k]; box.hi[k] = bound[3 + k]; }
			tokens[i] = ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_INSTANCE, instance);
		}
		else // PreparedSphere.BoxBound, SphereEntity.cs:66
		{
			const EchoSphere& s = spheres[pack.sphereOffset + local - pack.triangleCount];
			for (int k = 0; k < 3; k++) { box.lo[k] = f_sub(s.position[k], s.radius); box.hi[k] = f_add(s.position[k], s.radius); }
			tokens[i] = ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_SPHERE, local - pack.triangleCount);
		}

		boxes[i] = box;
		perm[i] = i;
		segmentOf[i] = p;
	}
};

struct RootPass // Build, SweepBuilder.cs:24-36, once per pack: the root segment over the pack's positions (binary node p) ...
{
	const PackRange* packs;
	Segment* segments;

	SWEEP_HD void operator()(uint32_t p) const { segments[p] = { packs[p].begin, range_size(packs[p]), p, 0u }; }
};

struct RootAxisPass // ... sorted by the major axis of the bound of everything in the pack: the segmented scan at the segment's end
{
	const ScanItem* heads;
	Segment* segments;
	unsigned long long* best;

	SWEEP_HD void operator()(uint32_t p) const
	{
		Segment segment = segments[p];
		segments[p].flags = major_axis(to_box(heads[segment.begin + segment.length - 1u])) | kNeedSort;
		best[p] = kNoCut;
	}
};

struct KeyPass
{
	const uint32_t* perm;
	const uint32_t* segmentOf;
	const Segment* segments;
	const Box* boxes;
	unsigned long long* keys;

	SWEEP_HD void operator()(uint32_t p) const
	{
		uint32_t index = segmentOf[p];
		uint32_t flags = segments[index].flags;
		uint32_t low = 0u;

		if (flags & kNeedSort) // Sorter.Sort, SweepBuilder.cs:199-212
		{
			const Box& box = boxes[perm[p]];
			uint32_t axis = flags & 3u;
			low = sort_key(f_add(box.lo[axis], box.hi[axis]));
		}

		keys[p] = (unsigned long long)index << 32 | low;
	}
};

struct GatherPass // forwards[p] and backwards[count - 1 - p]: the box at position p, flagged where its segment starts / ends
{
	uint32_t count;
	const uint32_t* perm;
	const uint32_t* segmentOf;
	const Segment* segments;
	const Box* boxes;
	ScanItem* forwards;
	ScanItem* backwards;

	SWEEP_HD void operator()(uint32_t p) const
	{
		Segment segment = segments[segmentOf[p]];
		const Box& box = boxes[perm[p]];
		forwards[p] = to_item(box, p == segment.begin ? 1u : 0u);
		backwards[count - 1u - p] = to_item(box, p == segment.begin + segment.length - 1u ? 1u : 0u);
	}
};

struct CostPass // SearchSurfaceAreaHeuristics, SweepBuilder.cs:132-160
{
	uint32_t count;
	const uint32_t* segmentOf;
	const Segment* segments;
	const ScanItem* heads; // inclusive forward scan
	const ScanItem* tails; // inclusive backward scan, reversed positions
	unsigned long long* best;

	SWEEP_HD void operator()(uint32_t p) const
	{
#if defined(__CUDA_ARCH__)
		const unsigned int active = __activemask(); // the lanes that run this pass (all 32 but in the last warp), taken before anything diverges
#endif
		uint32_t index = segmentOf[p];
		Segment segment = segments[index];
		uint32_t i = p - segment.begin;
		unsigned long long candidate = kNoCut;

		if (i != 0u)
		{
			float headArea = half_area(to_box(heads[p - 1u])), tailArea = half_area(to_box(tails[count - 1u - p]));
			float cost = f_add(f_mul(headArea, (float)(int32_t)i), f_mul(tailArea, (float)(int32_t)(segment.length - i)));
			if (cost == 0.0f) cost = 0.0f; // -0 and +0 are one cost
			if (cost < 3.402823466e+38f) candidate = (unsigned long long)sort_key(cost) << 32 | i;
		}

#if defined(__CUDA_ARCH__)
		// Consecutive lanes hold consecutive positions, so the lanes of one segment are a contiguous run of the warp: a segmented
		// shuffle reduction leaves the run's minimum in its first lane, and one atomic per (warp, segment) reaches memory. Per-lane
		// atomics serialise on the segment's word — a million of them on ONE address at the root: 41 % of the whole build (r2y).
		const unsigned int lane = threadIdx.x & 31u;

		for (unsigned int offset = 1u; offset < 32u; offset <<= 1)
		{
			unsigned long long other = __shfl_down_sync(active, candidate, offset);
			uint32_t otherIndex = __shfl_down_sync(active, index, offset);
			bool valid = lane + offset < 32u && ((active >> (lane + offset)) & 1u) != 0u;
			if (valid && otherIndex == index && other < candidate) candidate = other;
		}

		uint32_t before = __shfl_up_sync(active, index, 1u);
		bool leader = lane == 0u || ((active >> (lane - 1u)) & 1u) == 0u || before != index;
		if (leader && candidate != kNoCut) atomicMin(best + index, candidate);
#else
		if (candidate != kNoCut) atomic_min_u64(best + index, candidate);
#endif
	}
};

struct SplitPass // BuildLayer, SweepBuilder.cs:38-88 (+ BuildChild, :90-97, for the two halves)
{
	uint32_t count, nodeBase;
	const Segment* segments;
	const ScanItem* heads;
	const ScanItem* tails;
	const unsigned long long* best;
	const uint32_t* perm;
	const Box* boxes;
	const uint32_t* tokens;
	BinNode* nodes;
	Segment* slots;    // 2 per segment, in position order
	uint32_t* keep;    // slot lives on as a segment of the next level
	uint32_t* totals;  // [2]: some segment of the next level needs sorting

	SWEEP_HD void operator()(uint32_t s) const
	{
		Segment segment = segments[s];
		uint32_t begin = segment.begin, length = segment.length;

		unsigned long long found = best[s];
		uint32_t cut = found == kNoCut ? length / 2u : (uint32_t)(found & 0xFFFFFFFFull); // no finite cost at all: the host mirror's median split

		ScanItem firstItem = heads[begin + cut - 1u], secondItem = tails[count - 1u - (begin + cut)];
		Box bound = to_box(unite(firstItem, secondItem));
		uint32_t axis = major_axis(bound);

		Box volume[2] = { to_box(firstItem), to_box(secondItem) };
		uint32_t childNode[2] = { nodeBase + 2u * s, nodeBase + 2u * s + 1u };
		uint32_t head = cut > length / 2u ? 0u : 1u; // "headData is always larger than tailData"

		uint32_t child0 = childNode[head], child1 = childNode[head ^ 1u];
		if (half_area(volume[head]) < half_area(volume[head ^ 1u])) { uint32_t swap = child0; child0 = child1; child1 = swap; } // larger surface area first

		BinNode node;
		node.box = bound;
		node.child0 = child0;
		node.child1 = child1;
		node.axis = axis;
		node.token = ECHO_TOKEN_EMPTY;
		nodes[segment.node] = node;

		uint32_t childBegin[2] = { begin, begin + cut }, childLength[2] = { cut, length - cut };

		for (uint32_t k = 0; k < 2u; k++)
		{
			Segment slot = { childBegin[k], childLength[k], childNode[k], 0u };

			if (childLength[k] == 1u)
			{
				uint32_t primitive = perm[childBegin[k]];
				BinNode leaf;
				leaf.box = boxes[primitive];
				leaf.child0 = leaf.child1 = kNone;
				leaf.axis = 0u;
				leaf.token = tokens[primitive];
				nodes[childNode[k]] = leaf;
				keep[2u * s + k] = 0u;
			}
			else
			{
				uint32_t childAxis = major_axis(volume[k]);
				slot.flags = childAxis | (childAxis != axis ? kNeedSort : 0u);
				keep[2u * s + k] = 1u;
				if (childAxis != axis) atomic_or_u32(totals + 2, 1u);
			}

			slots[2u * s + k] = slot;
		}
	}
};

struct MarkPass
{
	const uint32_t* segmentOf;
	const Segment* slots;
	uint32_t* stay;

	SWEEP_HD void operator()(uint32_t p) const
	{
		uint32_t slot = 2u * segmentOf[p];
		if (p >= slots[slot + 1u].begin) ++slot;
		stay[p] = slots[slot].length > 1u ? 1u : 0u;
	}
};

struct MovePositionsPass
{
	uint32_t count;
	const uint32_t* segmentOf;
	const Segment* slots;
	const uint32_t* stay;
	const uint32_t* newPosition;
	const uint32_t* newSegment;
	const uint32_t* perm;
	uint32_t* nextPerm;
	uint32_t* nextSegmentOf;
	uint32_t* totals; // [0]: positions of the next level

	SWEEP_HD void operator()(uint32_t p) const
	{
		if (stay[p])
		{
			uint32_t slot = 2u * segmentOf[p];
			if (p >= slots[slot + 1u].begin) ++slot;
			uint32_t q = newPosition[p];
			nextPerm[q] = perm[p];
			nextSegmentOf[q] = newSegment[slot];
		}

		if (p == count - 1u) totals[0] = newPosition[p] + stay[p];
	}
};

struct MoveSegmentsPass
{
	uint32_t slotCount;
	const Segment* slots;
	const uint32_t* keep;
	const uint32_t* newPosition;
	const uint32_t* newSegment;
	Segment* nextSegments;
	unsigned long long* nextBest;
	uint32_t* totals; // [1]: segments of the next level

	SWEEP_HD void operator()(uint32_t c) const
	{
		if (keep[c])
		{
			Segment segment = slots[c];
			segment.begin = newPosition[segment.begin];
			uint32_t t = newSegment[c];
			nextSegments[t] = segment;
			nextBest[t] = kNoCut;
		}

		if (c == slotCount - 1u) totals[1] = newSegment[c] + keep[c];
	}
};

// ---- the collapse, QuadBoundingVolumeHierarchy.cs:363-565 ----

SWEEP_HD uint32_t children_sorted(const BinNode* nodes, uint32_t node, uint32_t& child0, uint32_t& child1) // GetChildrenSorted, :551-563
{
	uint32_t axis = nodes[node].axis;
	child0 = nodes[node].child0;
	child1 = nodes[node].child1;
	if (nodes[child0].box.lo[axis] > nodes[child1].box.lo[axis]) { uint32_t swap = child0; child0 = child1; child1 = swap; }
	return axis;
}

SWEEP_HD uint32_t add_children(const BinNode* nodes, uint32_t node, uint32_t* out) // AddChildren, :517-543: a leaf becomes [leaf, empty], axis 3
{
	if (nodes[node].child0 == kNone)
	{
		out[0] = node;
		out[1] = kNone;
		return 3u;
	}

	return children_sorted(nodes, node, out[0], out[1]);
}

struct QuadCountPass // quad nodes in the subtree of every internal binary node of one even level (the levels below are done), and the
{                     // subtree's depth as CreateNode counts it (:375-414): an empty slot 0, a leaf 1, a node 1 + the deepest of its slots
	uint32_t first;
	const BinNode* nodes;
	uint32_t* quadCount;
	uint32_t* quadDepth;

	SWEEP_HD void operator()(uint32_t i) const
	{
		uint32_t node = first + i;
		if (nodes[node].child0 == kNone) return;

		uint32_t child0, child1, slots[4];
		children_sorted(nodes, node, child0, child1);
		add_children(nodes, child0, slots);
		add_children(nodes, child1, slots + 2);

		uint32_t total = 1u, deepest = 0u;

		for (int k = 0; k < 4; k++)
		{
			if (slots[k] == kNone) continue;
			bool internal = nodes[slots[k]].child0 != kNone;
			if (internal) total += quadCount[slots[k]];
			uint32_t below = internal ? quadDepth[slots[k]] : 1u;
			if (below > deepest) deepest = below;
		}

		quadCount[node] = total;
		quadDepth[node] = deepest + 1u;
	}
};

struct QuadRootPass // the root of pack p is its quad node 0; the packs' nodes follow each other in pack order
{
	const uint32_t* rootBase; // exclusive sum of the roots' quad counts
	uint32_t* quadIndex;
	uint32_t* quadBase;

	SWEEP_HD void operator()(uint32_t p) const
	{
		quadIndex[p] = 0u;
		quadBase[p] = rootBase[p];
	}
};

struct QuadEmitPass // CreateNode, :363-404: pre-order indices (relative to the pack's root) for the internal slots, then the node itself
{
	uint32_t first;
	const BinNode* nodes;
	const uint32_t* quadCount;
	uint32_t* quadIndex;
	uint32_t* quadBase; // where the node's pack starts in `out`
	EchoQbvhNode* out;

	SWEEP_HD void operator()(uint32_t i) const
	{
		uint32_t node = first + i;
		if (nodes[node].child0 == kNone) return;

		uint32_t child0, child1, slots[4];
		uint32_t axisMajor = children_sorted(nodes, node, child0, child1);
		uint32_t axisMinor0 = add_children(nodes, child0, slots);
		uint32_t axisMinor1 = add_children(nodes, child1, slots + 2);

		uint32_t index = quadIndex[node], base = quadBase[node];
		uint32_t running = index + 1u;

		EchoQbvhNode quad;
		quad.axisMajor = (int32_t)axisMajor;
		quad.axisMinor0 = (int32_t)axisMinor0;
		quad.axisMinor1 = (int32_t)axisMinor1;
		quad.pad = 0u;

		const float infinity = bits_float(0x7F800000u);

		for (int k = 0; k < 4; k++)
		{
			Box box = { { infinity, infinity, infinity }, { infinity, infinity, infinity } }; // BoxBound.None, BoxBound.cs:94
			uint32_t token = ECHO_TOKEN_EMPTY;

			if (slots[k] != kNone)
			{
				const BinNode& source = nodes[slots[k]];
				box = source.box;

				if (source.child0 == kNone) token = source.token;
				else
				{
					quadIndex[slots[k]] = running;
					quadBase[slots[k]] = base;
					token = ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_NODE, running);
					running += quadCount[slots[k]];
				}
			}

			quad.minX[k] = box.lo[0]; quad.minY[k] = box.lo[1]; quad.minZ[k] = box.lo[2];
			quad.maxX[k] = box.hi[0]; quad.maxY[k] = box.hi[1]; quad.maxZ[k] = box.hi[2];
			quad.token4[k] = token;
		}

		out[base + index] = quad;
	}
};

// the same depth by a host pass over an emitted array (what the clustered builds use; the emulation checks QuadCountPass against it)
inline uint32_t quad_depth(const EchoQbvhNode* nodes, uint32_t nodeCount)
{
	std::vector<uint32_t> depth(nodeCount, 0u);
	std::vector<std::pair<uint32_t, int>> stack = { { 0u, 0 } };
	const uint32_t indexMask = (1u << ECHO_TOKEN_INDEX_BITS) - 1u;

	while (!stack.empty())
	{
		uint32_t index = stack.back().first;
		int slot = stack.back().second;

		if (slot == 4)
		{
			uint32_t deepest = 0u;
			for (uint32_t token : nodes[index].token4)
			{
				if (token == ECHO_TOKEN_EMPTY) continue;
				bool isNode = (token >> ECHO_TOKEN_INDEX_BITS) == ECHO_TOKEN_TYPE_NODE;
				uint32_t below = isNode ? depth[token & indexMask] : 1u;
				if (below > deepest) deepest = below;
			}
			depth[index] = deepest + 1u;
			stack.pop_back();
			continue;
		}

		stack.back().second = slot + 1;
		uint32_t token = nodes[index].token4[slot];
		if (token != ECHO_TOKEN_EMPTY && (token >> ECHO_TOKEN_INDEX_BITS) == ECHO_TOKEN_TYPE_NODE) stack.push_back({ token & indexMask, 0 });
	}

	return depth[0];
}

// ---- memory: one arena carved twice (first with a null base to measure) ----

struct Arena
{
	char* base = nullptr;
	size_t used = 0;

	template<class T>
	T* take(uint64_t count)
	{
		size_t offset = used;
		used += (sizeof(T) * (count ? count : 1) + 255) & ~size_t(255);
		return base ? (T*)(base + offset) : nullptr;
	}
};

struct Buffers
{
	Box* boxes;
	uint32_t *tokens, *perm[2], *segmentOf[2], *stay, *newPosition, *keep, *newSegment, *totals, *quadCount, *quadDepth, *quadIndex, *quadBase, *rootBase;
	unsigned long long *keys[2], *best[2];
	ScanItem *forwards, *backwards, *heads, *tails;
	Segment *segments[2], *slots;
	BinNode* nodes;
	EchoQbvhNode* quads;

	PackRange* packs;

	void carve(Arena& arena, uint64_t total, uint32_t packCount)
	{
		packs = arena.take<PackRange>(packCount);
		rootBase = arena.take<uint32_t>(packCount);
		boxes = arena.take<Box>(total);
		tokens = arena.take<uint32_t>(total);
		for (int k = 0; k < 2; k++)
		{
			perm[k] = arena.take<uint32_t>(total);
			segmentOf[k] = arena.take<uint32_t>(total);
			keys[k] = arena.take<unsigned long long>(total);
			best[k] = arena.take<unsigned long long>(total / 2 + 1);
			segments[k] = arena.take<Segment>(total / 2 + 1);
		}
		stay = arena.take<uint32_t>(total);
		newPosition = arena.take<uint32_t>(total);
		keep = arena.take<uint32_t>(total + 2);
		newSegment = arena.take<uint32_t>(total + 2);
		totals = arena.take<uint32_t>(4);
		forwards = arena.take<ScanItem>(total);
		backwards = arena.take<ScanItem>(total);
		heads = arena.take<ScanItem>(total);
		tails = arena.take<ScanItem>(total);
		slots = arena.take<Segment>(total + 2);
		nodes = arena.take<BinNode>(2 * total);
		quadCount = arena.take<uint32_t>(2 * total);
		quadDepth = arena.take<uint32_t>(2 * total);
		quadIndex = arena.take<uint32_t>(2 * total);
		quadBase = arena.take<uint32_t>(2 * total);
		quads = arena.take<EchoQbvhNode>(total);
	}
};

struct Result
{
	bool ok = false;       // false: a backend call failed (its error is set) ...
	bool gaveUp = false;   // ... or some tree chains deeper than kMaxLevels
	uint32_t nodeCount = 0, maxDepth = 0, levels = 0; // nodeCount: all packs; maxDepth: pack 0's
	std::vector<uint32_t> packNodeCount, packMaxDepth, packNodeBase; // per pack: its quad nodes are quads[packNodeBase, + packNodeCount)
	const EchoQbvhNode* quads = nullptr; // backend memory
};

// Backend concept:
//   char* allocate(size_t bytes)                                   one block, released by the backend's owner
//   template<class F> bool for_each(uint32_t n, const F& f)        f(0) ... f(n - 1), any order, possibly concurrently
//   bool sort_pairs(const u64* keysIn, u64* keysOut, const u32* valuesIn, u32* valuesOut, uint32_t n, int endBit)   STABLE, by bits [0, endBit)
//   bool scan_items(const ScanItem* in, ScanItem* out, uint32_t n) inclusive, ScanOp
//   bool exclusive_sum(const uint32_t* in, uint32_t* out, uint32_t n)
//   template<class T> bool read(const T* source, T* destination, uint32_t n)    backend -> host, complete on return
//   template<class T> bool write(T* destination, const T* source, uint32_t n)   host -> backend
//   bool fill_zero(void* pointer, size_t bytes)
//
// A FOREST: the trees of `packCount` packs in one run. Nothing couples two segments of one level, so each pack is one more root
// segment; every level of the loop serves all packs at once, and the run reads back as many levels as its deepest tree has. `packs`
// (host memory) gives each pack's ranges of the shared arrays (backend memory) and its first position; the positions of the packs
// follow each other without gaps. Every tree is emitted as the single-pack build emits it — tokens and child indices relative to the
// pack — and the trees lie back to back in `quads`. A single pack is the forest of one tree.
template<class Backend>
Result build_forest(Backend& backend, const PackRange* packs, uint32_t packCount, const EchoTriangle* triangles, const EchoSphere* spheres, const float* instanceBounds)
{
	Result result;
	if (packCount == 0u) { result.ok = true; return result; }
	const uint32_t total = packs[packCount - 1u].begin + range_size(packs[packCount - 1u]);

	Buffers b;
	Arena measure;
	b.carve(measure, total, packCount);
	Arena arena;
	arena.base = backend.allocate(measure.used);
	if (!arena.base) return result;
	b.carve(arena, total, packCount);

	if (!backend.write(b.packs, packs, packCount)) return result;
	if (!backend.for_each(total, BoundsPass{ b.packs, packCount, triangles, spheres, instanceBounds, b.boxes, b.tokens, b.perm[0], b.segmentOf[0] })) return result;

	// Build, SweepBuilder.cs:24-36: each root is sorted by the major axis of the bound of everything in its pack
	if (!backend.for_each(packCount, RootPass{ b.packs, b.segments[0] })) return result;
	if (!backend.for_each(total, GatherPass{ total, b.perm[0], b.segmentOf[0], b.segments[0], b.boxes, b.forwards, b.backwards })) return result;
	if (!backend.scan_items(b.forwards, b.heads, total)) return result;
	if (!backend.for_each(packCount, RootAxisPass{ b.heads, b.segments[0], b.best[0] })) return result;

	std::vector<std::pair<uint32_t, uint32_t>> levels = { { 0u, packCount } }; // node id range {first, count} of every binary depth
	uint32_t count = total, segmentCount = packCount, nodeBase = packCount;
	bool anySort = true;
	int side = 0;                                     // which of the segmentOf / segments / best pairs holds the current level
	uint32_t *current = b.perm[0], *other = b.perm[1]; // position -> primitive of the current level, and the spare buffer

	while (segmentCount > 0u)
	{
		if ((int)levels.size() > kMaxLevels) { result.ok = true; result.gaveUp = true; return result; }

		const uint32_t* sorted = current;
		uint32_t* spare = other;

		if (anySort)
		{
			int segmentBits = 1;
			while ((1ull << segmentBits) < segmentCount) ++segmentBits;
			if (!backend.for_each(count, KeyPass{ current, b.segmentOf[side], b.segments[side], b.boxes, b.keys[0] })) return result;
			if (!backend.sort_pairs(b.keys[0], b.keys[1], current, other, count, 32 + segmentBits)) return result;
			sorted = other;
			spare = current;
		}

		uint32_t zeros[4] = { 0u, 0u, 0u, 0u };
		if (!backend.write(b.totals, zeros, 4)) return result;

		if (!backend.for_each(count, GatherPass{ count, sorted, b.segmentOf[side], b.segments[side], b.boxes, b.forwards, b.backwards })) return result;
		if (!backend.scan_items(b.forwards, b.heads, count) || !backend.scan_items(b.backwards, b.tails, count)) return result;
		if (!backend.for_each(count, CostPass{ count, b.segmentOf[side], b.segments[side], b.heads, b.tails, b.best[side] })) return result;
		if (!backend.for_each(segmentCount, SplitPass{ count, nodeBase, b.segments[side], b.heads, b.tails, b.best[side], sorted, b.boxes, b.tokens, b.nodes, b.slots, b.keep, b.totals })) return result;
		if (!backend.for_each(count, MarkPass{ b.segmentOf[side], b.slots, b.stay })) return result;
		if (!backend.exclusive_sum(b.stay, b.newPosition, count) || !backend.exclusive_sum(b.keep, b.newSegment, 2u * segmentCount)) return result;
		if (!backend.for_each(count, MovePositionsPass{ count, b.segmentOf[side], b.slots, b.stay, b.newPosition, b.newSegment, sorted, spare, b.segmentOf[side ^ 1], b.totals })) return result;
		if (!backend.for_each(2u * segmentCount, MoveSegmentsPass{ 2u * segmentCount, b.slots, b.keep, b.newPosition, b.newSegment, b.segments[side ^ 1], b.best[side ^ 1], b.totals })) return result;

		uint32_t totals[4];
		if (!backend.read(b.totals, totals, 4)) return result;

		levels.push_back({ nodeBase, 2u * segmentCount });
		nodeBase += 2u * segmentCount;

		if (spare == other) { other = current; current = spare; } // the survivors went to the spare buffer: it is the next level's order

		count = totals[0];
		segmentCount = totals[1];
		anySort = totals[2] != 0u;
		side ^= 1;
	}

	// collapse: sizes bottom-up over the even levels, then every root's place (the packs back to back), indices and nodes top-down
	int last = (int)levels.size() - 1;
	for (int level = last - (last & 1); level >= 0; level -= 2)
		if (!backend.for_each(levels[level].second, QuadCountPass{ levels[level].first, b.nodes, b.quadCount, b.quadDepth })) return result;

	result.packNodeCount.resize(packCount);
	result.packMaxDepth.resize(packCount);
	result.packNodeBase.resize(packCount);
	if (!backend.exclusive_sum(b.quadCount, b.rootBase, packCount)) return result; // the roots are binary nodes 0 .. packCount - 1
	if (!backend.read(b.quadCount, result.packNodeCount.data(), packCount) || !backend.read(b.quadDepth, result.packMaxDepth.data(), packCount)
		|| !backend.read(b.rootBase, result.packNodeBase.data(), packCount)) return result;
	if (!backend.for_each(packCount, QuadRootPass{ b.rootBase, b.quadIndex, b.quadBase })) return result;

	for (int level = 0; level <= last; level += 2)
		if (!backend.for_each(levels[level].second, QuadEmitPass{ levels[level].first, b.nodes, b.quadCount, b.quadIndex, b.quadBase, b.quads })) return result;

	result.ok = true;
	result.nodeCount = result.packNodeBase[packCount - 1u] + result.packNodeCount[packCount - 1u];
	result.maxDepth = result.packMaxDepth[0];
	result.levels = (uint32_t)levels.size();
	result.quads = b.quads;
	return result;
}

// one pack: the tree of GeometryCollection.CreateBounds' triangles, spheres and placements
template<class Backend>
Result build(Backend& backend, const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
             const float* instanceBounds, uint32_t instanceCount)
{
	const PackRange pack = { 0u, triangleCount, 0u, sphereCount, 0u, instanceCount, 0u };
	return build_forest(backend, &pack, 1u, triangles, spheres, instanceBounds);
}

} // namespace sweep
} // namespace echo
