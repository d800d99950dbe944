// render.cu — the wavefront path tracer behind echo_b200_render_tiles: one EvaluationOperation worth of tiles
// (Processes/Evaluation/EvaluationOperation.cs:83-148) evaluated by PathTracedEvaluator.Evaluate
// (Evaluation/Evaluators/PathTracedEvaluator.cs:43-207) re-organised as kernels over SoA path state:
//
//   raygen  ->  [ extend (QBVH closest hit, classifies the hit by material into per-class queues)
//                 shade<class> (emission + MIS bookkeeping, BSDF sample, light pick/sample, shadow-ray emit, RR)
//                 shadow (QBVH occlusion, adds the pending NEE contribution) ]*  ->  accumulate (Kahan-Welford per pixel)
//
// Every path keeps the reference's draw order of random numbers and its order of floating-point accumulation, so a
// sample's radiance is bit-identical to the oracle's. Queue management uses warp-aggregated atomics (ballot + popc).
#include <algorithm>
#include <atomic>
#include <string>
#include <cstring>
#include <thread>
#include <type_traits>
#include <sched.h>
#include <cstdio>
#include <cstdlib>

#include "echo_internal.h"
#include "echo_shading.cuh"
#include "echo_instanced.cuh"
#include "echo_traverse.cuh"

namespace echo
{

constexpr int kBlock = 128;

enum PathMode : uint32_t { MODE_FIRST = 0, MODE_NO_MIS = 1, MODE_MIS = 2 };
// material classes of the shading queues. CLASS_SMOOTH holds the dielectrics whose roughness makes them purely specular: their
// kernel carries no microfacet code and its lanes do not wait for the glossy lanes of a mixed queue (C3: the dielectric kernel ran
// at 14.6 active threads per warp with both kinds in one queue, ncu r1m)
enum ShadeClass : int { CLASS_MISS = 0, CLASS_DIFFUSE = 1, CLASS_DIELECTRIC = 2, CLASS_CONDUCTOR = 3, CLASS_TERMINAL = 4, CLASS_SMOOTH = 5, CLASS_COUNT = 6 };

// counter slots in RenderState::counters
// (the class counts are double-buffered by iteration parity: classify of iteration k + 1 fills one set while the other, consumed by
// the shading kernels of iteration k, waits to be cleared by the rotate kernel)
enum : int { COUNTER_NEXT = 0, COUNTER_SHADOW = 1, COUNTER_CLASS = 2, COUNTER_PIXELS = COUNTER_CLASS + 2 * CLASS_COUNT, COUNTER_TOTAL = COUNTER_PIXELS + 1 };
static_assert(COUNTER_TOTAL <= 32, "counters[32] is the saved active count");

struct PathBuffers
{
	// rays in flight, compacted: slot i of rayQueue[q] holds 32 bytes {origin.xyz, direction.x | direction.yz, limit, ignore}
	// (the EchoRay layout, so the persistent traversal core streams it exactly like a batch) and rayPath[q][i] its path id
	float4* rayQueue[2];
	uint32_t* rayPath[2];
	float4* hitQueue;     // per ray slot: token bits, distance, uv

	// per path id
	float4* energy;       // rgb, w = scatterPdf of the bounce that spawned the current ray (MIS)
	float4* result;       // rgb, w = bits: bounces done | mode << 16
	float4* oldPosition;  // MIS: GeometryPoint oldPoint
	float4* oldNormal;
	uint32_t* key;        // sample_key(seed, pixel, sample); stratified: stratified_series(seed, pixel, epoch)

	// shadow rays of the current bounce, compacted: {origin.xyz, direction.x | direction.yz, travel, ignore} + pending value
	float4* shadowQueue;
	float4* shadowValue;  // pending energy * radiant, w = path id bits

	// instanced scenes only (null otherwise): the instance layers of each ray's ignore hierarchy, of each hit and of each
	// shadow ray's ignore hierarchy, 8 words per slot (echo_instanced.cuh PathLayers)
	uint4* rayLayers[2];
	uint4* hitLayers;
	uint4* shadowLayers;

	uint32_t* classQueue[CLASS_COUNT]; // ray slots sorted by the material class of what they hit
	uint32_t* counters;
	unsigned long long* stats; // EchoStats layout

	const uint32_t* sampleIndex; // per path id (WorkerState::sampleIndex): stratified draws take the sample's position in its epoch from it
};

// ECHO_B200_PROFILE=1: per-kernel device time of the wavefront (CUDA events around every launch, synchronised; the
// numbers printed by a run with this switch on are diagnostics, never bench values).
struct KernelTimer
{
	enum { RAYGEN, EXTEND, SHADE_MISS, SHADE_DIFFUSE, SHADE_DIELECTRIC, SHADE_CONDUCTOR, SHADE_TERMINAL, SHADE_SMOOTH, SHADOW, ROTATE, FINISH, ACCUMULATE, OTHER, COUNT };
	bool enabled = false;
	double milliseconds[COUNT] = {};
	uint64_t launches[COUNT] = {};
	cudaEvent_t begin = nullptr, end = nullptr;

	KernelTimer()
	{
		const char* value = std::getenv("ECHO_B200_PROFILE");
		enabled = value && value[0] == '1';
	}

	~KernelTimer()
	{
		if (begin) cudaEventDestroy(begin);
		if (end) cudaEventDestroy(end);
	}

	void start(cudaStream_t stream)
	{
		if (!enabled) return;
		if (!begin) { cudaEventCreate(&begin); cudaEventCreate(&end); } // on the worker's own device
		cudaEventRecord(begin, stream);
	}

	float last = 0.0f;

	void stop(int slot, cudaStream_t stream)
	{
		if (!enabled) return;
		cudaEventRecord(end, stream);
		cudaEventSynchronize(end);
		float ms = 0.0f;
		cudaEventElapsedTime(&ms, begin, end);
		milliseconds[slot] += ms;
		++launches[slot];
		last = ms;
	}

	void report()
	{
		if (!enabled) return;
		static const char* names[COUNT] = { "raygen", "extend", "shade<miss>", "shade<diffuse>", "shade<dielectric>", "shade<conductor>", "shade<terminal>", "shade<smooth>", "shadow", "rotate", "finish", "accumulate", "classify" };
		double total = 0.0;
		for (double ms : milliseconds) total += ms;
		for (int i = 0; i < COUNT; i++)
			if (launches[i]) std::fprintf(stderr, "[echo_b200 profile] %-18s %8llu launches %10.3f ms %5.1f %%\n", names[i], (unsigned long long)launches[i], milliseconds[i], 100.0 * milliseconds[i] / total);
		std::fprintf(stderr, "[echo_b200 profile] total %.3f ms\n", total);
		for (int i = 0; i < COUNT; i++) { milliseconds[i] = 0.0; launches[i] = 0; }
	}
};

struct WorkerState
{
	cudaStream_t stream = nullptr;
	uint64_t capacity = 0;
	PathBuffers paths = {};
	std::vector<void*> allocations;

	int2* pixelXY = nullptr;        // per path slot
	uint32_t* sampleIndex = nullptr;
	float4* sampleOut = nullptr;    // per path slot radiance

	// per-pixel accumulators of the current tile batch
	uint64_t pixelCapacity = 0;
	float4* accumulator = nullptr;  // 4 x float4 per pixel: average total/error, squared total/error
	uint32_t* sampleCount = nullptr;
	uint32_t* activePixels[2] = { nullptr, nullptr };
	int2* batchPixelXY = nullptr;
	int32_t* tileXYDevice = nullptr;
	uint64_t tileCapacity = 0;

	uint32_t* hostCounters = nullptr; // pinned, mapped: [0..1] the 8-byte iteration mirror the device writes, [8] active pixels of an epoch

	// Run-ahead launching (evaluate_paths): the pipeline thread queues wavefront iterations without waiting for their counts;
	// `serial` numbers every iteration this worker ever launched, the rotate kernel publishes {serial, rays left} in the mirror
	static constexpr int kEventRing = 8;
	cudaEvent_t iterationDone[kEventRing] = {};
	bool eventsBlocking = false;
	uint32_t serial = 0;

	KernelTimer timer; // ECHO_B200_PROFILE=1 diagnostics (one pipeline, lock step)
};

// Tile batches are rendered by up to kWorkers concurrent pipelines (host thread + stream + wavefront buffers each): the
// long, narrow tail of one batch's late bounces overlaps the wide first bounces of another, keeping the SMs busy.
// below this many rays a bounce uses the one-thread-per-ray kernels: a persistent launch only pays off while every resident
// thread (148 x 7 x 128) gets several rays to replace finished ones with. A/B r2g with the exact class grids in place,
// 64 Ki / 256 Ki / 1 Mi: C1 340 / 355 / 407, C4 344 / 345 / 344, C5 458 / 460 / 460 M samples/s
constexpr uint32_t kNarrowLimit = 1048576;
// below this many live paths one kernel finishes them (tail_kernel). A/B of the threshold on C1 / C4 / C5 (variants/ab8.sh):
// 0 -> 260 / 302 / 314 M samples/s, 4096 -> 317 / 313 / 325, 16384 -> 314 / 314 / 323, 65536 -> 250 / 308 / 264 (the longest path
// of a big tail then runs alone for milliseconds), 262144 -> 140 / 277 / 187
constexpr uint32_t kTailLimit = 8192;
constexpr int kWorkers = 8; // A/B on C3/C4/C5: 1 -> 134, 2 -> 207, 4 -> 280, 8 -> 329, 12 -> 330 M samples/s on C5 (profiles/README.md)

// At most 16 Mi paths per batch and pipeline (250 B of wavefront state per path: about 4 GB each); render_tiles splits smaller
// jobs so that every pipeline gets a share. A/B at 64 spp per step, 4 / 8 / 16 Mi: C3 439 / 459 / 456, C4 321 / 330 / 332, C5 (16 spp)
// 337 / 350 / 368 M samples/s — wider launches per bounce and 2-4x fewer of them (variants/ab10.sh, ECHO_B200_BATCH_PATHS).
constexpr uint64_t kPathsPerBatch = 1ull << 24;

struct RenderState
{
	std::vector<WorkerState*> workers;
};

// ---------------------------------------------------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------------------------------------------------

// Wavefront state (ray / hit / class / shadow queues, per-path records) is written by one kernel and read by the next, gigabytes
// later: it cannot be reused out of L2 and only evicts the tree, which can (C5: 630 MB of nodes against 126 MB of L2). With
// ECHO_STREAM_STATE these accesses carry the streaming hint (ld.global.cs / st.global.cs: evict first). A/B in profiles/README.md.
#ifndef ECHO_STREAM_STATE
#define ECHO_STREAM_STATE 0
#endif

template<class T>
ECHO_DEVICE T stream_load(const T* pointer)
{
#if ECHO_STREAM_STATE
	return __ldcs(pointer);
#else
	return *pointer;
#endif
}

template<class T>
ECHO_DEVICE void stream_store(T* pointer, T value)
{
#if ECHO_STREAM_STATE
	__stcs(pointer, value);
#else
	*pointer = value;
#endif
}

// warp-aggregated append: one atomic per warp (ballot + popc + shuffle)
ECHO_DEVICE uint32_t queue_slot(uint32_t* counter, bool predicate)
{
	uint32_t mask = __ballot_sync(0xFFFFFFFFu, predicate);
	if (mask == 0u) return 0u;

	uint32_t lane = threadIdx.x & 31u;
	int leader = __ffs(mask) - 1;
	uint32_t base = 0u;
	if ((int)lane == leader) base = atomicAdd(counter, (uint32_t)__popc(mask));
	base = __shfl_sync(0xFFFFFFFFu, base, leader);
	return base + (uint32_t)__popc(mask & ((1u << lane) - 1u));
}

ECHO_DEVICE void stat_add(unsigned long long* stats, int slot, bool predicate)
{
	uint32_t mask = __ballot_sync(0xFFFFFFFFu, predicate);
	if (mask != 0u && (threadIdx.x & 31u) == (uint32_t)(__ffs(mask) - 1)) atomicAdd(stats + slot, (unsigned long long)__popc(mask));
}

// EchoStats slots
enum : int
{
	STAT_SAMPLE_EVALUATED = 0, STAT_SAMPLE_REJECTED, STAT_PIXEL_EVALUATED, STAT_BOUNCE_CREATED, STAT_BOUNCE_SPECULAR, STAT_BOUNCE_MIS,
	STAT_LIGHT_SAMPLED, STAT_LIGHT_OCCLUSION_CHECKED, STAT_LIGHT_OCCLUSION_PASSED, STAT_LIGHT_EVALUATED_INFINITE,
	STAT_TRACE_QUERIES, STAT_OCCLUDE_QUERIES, STAT_KERNEL_LAUNCHES,
	STAT_NODE_VISITS, STAT_TRIANGLE_VISITS, STAT_SPHERE_VISITS, STAT_LIGHT_NODE_VISITS, // counted passes only
	STAT_COUNT = 24
};
static_assert(sizeof(EchoStats) == sizeof(unsigned long long) * STAT_COUNT, "EchoStats layout");

ECHO_DEVICE vec3 xyz(float4 v) { return { v.x, v.y, v.z }; }
ECHO_DEVICE rgb as_rgb(float4 v) { return { v.x, v.y, v.z }; }
ECHO_DEVICE float4 make4(vec3 v, float w) { return make_float4(v.x, v.y, v.z, w); }
ECHO_DEVICE float4 make4(rgb v, float w) { return make_float4(v.r, v.g, v.b, w); }

ECHO_DEVICE uint32_t token_light_type(uint32_t token) { return token_index(token) >> ECHO_LIGHT_INDEX_BITS; }
ECHO_DEVICE uint32_t token_light_index(uint32_t token) { return token & ((1u << ECHO_LIGHT_INDEX_BITS) - 1u); }
ECHO_DEVICE bool token_is_raw_geometry(uint32_t token) { uint32_t t = token_type(token); return t == ECHO_TOKEN_TYPE_TRIANGLE || t == ECHO_TOKEN_TYPE_SPHERE; }

ECHO_DEVICE bool token_is_infinite_light(uint32_t token) // EntityToken.cs:194-202
{
	if (token_type(token) != ECHO_TOKEN_TYPE_LIGHT) return false;
	return token_light_type(token) <= ECHO_LIGHT_TYPE_INFINITE_DELTA;
}

ECHO_DEVICE bool token_is_area_light(uint32_t token) // EntityToken.cs:187-192
{
	if (token_is_raw_geometry(token)) return true;
	if (token_type(token) != ECHO_TOKEN_TYPE_LIGHT) return false;
	return token_light_type(token) == ECHO_LIGHT_TYPE_INFINITE;
}

// ---------------------------------------------------------------------------------------------------------------------
// geometry records
// ---------------------------------------------------------------------------------------------------------------------

struct TriangleData
{
	vec3 vertex0, edge1, edge2, normal0, normal1, normal2;
	uint32_t material;
};

ECHO_DEVICE TriangleData load_triangle(const DeviceScene& scene, uint32_t index)
{
	ECHO_CHECK(scene, index < scene.triangleCount, CHECK_TRIANGLE);
	const float4* hot = scene.triHot + (size_t)index * 3;
	const float4* shade = scene.triShade + (size_t)index * 3;
	float4 a = __ldg(hot), b = __ldg(hot + 1), c = __ldg(hot + 2);
	float4 d = __ldg(shade), e = __ldg(shade + 1), f = __ldg(shade + 2);
	return { xyz(a), xyz(b), xyz(c), xyz(d), xyz(e), xyz(f), __float_as_uint(d.w) };
}

ECHO_DEVICE vec3 triangle_normal(const TriangleData& t) { return normalized(cross(t.edge1, t.edge2)); }           // TriangleEntity.cs:136
ECHO_DEVICE float triangle_area(const TriangleData& t) { return div(magnitude(cross(t.edge1, t.edge2)), 2.0f); }  // TriangleEntity.cs:148

ECHO_DEVICE vec3 triangle_shading_normal(const TriangleData& t, vec2 uv) // TriangleEntity.cs:187
{
	return normalized((1.0f - uv.x - uv.y) * t.normal0 + uv.x * t.normal1 + uv.y * t.normal2);
}

ECHO_DEVICE vec3 triangle_point(const TriangleData& t, vec2 uv) { return t.vertex0 + uv.x * t.edge1 + uv.y * t.edge2; } // TriangleEntity.cs:265

ECHO_DEVICE vec3 sphere_normal(vec2 uv) // SphereEntity.cs:229-234,252-266
{
	float sinT = uv.x, sinP = uv.y, sign = 1.0f;

	if (sinT > 1.5f)
	{
		sinT -= 3.0f;
		sign = -1.0f;
	}

	float cosT = identity(sinT) * sign;
	float cosP = identity(sinP);
	return normalized(vec3{ sinT * cosP, sinP, cosT * cosP });
}

ECHO_DEVICE vec2 triangle_texcoord(const DeviceScene& scene, uint32_t index, vec2 uv) // PreparedTriangle.GetTexcoord, TriangleEntity.cs:188
{
	float4 a = __ldg(scene.triTexcoord + (size_t)index * 2), b = __ldg(scene.triTexcoord + (size_t)index * 2 + 1);
	float w = 1.0f - uv.x - uv.y;
	return { w * a.x + uv.x * a.z + uv.y * b.x, w * a.y + uv.x * a.w + uv.y * b.y };
}

ECHO_DEVICE vec2 sphere_texcoord(vec2 uv) // PreparedSphere.GetTexcoord, SphereEntity.cs:236-245 (Atan2 / Asin pinned)
{
	float sinT = uv.x, sinP = uv.y, sign = 1.0f;

	if (sinT > 1.5f)
	{
		sinT -= 3.0f;
		sign = -1.0f;
	}

	float cosT = identity(sinT) * sign;
	return { fma_f(atan2_det(sinT, cosT), kTauR, 0.5f), fma_f(asin_det(clamp11(sinP)), kPiR, 0.5f) };
}

ECHO_DEVICE float sphere_area(float radius) { return 4.0f * kPi * radius * radius; } // SphereEntity.cs:72

struct SurfacePoint // GeometryPoint
{
	vec3 position, normal;
};

ECHO_DEVICE float geometry_point_pdf(const SurfacePoint& point, vec3 origin, float area) // GeometryPoint.cs:28-39
{
	vec3 delta = point.position - origin;
	float length2 = squared_magnitude(delta);
	float length = sqrt0(length2);

	float d = abs_bits(dot(point.normal, delta));
	if (!positive(d)) return 0.0f;
	return div(length2 * length, d * area);
}

// ---------------------------------------------------------------------------------------------------------------------
// light tree (Aggregation/Selection/LightTree.cs, Aggregation/Bounds/LightBound.cs)
// ---------------------------------------------------------------------------------------------------------------------

struct LightNode
{
	vec3 boxMin, boxMax, coneAxis;
	float cosOffset, cosExtend, power;
	uint32_t child0, child1;
};

ECHO_DEVICE LightNode load_light_node(const DeviceScene& scene, const PackInfo& info, uint32_t index)
{
	ECHO_CHECK(scene, index < info.lightNodeCount && info.lightNodeOffset + index < scene.lightNodeCount, CHECK_LIGHT_NODE);
	const float4* p = scene.lightNodes + ((size_t)info.lightNodeOffset + index) * 4;
	float4 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2), d = __ldg(p + 3);
	LightNode n;
	n.boxMin = { a.x, a.y, a.z };
	n.boxMax = { a.w, b.x, b.y };
	n.coneAxis = { b.z, b.w, c.x };
	n.cosOffset = c.y;
	n.cosExtend = c.z;
	n.power = c.w;
	n.child0 = __float_as_uint(d.x);
	n.child1 = __float_as_uint(d.y);
	return n;
}

ECHO_DEVICE float clamp_subtract_cos(float sin0, float cos0, float sin1, float cos1) { return cos0 > cos1 ? 1.0f : cos0 * cos1 + sin0 * sin1; } // LightBound.cs:79
ECHO_DEVICE float clamp_subtract_sin(float sin0, float cos0, float sin1, float cos1) { return cos0 > cos1 ? 0.0f : sin0 * cos1 - cos0 * sin1; } // LightBound.cs:80

ECHO_DEVICE float light_importance(const LightNode& bound, const SurfacePoint& origin) // LightBound.cs:30-60
{
	vec3 center = (bound.boxMax + bound.boxMin) / 2.0f;
	vec3 incident = origin.position - center;

	float length2 = squared_magnitude(incident);

	if (almost_zero(length2)) incident = { 0.0f, 0.0f, 0.0f };
	else incident = incident * sqrt_r0(length2);

	float cosAxis = dot(bound.coneAxis, incident);
	float sinAxis = identity(cosAxis);

	float cosOffset = bound.cosOffset;
	float sinOffset = identity(cosOffset);

	float sinRadius, cosRadius; // FindSubtendedAngles, :62-77
	vec3 size = bound.boxMax - bound.boxMin;
	float radius2 = div(squared_magnitude(size), 4.0f);

	if (length2 < radius2)
	{
		sinRadius = 0.0f;
		cosRadius = -1.0f;
	}
	else
	{
		float sinRadius2 = div(radius2, length2);
		sinRadius = sqrt0(sinRadius2);
		cosRadius = sqrt0(1.0f - sinRadius2);
	}

	float cosRemain = clamp_subtract_cos(sinAxis, cosAxis, sinOffset, cosOffset);
	float sinRemain = clamp_subtract_sin(sinAxis, cosAxis, sinOffset, cosOffset);
	float cosFinal = clamp_subtract_cos(sinRemain, cosRemain, sinRadius, cosRadius);
	if (cosFinal <= bound.cosExtend) return 0.0f;

	float cosIncident = abs_bits(dot(origin.normal, incident));
	float sinIncident = identity(cosIncident);
	float cosReflect = clamp_subtract_cos(sinIncident, cosIncident, sinRadius, cosRadius);

	length2 = max_net(length2, div(magnitude(size), 2.0f));
	return max0(div(bound.power, length2) * cosFinal * cosReflect);
}

// LightTree.Pick, LightTree.cs:115-134 (tail recursion as a loop). Returns the token; pdf == 0 means impossible.
// COUNT (counted passes only, see shade_counted_kernel): LightBound.Importance evaluations go to scene.lightVisits
template<bool COUNT = false>
ECHO_DEVICE uint32_t light_tree_pick(const DeviceScene& scene, const PackInfo& info, const SurfacePoint& origin, float& sample, float& outPdf)
{
	outPdf = 0.0f;
	if (info.lightNodeCount == 0u) return ECHO_TOKEN_EMPTY;

	LightNode node = load_light_node(scene, info, 0u);
	float pdf = 1.0f;

	while (true)
	{
		if (node.child0 == ECHO_TOKEN_EMPTY)
		{
			outPdf = pdf;
			return node.child1;
		}

		LightNode left = load_light_node(scene, info, node.child0);
		LightNode right = load_light_node(scene, info, node.child1);
		float importance0 = light_importance(left, origin);
		float importance1 = light_importance(right, origin);
		if (COUNT) atomicAdd(scene.lightVisits, 2ull);

		if (!positive(importance0) && !positive(importance1)) return ECHO_TOKEN_EMPTY;

		float split = div(importance0, importance0 + importance1);

		if (sample < split)
		{
			sample = sample_stretch(sample, 0.0f, split);
			node = left;
			pdf = pdf * split;
		}
		else
		{
			sample = sample_stretch(sample, split, 1.0f);
			node = right;
			pdf = pdf * (1.0f - split);
		}
	}
}

// LightTree.ProbabilityMass, LightTree.cs:53-57,136-154: the recursion multiplies split factors from the leaf upward,
// so the factors of the root-to-leaf walk are kept and folded right to left.
template<bool COUNT = false>
ECHO_DEVICE float light_tree_mass(const DeviceScene& scene, const PackInfo& info, uint32_t token, const SurfacePoint& origin)
{
	// map.TryGetValue: binary search over the pack's sorted emitter tokens
	ECHO_CHECK(scene, info.emitterOffset + info.emitterCount <= scene.emitterCount, CHECK_EMITTER);
	int low = (int)info.emitterOffset, high = (int)(info.emitterOffset + info.emitterCount) - 1, found = -1;

	while (low <= high)
	{
		int middle = (low + high) >> 1;
		uint32_t value = __ldg(scene.emitterTokens + middle);
		if (value == token) { found = middle; break; }
		if (value < token) low = middle + 1;
		else high = middle - 1;
	}

	if (found < 0) return 0.0f;
	unsigned long long branches = __ldg(scene.emitterPaths + found);

	float factors[64];
	int depth = 0;
	LightNode node = load_light_node(scene, info, 0u);

	while (node.child0 != ECHO_TOKEN_EMPTY && depth < 64)
	{
		LightNode left = load_light_node(scene, info, node.child0);
		LightNode right = load_light_node(scene, info, node.child1);
		float importance0 = light_importance(left, origin);
		float importance1 = light_importance(right, origin);
		if (COUNT) atomicAdd(scene.lightVisits, 2ull);
		float split = div(importance0, importance0 + importance1);

		if ((branches & 1ull) == 0ull)
		{
			factors[depth++] = split;
			node = left;
		}
		else
		{
			factors[depth++] = 1.0f - split;
			node = right;
		}

		branches >>= 1;
	}

	float mass = 1.0f;
	for (int i = depth - 1; i >= 0; i--) mass = factors[i] * mass;
	return mass;
}

// ---------------------------------------------------------------------------------------------------------------------
// infinite lights: AmbientLight over a Pure texture (AmbientLight.cs:53-67) and DirectionalLight (DirectionalLight.cs:78-108).
// EchoInfiniteLight = 10 float4: {radiance, directlyVisible} {type, isDelta, cosAngle, -} {intensity, -} {direction, -}
// rotation[9] texture distribution - | inverseRotation[9] + pad
// ---------------------------------------------------------------------------------------------------------------------

constexpr int kInfiniteStride = 10;

struct InfiniteLight
{
	rgb radiance;
	bool directlyVisible, directional, delta, environment, cubemap;
	float cosAngle;
	const float4* data;
};

ECHO_DEVICE InfiniteLight load_infinite(const DeviceScene& scene, uint32_t index)
{
	ECHO_CHECK(scene, index < scene.infiniteLightCount, CHECK_INFINITE_LIGHT);
	const float4* p = scene.infiniteLights + (size_t)index * kInfiniteStride;
	float4 a = __ldg(p), b = __ldg(p + 1);
	uint32_t type = __float_as_uint(b.x);
	return { as_rgb(a), __float_as_uint(a.w) != 0u, type == ECHO_INFINITE_DIRECTIONAL, __float_as_uint(b.y) != 0u, type == ECHO_INFINITE_ENVIRONMENT,
	         type == ECHO_INFINITE_CUBEMAP, b.z, p };
}

ECHO_DEVICE vec3 rotate3x3(float4 r0, float4 r1, float r8, vec3 v) // Float3x3 * Float3 (Float3x3.cs:264-269), nine row-major floats
{
	return { r0.x * v.x + r0.y * v.y + r0.z * v.z, r0.w * v.x + r1.x * v.y + r1.y * v.z, r1.z * v.x + r1.w * v.y + r8 * v.z };
}

ECHO_DEVICE vec3 infinite_to_world(const InfiniteLight& light, vec3 v) // LocalToWorldRotation: words 16..24
{
	return rotate3x3(__ldg(light.data + 4), __ldg(light.data + 5), __ldg(light.data + 6).x, v);
}

ECHO_DEVICE vec3 infinite_to_local(const InfiniteLight& light, vec3 v) // WorldToLocalRotation: words 28..36
{
	return rotate3x3(__ldg(light.data + 7), __ldg(light.data + 8), __ldg(light.data + 9).x, v);
}

// ---- Evaluation/Sampling/DiscreteDistribution1D.cs:58-166 over a stored cdf ----
struct Distribution1D
{
	const float* cdf;
	int count;

	ECHO_DEVICE void bounds(int index, float& lower, float& upper) const
	{
		lower = index == 0 ? 0.0f : __ldg(cdf + index - 1);
		upper = __ldg(cdf + index);
	}

	ECHO_DEVICE int find_index(float sample) const // FindIndex / FixIndex / BinarySearch
	{
		uint32_t head = 0u, tail = (uint32_t)count;
		int index = -1;

		while (head < tail)
		{
			uint32_t middle = (tail + head) >> 1;
			float current = __ldg(cdf + middle);
			if (current == sample) { index = (int)middle; break; }
			if (current > sample) tail = middle;
			else head = middle + 1u;
		}

		if (index < 0) return (int)head;

		float lower, upper;
		bounds(index, lower, upper);
		if (upper - lower > 0.0f) return index + 1;

		do
		{
			lower = upper;
			upper = __ldg(cdf + ++index);
		}
		while (lower == upper);

		return index;
	}

	ECHO_DEVICE float sample(float u, float& pdf) const
	{
		int index = find_index(u);
		float lower, upper;
		bounds(index, lower, upper);

		float gap = upper - lower;
		float countR = rcp((float)count);
		float shift = div(u - lower, gap) + (float)index;
		pdf = gap * (float)count;
		return sample1d(shift * countR);
	}

	ECHO_DEVICE float probability_density(float result) const
	{
		float lower, upper;
		bounds(sample_range(result, count), lower, upper);
		return (upper - lower) * (float)count;
	}
};

// ---- Textures/Directional/CylindricalTexture.cs:98-165 ----
ECHO_DEVICE vec2 cylindrical_to_uv(vec3 direction) // ToUV, :142-151 (Atan2 / Acos pinned)
{
	return { fma_f(atan2_det(direction.x, direction.z), kTauR, 0.5f), fma_f(acos_det(clamp11(direction.y)), -kPiR, 1.0f) };
}

struct EnvironmentGrid
{
	uint32_t texture;
	const float* values;
	int width, height;
};

ECHO_DEVICE EnvironmentGrid environment_grid(const DeviceScene& scene, const InfiniteLight& light)
{
	float4 tail = __ldg(light.data + 6); // rotation[8], texture, distribution, pad
	uint32_t texture = __float_as_uint(tail.y);
	ECHO_CHECK(scene, texture < scene.textureCount, CHECK_TEXTURE);
	uint4 header = __ldg(scene.textures + (size_t)texture * 2);
	ECHO_CHECK(scene, (uint64_t)__float_as_uint(tail.z) + (uint64_t)header.y * (header.x + 1ull) <= scene.distributionCount, CHECK_DISTRIBUTION);
	return { texture, scene.distributions + __float_as_uint(tail.z), (int)header.x, (int)header.y };
}

ECHO_DEVICE float cylindrical_pdf(const DeviceScene& scene, const InfiniteLight& light, vec3 incident) // :100-110
{
	vec2 uv = cylindrical_to_uv(incident);
	float cosP = -incident.y;
	float sinP = identity(cosP);
	if (!positive(sinP)) return 0.0f;

	EnvironmentGrid grid = environment_grid(scene, light);
	float x = sample1d(uv.x), y = sample1d(uv.y); // (Sample2D)uv

	Distribution1D vertical{ grid.values, grid.height };
	Distribution1D slice{ grid.values + grid.height + (size_t)sample_range(y, grid.height) * grid.width, grid.width };
	float pdfX = slice.probability_density(x);
	float pdfY = vertical.probability_density(y);
	return div(pdfX * pdfY * (kTauR / kPi), sinP);
}

ECHO_DEVICE Sampled cylindrical_sample(const DeviceScene& scene, const InfiniteLight& light, vec2 sample, vec3& incident) // :112-140
{
	EnvironmentGrid grid = environment_grid(scene, light);

	float pdfY, pdfX;
	float y = Distribution1D{ grid.values, grid.height }.sample(sample.y, pdfY);
	float x = Distribution1D{ grid.values + grid.height + (size_t)sample_range(y, grid.height) * grid.width, grid.width }.sample(sample.x, pdfX);
	float pdf = pdfX * pdfY;

	incident = { 0.0f, 0.0f, 0.0f };
	if (!positive(pdf)) return impossible();

	float sinT, cosT, sinP, cosP;
	sincos_det(x * kTau, sinT, cosT);
	sincos_det(y * kPi, sinP, cosP);
	if (!positive(sinP)) return impossible();

	incident = { -sinP * sinT, -cosP, -sinP * cosT };
	return { as_rgb(texture_sample(scene, grid.texture, vec2{ x, y })), div(pdf * (kTauR / kPi), sinP) };
}

// Textures/Directional/Cubemap.cs:62-82 with (Direction)incident (Direction.cs:325-333)
ECHO_DEVICE rgb cubemap_evaluate(const DeviceScene& scene, const InfiniteLight& light, vec3 incident)
{
	float ax = fabsf(incident.x), ay = fabsf(incident.y), az = fabsf(incident.z);
	int axis = ax > ay ? (ax > az ? 0 : 2) : (ay > az ? 1 : 2);
	float part = axis == 0 ? incident.x : (axis == 1 ? incident.y : incident.z);
	bool negative = part < 0.0f;
	int index = axis * 2 + (negative ? 1 : 0);

	vec2 uv;
	switch (index)
	{
		case 0: uv = { -incident.z, incident.y }; break;
		case 1: uv = { incident.z, incident.y }; break;
		case 2: uv = { incident.x, -incident.z }; break;
		case 3: uv = { incident.x, incident.z }; break;
		case 4: uv = { incident.x, incident.y }; break;
		default: uv = { -incident.x, incident.y }; break;
	}

	float scale = div(0.5f, negative ? -part : part); // target.ExtractComponent(incident)
	uv = { uv.x * scale + 0.5f, uv.y * scale + 0.5f };
	uint32_t first = __float_as_uint(__ldg(light.data + 6).y);
	return as_rgb(texture_sample(scene, first + (uint32_t)index, uv));
}

ECHO_DEVICE rgb infinite_evaluate(const DeviceScene& scene, const InfiniteLight& light, vec3 incident)
{
	if (light.cubemap) return light.radiance * cubemap_evaluate(scene, light, infinite_to_local(light, incident));

	if (light.environment) // AmbientLight.Evaluate, AmbientLight.cs:53-54
	{
		uint32_t texture = __float_as_uint(__ldg(light.data + 6).y);
		return light.radiance * as_rgb(texture_sample(scene, texture, cylindrical_to_uv(infinite_to_local(light, incident))));
	}

	if (!light.directional) return light.radiance;
	if (light.delta) return make_rgb(0.0f);

	float cosIncident = dot(xyz(__ldg(light.data + 3)), incident);
	if (cosIncident <= light.cosAngle) return make_rgb(0.0f);
	return light.radiance; // scaledIntensity
}

ECHO_DEVICE float infinite_pdf(const DeviceScene& scene, const InfiniteLight& light, vec3 incident)
{
	if (light.environment) return cylindrical_pdf(scene, light, infinite_to_local(light, incident)); // AmbientLight.cs:56-57
	if (!light.directional) return kUniformSpherePdf;
	if (light.delta) return 0.0f;
	return uniform_cone_pdf(light.cosAngle);
}

ECHO_DEVICE Sampled infinite_sample(const DeviceScene& scene, const InfiniteLight& light, vec2 sample, vec3& incident, float& travel)
{
	travel = kInfinity;

	if (light.environment) // AmbientLight.Sample, AmbientLight.cs:59-66
	{
		Sampled sampled = cylindrical_sample(scene, light, sample, incident);
		incident = infinite_to_world(light, incident);
		return { sampled.content * light.radiance, sampled.pdf };
	}

	if (light.cubemap) // IDirectionalTexture.Sample's default inside AmbientLight.Sample
	{
		vec3 local = uniform_sphere(sample);
		incident = infinite_to_world(light, local);
		return { cubemap_evaluate(scene, light, local) * light.radiance, kUniformSpherePdf };
	}

	if (!light.directional)
	{
		incident = uniform_sphere(sample); // IDirectionalTexture.Sample default, Textures/Directional/IDirectionalTexture.cs
		return { light.radiance, kUniformSpherePdf };
	}

	if (light.delta)
	{
		incident = xyz(__ldg(light.data + 3));
		return { as_rgb(__ldg(light.data + 2)), 1.0f };
	}

	vec3 local = uniform_cone(sample, light.cosAngle);
	local.z = -local.z; // Utility.NegateZ
	incident = infinite_to_world(light, local);
	return { light.radiance, uniform_cone_pdf(light.cosAngle) };
}

// PreparedScene.Pick, PreparedScene.cs:113-150; outLayers receives the instance layers of the picked light's hierarchy
template<bool INST, bool COUNT = false>
ECHO_DEVICE uint32_t scene_pick(const DeviceScene& scene, const SurfacePoint& origin, float sample, float& outPdf, PathLayers& outLayers)
{
	outLayers = no_layers();

	if (sample < scene.infiniteThreshold)
	{
		sample = sample_stretch(sample, 0.0f, scene.infiniteThreshold);
		int index = sample_range(sample, (int)scene.infiniteLightCount);
		outPdf = scene.infinitePdf;
		bool delta = __float_as_uint(__ldg(scene.infiniteLights + (size_t)index * kInfiniteStride + 1).y) != 0u;
		return ECHO_LIGHT_TOKEN_MAKE(delta ? ECHO_LIGHT_TYPE_INFINITE_DELTA : ECHO_LIGHT_TYPE_INFINITE, (uint32_t)index); // :120
	}

	sample = sample_stretch(sample, scene.infiniteThreshold, 1.0f);
	float pdf = 1.0f - scene.infiniteThreshold;
	PackInfo info = INST ? load_pack_info(scene, 0u) : whole_scene_pack(scene);

	while (true) // :132-147: the same `origin` serves every layer (it is not moved into the placement's space)
	{
		float tokenPdf;
		uint32_t token = light_tree_pick<COUNT>(scene, info, origin, sample, tokenPdf);

		if (almost_zero(tokenPdf))
		{
			outPdf = 0.0f;
			return ECHO_TOKEN_EMPTY;
		}

		pdf *= tokenPdf;

		if (!INST || token_type(token) != ECHO_TOKEN_TYPE_INSTANCE || outLayers.count >= ECHO_MAX_INSTANCE_LAYERS)
		{
			outPdf = pdf;
			return token;
		}

		float4 tail = __ldg(instance_data(scene, info.instanceOffset + token_index(token)) + 6);
		outLayers.tokens[outLayers.count++] = token;
		info = load_pack_info(scene, __float_as_uint(tail.z));
	}
}

// PreparedScene.ProbabilityMass, PreparedScene.cs:158-179
template<bool INST, bool COUNT = false>
ECHO_DEVICE float scene_probability_mass(const DeviceScene& scene, uint32_t light, const PathLayers& layers, const SurfacePoint& origin)
{
	if (token_is_infinite_light(light)) return scene.infinitePdf;
	float pdf = 1.0f - scene.infiniteThreshold;
	PackInfo info = INST ? load_pack_info(scene, 0u) : whole_scene_pack(scene);

	if (INST)
	{
		for (uint32_t k = 0; k < layers.count; k++)
		{
			pdf *= light_tree_mass<COUNT>(scene, info, layers.tokens[k], origin);
			float4 tail = __ldg(instance_data(scene, info.instanceOffset + token_index(layers.tokens[k])) + 6);
			info = load_pack_info(scene, __float_as_uint(tail.z));
			if (almost_zero(pdf)) return 0.0f;
		}
	}

	return pdf * light_tree_mass<COUNT>(scene, info, light, origin);
}

// ---------------------------------------------------------------------------------------------------------------------
// light sampling (Aggregation/Preparation/LightCollection.cs, TriangleEntity.cs:166-185, SphereEntity.cs:151-225)
// ---------------------------------------------------------------------------------------------------------------------

// index inside the swatch the geometry's pack (or placement) uses
ECHO_DEVICE uint32_t geometry_material(const DeviceScene& scene, const PackInfo& info, uint32_t token)
{
	ECHO_CHECK(scene, token_type(token) == ECHO_TOKEN_TYPE_TRIANGLE ? info.triangleOffset + token_index(token) < scene.triangleCount
	                                                               : info.sphereOffset + token_index(token) < scene.sphereCount, CHECK_SPHERE);
	if (token_type(token) == ECHO_TOKEN_TYPE_TRIANGLE) return __float_as_uint(__ldg(scene.triShade + ((size_t)info.triangleOffset + token_index(token)) * 3).w);
	return __ldg(scene.sphereMaterial + info.sphereOffset + token_index(token));
}

ECHO_DEVICE bool geometry_sample(const DeviceScene& scene, const PackInfo& info, uint32_t token, vec3 origin, vec2 sample, SurfacePoint& point, float& pdf)
{
	if (token_type(token) == ECHO_TOKEN_TYPE_TRIANGLE)
	{
		TriangleData triangle = load_triangle(scene, info.triangleOffset + token_index(token));
		vec2 uv = uniform_triangle(sample);
		point.position = triangle_point(triangle, uv);
		point.normal = triangle_shading_normal(triangle, uv);
		pdf = geometry_point_pdf(point, origin, triangle_area(triangle));
		return true;
	}

	float4 sphere = __ldg(scene.spheres + info.sphereOffset + token_index(token));
	vec3 position = { sphere.x, sphere.y, sphere.z };
	float radius = sphere.w;

	vec3 offset = origin - position;
	float radius2 = radius * radius;
	float length2 = squared_magnitude(offset);

	if (length2 < radius2)
	{
		vec3 normal = uniform_sphere(sample);
		point = { normal * radius + position, normal }; // GetPoint, SphereEntity.cs:227
		pdf = geometry_point_pdf(point, origin, sphere_area(radius));
		return true;
	}

	float sinMaxT2 = div(radius2, length2);
	float cosMaxT = sqrt0(1.0f - sinMaxT2);

	if (almost_zero(1.0f - cosMaxT))
	{
		pdf = 0.0f;
		return false;
	}

	float cosT = fma_f(cosMaxT - 1.0f, sample.x, 1.0f);
	float sinT = identity(cosT);
	float phi = sample.y * kTau;

	float length = sqrt0(length2);
	float project = length * cosT - sqrt0(radius2 - length2 * sinT * sinT);
	float cosA = div(length2 + radius2 - project * project, 2.0f * length * radius);
	float sinA = identity(cosA);

	float sinP, cosP;
	sincos_det(phi, sinP, cosP);
	vec3 normal = normalized(vec3{ sinA * cosP, sinA * sinP, cosA });
	pdf = uniform_cone_pdf(cosMaxT);

	frame transform = make_frame(offset / length);
	vec3 world = apply_forward(transform, normal);
	point = { world * radius + position, world };
	return true;
}

ECHO_DEVICE float geometry_pdf(const DeviceScene& scene, const PackInfo& info, uint32_t token, vec3 origin, vec3 incident)
{
	if (token_type(token) == ECHO_TOKEN_TYPE_TRIANGLE)
	{
		TriangleData triangle = load_triangle(scene, info.triangleOffset + token_index(token));
		vec2 uv = { 0.0f, 0.0f };
		float distance = triangle_intersect(triangle.vertex0, triangle.edge1, triangle.edge2, origin, incident, uv);
		if (distance == kInfinity) return 0.0f;
		return div(distance * distance, abs_bits(dot(triangle_shading_normal(triangle, uv), incident) * triangle_area(triangle)));
	}

	float4 sphere = __ldg(scene.spheres + info.sphereOffset + token_index(token));
	float radius = sphere.w;
	vec3 offset = origin - vec3{ sphere.x, sphere.y, sphere.z };
	float radius2 = radius * radius;
	float length2 = squared_magnitude(offset);

	if (length2 <= radius2)
	{
		float projected = dot(offset, incident);
		float extend2 = fma_f(projected, projected, radius2 - length2);

		float distance = sqrt0(extend2) - projected;
		vec3 normal = offset + incident * distance;

		float cosWeight = dot(incident, normal) * radius;
		if (almost_zero(cosWeight)) return 0.0f;

		return div(distance * distance, abs_bits(cosWeight)) * kUniformSpherePdf;
	}

	float sinMaxT2 = div(radius2, length2);
	float cosMaxT = sqrt0(1.0f - sinMaxT2);
	return almost_zero(1.0f - cosMaxT) ? 0.0f : uniform_cone_pdf(cosMaxT);
}

// PreparedScene.Sample, PreparedScene.cs:182-204 -> LightCollection.Sample (:141-193) / PointLight.cs:48-66 / AmbientLight.cs:60-67
template<bool INST>
ECHO_DEVICE Sampled scene_sample_light(const DeviceScene& scene, uint32_t light, const PathLayers& layers, const SurfacePoint& origin, vec2 sample, vec3& incident, float& travel)
{
	incident = { 0.0f, 0.0f, 0.0f };
	travel = 0.0f;

	if (token_is_infinite_light(light))
	{
		return infinite_sample(scene, load_infinite(scene, token_light_index(light)), sample, incident, travel);
	}

	// FindLayer + `forwardTransform * origin` (:192-198, GeometryPoint.cs:41-45): the shading point in the space of the pack
	// that owns the light (without layers: the identity, still multiplied through)
	Layer layer = find_layer<INST>(scene, layers);
	vec3 position = transform_point(layer.forward, origin.position);
	Sampled result;

	if (token_type(light) == ECHO_TOKEN_TYPE_LIGHT)
	{
		ECHO_CHECK(scene, layer.info.pointLightOffset + token_light_index(light) < scene.pointLightCount, CHECK_POINT_LIGHT);
		const float4* p = scene.pointLights + ((size_t)layer.info.pointLightOffset + token_light_index(light)) * 2;
		float4 intensity = __ldg(p), lightPosition = __ldg(p + 1);
		vec3 offset = xyz(lightPosition) - position;
		float travel2 = squared_magnitude(offset);

		if (!positive(travel2)) return impossible();

		travel = sqrt0(travel2);
		float travelR = rcp(travel);
		incident = offset * travelR;
		result = { as_rgb(intensity) * travelR * travelR, 1.0f };
	}
	else
	{
		// the material comes from the PACK's swatch (geometries.swatch, LightCollection.cs:145,151), not from the placement's
		MaterialRecord material = load_material(scene, layer.info.materialOffset + geometry_material(scene, layer.info, light));
		if (material.type != ECHO_MATERIAL_EMISSIVE) return impossible();

		SurfacePoint point;
		float pdf;
		if (!geometry_sample(scene, layer.info, light, position, sample, point, pdf)) return impossible();
		if (!positive(pdf)) return impossible();

		vec3 delta = point.position - position;
		float travel2 = squared_magnitude(delta);
		if (!positive(travel2)) return impossible();

		travel = sqrt0(travel2);
		incident = delta * rcp(travel);
		travel *= 1.0f - 2E-5f; // TravelMultiplier, LightCollection.cs:89

		rgb emitted = dot(-incident, point.normal) > 0.0f ? material_emission(material) : make_rgb(0.0f); // Emissive.Emit, Emissive.cs:64
		result = { emitted, pdf };
	}

	// back to world space, :200-201
	incident = normalized(transform_direction(layer.inverse, incident));
	travel *= transform_scale(layer.inverse);
	return result;
}

// PreparedScene.ProbabilityDensity, PreparedScene.cs:207-225
template<bool INST>
ECHO_DEVICE float scene_light_pdf(const DeviceScene& scene, uint32_t light, const PathLayers& layers, const SurfacePoint& origin, vec3 incident)
{
	if (token_is_infinite_light(light)) return infinite_pdf(scene, load_infinite(scene, token_light_index(light)), incident);
	if (token_type(light) == ECHO_TOKEN_TYPE_LIGHT) return 1.0f;

	Layer layer = find_layer<INST>(scene, layers);
	vec3 position = transform_point(layer.forward, origin.position);
	vec3 direction = normalized(transform_direction(layer.forward, incident));
	return geometry_pdf(scene, layer.info, light, position, direction);
}

ECHO_DEVICE rgb evaluate_infinite(const DeviceScene& scene, vec3 direction, bool direct) // PreparedScene.cs:233-253
{
	rgb total = make_rgb(0.0f);

	for (uint32_t i = 0; i < scene.infiniteLightCount; i++)
	{
		InfiniteLight light = load_infinite(scene, i);
		if (direct && !light.directlyVisible) continue;
		total = total + infinite_evaluate(scene, light, direction);
	}

	return total;
}

ECHO_DEVICE float power_heuristic(float pdf0, float pdf1) // PathTracedEvaluator.cs:213-217
{
	float squared = pdf0 * pdf0;
	return div(squared, squared + pdf1 * pdf1);
}

// ---------------------------------------------------------------------------------------------------------------------
// camera (Scenic/Cameras/PerspectiveCamera.cs:51-98, RaySpawner.cs:19-46)
// ---------------------------------------------------------------------------------------------------------------------

ECHO_DEVICE vec3 camera_direction(const EchoCamera& c, vec3 d)
{
	const float* m = c.transform;
	return { m[0] * d.x + m[1] * d.y + m[2] * d.z, m[4] * d.x + m[5] * d.y + m[6] * d.z, m[8] * d.x + m[9] * d.y + m[10] * d.z };
}

ECHO_DEVICE vec3 camera_point(const EchoCamera& c, vec3 p)
{
	const float* m = c.transform;
	return { m[0] * p.x + m[1] * p.y + m[2] * p.z + m[3], m[4] * p.x + m[5] * p.y + m[6] * p.z + m[7], m[8] * p.x + m[9] * p.y + m[10] * p.z + m[11] };
}

ECHO_DEVICE void camera_spawn(const EchoCamera& camera, int width, int height, int px, int py, vec2 shift, vec2 lens, vec3& origin, vec3& direction)
{
	float sizeRX = rcp((float)width);                       // TextureGrid.cs:22
	float offsetY = div(div((float)height, (float)width), -2.0f); // aspects.Y / -2, RaySpawner.cs:22
	float sx = shift.x + (float)px, sy = shift.y + (float)py;
	vec2 uv = { fma_f(sx, sizeRX, 1.0f / -2.0f), fma_f(sy, sizeRX, offsetY) }; // SpawnX, RaySpawner.cs:37-46

	if (camera.type == ECHO_CAMERA_ORTHOGRAPHIC) // OrthographicCamera.cs:33-38
	{
		origin = camera_point(camera, vec3{ uv.x * camera.width, uv.y * camera.width, 0.0f });
		direction = { camera.direction[0], camera.direction[1], camera.direction[2] };
		return;
	}

	if (camera.type == ECHO_CAMERA_CYLINDRICAL) // CylindricalCamera.cs:27-33 + CylindricalTexture.ToDirection (CylindricalTexture.cs:153-164)
	{
		float sizeRY = rcp((float)height);
		float sinT, cosT, sinP, cosP;
		sincos_det(sx * sizeRX * kTau, sinT, cosT);
		sincos_det(sy * sizeRY * kPi, sinP, cosP);
		vec3 local = normalized(vec3{ -sinP * sinT, -cosP, -sinP * cosT });
		origin = { camera.transform[3], camera.transform[7], camera.transform[11] };
		direction = normalized(camera_direction(camera, local));
		return;
	}

	bool hasDepthOfField = positive(camera.lensRadius) && positive(camera.focalDistance);

	if (!hasDepthOfField)
	{
		origin = { camera.transform[3], camera.transform[7], camera.transform[11] };
		direction = normalized(camera_direction(camera, vec3{ uv.x, uv.y, camera.forwardLength }));
		return;
	}

	float focusScale = div(camera.focalDistance, camera.forwardLength);
	vec2 disk = concentric_disk(lens);
	vec3 lensPoint = { disk.x * camera.lensRadius, disk.y * camera.lensRadius, 0.0f };
	vec3 focus = { uv.x * focusScale, uv.y * focusScale, camera.focalDistance };

	origin = camera_point(camera, lensPoint);
	direction = normalized(camera_direction(camera, focus - lensPoint));
}

// ---------------------------------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------------------------------

// The draws of one sample in the reference's pairing (CameraSample.cs:19-23; PathTracedEvaluator.cs:60-66): the uniform sequence
// (sample_value), or with STRAT the stratified one (ECHO_DISTRIBUTION_STRATIFIED). STRAT is a template parameter of every kernel
// that draws, so the uniform instantiations carry no trace of the stratified code (the shading kernels run at the register cap).
template<bool STRAT>
ECHO_DEVICE float draw1d(uint32_t key, const Strata& strata, uint32_t dimension)
{
	if (STRAT) return stratified_1d(key, dimension, strata);
	return sample_value(key, dimension);
}

template<bool STRAT>
ECHO_DEVICE vec2 draw2d(uint32_t key, const Strata& strata, uint32_t dimension)
{
	if (STRAT) return stratified_2d(key, dimension, strata);
	return { sample_value(key, dimension), sample_value(key, dimension + 1u) };
}

// the sample's place in its epoch, read only by the stratified instantiations
template<bool STRAT>
ECHO_DEVICE Strata path_strata(const EchoRenderParams& params, const PathBuffers& paths, uint32_t id)
{
	if (STRAT) return make_strata((uint32_t)params.extend, paths.sampleIndex[id]);
	return { 0u, 0u, 0u };
}

template<bool STRAT>
__global__ void __launch_bounds__(kBlock) raygen_kernel(DeviceScene scene, EchoRenderParams params, uint32_t count, const int2* __restrict__ pixelXY,
                                                       const uint32_t* __restrict__ sampleIndex, PathBuffers paths)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	if (i >= count) return;

	int2 pixel = pixelXY[i];
	const uint32_t pixelIndex = (uint32_t)pixel.y * (uint32_t)params.width + (uint32_t)pixel.x;
	const Strata strata = path_strata<STRAT>(params, paths, i);
	uint32_t key = STRAT ? stratified_series(params.seed, pixelIndex, sampleIndex[i] / (uint32_t)params.extend) // Distribution.BeginSeries per epoch
	                     : sample_key(params.seed, pixelIndex, sampleIndex[i]);

	vec2 shift = draw2d<STRAT>(key, strata, 0u); // CameraSample.Create, CameraSample.cs:19-23
	vec2 lens = draw2d<STRAT>(key, strata, 2u);

	vec3 origin, direction;
	camera_spawn(scene.camera, params.width, params.height, pixel.x, pixel.y, shift, lens, origin, direction);

	stream_store(paths.rayQueue[0] + i * 2u, make_float4(origin.x, origin.y, origin.z, direction.x));
	stream_store(paths.rayQueue[0] + i * 2u + 1u, make_float4(direction.y, direction.z, kInfinity, __uint_as_float(ECHO_TOKEN_EMPTY)));
	stream_store(paths.rayPath[0] + i, i);
	if (paths.rayLayers[0]) store_layers(paths.rayLayers[0], i, no_layers());
	stream_store(paths.energy + i, make_float4(1.0f, 1.0f, 1.0f, 0.0f));
	stream_store(paths.result + i, make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(MODE_FIRST << 16)));
	stream_store(paths.key + i, key);
}

ECHO_DEVICE int classify_material(const DeviceScene& scene, uint32_t materialIndex)
{
	const float4* p = scene.materials + (size_t)materialIndex * 4;
	uint32_t type = __float_as_uint(__ldg(p).x);

	for (int level = 0; level < 4 && type == ECHO_MATERIAL_ONESIDED; level++)
	{
		materialIndex = __float_as_uint(__ldg(p + 3).w);
		p = scene.materials + (size_t)materialIndex * 4;
		type = __float_as_uint(__ldg(p).x);
	}

	switch (type)
	{
		case ECHO_MATERIAL_DIFFUSE: return CLASS_DIFFUSE;
		case ECHO_MATERIAL_DIELECTRIC:
		{
			// Dielectric.Scatter builds SpecularFresnel iff both alphas are specular (Dielectric.cs:29-47, IMicrofacet.cs:43-51); a textured
			// roughness is only known per hit, so such materials stay in the class that carries both kinds
			if (scene.textureCount != 0u && __ldg(scene.materialTextures + (size_t)materialIndex * 2).z != ECHO_TEXTURE_NONE) return CLASS_DIELECTRIC;
			float4 second = __ldg(p + 1); // albedo.zw, roughness.xy
			bool specularX, specularY;
			microfacet_alpha(second.z, specularX);
			microfacet_alpha(second.w, specularY);
			return specularX && specularY ? CLASS_SMOOTH : CLASS_DIELECTRIC;
		}
		case ECHO_MATERIAL_COATED_DIFFUSE: return CLASS_DIELECTRIC; // shares the GlossyReflection<TR, RealFresnel> code
		case ECHO_MATERIAL_CONDUCTOR: return CLASS_CONDUCTOR;
		default: return CLASS_TERMINAL;
	}
}

// Path.Advance's scene.Trace (PathTracedEvaluator.cs:261-271 -> PreparedScene.cs:66-75) over the compacted ray queue
struct ExtendIO
{
	const float4* __restrict__ rays;
	float4* __restrict__ hits;

	ECHO_DEVICE const float4* ray_pointer(uint32_t index) const { return rays + (size_t)index * 2; }
	ECHO_DEVICE float4* prepared_pointer(uint32_t index) const { return hits + index; }

	ECHO_DEVICE void store_closest(uint32_t index, bool hit, uint32_t token, float distance, vec2 uv, float limit) const
	{
		stream_store(hits + index, make_float4(__uint_as_float(hit ? token : ECHO_TOKEN_EMPTY), hit ? distance : limit, uv.x, uv.y));
	}

	ECHO_DEVICE void store_any(uint32_t, bool) const {}
};

// the instance layers of the wavefront's queues, in the IO form the instanced traversal core asks for
struct ExtendLayersIO : ExtendIO
{
	const uint4* __restrict__ rayLayers;
	uint4* __restrict__ hitLayers;

	ECHO_DEVICE uint32_t load_ignore_layers(uint32_t index, uint32_t* tokens) const
	{
		PathLayers layers = load_layers(rayLayers, index);
		for (uint32_t k = 0; k < ECHO_MAX_INSTANCE_LAYERS; k++) tokens[k] = layers.tokens[k];
		return min(layers.count, ECHO_MAX_INSTANCE_LAYERS);
	}

	ECHO_DEVICE void store_hit_layers(uint32_t index, bool hit, const uint32_t* tokens, uint32_t count) const
	{
		PathLayers layers = no_layers();
		if (hit)
		{
			layers.count = count;
			for (uint32_t k = 0; k < count; k++) layers.tokens[k] = tokens[k];
		}
		store_layers(hitLayers, index, layers);
	}
};

template<bool PACKS>
using ExtendIOFor = std::conditional_t<PACKS, ExtendLayersIO, ExtendIO>;

// PACKS: through the instanced packs, with the ignore hierarchy's instance layers in and the hit's instance layers out
template<int STACK, bool PACKS>
__global__ void __launch_bounds__(kTraverseBlock, PACKS ? ECHO_INST_MIN_BLOCKS : ECHO_MIN_BLOCKS) extend_kernel(DeviceScene scene, ExtendIOFor<PACKS> io, const uint32_t* __restrict__ queueCount,
                                                                                                               unsigned long long* __restrict__ nextRay)
{
	__shared__ float4 stagedRays[kTraverseBlock * kStagedFloat4];
	persistent_traverse<STACK, false, PACKS>(scene, io, *queueCount, nextRay, stagedRays);
	persistent_finish(nextRay);
}

// Narrow wavefronts (late bounces) have fewer rays than resident lanes: work replacement has nothing to replace with and
// the launch is bound by the latency of its longest ray, so the leaner one-thread-per-ray loop is used instead.
template<int STACK, bool PACKS, bool COUNT>
__global__ void __launch_bounds__(kBlock) extend_narrow_kernel(DeviceScene scene, ExtendIOFor<PACKS> io, const uint32_t* __restrict__ queueCount, unsigned long long* __restrict__ stats)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	VisitCounts local = { 0u, 0u, 0u };

	if (i < *queueCount)
	{
		float4 a = io.rays[i * 2u], b = io.rays[i * 2u + 1u];
		float distance = b.z;
		uint32_t token = ECHO_TOKEN_EMPTY;
		vec2 uv = { 0.0f, 0.0f };
		PathLayers hitLayers = no_layers();
		bool hit;

		if constexpr (PACKS)
			hit = scene_trace_layers<STACK, COUNT>(scene, { a.x, a.y, a.z }, { a.w, b.x, b.y }, __float_as_uint(b.w), load_layers(io.rayLayers, i),
			                                       distance, token, uv, hitLayers, COUNT ? &local : nullptr);
		else hit = scene_trace<STACK, COUNT>(scene, { a.x, a.y, a.z }, { a.w, b.x, b.y }, __float_as_uint(b.w), distance, token, uv, COUNT ? &local : nullptr);

		io.store_closest(i, hit, token, distance, uv, b.z);
		if constexpr (PACKS) store_layers(io.hitLayers, i, hit ? hitLayers : no_layers());
	}

	if (COUNT) visit_flush(stats, STAT_NODE_VISITS, local);
}

// The material-class sort: one thread per traced ray appends its slot to the queue of the class it hit. The appends of a whole CTA
// are gathered in shared memory first and reach each global class counter as ONE atomic per CTA: with one atomic per warp the
// kernel was bound by the serialisation of a quarter million same-address atomics per launch (IPC 0.37, 0.38 ms for 8.3 M rays).
constexpr int kClassifyBlock = 512;

template<bool INST>
__global__ void __launch_bounds__(kClassifyBlock) classify_kernel(DeviceScene scene, const uint32_t* __restrict__ queueCount, uint32_t* __restrict__ classCounts, PathBuffers paths)
{
	__shared__ uint32_t blockCount[CLASS_COUNT], blockBase[CLASS_COUNT];
	if (threadIdx.x < CLASS_COUNT) blockCount[threadIdx.x] = 0u;
	__syncthreads();

	uint32_t i = blockIdx.x * kClassifyBlock + threadIdx.x;
	bool active = i < *queueCount;
	int shadeClass = -1;

	if (active)
	{
		uint32_t token = __float_as_uint(stream_load(paths.hitQueue + i).x);
		shadeClass = CLASS_MISS;

		if (token != ECHO_TOKEN_EMPTY)
		{
			// the hit's pack and the swatch of its placement (PreparedScene.Interact: instance.swatch[info.material])
			PackInfo info = whole_scene_pack(scene);
			uint32_t materialOffset = 0u;

			if (INST)
			{
				PathLayers layers = load_layers(paths.hitLayers, i);
				info = load_pack_info(scene, 0u);
				materialOffset = info.materialOffset;

				for (uint32_t k = 0; k < layers.count; k++)
				{
					float4 tail = __ldg(instance_data(scene, info.instanceOffset + token_index(layers.tokens[k])) + 6);
					materialOffset = __float_as_uint(tail.w);
					info = load_pack_info(scene, __float_as_uint(tail.z));
				}
			}

			shadeClass = classify_material(scene, materialOffset + geometry_material(scene, info, token));
		}
	}

	stat_add(paths.stats, STAT_TRACE_QUERIES, active);

	// position inside the CTA's share of each class queue: one shared-memory atomic per warp and class
	const uint32_t lane = threadIdx.x & 31u;
	uint32_t offset = 0u;

#pragma unroll
	for (int c = 0; c < CLASS_COUNT; c++)
	{
		uint32_t mask = __ballot_sync(0xFFFFFFFFu, shadeClass == c);
		if (mask == 0u) continue;
		uint32_t warpBase = 0u;
		int leader = __ffs(mask) - 1;
		if ((int)lane == leader) warpBase = atomicAdd(&blockCount[c], (uint32_t)__popc(mask));
		warpBase = __shfl_sync(0xFFFFFFFFu, warpBase, leader);
		if (shadeClass == c) offset = warpBase + (uint32_t)__popc(mask & ((1u << lane) - 1u));
	}

	__syncthreads();
	if (threadIdx.x < CLASS_COUNT && blockCount[threadIdx.x] != 0u) blockBase[threadIdx.x] = atomicAdd(classCounts + threadIdx.x, blockCount[threadIdx.x]);
	__syncthreads();

	if (shadeClass >= 0) stream_store(paths.classQueue[shadeClass] + blockBase[shadeClass] + offset, i);
}

// ---- PreparedScene.Interact (PreparedScene.cs:95-105) + GeometryCollection.GetContactInfo (:200-232) + material.Scatter ----
// What a hit becomes: its shading point, material and BSDF. Every evaluator shades its hits through this one function.
struct Contact
{
	SurfacePoint point;
	vec3 shadeNormal, outgoing;
	uint32_t materialIndex;
	vec2 texcoord;
	MaterialRecord material;
	Bsdf bsdf;
};

template<bool INST>
ECHO_DEVICE void interact(const DeviceScene& scene, uint32_t token, vec2 uv, float distance, const PathLayers& layers, vec3 origin, vec3 direction, Contact& c)
{
	Layer layer = find_layer<INST>(scene, layers); // FindLayer, :97
	const bool textured = INST && scene.textureCount != 0u;
	vec3 infoNormal, infoShading;
	c.texcoord = { 0.0f, 0.0f };

	if (token_type(token) == ECHO_TOKEN_TYPE_TRIANGLE)
	{
		TriangleData triangle = load_triangle(scene, layer.info.triangleOffset + token_index(token));
		c.materialIndex = layer.materialOffset + triangle.material; // instance.swatch[info.material], :102
		infoNormal = triangle_normal(triangle);
		infoShading = triangle_shading_normal(triangle, uv);
		if (textured) c.texcoord = triangle_texcoord(scene, layer.info.triangleOffset + token_index(token), uv);
	}
	else
	{
		c.materialIndex = layer.materialOffset + __ldg(scene.sphereMaterial + layer.info.sphereOffset + token_index(token));
		infoNormal = infoShading = sphere_normal(uv);
		if (textured) c.texcoord = sphere_texcoord(uv);
	}

	c.point.position = direction * max_net(distance, kEpsilon) + origin; // TraceQuery.Position, TraceQuery.cs:76-82
	c.point.normal = normalized(transform_direction(layer.inverse, infoNormal)); // :100-101 (the identity without layers)
	c.shadeNormal = normalized(transform_direction(layer.inverse, infoShading));
	c.outgoing = -direction;
	if (textured) apply_normal_mapping(scene, c.materialIndex, c.texcoord, c.shadeNormal); // GeometryShade's constructor, GeometryShade.cs:17

	c.material = load_material(scene, c.materialIndex);
	material_scatter<INST>(scene, c.material, c.outgoing, c.point.normal, c.shadeNormal, c.bsdf, c.materialIndex, c.texcoord);
}

// What one loop body of PathTracedEvaluator.Evaluate produces for a path: statistics, the next ray if the path goes on, the
// shadow ray of its light sample if one is needed.
struct ShadeOut
{
	bool statInfinite = false, statBounce = false, statSpecular = false, statMis = false, statSampled = false, statChecked = false;
	bool survive = false, shadow = false;
	uint32_t id = 0u;
	float4 nextOrigin = make_float4(0, 0, 0, 0), nextDirection = make_float4(0, 0, 0, 0), nextEnergy = make_float4(0, 0, 0, 0);
	float4 shadowOrigin = make_float4(0, 0, 0, 0), shadowDirection = make_float4(0, 0, 0, 0), shadowValue = make_float4(0, 0, 0, 0);
	PathLayers hitLayers = no_layers(); // the instance layers of the hit: the ignore hierarchy of both spawned rays
};

// One loop body of PathTracedEvaluator.Evaluate for the path whose ray sits in slot `raySlot` of the current queue and whose hit
// record is in hitQueue[raySlot]. CLASS / KINDS prune the code to what a material-class queue can contain; CLASS < 0 keeps
// everything (the tail kernel), `missed` then says whether the ray hit anything.
template<int CLASS, uint32_t KINDS, bool INST, bool STRAT, bool COUNT = false>
ECHO_DEVICE void shade_body(const DeviceScene& scene, const EchoRenderParams& params, const PathBuffers& paths, int current, uint32_t raySlot, bool missed, ShadeOut& o)
{
	bool &statInfinite = o.statInfinite, &statBounce = o.statBounce, &statSpecular = o.statSpecular, &statMis = o.statMis;
	bool &statSampled = o.statSampled, &statChecked = o.statChecked, &survive = o.survive, &shadow = o.shadow;
	uint32_t& id = o.id;
	float4 &nextOrigin = o.nextOrigin, &nextDirection = o.nextDirection, &nextEnergy = o.nextEnergy;
	float4 &shadowOrigin = o.shadowOrigin, &shadowDirection = o.shadowDirection, &shadowValue = o.shadowValue;
	PathLayers& hitLayers = o.hitLayers;
	(void)missed;

	id = stream_load(paths.rayPath[current] + raySlot);

	float4 rayA = stream_load(paths.rayQueue[current] + raySlot * 2u), rayB = stream_load(paths.rayQueue[current] + raySlot * 2u + 1u);
	float4 energy4 = stream_load(paths.energy + id);
	float4 result4 = stream_load(paths.result + id);

	vec3 direction = { rayA.w, rayB.x, rayB.y };
	rgb energy = as_rgb(energy4);
	rgb result = as_rgb(result4);
	float scatterPdfPrevious = energy4.w;
	uint32_t state = __float_as_uint(result4.w);
	uint32_t bounces = state & 0xFFFFu, mode = state >> 16;

	if (CLASS == CLASS_MISS || (CLASS < 0 && missed))
	{
		// no intersection: PathTracedEvaluator.cs:48-52 (first), :112-130 (MIS), :137-143 (fallback)
		statInfinite = true;

		if (mode == MODE_FIRST) result = evaluate_infinite(scene, direction, true);
		else if (mode == MODE_NO_MIS) result = result + energy * evaluate_infinite(scene, direction, false);
		else
		{
			SurfacePoint oldPoint = { xyz(stream_load(paths.oldPosition + id)), xyz(stream_load(paths.oldNormal + id)) };
			(void)oldPoint;

			for (uint32_t index = 0; index < scene.infiniteLightCount; index++)
			{
				InfiniteLight light = load_infinite(scene, index);
				if (light.delta) continue; // "Skip delta lights; they do not like MIS", :118

				float pdf = scene.infinitePdf * infinite_pdf(scene, light, direction); // ProbabilityMass * light.ProbabilityDensity, :121-122
				if (!positive(pdf)) continue;
				float weight = power_heuristic(scatterPdfPrevious, pdf);
				result = result + energy * (infinite_evaluate(scene, light, direction) * weight);
			}
		}

		stream_store(paths.result + id, make4(result, result4.w));
	}
	else
	{
		float4 hit4 = stream_load(paths.hitQueue + raySlot);
		uint32_t token = __float_as_uint(hit4.x);

		if (INST) hitLayers = load_layers(paths.hitLayers, raySlot);
		Contact contact;
		interact<INST>(scene, token, { hit4.z, hit4.w }, hit4.y, hitLayers, xyz(rayA), direction, contact);
		const SurfacePoint& point = contact.point;
		const vec3 &shadeNormal = contact.shadeNormal, &outgoing = contact.outgoing;
		const MaterialRecord& material = contact.material;
		const Bsdf& bsdf = contact.bsdf;

		// ---- emission of the new vertex: ContributeEmissive (:305-311), MIS-weighted after a MIS bounce (:96-109) ----
		if ((CLASS == CLASS_TERMINAL || CLASS < 0) && material.type == ECHO_MATERIAL_EMISSIVE && positive(emissive_power(material)))
		{
			float weight = 1.0f;
			bool contribute = true;

			if (mode == MODE_MIS)
			{
				SurfacePoint oldPoint = { xyz(stream_load(paths.oldPosition + id)), xyz(stream_load(paths.oldNormal + id)) };
				float pmf = scene_probability_mass<INST, COUNT>(scene, token, hitLayers, oldPoint);
				contribute = positive(pmf);

				if (contribute)
				{
					float pdf = scene_light_pdf<INST>(scene, token, hitLayers, oldPoint, direction);
					contribute = positive(pdf);
					if (contribute) weight = power_heuristic(scatterPdfPrevious, pmf * pdf);
				}
			}

			if (contribute)
			{
				rgb emitted = dot(outgoing, point.normal) > 0.0f ? material_emission(material) : make_rgb(0.0f);
				result = result + energy * (emitted * weight);
			}
		}

		// ---- the loop body: `for (int depth = 0; depth < BounceLimit; depth++)`, :57 ----
		if (bounces < (uint32_t)params.bounceLimit)
		{
			uint32_t key = stream_load(paths.key + id);
			const Strata strata = path_strata<STRAT>(params, paths, id);
			uint32_t dimension = 4u + 6u * bounces;
			vec2 bounceSample = draw2d<STRAT>(key, strata, dimension);
			float survivalSample = draw1d<STRAT>(key, strata, dimension + 2u);
			float lightSample = draw1d<STRAT>(key, strata, dimension + 3u);
			vec2 radiantSample = draw2d<STRAT>(key, strata, dimension + 4u);

			// Bounce, :326-354
			vec3 incident;
			int selectedType;
			Sampled bounced = bsdf_sample<KINDS>(bsdf, outgoing, bounceSample, incident, selectedType);
			rgb scatter = bounced.content * abs_bits(dot(incident, shadeNormal));
			float scatterPdf = bounced.pdf;
			statBounce = true;

			bool mis = false;

			if (!positive(scatterPdf) || (selectedType & FT_SPECULAR)) statSpecular = true;
			else
			{
				// ---- ImportanceSampleRadiant, :162-207 ----
				float lightPdf;
				PathLayers lightLayers;
				uint32_t light = scene_pick<INST, COUNT>(scene, point, lightSample, lightPdf, lightLayers);

				if (positive(lightPdf))
				{
					vec3 lightIncident;
					float travel;
					Sampled radiantSampled = scene_sample_light<INST>(scene, light, lightLayers, point, radiantSample, lightIncident, travel);
					rgb radiant = radiantSampled.content;

					float pdf = lightPdf * radiantSampled.pdf;
					mis = token_is_area_light(light);

					if (positive(pdf) && !is_zero(radiant))
					{
						statSampled = true;

						rgb lightScatter = bsdf_evaluate<KINDS>(bsdf, outgoing, lightIncident);
						lightScatter = lightScatter * abs_bits(dot(lightIncident, shadeNormal));

						if (!is_zero(lightScatter))
						{
							statChecked = true;

							radiant = radiant * (lightScatter / pdf);
							if (mis) radiant = radiant * power_heuristic(pdf, bsdf_pdf<KINDS>(bsdf, outgoing, lightIncident));

							shadow = true;
							shadowOrigin = make_float4(point.position.x, point.position.y, point.position.z, lightIncident.x);
							shadowDirection = make_float4(lightIncident.y, lightIncident.z, travel, __uint_as_float(token)); // SpawnOcclude: ignore = hit token
							shadowValue = make4(energy * radiant, __uint_as_float(id));
						}
					}
				}
			}

			// ---- Path.Continue, :282-293 ----
			if (positive(scatterPdf))
			{
				energy = energy * (scatter / scatterPdf);

				float rate = clamp01(params.survivability * luminance(energy)); // RussianRoulette, :313-320

				if (!(survivalSample >= rate))
				{
					energy = energy / rate;
					survive = true;

					if (mis && !statSpecular)
					{
						statMis = true;
						stream_store(paths.oldPosition + id, make4(point.position, 0.0f));
						stream_store(paths.oldNormal + id, make4(point.normal, 0.0f));
					}

					uint32_t nextMode = (mis && !statSpecular) ? MODE_MIS : MODE_NO_MIS;
					nextOrigin = make_float4(point.position.x, point.position.y, point.position.z, incident.x);
					nextDirection = make_float4(incident.y, incident.z, kInfinity, __uint_as_float(token)); // SpawnTrace: ignore = hit token, TraceQuery.cs:88
					nextEnergy = make4(energy, scatterPdf);
					result4.w = __uint_as_float((bounces + 1u) | (nextMode << 16));
				}
			}
		}

		stream_store(paths.result + id, make4(result, result4.w));
		if (survive) stream_store(paths.energy + id, nextEnergy);
	}
}

// One loop body of PathTracedEvaluator.Evaluate for every path in a material-class queue.
#ifndef ECHO_SHADE_MIN_BLOCKS
#define ECHO_SHADE_MIN_BLOCKS 6 // resident CTAs per SM asked of the shading kernels: 80 registers and a few hundred bytes of spills instead of 100-110 registers at 4 CTAs; no target / 5 / 6 / 7 / 8: C3 474 / 477 / 483 / 483 / 485, C4 329 / 338 / 342 / 345 / 347, textured 719 / 721 / 733 / 725 / 712 M samples/s (variants/ab15.sh)
#endif
// what a shading thread leaves behind: its next ray and its shadow ray appended to their queues, its statistics (every lane of the warp calls)
template<bool INST>
ECHO_DEVICE void shade_emit(const PathBuffers& paths, int current, const ShadeOut& o)
{
	const bool survive = o.survive, shadow = o.shadow;
	uint32_t nextSlot = queue_slot(paths.counters + COUNTER_NEXT, survive);

	if (survive)
	{
		stream_store(paths.rayQueue[current ^ 1] + nextSlot * 2u, o.nextOrigin);
		stream_store(paths.rayQueue[current ^ 1] + nextSlot * 2u + 1u, o.nextDirection);
		stream_store(paths.rayPath[current ^ 1] + nextSlot, o.id);
		if (INST) store_layers(paths.rayLayers[current ^ 1], nextSlot, o.hitLayers);
	}

	uint32_t shadowSlot = queue_slot(paths.counters + COUNTER_SHADOW, shadow);

	if (shadow)
	{
		stream_store(paths.shadowQueue + shadowSlot * 2u, o.shadowOrigin);
		stream_store(paths.shadowQueue + shadowSlot * 2u + 1u, o.shadowDirection);
		stream_store(paths.shadowValue + shadowSlot, o.shadowValue);
		if (INST) store_layers(paths.shadowLayers, shadowSlot, o.hitLayers);
	}

	stat_add(paths.stats, STAT_LIGHT_EVALUATED_INFINITE, o.statInfinite);
	stat_add(paths.stats, STAT_BOUNCE_CREATED, o.statBounce);
	stat_add(paths.stats, STAT_BOUNCE_SPECULAR, o.statSpecular);
	stat_add(paths.stats, STAT_BOUNCE_MIS, o.statMis);
	stat_add(paths.stats, STAT_LIGHT_SAMPLED, o.statSampled);
	stat_add(paths.stats, STAT_LIGHT_OCCLUSION_CHECKED, o.statChecked);
}

template<int CLASS, uint32_t KINDS, bool INST, bool STRAT>
__global__ void __launch_bounds__(kBlock, ECHO_SHADE_MIN_BLOCKS) shade_kernel(DeviceScene scene, EchoRenderParams params, const uint32_t* __restrict__ queue,
                                                      const uint32_t* __restrict__ queueCount, PathBuffers paths, int current)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	bool active = i < *queueCount;

	ShadeOut o;
	if (active) shade_body<CLASS, KINDS, INST, STRAT>(scene, params, paths, current, stream_load(queue + i), false, o);
	shade_emit<INST>(paths, current, o);
}

// Counted passes (ECHO_EVALUATOR_COUNT_VISITS) shade every ray of the queue with this one kernel instead of the six class kernels:
// the all-lobes body the tail kernel uses (same operations per path, same bits), instantiated with the light-tree visit counter, so
// the class kernels of ordinary renders carry no counting code at all (a never-taken branch in the light-tree descent cost the
// diffuse class 2.4x on the instanced scene: registers at the 80-register cap).
template<bool INST, bool STRAT>
__global__ void __launch_bounds__(kBlock) shade_counted_kernel(DeviceScene scene, EchoRenderParams params, const uint32_t* __restrict__ rayCount, PathBuffers paths, int current)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	bool active = i < *rayCount;

	ShadeOut o;
	if (active) shade_body<-1, KINDS_ALL, INST, STRAT, true>(scene, params, paths, current, i, __float_as_uint(paths.hitQueue[i].x) == ECHO_TOKEN_EMPTY, o);
	shade_emit<INST>(paths, current, o);
}

// scene.Occlude of ImportanceSampleRadiant (:196-197); unoccluded pending contributions go into Path.Result (:80-84).
// A path has at most one shadow ray per bounce, so the read-modify-write of its result needs no atomic.
struct ShadowIO
{
	const float4* __restrict__ rays;
	const float4* __restrict__ values;
	float4* __restrict__ result;
	uint32_t passed;

	ECHO_DEVICE const float4* ray_pointer(uint32_t index) const { return rays + (size_t)index * 2; }
	ECHO_DEVICE float4* prepared_pointer(uint32_t) const { return nullptr; }
	ECHO_DEVICE void store_closest(uint32_t, bool, uint32_t, float, vec2, float) const {}

	ECHO_DEVICE void store_any(uint32_t index, bool occluded)
	{
		if (occluded) return;
		float4 value = stream_load(values + index);
		uint32_t id = __float_as_uint(value.w);
		float4 total = stream_load(result + id);
		total.x += value.x;
		total.y += value.y;
		total.z += value.z;
		stream_store(result + id, total);
		++passed;
	}
};

struct ShadowLayersIO : ShadowIO
{
	const uint4* __restrict__ shadowLayers;

	ECHO_DEVICE uint32_t load_ignore_layers(uint32_t index, uint32_t* tokens) const
	{
		PathLayers layers = load_layers(shadowLayers, index);
		for (uint32_t k = 0; k < ECHO_MAX_INSTANCE_LAYERS; k++) tokens[k] = layers.tokens[k];
		return min(layers.count, ECHO_MAX_INSTANCE_LAYERS);
	}

	ECHO_DEVICE void store_hit_layers(uint32_t, bool, const uint32_t*, uint32_t) const {}
};

template<bool PACKS>
using ShadowIOFor = std::conditional_t<PACKS, ShadowLayersIO, ShadowIO>;

template<int STACK, bool PACKS>
__global__ void __launch_bounds__(kTraverseBlock, PACKS ? ECHO_INST_MIN_BLOCKS : ECHO_MIN_BLOCKS) shadow_kernel(DeviceScene scene, ShadowIOFor<PACKS> io, const uint32_t* __restrict__ shadowCount,
                                                                                                               unsigned long long* __restrict__ nextRay, unsigned long long* __restrict__ stats)
{
	__shared__ float4 stagedRays[kTraverseBlock * kStagedFloat4];
	io.passed = 0u;
	persistent_traverse<STACK, true, PACKS>(scene, io, *shadowCount, nextRay, stagedRays);
	persistent_finish(nextRay);

	warp_add(stats, STAT_LIGHT_OCCLUSION_PASSED, io.passed);
	if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(stats + STAT_OCCLUDE_QUERIES, (unsigned long long)*shadowCount);
}

template<int STACK, bool PACKS, bool COUNT>
__global__ void __launch_bounds__(kBlock) shadow_narrow_kernel(DeviceScene scene, ShadowIOFor<PACKS> io, const uint32_t* __restrict__ shadowCount, unsigned long long* __restrict__ stats)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	bool active = i < *shadowCount;
	io.passed = 0u;
	VisitCounts local = { 0u, 0u, 0u };

	if (active)
	{
		float4 a = io.rays[i * 2u], b = io.rays[i * 2u + 1u];
		bool occluded;

		if constexpr (PACKS)
			occluded = scene_occlude_layers<STACK, COUNT>(scene, { a.x, a.y, a.z }, { a.w, b.x, b.y }, __float_as_uint(b.w), load_layers(io.shadowLayers, i), b.z, COUNT ? &local : nullptr);
		else occluded = scene_occlude<STACK, COUNT>(scene, { a.x, a.y, a.z }, { a.w, b.x, b.y }, __float_as_uint(b.w), b.z, COUNT ? &local : nullptr);

		io.store_any(i, occluded);
	}

	stat_add(stats, STAT_OCCLUDE_QUERIES, active);
	stat_add(stats, STAT_LIGHT_OCCLUSION_PASSED, io.passed != 0u);
	if (COUNT) visit_flush(stats, STAT_NODE_VISITS, local);
}

// ---- Scalars.AlmostEquals (Scalars.cs:153-168) and Float3.Equals (Float3.cs:369) ----
ECHO_DEVICE bool almost_equals(float value, float other)
{
	if (value == other) return true;
	const float epsilon = 1E-5f, normal = 1.17549435E-38f; // (1L << 23) * float.Epsilon

	float difference = fabsf(value - other);
	if (value == 0.0f || other == 0.0f || difference < normal) return difference < epsilon * normal;

	float sum = fabsf(value) + fabsf(other);
	float capped = sum != sum ? sum : (sum < 3.40282347E+38f ? sum : 3.40282347E+38f); // Math.Min(sum, float.MaxValue)
	return difference < epsilon * capped;
}

ECHO_DEVICE bool float3_equals(vec3 a, vec3 b) { return almost_equals(a.x, b.x) && almost_equals(a.y, b.y) && almost_equals(a.z, b.z); }

constexpr uint32_t KINDS_AUXILIARY = kind_bit(BSDF_EMPTY) | kind_bit(BSDF_DIELECTRIC_SPECULAR) | kind_bit(BSDF_CONDUCTOR_SPECULAR) | kind_bit(BSDF_INVISIBLE);
constexpr int kAuxiliaryBounceCap = 1024; // both evaluators loop `while (scene.Trace(...))`; the cap only guards the GPU against a hall of mirrors (the oracle has the same one)

// AlbedoEvaluator.Evaluate (AlbedoEvaluator.cs:18-55) / NormalDepthEvaluator.Evaluate (NormalDepthEvaluator.cs:20-60): one
// thread per sample follows purely specular bounces from the camera ray raygen_kernel left in rayQueue[0] and reports the
// first other surface. These passes run at a few samples per pixel for the denoiser: a plain loop, no wavefront.
template<int STACK, bool INST, bool STRAT>
__global__ void __launch_bounds__(kBlock) auxiliary_kernel(DeviceScene scene, EchoRenderParams params, uint32_t count, PathBuffers paths, float4* __restrict__ out)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	if (i >= count) return;

	float4 rayA = paths.rayQueue[0][i * 2u], rayB = paths.rayQueue[0][i * 2u + 1u];
	vec3 origin = xyz(rayA), direction = { rayA.w, rayB.x, rayB.y };
	const vec3 cameraDirection = direction;
	const uint32_t key = paths.key[i];
	const Strata strata = path_strata<STRAT>(params, paths, i);
	const int kind = params.evaluator & ECHO_EVALUATOR_KIND_MASK;
	const bool divergeOnce = (params.evaluator & ECHO_EVALUATOR_DIVERGE_ONCE) != 0;

	uint32_t dimension = 4u; // after CameraSample's four (CameraSample.cs:19-23); one Next2D per specular bounce
	uint32_t ignore = ECHO_TOKEN_EMPTY;
	PathLayers ignoreLayers = no_layers();
	bool direct = true; // whether the path is still going in its original direction
	bool exited = false;
	float depth = 0.0f;
	float4 result = make_float4(0.0f, 0.0f, 0.0f, 0.0f);

	for (int bounce = 0; bounce < kAuxiliaryBounceCap && !exited; bounce++)
	{
		float distance = kInfinity;
		uint32_t token = ECHO_TOKEN_EMPTY;
		vec2 uv = { 0.0f, 0.0f };
		PathLayers hitLayers = no_layers();
		bool hit;

		if (INST && scene.packCount != 0u) hit = scene_trace_layers<STACK, false>(scene, origin, direction, ignore, ignoreLayers, distance, token, uv, hitLayers, nullptr);
		else hit = scene_trace<STACK, false>(scene, origin, direction, ignore, distance, token, uv, nullptr); // INST without packs is a textured scene: one pack

		if (!hit) break;

		Contact contact;
		interact<INST>(scene, token, uv, distance, hitLayers, origin, direction, contact);
		if (INST && scene.textureCount != 0u) resolve_material_textures(scene, contact.materialIndex, contact.texcoord, contact.material); // (RGB128)material.SampleAlbedo(contact)

		// Exit(): (RGB128)material.SampleAlbedo(contact) / new NormalDepth128(contact.shade.Normal, depth).ToFloat4()
		auto leave = [&]()
		{
			result = kind == ECHO_EVALUATOR_ALBEDO ? make_float4(contact.material.albedo[0], contact.material.albedo[1], contact.material.albedo[2], 0.0f)
			                                       : make_float4(contact.shadeNormal.x, contact.shadeNormal.y, contact.shadeNormal.z, depth);
			exited = true;
		};

		if (!direct) { leave(); continue; }
		if (kind == ECHO_EVALUATOR_NORMAL_DEPTH) depth += distance;

		if (((KINDS_AUXILIARY >> contact.bsdf.kind) & 1u) == 0u) { leave(); continue; } // bsdf.Count != bsdf.CountSpecular: not fully specular

		vec2 sample = draw2d<STRAT>(key, strata, dimension);
		dimension += 2u;

		vec3 incident;
		int selectedType;
		Sampled sampled = bsdf_sample<KINDS_AUXILIARY>(contact.bsdf, contact.outgoing, sample, incident, selectedType);
		if (!positive(sampled.pdf)) { leave(); continue; } // sample.NotPossible

		if (!float3_equals(incident, cameraDirection)) direct = false; // compared with the CAMERA ray's direction
		if (!divergeOnce && !direct) { leave(); continue; }

		// query.SpawnTrace(incident), TraceQuery.cs:88
		origin = contact.point.position;
		direction = incident;
		ignore = token;
		ignoreLayers = hitLayers;
	}

	if (!exited)
	{
		if (kind == ECHO_EVALUATOR_ALBEDO) result = make4(evaluate_infinite(scene, direction, direct), 0.0f); // scene.EvaluateInfinite(query.ray.direction, direct)
		else
		{
			if (direct) depth = scene.boundRadius * 2.0f; // negative direction and scene diameter for escaped rays
			result = make_float4(-cameraDirection.x, -cameraDirection.y, -cameraDirection.z, depth);
		}
	}

	out[i] = result;
}

// The tail of a wavefront: once only a few thousand paths are alive, every further bounce still costs nine dependent kernel
// launches whose duration no longer depends on the ray count. This kernel finishes those paths instead: one thread per path
// loops trace -> shade -> shadow -> next bounce until its path ends, with the same device functions as the wavefront
// kernels (shade_body with every lobe compiled in) and the same per-path buffers, so every path sees the same sequence of
// operations and its radiance keeps its bits.
template<int STACK, bool INST, bool STRAT>
__global__ void __launch_bounds__(kBlock) tail_kernel(DeviceScene scene, EchoRenderParams params, const uint32_t* __restrict__ queueCount, PathBuffers paths, int current)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	bool active = i < *queueCount;
	const bool packs = INST && scene.packCount != 0u;
	uint32_t counted[9] = { 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u }; // trace, occlude, passed, infinite, bounce, specular, mis, sampled, checked

	// The wavefront queued extend (and classify) of this iteration before it decided for the tail: the first hit of every path is
	// already in hitQueue (and counted), only later bounces are traced here.
	bool traced = true;

	while (active)
	{
		bool hit = false;

		if (traced)
		{
			hit = __float_as_uint(paths.hitQueue[i].x) != ECHO_TOKEN_EMPTY;
			traced = false;
		}
		else
		{
			// ---- Path.Advance: scene.Trace (PathTracedEvaluator.cs:261-271) ----
			float4 a = paths.rayQueue[current][i * 2u], b = paths.rayQueue[current][i * 2u + 1u];
			float distance = b.z;
			uint32_t token = ECHO_TOKEN_EMPTY;
			vec2 uv = { 0.0f, 0.0f };

			if (packs)
			{
				PathLayers hitLayers = no_layers();
				hit = scene_trace_layers<STACK, false>(scene, { a.x, a.y, a.z }, { a.w, b.x, b.y }, __float_as_uint(b.w), load_layers(paths.rayLayers[current], i),
				                                       distance, token, uv, hitLayers, nullptr);
				store_layers(paths.hitLayers, i, hit ? hitLayers : no_layers());
			}
			else hit = scene_trace<STACK, false>(scene, { a.x, a.y, a.z }, { a.w, b.x, b.y }, __float_as_uint(b.w), distance, token, uv, nullptr);

			paths.hitQueue[i] = make_float4(__uint_as_float(hit ? token : ECHO_TOKEN_EMPTY), hit ? distance : b.z, uv.x, uv.y);
			++counted[0];
		}

		// ---- one loop body of Evaluate ----
		ShadeOut o;
		shade_body<-1, KINDS_ALL, INST, STRAT>(scene, params, paths, current, i, !hit, o);
		counted[3] += o.statInfinite; counted[4] += o.statBounce; counted[5] += o.statSpecular;
		counted[6] += o.statMis; counted[7] += o.statSampled; counted[8] += o.statChecked;

		// ---- scene.Occlude of ImportanceSampleRadiant (:196-197) ----
		if (o.shadow)
		{
			vec3 origin = xyz(o.shadowOrigin), direction = { o.shadowOrigin.w, o.shadowDirection.x, o.shadowDirection.y };
			float travel = o.shadowDirection.z;
			uint32_t ignore = __float_as_uint(o.shadowDirection.w);
			bool occluded = packs ? scene_occlude_layers<STACK, false>(scene, origin, direction, ignore, o.hitLayers, travel, nullptr)
			                      : scene_occlude<STACK, false>(scene, origin, direction, ignore, travel, nullptr);

			++counted[1];

			if (!occluded)
			{
				uint32_t id = __float_as_uint(o.shadowValue.w);
				float4 total = paths.result[id];
				total.x += o.shadowValue.x;
				total.y += o.shadowValue.y;
				total.z += o.shadowValue.z;
				paths.result[id] = total;
				++counted[2];
			}
		}

		if (!o.survive) break;

		// query.SpawnTrace: the path keeps its slot of the current queue
		paths.rayQueue[current][i * 2u] = o.nextOrigin;
		paths.rayQueue[current][i * 2u + 1u] = o.nextDirection;
		if (INST) store_layers(paths.rayLayers[current], i, o.hitLayers);
	}

	const int slots[9] = { STAT_TRACE_QUERIES, STAT_OCCLUDE_QUERIES, STAT_LIGHT_OCCLUSION_PASSED, STAT_LIGHT_EVALUATED_INFINITE, STAT_BOUNCE_CREATED,
	                       STAT_BOUNCE_SPECULAR, STAT_BOUNCE_MIS, STAT_LIGHT_SAMPLED, STAT_LIGHT_OCCLUSION_CHECKED };

	// spelled out rather than nine warp_add calls, which compile this kernel to a different register allocation
#pragma unroll
	for (int k = 0; k < 9; k++)
	{
		uint32_t value = counted[k];
		for (int offset = 16; offset > 0; offset >>= 1) value += __shfl_down_sync(0xFFFFFFFFu, value, offset);
		if ((threadIdx.x & 31u) == 0u && value) atomicAdd(paths.stats + slots[k], (unsigned long long)value);
	}
}

// StandardNaiveEvaluator.Evaluate (StandardNaiveEvaluator.cs:16-55): `scatter * Evaluate(depth + 1) + emission`, no light sampling,
// no roulette. The recursion multiplies from the innermost bounce outwards, so the thread keeps every bounce's scatter and
// emission (bounceLimit <= 128) and folds them backwards once the path has ended.
constexpr int kNaiveBounceCap = 128;

template<int STACK, bool INST, bool STRAT>
__global__ void __launch_bounds__(kBlock) naive_kernel(DeviceScene scene, EchoRenderParams params, uint32_t count, PathBuffers paths, float4* __restrict__ out)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	bool active = i < count;
	uint32_t traced = 0u, bounced = 0u;

	if (active)
	{
		float4 rayA = paths.rayQueue[0][i * 2u], rayB = paths.rayQueue[0][i * 2u + 1u];
		vec3 origin = xyz(rayA), direction = { rayA.w, rayB.x, rayB.y };
		const uint32_t key = paths.key[i];
		const Strata strata = path_strata<STRAT>(params, paths, i);
		const bool packs = INST && scene.packCount != 0u;
		const int limit = params.bounceLimit < kNaiveBounceCap ? params.bounceLimit : kNaiveBounceCap;

		rgb scatters[kNaiveBounceCap], emissions[kNaiveBounceCap];
		int depth = 0;
		uint32_t ignore = ECHO_TOKEN_EMPTY;
		PathLayers ignoreLayers = no_layers();
		rgb value = make_rgb(0.0f);

		while (true)
		{
			bool hit = false;
			float distance = kInfinity;
			uint32_t token = ECHO_TOKEN_EMPTY;
			vec2 uv = { 0.0f, 0.0f };
			PathLayers hitLayers = no_layers();

			if (depth != limit)
			{
				++traced;

				if (packs) hit = scene_trace_layers<STACK, false>(scene, origin, direction, ignore, ignoreLayers, distance, token, uv, hitLayers, nullptr);
				else hit = scene_trace<STACK, false>(scene, origin, direction, ignore, distance, token, uv, nullptr);
			}

			if (!hit) // depth exhausted or escaped: scene.EvaluateInfinite(query.ray.direction, direct), :27-31
			{
				value = evaluate_infinite(scene, direction, depth == 0);
				break;
			}

			Contact contact;
			interact<INST>(scene, token, uv, distance, hitLayers, origin, direction, contact);

			// `material is Emissive emissive ? emissive.Emit(contact.point, contact.outgoing) : RGB128.Black`, :42
			rgb emission = contact.material.type == ECHO_MATERIAL_EMISSIVE && dot(contact.outgoing, contact.point.normal) > 0.0f ? material_emission(contact.material) : make_rgb(0.0f);

			vec2 sample = draw2d<STRAT>(key, strata, 4u + 2u * (uint32_t)depth);
			vec3 incident;
			int selectedType;
			Sampled sampled = bsdf_sample<KINDS_ALL>(contact.bsdf, contact.outgoing, sample, incident, selectedType);
			++bounced;

			if (!positive(sampled.pdf) || is_zero(sampled.content)) // "Exit if the BSDF sample is not promising", :46
			{
				value = emission;
				break;
			}

			scatters[depth] = (sampled.content / sampled.pdf) * abs_bits(dot(incident, contact.shadeNormal));
			emissions[depth] = emission;
			++depth;

			origin = contact.point.position; // query.SpawnTrace(incident)
			direction = incident;
			ignore = token;
			ignoreLayers = hitLayers;
		}

		for (int d = depth - 1; d >= 0; d--) value = scatters[d] * value + emissions[d]; // :54, innermost first
		out[i] = make4(value, 0.0f);
	}

	// both sums in one loop rather than two warp_add calls, which compile this kernel to a different register allocation
	for (int offset = 16; offset > 0; offset >>= 1)
	{
		traced += __shfl_down_sync(0xFFFFFFFFu, traced, offset);
		bounced += __shfl_down_sync(0xFFFFFFFFu, bounced, offset);
	}

	if ((threadIdx.x & 31u) == 0u)
	{
		if (traced) atomicAdd(paths.stats + STAT_TRACE_QUERIES, (unsigned long long)traced);
		if (bounced) atomicAdd(paths.stats + STAT_BOUNCE_CREATED, (unsigned long long)bounced);
	}
}

__global__ void __launch_bounds__(kBlock) finish_kernel(uint32_t count, PathBuffers paths, float4* __restrict__ out)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	if (i >= count) return;
	float4 result = paths.result[i];
	out[i] = make_float4(result.x, result.y, result.z, 0.0f);
}

// Iteration bookkeeping, launched right after classify of iteration k: the count of the ray queue that extend and classify of k
// just consumed (COUNTER_NEXT) is saved as the active count, and goes to the pipeline thread together with the class counts of k as
// one record in mapped pinned memory — class counts first, then {serial of k, rays} as ONE 8-byte store. The per-iteration counters
// are cleared for the shading kernels of k, and so is the other parity's set of class counts (consumed by the shading of k - 1).
__global__ void rotate_counters_kernel(uint32_t* counters, uint32_t* activeCount, unsigned long long* hostMirror, uint32_t serial, int parity)
{
	uint32_t rays = counters[COUNTER_NEXT];
	*activeCount = rays;

	volatile uint32_t* classMirror = reinterpret_cast<volatile uint32_t*>(hostMirror + 1);
	for (int c = 0; c < CLASS_COUNT; c++) classMirror[c] = counters[COUNTER_CLASS + parity * CLASS_COUNT + c];
	__threadfence_system();
	*reinterpret_cast<volatile unsigned long long*>(hostMirror) = ((unsigned long long)serial << 32) | (unsigned long long)rays;

	counters[COUNTER_NEXT] = 0u;
	counters[COUNTER_SHADOW] = 0u;
	for (int c = 0; c < CLASS_COUNT; c++) counters[COUNTER_CLASS + (parity ^ 1) * CLASS_COUNT + c] = 0u;
}

// ---- Kahan summation + Welford accumulation, Summation.cs:8-58 + Accumulator.cs:11-71 ----
struct Sum4
{
	float4 total, error;
};

ECHO_DEVICE float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
ECHO_DEVICE float4 sub4(float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
ECHO_DEVICE float4 mul4(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
ECHO_DEVICE float4 neg4(float4 a) { return make_float4(-a.x, -a.y, -a.z, -a.w); }

ECHO_DEVICE Sum4 sum_add(Sum4 s, float4 value) // Summation.cs:31-38
{
	float4 delta = sub4(value, s.error);
	float4 total = add4(s.total, delta);
	float4 error = sub4(sub4(total, s.total), delta);
	return { total, error };
}

ECHO_DEVICE Sum4 sum_add(Sum4 s, Sum4 value) // Summation.cs:42-51
{
	float4 error = add4(s.error, value.error);
	float4 delta = sub4(value.total, error);
	float4 total = add4(s.total, delta);
	error = sub4(sub4(total, s.total), delta);
	return { total, error };
}

ECHO_DEVICE Sum4 sum_scale(Sum4 s, float4 value) { return { mul4(s.total, value), mul4(s.error, value) }; } // Summation.cs:40
ECHO_DEVICE Sum4 sum_negate(Sum4 s) { return { neg4(s.total), neg4(s.error) }; }

// one thread per pixel walks its `extend` samples of this epoch in sample order (EvaluationOperation.cs:117-135)
__global__ void __launch_bounds__(kBlock) accumulate_kernel(EchoRenderParams params, uint32_t pixelCount, const uint32_t* __restrict__ activePixels,
                                                           const float4* __restrict__ samples, float4* __restrict__ accumulator, uint32_t* __restrict__ sampleCount,
                                                           uint32_t epoch, uint32_t* __restrict__ nextActive, uint32_t* __restrict__ counters, unsigned long long* __restrict__ stats)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	bool valid = i < pixelCount;
	bool again = false;
	uint32_t rejected = 0u;
	uint32_t pixel = 0u;

	if (valid)
	{
		pixel = activePixels[i];
		Sum4 average = { accumulator[pixel * 4u], accumulator[pixel * 4u + 1u] };
		Sum4 squared = { accumulator[pixel * 4u + 2u], accumulator[pixel * 4u + 3u] };
		uint32_t count = sampleCount[pixel];

		for (int s = 0; s < params.extend; s++)
		{
			float4 sample = samples[(size_t)i * params.extend + s];
			float sum = (sample.x + sample.y) + (sample.z + sample.w); // Float4.Sum

			if (!isfinite(sum)) // Accumulator.Add gate, Accumulator.cs:57
			{
				++rejected;
				continue;
			}

			++count;

			Sum4 delta = sum_add(average, neg4(sample));                       // average - sample
			float countR = rcp((float)count);
			average = sum_add(average, sum_negate(sum_scale(delta, make_float4(countR, countR, countR, countR)))); // average -= delta / count
			Sum4 after = sum_add(average, neg4(sample));
			squared = sum_add(squared, sum_scale(delta, after.total));         // squared += delta * (average - sample).Result
		}

		accumulator[pixel * 4u] = average.total;
		accumulator[pixel * 4u + 1u] = average.error;
		accumulator[pixel * 4u + 2u] = squared.total;
		accumulator[pixel * 4u + 3u] = squared.error;
		sampleCount[pixel] = count;

		// epoch loop condition, EvaluationOperation.cs:137; Accumulator.Noise (:28-51) with exact 1/x and 1/sqrt
		if (epoch < (uint32_t)params.maxEpoch)
		{
			if (epoch < (uint32_t)params.minEpoch) again = true;
			else if (count >= 2u)
			{
				float oneLess = (float)(count - 1u);
				oneLess *= oneLess * oneLess;

				float mean[4] = { average.total.x, average.total.y, average.total.z, average.total.w };
				float m2[4] = { squared.total.x, squared.total.y, squared.total.z, squared.total.w };
				float noiseMax = 0.0f;

				for (int c = 0; c < 4; c++)
				{
					float numerator = mean[c] * mean[c] * oneLess;
					float denominator = rcp(m2[c]);
					float noise = numerator != 0.0f ? rcp(__fsqrt_rn(numerator * denominator)) : 0.0f;
					if (c == 0 || noise > noiseMax) noiseMax = noise;
				}

				again = noiseMax > params.noiseThreshold;
			}
		}
	}

	uint32_t slot = queue_slot(counters + COUNTER_PIXELS, again);
	if (again) nextActive[slot] = pixel;

	if (valid)
	{
		atomicAdd(stats + STAT_SAMPLE_EVALUATED, (unsigned long long)params.extend);
		if (rejected) atomicAdd(stats + STAT_SAMPLE_REJECTED, (unsigned long long)rejected);
	}
}

// fills the per-slot (pixel, sample index) descriptors of one epoch from the active pixel list
__global__ void __launch_bounds__(kBlock) epoch_slots_kernel(EchoRenderParams params, uint32_t pixelCount, const uint32_t* __restrict__ activePixels,
                                                            const int2* __restrict__ batchPixelXY, uint32_t epoch, int2* __restrict__ pixelXY, uint32_t* __restrict__ sampleIndex)
{
	uint64_t i = (uint64_t)blockIdx.x * kBlock + threadIdx.x;
	uint64_t total = (uint64_t)pixelCount * params.extend;
	if (i >= total) return;

	uint32_t p = (uint32_t)(i / params.extend), s = (uint32_t)(i % params.extend);
	pixelXY[i] = batchPixelXY[activePixels[p]];
	sampleIndex[i] = (uint32_t)(params.epochOffset + (int)epoch - 1) * (uint32_t)params.extend + s;
}

// lays out the pixels of a batch of tiles; pixels outside the image are not listed
__global__ void __launch_bounds__(kBlock) batch_pixels_kernel(EchoRenderParams params, const int32_t* __restrict__ tileXY, uint32_t tileCount,
                                                             int2* __restrict__ batchPixelXY, uint32_t* __restrict__ activePixels, uint32_t* __restrict__ counters,
                                                             float4* __restrict__ accumulator, uint32_t* __restrict__ sampleCount)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	uint32_t perTile = (uint32_t)(params.tileSize * params.tileSize);
	bool inside = false;

	if (i < tileCount * perTile)
	{
		uint32_t tile = i / perTile, local = i % perTile;
		int px = tileXY[tile * 2u] * params.tileSize + (int)(local % (uint32_t)params.tileSize);
		int py = tileXY[tile * 2u + 1u] * params.tileSize + (int)(local / (uint32_t)params.tileSize);
		inside = px < params.width && py < params.height;

		batchPixelXY[i] = make_int2(px, py);
		accumulator[i * 4u] = accumulator[i * 4u + 1u] = accumulator[i * 4u + 2u] = accumulator[i * 4u + 3u] = make_float4(0, 0, 0, 0);
		sampleCount[i] = 0u;
	}

	uint32_t slot = queue_slot(counters + COUNTER_PIXELS, inside);
	if (inside) activePixels[slot] = i;
}

__global__ void __launch_bounds__(kBlock) resolve_tiles_kernel(EchoRenderParams params, uint32_t pixelTotal, const int2* __restrict__ batchPixelXY,
                                                              const float4* __restrict__ accumulator, const uint32_t* __restrict__ sampleCount,
                                                              float4* __restrict__ tilesOut, float4* __restrict__ frame, unsigned long long* __restrict__ stats)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	if (i >= pixelTotal) return;

	int2 pixel = batchPixelXY[i];
	bool inside = pixel.x < params.width && pixel.y < params.height;
	float4 value = inside ? accumulator[i * 4u] : make_float4(0, 0, 0, 0); // Accumulator.Value = average.Result

	if (tilesOut) tilesOut[i] = value;
	if (frame && inside)
	{
		// (mean * n, n) with n = samples accumulated, ADDED: frames of devices that rendered other tiles (zeros here) or other
		// epochs of the same pixel (sample sharding) sum to (sum of samples, count); exact whenever n is a power of two
		float weight = (float)sampleCount[i];
		float4& target = frame[(size_t)pixel.y * params.width + pixel.x];
		target = make_float4(target.x + value.x * weight, target.y + value.y * weight, target.z + value.z * weight, target.w + weight);
	}
	if (inside) atomicAdd(stats + STAT_PIXEL_EVALUATED, 1ull);
}

__global__ void __launch_bounds__(kBlock) frame_resolve_kernel(float4* frame, uint32_t count)
{
	uint32_t i = blockIdx.x * kBlock + threadIdx.x;
	if (i >= count) return;
	float4 value = frame[i];
	if (value.w > 0.0f) frame[i] = make_float4(div(value.x, value.w), div(value.y, value.w), div(value.z, value.w), 0.0f);
	else frame[i] = make_float4(0, 0, 0, 0);
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------

RenderState* render_state_create() { return new RenderState(); }

static void release(WorkerState* state)
{
	for (void* p : state->allocations) cudaFree(p);
	state->allocations.clear();
	state->paths.rayLayers[0] = state->paths.rayLayers[1] = state->paths.hitLayers = state->paths.shadowLayers = nullptr;
	state->capacity = 0;
	state->pixelCapacity = 0;
	state->tileCapacity = 0;
}

void render_state_destroy(RenderState* state)
{
	if (!state) return;

	for (WorkerState* worker : state->workers)
	{
		release(worker);
		if (worker->hostCounters) cudaFreeHost(worker->hostCounters);
		for (cudaEvent_t event : worker->iterationDone)
			if (event) cudaEventDestroy(event);
		if (worker->stream) cudaStreamDestroy(worker->stream);
		delete worker;
	}

	delete state;
}

static WorkerState* get_worker(RenderState* state, size_t index)
{
	while (state->workers.size() <= index)
	{
		WorkerState* worker = new WorkerState();

		if (!check_cuda(cudaStreamCreateWithFlags(&worker->stream, cudaStreamNonBlocking), "cudaStreamCreate(render worker)"))
		{
			delete worker;
			return nullptr;
		}

		state->workers.push_back(worker);
	}

	return state->workers[index];
}

template<class T>
static bool allocate(WorkerState* state, T*& pointer, uint64_t count)
{
	void* p = nullptr;
	if (!check_cuda(cudaMalloc(&p, sizeof(T) * std::max<uint64_t>(count, 1)), "cudaMalloc(render state)")) return false;
	state->allocations.push_back(p);
	pointer = (T*)p;
	return true;
}

static bool ensure_capacity(WorkerState* state, uint64_t paths, uint64_t pixels, uint64_t tiles, bool instanced)
{
	if (!state->hostCounters)
	{
		if (!check_cuda(cudaMallocHost((void**)&state->hostCounters, sizeof(uint32_t) * 64), "cudaMallocHost")) return false;
		std::memset(state->hostCounters, 0, sizeof(uint32_t) * 64); // the iteration mirror starts at serial 0 = "nothing finished"
	}
	bool layersReady = !instanced || state->paths.hitLayers != nullptr;
	if (paths <= state->capacity && pixels <= state->pixelCapacity && tiles <= state->tileCapacity && layersReady) return true;

	paths = std::max(paths, state->capacity);
	pixels = std::max(pixels, state->pixelCapacity);
	tiles = std::max(tiles, state->tileCapacity);
	release(state);

	PathBuffers& b = state->paths;
	bool ok = allocate(state, b.rayQueue[0], paths * 2) && allocate(state, b.rayQueue[1], paths * 2) && allocate(state, b.rayPath[0], paths)
		&& allocate(state, b.rayPath[1], paths) && allocate(state, b.hitQueue, paths)
		&& allocate(state, b.energy, paths) && allocate(state, b.result, paths) && allocate(state, b.oldPosition, paths)
		&& allocate(state, b.oldNormal, paths) && allocate(state, b.key, paths) && allocate(state, b.shadowQueue, paths * 2)
		&& allocate(state, b.shadowValue, paths) && allocate(state, b.counters, 64) && allocate(state, b.stats, STAT_COUNT)
		&& allocate(state, state->pixelXY, paths) && allocate(state, state->sampleIndex, paths) && allocate(state, state->sampleOut, paths)
		&& allocate(state, state->accumulator, pixels * 4) && allocate(state, state->sampleCount, pixels)
		&& allocate(state, state->activePixels[0], pixels) && allocate(state, state->activePixels[1], pixels)
		&& allocate(state, state->batchPixelXY, pixels) && allocate(state, state->tileXYDevice, tiles * 2);

	for (int c = 0; ok && c < CLASS_COUNT; c++) ok = allocate(state, b.classQueue[c], paths);

	if (instanced)
		ok = ok && allocate(state, b.rayLayers[0], paths * 2) && allocate(state, b.rayLayers[1], paths * 2) && allocate(state, b.hitLayers, paths * 2)
			&& allocate(state, b.shadowLayers, paths * 2)
			&& check_cuda(cudaMemset(b.hitLayers, 0, sizeof(uint4) * paths * 2), "cudaMemset(hit layers)"); // only instanced traversal writes them

	if (!ok) return false;

	b.sampleIndex = state->sampleIndex;
	state->capacity = paths;
	state->pixelCapacity = pixels;
	state->tileCapacity = tiles;
	return true;
}

static bool profiling()
{
	static const bool enabled = []
	{
		const char* value = std::getenv("ECHO_B200_PROFILE");
		return value && value[0] == '1';
	}();
	return enabled;
}

// Tuning switches of the wavefront: read once from the environment (ECHO_B200_<NAME>), changeable at run time through
// echo_b200_debug_set_option so that one process can A/B them without rebuilding its scene (variants/r2_sweep_c5.py).
struct RenderOptions
{
	std::atomic<long long> renderWorkers, batchPaths, narrowLimit, tailLimit, runAhead, blockingSync, guidedBatches;

	RenderOptions()
	{
		renderWorkers = from_environment("ECHO_B200_RENDER_WORKERS", kWorkers);      // concurrent tile-batch pipelines
		batchPaths = from_environment("ECHO_B200_BATCH_PATHS", (long long)kPathsPerBatch); // paths per batch and pipeline
		narrowLimit = from_environment("ECHO_B200_NARROW_LIMIT", kNarrowLimit);      // rays below which a bounce uses the one-thread-per-ray kernels
		tailLimit = from_environment("ECHO_B200_TAIL_LIMIT", kTailLimit);            // live paths below which tail_kernel finishes a batch (0 = never)
		runAhead = from_environment("ECHO_B200_RUN_AHEAD", -1);                      // -1 = automatic, see run_ahead()
		blockingSync = from_environment("ECHO_B200_BLOCKING_SYNC", -1);              // -1 = automatic, see wait_mode()
		guidedBatches = from_environment("ECHO_B200_GUIDED_BATCHES", 0);             // batches shrink towards the end of a call, see render_tiles
	}

	static long long from_environment(const char* name, long long fallback)
	{
		const char* value = std::getenv(name);
		return value ? std::atoll(value) : fallback;
	}
};

static RenderOptions& options()
{
	static RenderOptions instance;
	return instance;
}

bool set_render_option(const char* name, long long value)
{
	RenderOptions& o = options();
	const std::string key = name ? name : "";
	if (key == "RENDER_WORKERS") o.renderWorkers = value;
	else if (key == "BATCH_PATHS") o.batchPaths = value;
	else if (key == "NARROW_LIMIT") o.narrowLimit = value;
	else if (key == "TAIL_LIMIT") o.tailLimit = value;
	else if (key == "RUN_AHEAD") o.runAhead = value;
	else if (key == "BLOCKING_SYNC") o.blockingSync = value;
	else if (key == "GUIDED_BATCHES") o.guidedBatches = value;
	else return false;
	return true;
}

// How a pipeline thread waits for the counts of a unit (ECHO_B200_BLOCKING_SYNC):
//   0  cudaEventSynchronize on a spinning event: the fastest wake-up while every pipeline thread has a core of its own;
//   1  a blocking-sync event: the thread sleeps in the driver; a wake-up costs tens of microseconds, once per bounce in lock step;
//   2  poll the mirror record in pinned memory, yielding the core between polls (sched_yield): when N ranks x 8 pipelines outnumber the
//      host's cores (8 ranks on a 32-core box) a waiting thread hands its core to a runnable one at once and is back within
//      microseconds of its counts arriving, so the loop can stay in lock step with exactly sized launches.
// Automatic choice: 0 when the pipelines of all visible devices fit the cores, else the measured best of 1 / 2 (kOversubscribedWait).
enum WaitMode : int { WAIT_SPIN = 0, WAIT_BLOCK = 1, WAIT_YIELD = 2 };
constexpr int kOversubscribedWait = WAIT_YIELD;

static int wait_mode()
{
	long long configured = options().blockingSync;
	if (configured >= 0) return (int)std::min<long long>(configured, 2);

	static const bool oversubscribed = []
	{
		int devices = 1;
		cudaGetDeviceCount(&devices);
		return (unsigned int)(devices * kWorkers) > std::thread::hardware_concurrency();
	}();
	return oversubscribed ? kOversubscribedWait : WAIT_SPIN;
}

static bool blocking_waits() { return wait_mode() == WAIT_BLOCK; }

static bool ensure_events(WorkerState* state)
{
	const bool blocking = blocking_waits();
	if (state->iterationDone[0] && state->eventsBlocking == blocking) return true;

	for (cudaEvent_t& event : state->iterationDone)
	{
		if (event) cudaEventDestroy(event);
		event = nullptr;
	}

	unsigned int flags = cudaEventDisableTiming | (blocking ? cudaEventBlockingSync : 0u);
	for (cudaEvent_t& event : state->iterationDone)
		if (!check_cuda(cudaEventCreateWithFlags(&event, flags), "cudaEventCreate(iteration)")) return false;
	state->eventsBlocking = blocking;
	return true;
}

static unsigned int blocks_for(uint64_t count) { return (unsigned int)std::max<uint64_t>((count + kBlock - 1) / kBlock, 1); }

// How many wavefront iterations a pipeline may have queued beyond the newest one whose ray count the host has seen
// (ECHO_B200_RUN_AHEAD; 0 = lock step: launch, wait, read the count, launch). Running ahead sizes grids with counts that are one
// to three bounces old — more CTAs that find nothing to do — which on one GPU with spinning waits costs more than the wake-up
// latency it hides (A/B r2a, run-ahead 0 / 1 / 3 / 6: C1 323 / 318 / 303 / 283, C3 455 / 448 / 435 / 421, C4 344 / 340 / 332 / 322,
// C5 394 / 390 / 379 / 367 M samples/s). Automatic choice: lock step while the pipeline threads can spin on cores of their own,
// kRunAhead when they sleep in blocking waits (8 ranks x 8 pipelines on one host), where a wake-up costs tens of microseconds.
constexpr uint32_t kRunAhead = 2;

static uint32_t run_ahead()
{
	long long configured = options().runAhead;
	if (configured < 0) configured = blocking_waits() ? kRunAhead : 0;
	return (uint32_t)std::min<long long>(configured, WorkerState::kEventRing - 2);
}

// Evaluates `count` path slots already described in state->pixelXY / sampleIndex; radiance lands in state->sampleOut.
//
// The bounce loop runs AHEAD of the device. Every kernel of an iteration reads its ray / class / shadow counts from device
// memory and exits past them, so the host only needs an UPPER BOUND of the live rays to size the grids — and the live count
// never grows from one bounce to the next (a path spawns at most one ray). The rotate kernel that closes iteration k publishes
// {serial of k, rays left} as one 8-byte word in mapped pinned memory; the pipeline thread reads the newest word it can see,
// sizes the next iteration with it and keeps launching, at most `runAhead` iterations beyond the last count it has seen. It
// blocks only when that window is full. The device therefore never idles between bounces waiting for a host thread to wake
// up and launch (8 ranks x 8 pipelines share the box's host cores), and when the wavefront empties at most `runAhead`
// surplus iterations were queued, each nine launches of kernels that find zero counts.
template<int STACK, bool INST, bool STRAT>
static bool evaluate_paths(WorkerState* state, const DeviceScene& sceneIn, const EchoRenderParams& params, uint32_t count, uint64_t& launches, cudaStream_t stream)
{
	PathBuffers& paths = state->paths;
	uint32_t* counters = paths.counters;
	uint32_t* activeCount = counters + 32; // separate slot read by the kernels of one iteration
	KernelTimer& timer = state->timer;

	if (count == 0u) return true;
	if (!check_cuda(cudaMemsetAsync(counters, 0, sizeof(uint32_t) * 64, stream), "cudaMemsetAsync(counters)")) return false;

	timer.start(stream);
	raygen_kernel<STRAT><<<blocks_for(count), kBlock, 0, stream>>>(sceneIn, params, count, state->pixelXY, state->sampleIndex, paths);
	timer.stop(KernelTimer::RAYGEN, stream);
	++launches;

	if ((params.evaluator & ECHO_EVALUATOR_KIND_MASK) == ECHO_EVALUATOR_NAIVE)
	{
		naive_kernel<STACK, INST, STRAT><<<blocks_for(count), kBlock, 0, stream>>>(sceneIn, params, count, paths, state->sampleOut);
		++launches;
		return check_cuda(cudaGetLastError(), "naive_kernel launch");
	}

	if ((params.evaluator & ECHO_EVALUATOR_KIND_MASK) != ECHO_EVALUATOR_PATH_TRACED)
	{
		auxiliary_kernel<STACK, INST, STRAT><<<blocks_for(count), kBlock, 0, stream>>>(sceneIn, params, count, paths, state->sampleOut);
		++launches;
		return check_cuda(cudaGetLastError(), "auxiliary_kernel launch");
	}

	// a counted pass (ECHO_EVALUATOR_COUNT_VISITS): the one-thread-per-query kernels with visit counters for every bounce, no
	// tail kernel; same per-ray operations, so the same results and the visit counts of the persistent kernels
	const bool counted = (params.evaluator & ECHO_EVALUATOR_COUNT_VISITS) != 0;
	DeviceScene scene = sceneIn;
	if (counted) scene.lightVisits = paths.stats + STAT_LIGHT_NODE_VISITS;

	// what the shading kernels read of the parameters does not include the epoch (it only numbers the samples, in raygen)
	EchoRenderParams iterationParams = params;
	iterationParams.epochOffset = 0;

	const uint32_t narrowLimit = (uint32_t)options().narrowLimit;
	const uint32_t tailLimit = (uint32_t)options().tailLimit;
	const uint32_t runAhead = timer.enabled ? 0u : run_ahead();
	const int waitMode = wait_mode();

	if (!ensure_events(state)) return false;

	volatile unsigned long long* mirror = reinterpret_cast<volatile unsigned long long*>(state->hostCounters);
	volatile uint32_t* classMirror = reinterpret_cast<volatile uint32_t*>(state->hostCounters + 2);
	const uint32_t firstSerial = state->serial + 1u;  // serial of this call's unit 0
	uint32_t launched = 0u;                           // units queued so far
	uint32_t bound = count;                           // upper bound of the rays of every iteration not yet known exactly
	const bool packs = INST && scene.packCount != 0u; // INST without packs: a textured scene, ordinary traversal, zeroed hit layers
	uint32_t* const rayCount = counters + COUNTER_NEXT; // rays in the queue extend / classify are about to consume

	// A UNIT of work is [shade x6, shadow] of iteration k - 1 followed by [extend, classify, rotate] of iteration k (unit 0 has only the
	// second half): extend and classify of the NEXT bounce are queued before the host looks at any count, so that when it does
	// look — rotate k published {rays, class counts of k} — it can size the six shading launches of k exactly (and skip the empty
	// ones) instead of covering each class with a grid for all live rays.
	auto launch_trace_half = [&](uint32_t k, unsigned int blocks, bool narrow) -> bool
	{
		const int current = (int)(k & 1u);
		unsigned long long* rayCounters = narrow ? nullptr : ray_counters(stream);
		if (!narrow && !rayCounters) return false;

		// one-thread-per-ray for narrow and counted passes, persistent otherwise; `io` names the instantiation (with or without packs)
		auto extend = [&](auto io)
		{
			constexpr bool PACKS = std::is_same<decltype(io), ExtendLayersIO>::value;
			if (counted) extend_narrow_kernel<STACK, PACKS, true><<<blocks, kBlock, 0, stream>>>(scene, io, rayCount, paths.stats);
			else if (narrow) extend_narrow_kernel<STACK, PACKS, false><<<blocks, kBlock, 0, stream>>>(scene, io, rayCount, paths.stats);
			else
			{
				const int grid = persistent_grid((const void*)extend_kernel<STACK, PACKS>);
				extend_kernel<STACK, PACKS><<<std::min<unsigned int>(blocks, (unsigned int)grid), kTraverseBlock, 0, stream>>>(scene, io, rayCount, rayCounters);
			}
		};

		timer.start(stream);
		ExtendIO extendIO = { paths.rayQueue[current], paths.hitQueue };
		if (packs) extend(ExtendLayersIO{ extendIO, paths.rayLayers[current], paths.hitLayers });
		else extend(extendIO);
		timer.stop(KernelTimer::EXTEND, stream);

		timer.start(stream);
		unsigned int classifyBlocks = (blocks * (unsigned int)kBlock + kClassifyBlock - 1) / kClassifyBlock;
		classify_kernel<INST><<<classifyBlocks, kClassifyBlock, 0, stream>>>(scene, rayCount, counters + COUNTER_CLASS + current * CLASS_COUNT, paths);
		timer.stop(KernelTimer::OTHER, stream);

		timer.start(stream);
		rotate_counters_kernel<<<1, 1, 0, stream>>>(counters, activeCount, const_cast<unsigned long long*>(mirror), firstSerial + k, current);
		timer.stop(KernelTimer::ROTATE, stream);
		launches += 3;

		if (!check_cuda(cudaGetLastError(), "wavefront launch")) return false;
		return check_cuda(cudaEventRecord(state->iterationDone[k % WorkerState::kEventRing], stream), "cudaEventRecord(iteration)");
	};

	// unit 0: the camera rays
	if (!check_cuda(cudaMemcpyAsync(rayCount, &count, sizeof(uint32_t), cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(count)")) return false;
	if (!launch_trace_half(0u, blocks_for(count), counted || count < narrowLimit)) return false;
	launched = 1u;

	while (true)
	{
		// the newest finished unit the host can see (a word left by an earlier call fails the range test)
		unsigned long long seen = *mirror;
		uint32_t finished = (uint32_t)(seen >> 32) - firstSerial + 1u; // units of this call known to be finished
		if (finished > launched) finished = 0u;

		if (finished > 0u)
		{
			bound = std::min(bound, (uint32_t)seen);
			if ((uint32_t)seen == 0u) break; // the wavefront is empty; whatever was queued beyond finds zero counts
		}

		if (launched - finished > runAhead)
		{
			// window full: wait until the oldest unit the host has not seen yet is done, then look again
			if (waitMode == WAIT_YIELD)
			{
				for (uint32_t polls = 0; (uint32_t)(*mirror >> 32) - firstSerial + 1u <= finished || (uint32_t)(*mirror >> 32) - firstSerial + 1u > launched; polls++)
				{
					sched_yield();
					// a failed launch never publishes its record: look at the stream now and then instead of polling forever
					if ((polls & 0xFFFu) == 0xFFFu && cudaStreamQuery(stream) != cudaErrorNotReady) break;
				}

				if (!check_cuda(cudaGetLastError(), "wavefront iteration")) return false;
			}
			else if (!check_cuda(cudaEventSynchronize(state->iterationDone[finished % WorkerState::kEventRing]), "wavefront iteration")) return false;

			continue;
		}

		const uint32_t k = launched - 1u;           // the iteration this unit shades; its rays sit in queue k & 1
		const int current = (int)(k & 1u);
		const bool exact = finished == launched;    // nothing in flight: `bound` IS the ray count of k and the class counts are k's
		const unsigned int blocks = blocks_for(bound);

		// the tail: finish the few paths that are left in one launch (it traces for itself: the hits of k are simply not used)
		if (!timer.enabled && !counted && bound < tailLimit)
		{
			tail_kernel<STACK, INST, STRAT><<<blocks, kBlock, 0, stream>>>(scene, iterationParams, activeCount, paths, current);
			if (!check_cuda(cudaGetLastError(), "tail_kernel launch")) return false;
			++launches;
			break;
		}

		uint32_t classRays[CLASS_COUNT];
		for (int c = 0; c < CLASS_COUNT; c++) classRays[c] = counted ? 0u : (exact ? classMirror[c] : bound);
		const uint32_t missRays = exact ? classMirror[CLASS_MISS] : 0u;

		if (counted)
		{
			shade_counted_kernel<INST, STRAT><<<blocks, kBlock, 0, stream>>>(scene, iterationParams, activeCount, paths, current);
			++launches;
		}

		const uint32_t* classCounts = counters + COUNTER_CLASS + current * CLASS_COUNT;

#define ECHO_SHADE(CLASS_VALUE, KINDS_VALUE, SLOT)                                                                                                       \
		if (classRays[CLASS_VALUE] != 0u)                                                                                                                \
		{                                                                                                                                                \
			timer.start(stream);                                                                                                                         \
			shade_kernel<CLASS_VALUE, KINDS_VALUE, INST, STRAT><<<blocks_for(classRays[CLASS_VALUE]), kBlock, 0, stream>>>(scene, iterationParams,       \
			                                                              paths.classQueue[CLASS_VALUE], classCounts + CLASS_VALUE, paths, current);     \
			timer.stop(SLOT, stream);                                                                                                                    \
			++launches;                                                                                                                                  \
		}

		ECHO_SHADE(CLASS_MISS, 0u, KernelTimer::SHADE_MISS)
		ECHO_SHADE(CLASS_DIFFUSE, KINDS_DIFFUSE, KernelTimer::SHADE_DIFFUSE)
		ECHO_SHADE(CLASS_SMOOTH, KINDS_SMOOTH, KernelTimer::SHADE_SMOOTH)
		ECHO_SHADE(CLASS_DIELECTRIC, KINDS_DIELECTRIC, KernelTimer::SHADE_DIELECTRIC)
		ECHO_SHADE(CLASS_CONDUCTOR, KINDS_CONDUCTOR, KernelTimer::SHADE_CONDUCTOR)
		ECHO_SHADE(CLASS_TERMINAL, KINDS_TERMINAL, KernelTimer::SHADE_TERMINAL)
#undef ECHO_SHADE

		// shadow rays of k: at most one per ray that hit something
		const uint32_t shadowBound = exact ? bound - missRays : bound;
		const bool narrow = counted || bound < narrowLimit;

		if (shadowBound != 0u)
		{
			const unsigned int shadowBlocks = blocks_for(shadowBound);
			unsigned long long* rayCounters = narrow ? nullptr : ray_counters(stream);
			if (!narrow && !rayCounters) return false;

			auto shadow = [&](auto io)
			{
				constexpr bool PACKS = std::is_same<decltype(io), ShadowLayersIO>::value;
				if (counted) shadow_narrow_kernel<STACK, PACKS, true><<<shadowBlocks, kBlock, 0, stream>>>(scene, io, counters + COUNTER_SHADOW, paths.stats);
				else if (narrow) shadow_narrow_kernel<STACK, PACKS, false><<<shadowBlocks, kBlock, 0, stream>>>(scene, io, counters + COUNTER_SHADOW, paths.stats);
				else
				{
					const int grid = persistent_grid((const void*)shadow_kernel<STACK, PACKS>);
					shadow_kernel<STACK, PACKS><<<std::min<unsigned int>(shadowBlocks, (unsigned int)grid), kTraverseBlock, 0, stream>>>(scene, io, counters + COUNTER_SHADOW, rayCounters, paths.stats);
				}
			};

			timer.start(stream);
			ShadowIO shadowIO = { paths.shadowQueue, paths.shadowValue, paths.result, 0u };
			if (packs) shadow(ShadowLayersIO{ shadowIO, paths.shadowLayers });
			else shadow(shadowIO);

			timer.stop(KernelTimer::SHADOW, stream);
			++launches;
		}

		if (!check_cuda(cudaGetLastError(), "wavefront launch")) return false;

		// extend + classify + rotate of iteration k + 1: at most the rays of k that hit something go on
		const uint32_t nextBound = std::max(shadowBound, 1u);
		if (!launch_trace_half(launched, blocks_for(nextBound), counted || nextBound < narrowLimit)) return false;
		++launched;
	}

	state->serial += launched;

	timer.start(stream);
	finish_kernel<<<blocks_for(count), kBlock, 0, stream>>>(count, paths, state->sampleOut);
	timer.stop(KernelTimer::FINISH, stream);
	++launches;
	return check_cuda(cudaGetLastError(), "finish_kernel launch");
}

// the instantiation a call needs: the tree's stack class, the full-featured shading kernels for packs or textures, and
// with ECHO_DISTRIBUTION_STRATIFIED the stratified instantiation of every kernel that draws
template<int STACK>
static bool evaluate_paths_stack(WorkerState* state, const DeviceScene& scene, const EchoRenderParams& params, uint32_t count, uint64_t& launches, cudaStream_t stream)
{
	const bool instanced = scene.packCount != 0u || scene.textureCount != 0u;
	const bool stratified = (params.evaluator & ECHO_DISTRIBUTION_STRATIFIED) != 0;

	if (instanced) return stratified ? evaluate_paths<STACK, true, true>(state, scene, params, count, launches, stream) : evaluate_paths<STACK, true, false>(state, scene, params, count, launches, stream);
	return stratified ? evaluate_paths<STACK, false, true>(state, scene, params, count, launches, stream) : evaluate_paths<STACK, false, false>(state, scene, params, count, launches, stream);
}

static bool evaluate_paths_dispatch(WorkerState* state, const DeviceScene& scene, const EchoRenderParams& params, uint32_t count, uint64_t& launches, cudaStream_t stream)
{
	switch (stack_class(scene.maxDepth))
	{
		case 0: return evaluate_paths_stack<48>(state, scene, params, count, launches, stream);
		case 1: return evaluate_paths_stack<96>(state, scene, params, count, launches, stream);
		case 2: return evaluate_paths_stack<192>(state, scene, params, count, launches, stream);
		default: set_error("QBVH deeper than 63 quad levels is not supported"); return false;
	}
}

static void collect_stats(WorkerState* state, EchoStats* stats, uint64_t launches, cudaStream_t stream)
{
	if (!stats) return;
	unsigned long long host[STAT_COUNT];
	cudaMemcpyAsync(host, state->paths.stats, sizeof(host), cudaMemcpyDeviceToHost, stream);
	cudaStreamSynchronize(stream);
	uint64_t* out = reinterpret_cast<uint64_t*>(stats);
	for (int i = 0; i < STAT_COUNT; i++) out[i] += host[i];
	stats->kernelLaunches += launches;
}

// one batch of tiles: pixel loop -> epoch loop -> sample loop of EvaluationOperation.Execute (EvaluationOperation.cs:100-141)
static bool render_batch(WorkerState* state, const DeviceScene& scene, const EchoRenderParams& params, const int32_t* tileXY, uint32_t tiles,
                         float4* tilesOut, float4* frame, uint64_t& launches)
{
	cudaStream_t stream = state->stream;
	uint64_t perTile = (uint64_t)params.tileSize * params.tileSize;
	uint32_t pixelTotal = (uint32_t)(tiles * perTile);

	if (!ensure_capacity(state, (uint64_t)pixelTotal * params.extend, pixelTotal, tiles, scene.packCount != 0u || scene.textureCount != 0u)) return false;
	if (!check_cuda(cudaMemcpyAsync(state->tileXYDevice, tileXY, sizeof(int32_t) * 2 * tiles, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(tiles)")) return false;
	if (!check_cuda(cudaMemsetAsync(state->paths.counters, 0, sizeof(uint32_t) * 64, stream), "cudaMemsetAsync(counters)")) return false;

	batch_pixels_kernel<<<blocks_for(pixelTotal), kBlock, 0, stream>>>(params, state->tileXYDevice, tiles, state->batchPixelXY, state->activePixels[0],
	                                                                 state->paths.counters, state->accumulator, state->sampleCount);
	++launches;

	if (!check_cuda(cudaMemcpyAsync(state->hostCounters + 8, state->paths.counters + COUNTER_PIXELS, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(pixels)")) return false;
	if (!check_cuda(cudaStreamSynchronize(stream), "batch setup")) return false;

	uint32_t activePixels = state->hostCounters[8];
	int list = 0;

	for (uint32_t epoch = 1; activePixels > 0 && epoch <= (uint32_t)params.maxEpoch; epoch++)
	{
		uint32_t slots = activePixels * (uint32_t)params.extend;

		epoch_slots_kernel<<<blocks_for(slots), kBlock, 0, stream>>>(params, activePixels, state->activePixels[list], state->batchPixelXY, epoch, state->pixelXY, state->sampleIndex);
		++launches;

		if (!evaluate_paths_dispatch(state, scene, params, slots, launches, stream)) return false;

		if (!check_cuda(cudaMemsetAsync(state->paths.counters + COUNTER_PIXELS, 0, sizeof(uint32_t), stream), "cudaMemsetAsync(pixel counter)")) return false;

		state->timer.start(stream);
		accumulate_kernel<<<blocks_for(activePixels), kBlock, 0, stream>>>(params, activePixels, state->activePixels[list], state->sampleOut, state->accumulator,
		                                                                 state->sampleCount, epoch, state->activePixels[list ^ 1], state->paths.counters, state->paths.stats);
		state->timer.stop(KernelTimer::ACCUMULATE, stream);
		++launches;

		if (!check_cuda(cudaMemcpyAsync(state->hostCounters + 8, state->paths.counters + COUNTER_PIXELS, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(pixels)")) return false;
		if (!check_cuda(cudaStreamSynchronize(stream), "epoch")) return false;

		activePixels = state->hostCounters[8];
		list ^= 1;
	}

	resolve_tiles_kernel<<<blocks_for(pixelTotal), kBlock, 0, stream>>>(params, pixelTotal, state->batchPixelXY, state->accumulator, state->sampleCount, tilesOut, frame, state->paths.stats);
	++launches;
	return check_cuda(cudaGetLastError(), "resolve_tiles_kernel launch");
}

bool stratified_extend_valid(const EchoRenderParams& params)
{
	return (params.evaluator & ECHO_DISTRIBUTION_STRATIFIED) == 0 || (params.extend > 0 && params.extend <= ECHO_DISTRIBUTION_STRATIFIED_EXTEND_MAX);
}

bool render_tiles(RenderState* state, const DeviceScene& scene, const EchoRenderParams& params, const int32_t* tileXY, uint32_t tileCount,
                  float4* tilesOut, float4* frame, EchoStats* stats, cudaStream_t stream)
{
	if (params.width <= 0 || params.height <= 0 || params.tileSize <= 0 || params.extend <= 0 || params.maxEpoch < 1 || params.minEpoch > params.maxEpoch)
	{
		set_error("invalid EchoRenderParams");
		return false;
	}

	if ((params.evaluator & ECHO_EVALUATOR_KIND_MASK) == ECHO_EVALUATOR_NAIVE && (params.bounceLimit < 0 || params.bounceLimit > kNaiveBounceCap))
	{
		set_error("the naive evaluator supports bounce limits up to 128");
		return false;
	}

	if ((params.evaluator & ECHO_EVALUATOR_KIND_MASK) > ECHO_EVALUATOR_NAIVE
	    || (params.evaluator & ~(ECHO_EVALUATOR_KIND_MASK | ECHO_EVALUATOR_DIVERGE_ONCE | ECHO_EVALUATOR_COUNT_VISITS | ECHO_DISTRIBUTION_STRATIFIED)) != 0)
	{
		set_error("unknown EchoRenderParams.evaluator");
		return false;
	}

	if ((params.evaluator & ECHO_EVALUATOR_COUNT_VISITS) != 0 && (params.evaluator & ECHO_EVALUATOR_KIND_MASK) != ECHO_EVALUATOR_PATH_TRACED)
	{
		set_error("ECHO_EVALUATOR_COUNT_VISITS is a switch of the path-traced evaluator");
		return false;
	}

	if (!stratified_extend_valid(params))
	{
		set_error("ECHO_DISTRIBUTION_STRATIFIED takes an extend of 1 to 2^23");
		return false;
	}

	// work submitted earlier on the caller's stream (e.g. clearing the frame) must be visible to the worker streams
	if (!check_cuda(cudaStreamSynchronize(stream), "render_tiles entry")) return false;

	const int configuredWorkers = (int)std::min<long long>(std::max<long long>(options().renderWorkers, 1), 16);

	// batch size: at most kPathsPerBatch paths, but small jobs are still split so that every pipeline gets a share
	// (never below 256 Ki paths per batch: smaller wavefronts are launch- and latency-bound from the first bounce)
	uint64_t perTile = (uint64_t)params.tileSize * params.tileSize;
	uint64_t pathsPerTile = perTile * params.extend;
	const uint64_t batchPaths = std::min<uint64_t>(std::max<uint64_t>((uint64_t)std::max<long long>(options().batchPaths, 1), 1ull << 16), 1ull << 26);
	uint64_t maxTiles = std::max<uint64_t>(1, batchPaths / pathsPerTile);
	uint64_t minTiles = std::max<uint64_t>(1, (1ull << 18) / pathsPerTile);
	uint64_t share = (tileCount + configuredWorkers - 1) / configuredWorkers;
	uint64_t tilesPerBatch = std::min<uint64_t>(std::max<uint64_t>(share, minTiles), maxTiles);
	tilesPerBatch = std::min<uint64_t>(tilesPerBatch, tileCount);
	uint64_t batchCount = (tileCount + tilesPerBatch - 1) / tilesPerBatch;

	int workerCount = (int)std::min<uint64_t>(profiling() ? 1 : configuredWorkers, batchCount);
	for (int i = 0; i < workerCount; i++)
		if (!get_worker(state, i)) return false;

	int device = 0;
	cudaGetDevice(&device);

	// Batches are claimed by the pipelines as they finish. GUIDED_BATCHES (off): a claim takes remaining / (2 x pipelines) tiles, capped by
	// the batch size and floored at the minimum, so that batches shrink towards the end of the call and the pipelines finish within one
	// small batch of each other. Measured (r2s, one GPU): worse everywhere — rank 0's eighth of C5 602 vs 567 ms, C3 253 vs 236 ms, C4 398 vs
	// 374 ms, C1 11.4 vs 10.3 ms: small batches cost more in launch-bound narrow bounces than an even finish saves. Kept as a switch.
	const bool guided = options().guidedBatches != 0;
	std::mutex claimGuard;
	uint64_t nextTile = 0;

	auto claim = [&](uint64_t& first, uint32_t& tiles) -> bool
	{
		std::lock_guard<std::mutex> lock(claimGuard);
		if (nextTile >= tileCount) return false;
		uint64_t remaining = tileCount - nextTile;
		uint64_t size = tilesPerBatch;
		if (guided) size = std::min<uint64_t>(tilesPerBatch, std::max<uint64_t>(minTiles, (remaining + 2 * workerCount - 1) / (2 * workerCount)));
		size = std::min<uint64_t>(size, remaining);
		first = nextTile;
		tiles = (uint32_t)size;
		nextTile += size;
		return true;
	};

	std::atomic<bool> failed{ false };
	std::vector<uint64_t> launches(workerCount, 0);
	std::vector<std::string> errors(workerCount);

	auto work = [&](int index)
	{
		WorkerState* worker = state->workers[index];
		bool ok = check_cuda(cudaSetDevice(device), "cudaSetDevice(render worker)");

		// the statistics buffer is allocated with the wavefront state: size the worker for a full batch up front
		ok = ok && ensure_capacity(worker, tilesPerBatch * perTile * params.extend, tilesPerBatch * perTile, tilesPerBatch, scene.packCount != 0u || scene.textureCount != 0u);
		ok = ok && check_cuda(cudaMemsetAsync(worker->paths.stats, 0, sizeof(unsigned long long) * STAT_COUNT, worker->stream), "cudaMemsetAsync(stats)");

		while (ok && !failed.load())
		{
			uint64_t first = 0;
			uint32_t tiles = 0;
			if (!claim(first, tiles)) break;
			ok = render_batch(worker, scene, params, tileXY + first * 2, tiles, tilesOut ? tilesOut + first * perTile : nullptr, frame, launches[index]);
		}

		ok = ok && check_cuda(cudaStreamSynchronize(worker->stream), "render worker");

		if (!ok)
		{
			failed.store(true);
			errors[index] = last_error_string();
		}
	};

	if (workerCount == 1) work(0);
	else
	{
		std::vector<std::thread> threads;
		for (int i = 0; i < workerCount; i++) threads.emplace_back(work, i);
		for (std::thread& thread : threads) thread.join();
	}

	if (failed.load())
	{
		for (const std::string& error : errors)
			if (!error.empty()) set_error(error);
		return false;
	}

	for (int i = 0; i < workerCount; i++) collect_stats(state->workers[i], stats, launches[i], state->workers[i]->stream);
	if (profiling()) state->workers[0]->timer.report();
	return true;
}

// debug: explicit (pixel, sample) lists -> per-sample radiance (device pointers in, device pointer out)
bool evaluate_sample_list(RenderState* renderState, const DeviceScene& scene, const EchoRenderParams& params, int channels, const int32_t* pixelXYHost, const uint32_t* sampleIndexHost,
                          uint64_t n, float* outRGBHost, cudaStream_t)
{
	if (!stratified_extend_valid(params))
	{
		set_error("ECHO_DISTRIBUTION_STRATIFIED takes an extend of 1 to 2^23");
		return false;
	}

	WorkerState* state = get_worker(renderState, 0);
	if (!state) return false;
	cudaStream_t stream = state->stream;
	std::vector<float4> staging;

	for (uint64_t first = 0; first < n; first += kPathsPerBatch)
	{
		uint32_t count = (uint32_t)std::min<uint64_t>(kPathsPerBatch, n - first);
		if (!ensure_capacity(state, count, 1, 1, scene.packCount != 0u || scene.textureCount != 0u)) return false;

		if (!check_cuda(cudaMemcpyAsync(state->pixelXY, pixelXYHost + first * 2, sizeof(int2) * count, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(pixels)")) return false;
		if (!check_cuda(cudaMemcpyAsync(state->sampleIndex, sampleIndexHost + first, sizeof(uint32_t) * count, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(samples)")) return false;
		if (!check_cuda(cudaMemsetAsync(state->paths.stats, 0, sizeof(unsigned long long) * STAT_COUNT, stream), "cudaMemsetAsync(stats)")) return false;

		uint64_t launches = 0;
		if (!evaluate_paths_dispatch(state, scene, params, count, launches, stream)) return false;

		staging.resize(count);
		if (!check_cuda(cudaMemcpyAsync(staging.data(), state->sampleOut, sizeof(float4) * count, cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(out)")) return false;
		if (!check_cuda(cudaStreamSynchronize(stream), "evaluate_sample_list")) return false;

		for (uint32_t i = 0; i < count; i++)
		{
			const float lanes[4] = { staging[i].x, staging[i].y, staging[i].z, staging[i].w };
			for (int c = 0; c < channels; c++) outRGBHost[(first + i) * channels + c] = lanes[c];
		}
	}

	return true;
}

bool launch_frame_resolve(float4* frame, int32_t width, int32_t height, cudaStream_t stream)
{
	uint32_t count = (uint32_t)width * (uint32_t)height;
	frame_resolve_kernel<<<blocks_for(count), kBlock, 0, stream>>>(frame, count);
	return check_cuda(cudaGetLastError(), "frame_resolve_kernel launch");
}

} // namespace echo
