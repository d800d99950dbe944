// echo_internal.h — host-side state behind the opaque EchoScene handle and the kernel launch entry points.
#pragma once
#include <cuda_runtime.h>

#include <mutex>
#include <string>
#include <vector>

#include "echo_scene.cuh"

namespace echo
{

void set_error(const std::string& message);
std::string last_error_string(); // the calling thread's last error (worker threads hand theirs to the caller)
bool check_cuda(cudaError_t status, const char* what);

// smallest compiled traversal stack that holds the reference's `maxDepth * 3 + 1` entries (QuadBoundingVolumeHierarchy.cs:34)
int stack_class(uint32_t maxDepth); // 0: 48, 1: 96, 2: 192 entries, -1: unsupported

// ---- trace.cu ----
// all launches are asynchronous on `stream`; counts (optional) receives 3 x uint64 totals {nodes, triangles, spheres}
bool launch_trace(const DeviceScene& scene, const EchoRay* rays, uint64_t n, EchoHit* hits, unsigned long long* counts, cudaStream_t stream);
bool launch_occlude(const DeviceScene& scene, const EchoRay* rays, uint64_t n, uint8_t* occluded, unsigned long long* counts, cudaStream_t stream);

// ---- instanced.cu: the same queries through instanced packs, with TokenHierarchy layers in and out (either may be null) ----
bool launch_trace_instanced(const DeviceScene& scene, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, EchoHit* hits,
                            EchoTokenHierarchy* hitLayers, unsigned long long* counts, cudaStream_t stream);
bool launch_occlude_instanced(const DeviceScene& scene, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, uint8_t* occluded,
                              unsigned long long* counts, cudaStream_t stream);

// trace.cu: the persistent, work-replacing form of the two calls above; `launched` = false when ECHO_B200_SIMPLE_TRACE asks for the simple kernels
bool launch_persistent_instanced(const DeviceScene& scene, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, EchoHit* hits,
                                 EchoTokenHierarchy* hitLayers, uint8_t* occluded, cudaStream_t stream, bool& launched);

unsigned long long* ray_counters(cudaStream_t stream); // the self-resetting work counter pair of persistent launches on this device and stream
int persistent_grid(const void* kernel);              // resident CTAs of a persistent kernel on the current device (cached per device)

// ---- build.cu / sweep.cu: device-side tree builds in the QBVH node format (host buffers in and out): the reference's SweepBuilder tree
// itself (sweep.cu, echo_sweep.h), or a clustered / Morton-ordered binary tree collapsed the same way (build.cu) ----
bool build_qbvh_sweep(const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
                      const float* instanceBounds, uint32_t instanceCount, EchoQbvhNode* outNodes, uint32_t* outNodeCount, uint32_t* outMaxDepth, bool* gaveUp);
void last_sweep_build(float* out4); // the calling thread's last build_qbvh_sweep: {upload, device build, download} ms, binary levels
bool build_qbvh_device(const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
                       const float* instanceBounds, uint32_t instanceCount, EchoQbvhNode* outNodes, uint32_t* outNodeCount, uint32_t* outMaxDepth);

// ---- lightbuild.cu: the reference's light tree (LightCollection.CreateBounds + LightTree.Build + AddToMap) built on the device, byte for
// byte the host mirror's (echo_light_build.h). Host buffers in, host vectors out; `refused` = deeper than a 64-bit path ----
namespace lightbuild { struct Sources; }
bool build_light_tree_device(const lightbuild::Sources& sources, std::vector<EchoLightNode>& nodes, std::vector<uint32_t>& tokens, std::vector<uint64_t>& paths, bool* refused);
void last_light_build(float* out4); // the calling thread's last build_light_tree_device: {upload, device build, download} ms, levels

// ---- packbuild.cu: every pack of an instanced scene, QBVH and light tree, in rounds of forests (echo_pack_build.h). Host memory in and
// out; returns an ECHO_B200_* status with the error set ----
namespace packbuild { struct Inputs; struct Output; }
int32_t build_packs_device(const packbuild::Inputs& inputs, packbuild::Output& output);
void last_pack_build(float* out8); // the calling thread's last build_packs_device: rounds, levels, read-backs, launches, ms

// ---- render.cu ----
struct RenderState; // wavefront buffers, owned per scene

RenderState* render_state_create();
void render_state_destroy(RenderState* state);

// Renders `tileCount` tiles. When `frame` is non-null the per-pixel means are ADDED into the full-frame device buffer
// (xyz = mean * epochs rendered, w += epochs) for multi-device sample/tile sharding; when `tilesOut` is non-null the
// tile-major Float4 means are written there (device pointer). Synchronises `stream` internally between wavefront steps.
bool stratified_extend_valid(const EchoRenderParams& params); // ECHO_DISTRIBUTION_STRATIFIED's extend limit (always true without the flag)
bool render_tiles(RenderState* state, const DeviceScene& scene, const EchoRenderParams& params, const int32_t* tileXY, uint32_t tileCount,
                  float4* tilesOut, float4* frame, EchoStats* stats, cudaStream_t stream);

bool launch_frame_resolve(float4* frame, int32_t width, int32_t height, cudaStream_t stream);

// tuning switches of the wavefront (the ECHO_B200_<NAME> environment variables), changeable at run time; false = unknown name
bool set_render_option(const char* name, long long value);
bool set_build_option(const char* name, long long value); // build.cu: BUILD_ALGORITHM (2 = SweepBuilder, 1 = PLOC, 0 = LBVH)

// ---- peaks.cu: on-chip ceilings measured on the current device: {L2 coalesced read, L2 random 32-byte sectors, L1 random sectors} GB/s
bool measure_peaks(float* out3);

// ---- debug.cu: device mirrors of the oracle's known-answer hooks ----
bool launch_debug_bxdf(int32_t kind, const float* params, const float* outgoing, const float* samples, uint64_t n,
                       float* sampled8, float* evaluated4, float* inverse4, cudaStream_t stream);
bool launch_debug_math(int32_t op, const float* a, const float* b, const float* c, uint64_t n, float* out, cudaStream_t stream);

} // namespace echo

struct EchoScene
{
	int device = 0;
	bool committed = false;
	cudaStream_t stream = nullptr;

	// host staging until commit
	std::vector<EchoQbvhNode> nodes;
	uint32_t maxDepth = 0;
	std::vector<EchoTriangle> triangles;
	std::vector<EchoSphere> spheres;
	std::vector<EchoMaterial> materials;
	std::vector<EchoLightNode> lightNodes;
	std::vector<uint32_t> emitterTokens;
	std::vector<uint64_t> emitterPaths;
	std::vector<EchoPointLight> pointLights;
	std::vector<EchoInfiniteLight> infiniteLights;
	float infiniteThreshold = 0.0f, infinitePdf = 0.0f;
	EchoCamera camera = {};
	float boundRadius = 0.0f;
	std::vector<float> distributions;
	std::vector<EchoTexture> textures;
	std::vector<float> texels; // RGBA
	std::vector<EchoMaterialTextures> materialTextures;
	std::vector<EchoPack> packs; // empty: the arrays are one pack
	std::vector<EchoInstance> instances;

	// device
	echo::DeviceScene d = {};
	std::vector<void*> allocations;

	// scratch for the host-buffer batch calls (grown on demand)
#ifndef ECHO_HOST_SLOTS
#define ECHO_HOST_SLOTS 8 // A/B r2p, 4 vs 8: page-locked callers 1 527 vs 1 531 Mrays/s, pageable callers (one staging thread per slot) 753 vs 969
#endif
	static constexpr int kSlots = ECHO_HOST_SLOTS; // chunk buffers (and, for pageable callers, host threads) of the host-buffer batch pipeline
	void* scratchRays[kSlots] = {};
	void* scratchOut[kSlots] = {};
	uint64_t scratchCapacity = 0; // rays per chunk buffer
	cudaStream_t copyStreams[kSlots] = {};
	cudaEvent_t chunkDone[kSlots] = {};
	void* stagingIn[kSlots] = {};  // page-locked staging of the same chunk size, allocated the first time a caller hands pageable buffers
	void* stagingOut[kSlots] = {};
	uint64_t stagingCapacity = 0;

	// device buffer of echo_b200_render_tiles' tile-major output, kept between calls (allocating and freeing it per call cost the first
	// calls hundreds of milliseconds at random: cudaFree hands the memory back to the system, the next cudaMalloc maps it again)
	void* tilesOut = nullptr;
	uint64_t tilesOutBytes = 0;
	void* hierarchyScratch[4] = {}; // rays, ignore layers, out, hit layers of the *_batch_hierarchy calls, for the same reason
	uint64_t hierarchyBytes[4] = {};

	echo::RenderState* render = nullptr;

	// Entry points that use the scene's own scratch (the host-buffer batches, the renderer's wavefront state) hold this for the length of
	// the call: concurrent calls on ONE handle — Echo's workers all enter Operation.Execute at once (Operation.cs:164-177) — are safe and
	// take turns; the asynchronous *_device batch calls on caller buffers do not need it.
	std::mutex compute;

	// echo_b200_scene_create_multi: this handle is the scene of the first device of the mask, `replicas` are the scenes of the
	// others. Uploads go to the primary's host staging; commit replicates to every device.
	std::vector<EchoScene*> replicas;
};
