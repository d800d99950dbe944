// api.cu — the C ABI of libecho_b200.so (include/echo_b200.h, include/echo_b200_debug.h): scene upload and layout
// conversion, the batched trace/occlude entry points with pipelined host<->device copies, and the tile renderer.
// There is no CPU fallback anywhere in this library: without a CUDA device every compute call fails.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <thread>

#include "../../include/echo_b200_debug.h"
#include "echo_internal.h"
#include "echo_light_build.h"
#include "echo_pack_build.h"

namespace echo
{

static thread_local std::string lastError;

void set_error(const std::string& message) { lastError = message; }
std::string last_error_string() { return lastError; }

bool check_cuda(cudaError_t status, const char* what)
{
	if (status == cudaSuccess) return true;
	lastError = std::string(what) + ": " + cudaGetErrorString(status);
	return false;
}

bool evaluate_sample_list(RenderState* state, const DeviceScene& scene, const EchoRenderParams& params, int channels, const int32_t* pixelXYHost, const uint32_t* sampleIndexHost,
                          uint64_t n, float* outRGBHost, cudaStream_t stream);

} // namespace echo

using namespace echo;

namespace
{

struct DeviceGuard
{
	int previous = -1;
	bool ok = false;

	explicit DeviceGuard(int device)
	{
		if (cudaGetDevice(&previous) != cudaSuccess) previous = -1;
		ok = check_cuda(cudaSetDevice(device), "cudaSetDevice");
	}

	~DeviceGuard()
	{
		if (previous >= 0) cudaSetDevice(previous);
	}
};

template<class T>
bool upload(EchoScene* scene, const std::vector<T>& host, const T*& device)
{
	void* p = nullptr;
	size_t bytes = sizeof(T) * std::max<size_t>(host.size(), 1);
	if (!check_cuda(cudaMalloc(&p, bytes), "cudaMalloc(scene)")) return false;
	scene->allocations.push_back(p);
	if (host.empty() && !check_cuda(cudaMemset(p, 0, bytes), "cudaMemset(scene)")) return false; // the placeholder of an empty array
	if (!host.empty() && !check_cuda(cudaMemcpy(p, host.data(), sizeof(T) * host.size(), cudaMemcpyHostToDevice), "cudaMemcpy(scene)")) return false;
	device = (const T*)p;
	return true;
}

void free_device(EchoScene* scene)
{
	for (void* p : scene->allocations) cudaFree(p);
	scene->allocations.clear();
	scene->committed = false;
}

int32_t fail(int32_t code, const char* message)
{
	set_error(message);
	return code;
}

bool require_committed(EchoScene* scene)
{
	if (!scene) { set_error("scene is null"); return false; }
	if (!scene->committed) { set_error("scene is not committed"); return false; }
	return true;
}

// Shading indexes the material array with what the geometry stores; commit only validates those indices against a non-empty
// array (a scene without materials is fine for trace / occlude batches), so the render entry points must refuse such a scene
// instead of reading the zeroed placeholder out of bounds.
bool require_renderable(EchoScene* scene)
{
	if (!require_committed(scene)) return false;
	if (scene->d.materialCount == 0u) { set_error("the scene has no materials: it can serve trace / occlude batches but cannot be rendered"); return false; }
	return true;
}

// rays per pipelined chunk of the host-buffer batch (1 Mi: 32 MB in, 16 MB out); the last chunk's kernel and download are
// the only work the PCIe upload cannot hide, so chunks are kept small, but large enough to fill one resident wave
uint64_t chunk_rays()
{
	static const uint64_t value = []
	{
		const char* text = getenv("ECHO_B200_CHUNK_RAYS");
		long long parsed = text ? atoll(text) : 0;
		return parsed >= 4096 ? (uint64_t)parsed : 1ull << 20;
	}();

	return value;
}

bool ensure_scratch(EchoScene* scene, uint64_t rays)
{
	if (scene->scratchCapacity >= rays) return true;

	for (int i = 0; i < EchoScene::kSlots; i++)
	{
		if (scene->scratchRays[i]) cudaFree(scene->scratchRays[i]);
		if (scene->scratchOut[i]) cudaFree(scene->scratchOut[i]);
		scene->scratchRays[i] = scene->scratchOut[i] = nullptr;
	}

	scene->scratchCapacity = 0;

	for (int i = 0; i < EchoScene::kSlots; i++)
	{
		if (!check_cuda(cudaMalloc(&scene->scratchRays[i], sizeof(EchoRay) * rays), "cudaMalloc(scratch rays)")) return false;
		if (!check_cuda(cudaMalloc(&scene->scratchOut[i], sizeof(EchoHit) * rays), "cudaMalloc(scratch out)")) return false;
		if (!scene->copyStreams[i] && !check_cuda(cudaStreamCreateWithFlags(&scene->copyStreams[i], cudaStreamNonBlocking), "cudaStreamCreate")) return false;
		if (!scene->chunkDone[i] && !check_cuda(cudaEventCreateWithFlags(&scene->chunkDone[i], cudaEventDisableTiming), "cudaEventCreate")) return false;
	}

	scene->scratchCapacity = rays;
	return true;
}

// ordinary (pageable) host memory, as opposed to cudaHostAlloc / cudaHostRegister memory? Unknown pointers count as pageable.
bool is_pageable(const void* pointer)
{
	cudaPointerAttributes attributes;
	if (cudaPointerGetAttributes(&attributes, pointer) != cudaSuccess) { cudaGetLastError(); return true; }
	return attributes.type == cudaMemoryTypeUnregistered;
}

bool ensure_staging(EchoScene* scene, uint64_t rays)
{
	if (scene->stagingCapacity >= rays) return true;

	for (int i = 0; i < EchoScene::kSlots; i++)
	{
		if (scene->stagingIn[i]) cudaFreeHost(scene->stagingIn[i]);
		if (scene->stagingOut[i]) cudaFreeHost(scene->stagingOut[i]);
		scene->stagingIn[i] = scene->stagingOut[i] = nullptr;
	}

	scene->stagingCapacity = 0;

	for (int i = 0; i < EchoScene::kSlots; i++)
		if (!check_cuda(cudaHostAlloc(&scene->stagingIn[i], sizeof(EchoRay) * rays, cudaHostAllocDefault), "cudaHostAlloc(staging)")
			|| !check_cuda(cudaHostAlloc(&scene->stagingOut[i], sizeof(EchoHit) * rays, cudaHostAllocDefault), "cudaHostAlloc(staging)")) return false;

	scene->stagingCapacity = rays;
	return true;
}

// Host-buffer batch from PAGEABLE memory — what a P/Invoke caller hands over when it pins a managed array with `fixed`
// (OidnDenoise.cs:109-110) instead of using echo_b200_host_alloc / _register. cudaMemcpyAsync from such memory is neither
// asynchronous nor fast (the driver stages it through one bounce buffer on the calling thread: 255 Mrays/s end to end against 1 530
// from page-locked memory). Here every slot of the pipeline gets a host thread of its own that copies its chunks into page-locked
// staging, runs upload / kernel / download on its stream and copies the results out: kSlots concurrent memcpys feed the link, and the
// chunks of different slots overlap on the device as in the page-locked path.
template<class Out, class Launch>
int32_t batch_host_staged(EchoScene* scene, const EchoRay* rays, uint64_t n, Out* out, uint64_t chunk, Launch launch)
{
	if (!ensure_staging(scene, chunk)) return ECHO_B200_ERR_CUDA;

	const uint64_t chunks = (n + chunk - 1) / chunk;
	std::vector<std::string> errors(EchoScene::kSlots);
	std::vector<char> failed(EchoScene::kSlots, 0);

	auto work = [&](int slot)
	{
		DeviceGuard guard(scene->device);
		bool ok = guard.ok;
		cudaStream_t stream = scene->copyStreams[slot];

		for (uint64_t index = (uint64_t)slot; ok && index < chunks; index += EchoScene::kSlots)
		{
			uint64_t first = index * chunk, count = std::min<uint64_t>(chunk, n - first);
			std::memcpy(scene->stagingIn[slot], rays + first, sizeof(EchoRay) * count);
			ok = check_cuda(cudaMemcpyAsync(scene->scratchRays[slot], scene->stagingIn[slot], sizeof(EchoRay) * count, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(rays)")
				&& launch((const EchoRay*)scene->scratchRays[slot], count, (Out*)scene->scratchOut[slot], stream)
				&& check_cuda(cudaMemcpyAsync(scene->stagingOut[slot], scene->scratchOut[slot], sizeof(Out) * count, cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(out)")
				&& check_cuda(cudaStreamSynchronize(stream), "batch");
			if (ok) std::memcpy(out + first, scene->stagingOut[slot], sizeof(Out) * count);
		}

		if (!ok)
		{
			cudaStreamSynchronize(stream);
			failed[slot] = 1;
			errors[slot] = last_error_string();
		}
	};

	std::vector<std::thread> threads;
	for (int slot = 1; slot < EchoScene::kSlots; slot++) threads.emplace_back(work, slot);
	work(0);
	for (std::thread& thread : threads) thread.join();

	for (int slot = 0; slot < EchoScene::kSlots; slot++)
	{
		if (!failed[slot]) continue;
		set_error(errors[slot]);
		return ECHO_B200_ERR_CUDA;
	}

	return ECHO_B200_OK;
}

// Host-buffer batch: chunks rotate over kSlots streams so that chunk k's upload overlaps the kernels and downloads of the
// chunks before it (H2D, compute and D2H engines run concurrently). With pinned host buffers the copies are truly asynchronous.
template<class Out, class Launch>
int32_t batch_host(EchoScene* scene, const EchoRay* rays, uint64_t n, Out* out, Launch launch)
{
	if (!require_committed(scene)) return ECHO_B200_ERR_INVALID;
	if (n == 0) return ECHO_B200_OK;
	if (!rays || !out) return fail(ECHO_B200_ERR_INVALID, "null buffer");

	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	std::lock_guard<std::mutex> turn(scene->compute);

	uint64_t chunk = std::min<uint64_t>(chunk_rays(), n);
	if (!ensure_scratch(scene, chunk)) return ECHO_B200_ERR_CUDA;

	// pageable caller memory: staged through page-locked buffers by one host thread per slot (small batches are not worth the threads)
	static const bool staging = [] { const char* text = getenv("ECHO_B200_STAGE_PAGEABLE"); return !text || text[0] != '0'; }();
	if (staging && n >= 4 * chunk && (is_pageable(rays) || is_pageable(out))) return batch_host_staged<Out>(scene, rays, n, out, chunk, launch);

	int slot = 0;
	bool ok = true;

	for (uint64_t first = 0; ok && first < n; first += chunk, slot = (slot + 1) % EchoScene::kSlots)
	{
		uint64_t count = std::min<uint64_t>(chunk, n - first);
		cudaStream_t stream = scene->copyStreams[slot];

		ok = check_cuda(cudaMemcpyAsync(scene->scratchRays[slot], rays + first, sizeof(EchoRay) * count, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(rays)")
			&& launch((const EchoRay*)scene->scratchRays[slot], count, (Out*)scene->scratchOut[slot], stream)
			&& check_cuda(cudaMemcpyAsync(out + first, scene->scratchOut[slot], sizeof(Out) * count, cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(out)");
	}

	// Also after a failed enqueue: downloads of earlier chunks may still be writing into the caller's buffer, which the caller
	// is free to release as soon as this call returns. The first error is the one reported.
	std::string firstError = ok ? std::string() : last_error_string();

	for (int i = 0; i < EchoScene::kSlots; i++)
		if (!check_cuda(cudaStreamSynchronize(scene->copyStreams[i]), "batch") && ok) { ok = false; firstError = last_error_string(); }

	if (!ok) set_error(firstError);
	return ok ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

// Multi-device scenes (echo_b200_scene_create_multi): runs `work(scene of device g, g)` for the primary and every replica, one host
// thread per device. Returns the first failing status with that thread's error text as the caller's last error.
template<class Work>
int32_t fan_out(EchoScene* scene, Work work)
{
	const size_t devices = 1 + scene->replicas.size();
	std::vector<int32_t> status(devices, ECHO_B200_OK);
	std::vector<std::string> errors(devices);

	auto run = [&](size_t g)
	{
		status[g] = work(g == 0 ? scene : scene->replicas[g - 1], g);
		if (status[g] != ECHO_B200_OK) errors[g] = last_error_string();
	};

	std::vector<std::thread> threads;
	for (size_t g = 1; g < devices; g++) threads.emplace_back(run, g);
	run(0);
	for (std::thread& thread : threads) thread.join();

	for (size_t g = 0; g < devices; g++)
	{
		if (status[g] == ECHO_B200_OK) continue;
		set_error(errors[g]);
		return status[g];
	}

	return ECHO_B200_OK;
}

bool single_device(EchoScene* scene)
{
	if (scene && !scene->replicas.empty()) { set_error("this entry point takes device memory of one device: it needs a single-device scene (echo_b200_scene_create)"); return false; }
	return true;
}

constexpr uint32_t kDealBlock = 64; // consecutive tiles of the caller's sequence that stay on one device (echo_b200.h, scene_create_multi)

} // namespace

extern "C"
{

const char* echo_b200_last_error(void) { return lastError.c_str(); }
const char* echo_b200_version(void) { return "echo-b200 0.1 (sm_100a)"; }

int32_t echo_b200_device_count(int32_t* out)
{
	if (!out) return fail(ECHO_B200_ERR_INVALID, "out is null");
	int count = 0;
	cudaError_t status = cudaGetDeviceCount(&count);

	if (status != cudaSuccess || count == 0)
	{
		*out = 0;
		cudaGetLastError();
		return fail(ECHO_B200_ERR_NO_DEVICE, "no usable CUDA device");
	}

	*out = count;
	return ECHO_B200_OK;
}

int32_t echo_b200_host_alloc(void** out, uint64_t bytes)
{
	if (!out) return fail(ECHO_B200_ERR_INVALID, "out is null");
	*out = nullptr;
	int32_t count = 0;
	int32_t status = echo_b200_device_count(&count);
	if (status != ECHO_B200_OK) return status;
	// portable: page-locked for every device of the process, not only the current one
	return check_cuda(cudaHostAlloc(out, std::max<uint64_t>(bytes, 1), cudaHostAllocPortable), "cudaHostAlloc") ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_host_free(void* pointer)
{
	if (!pointer) return ECHO_B200_OK;
	return check_cuda(cudaFreeHost(pointer), "cudaFreeHost") ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_host_register(void* pointer, uint64_t bytes)
{
	if (!pointer || bytes == 0) return fail(ECHO_B200_ERR_INVALID, "null or empty range");
	int32_t count = 0;
	int32_t status = echo_b200_device_count(&count);
	if (status != ECHO_B200_OK) return status;
	return check_cuda(cudaHostRegister(pointer, bytes, cudaHostRegisterPortable), "cudaHostRegister") ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_host_unregister(void* pointer)
{
	if (!pointer) return ECHO_B200_OK;
	return check_cuda(cudaHostUnregister(pointer), "cudaHostUnregister") ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_scene_create(EchoScene** out, int32_t device)
{
	if (!out) return fail(ECHO_B200_ERR_INVALID, "out is null");
	*out = nullptr;

	int32_t count = 0;
	int32_t status = echo_b200_device_count(&count);
	if (status != ECHO_B200_OK) return status;
	if (device < 0 || device >= count) return fail(ECHO_B200_ERR_INVALID, "device index out of range");

	EchoScene* scene = new EchoScene();
	scene->device = device;

	DeviceGuard guard(device);

	if (!guard.ok || !check_cuda(cudaStreamCreateWithFlags(&scene->stream, cudaStreamNonBlocking), "cudaStreamCreate"))
	{
		delete scene;
		return ECHO_B200_ERR_CUDA;
	}

	scene->render = render_state_create();
	*out = scene;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_create_multi(EchoScene** out, uint64_t deviceMask)
{
	if (!out) return fail(ECHO_B200_ERR_INVALID, "out is null");
	*out = nullptr;

	int32_t count = 0;
	int32_t status = echo_b200_device_count(&count);
	if (status != ECHO_B200_OK) return status;
	if (deviceMask == 0) return fail(ECHO_B200_ERR_INVALID, "device_mask is empty");
	if (count < 64 && (deviceMask >> count) != 0) return fail(ECHO_B200_ERR_INVALID, "device_mask names a device that does not exist");

	EchoScene* primary = nullptr;

	for (int32_t device = 0; device < count && device < 64; device++)
	{
		if (((deviceMask >> device) & 1ull) == 0) continue;
		EchoScene* scene = nullptr;
		status = echo_b200_scene_create(&scene, device);

		if (status != ECHO_B200_OK)
		{
			std::string error = last_error_string();
			echo_b200_scene_destroy(primary);
			set_error(error);
			return status;
		}

		if (!primary) primary = scene;
		else primary->replicas.push_back(scene);
	}

	*out = primary;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_gpu_count(EchoScene* scene, int32_t* out)
{
	if (!scene || !out) return fail(ECHO_B200_ERR_INVALID, "null argument");
	*out = 1 + (int32_t)scene->replicas.size();
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_destroy(EchoScene* scene)
{
	if (!scene) return ECHO_B200_OK;
	for (EchoScene* replica : scene->replicas) echo_b200_scene_destroy(replica);
	scene->replicas.clear();
	DeviceGuard guard(scene->device);
	free_device(scene);
	render_state_destroy(scene->render);

	for (int i = 0; i < EchoScene::kSlots; i++)
	{
		if (scene->scratchRays[i]) cudaFree(scene->scratchRays[i]);
		if (scene->scratchOut[i]) cudaFree(scene->scratchOut[i]);
		if (scene->copyStreams[i]) cudaStreamDestroy(scene->copyStreams[i]);
		if (scene->chunkDone[i]) cudaEventDestroy(scene->chunkDone[i]);
		if (scene->stagingIn[i]) cudaFreeHost(scene->stagingIn[i]);
		if (scene->stagingOut[i]) cudaFreeHost(scene->stagingOut[i]);
	}

	if (scene->tilesOut) cudaFree(scene->tilesOut);
	for (void* pointer : scene->hierarchyScratch) if (pointer) cudaFree(pointer);
	if (scene->stream) cudaStreamDestroy(scene->stream);
	delete scene;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_set_qbvh(EchoScene* scene, const EchoQbvhNode* nodes, uint32_t count, uint32_t maxDepth)
{
	if (!scene || (!nodes && count)) return fail(ECHO_B200_ERR_INVALID, "null argument");
	if (count == 0) return fail(ECHO_B200_ERR_INVALID, "a QBVH needs at least one node");
	if (stack_class(maxDepth) < 0) return fail(ECHO_B200_ERR_UNSUPPORTED, "QBVH deeper than 63 quad levels is not supported");
	scene->nodes.assign(nodes, nodes + count);
	scene->maxDepth = maxDepth;
	scene->committed = false;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_build_qbvh(EchoScene* scene, uint32_t* outNodeCount, uint32_t* outMaxDepth)
{
	if (!scene) return fail(ECHO_B200_ERR_INVALID, "null argument");
	if (!scene->packs.empty()) return fail(ECHO_B200_ERR_UNSUPPORTED, "scene_build_qbvh builds the accelerator of a scene without packs; build each pack with echo_b200_build_qbvh_instanced");
	uint64_t total = (uint64_t)scene->triangles.size() + scene->spheres.size();
	if (total < 2) return fail(ECHO_B200_ERR_INVALID, "upload at least two primitives (set_triangles / set_spheres) before scene_build_qbvh");
	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;

	std::vector<EchoQbvhNode> nodes(total - 1);
	uint32_t count = 0, depth = 0;
	if (!build_qbvh_device(scene->triangles.data(), (uint32_t)scene->triangles.size(), scene->spheres.data(), (uint32_t)scene->spheres.size(), nullptr, 0u, nodes.data(), &count, &depth))
		return ECHO_B200_ERR_CUDA;
	if (stack_class(depth) < 0) return fail(ECHO_B200_ERR_UNSUPPORTED, "QBVH deeper than 63 quad levels is not supported");

	nodes.resize(count);
	scene->nodes.swap(nodes);
	scene->maxDepth = depth;
	scene->committed = false;
	if (outNodeCount) *outNodeCount = count;
	if (outMaxDepth) *outMaxDepth = depth;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_set_triangles(EchoScene* scene, const EchoTriangle* triangles, uint32_t count)
{
	if (!scene || (!triangles && count)) return fail(ECHO_B200_ERR_INVALID, "null argument");
	scene->triangles.assign(triangles, triangles + count);
	scene->committed = false;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_set_spheres(EchoScene* scene, const EchoSphere* spheres, uint32_t count)
{
	if (!scene || (!spheres && count)) return fail(ECHO_B200_ERR_INVALID, "null argument");
	scene->spheres.assign(spheres, spheres + count);
	scene->committed = false;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_set_materials(EchoScene* scene, const EchoMaterial* materials, uint32_t count)
{
	if (!scene || (!materials && count)) return fail(ECHO_B200_ERR_INVALID, "null argument");

	for (uint32_t i = 0; i < count; i++)
	{
		if (materials[i].type > ECHO_MATERIAL_COATED_DIFFUSE) return fail(ECHO_B200_ERR_UNSUPPORTED, "material type outside the hot path");
		if (materials[i].type == ECHO_MATERIAL_ONESIDED && materials[i].base >= count) return fail(ECHO_B200_ERR_INVALID, "OneSided base index out of range");
	}

	scene->materials.assign(materials, materials + count);
	scene->committed = false;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_set_light_tree(EchoScene* scene, const EchoLightNode* nodes, uint32_t nodeCount, const uint32_t* tokens, const uint64_t* paths,
                                       uint32_t emitterCount, const EchoPointLight* points, uint32_t pointCount)
{
	if (!scene || (!nodes && nodeCount) || ((!tokens || !paths) && emitterCount) || (!points && pointCount)) return fail(ECHO_B200_ERR_INVALID, "null argument");
	scene->lightNodes.assign(nodes, nodes + nodeCount);

	// LightTree.map: kept as given here; commit sorts each pack's range for the device's binary search
	scene->emitterTokens.assign(tokens, tokens + emitterCount);
	scene->emitterPaths.assign(paths, paths + emitterCount);

	scene->pointLights.assign(points, points + pointCount);
	scene->committed = false;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_set_infinite(EchoScene* scene, const EchoInfiniteLight* lights, uint32_t count, float threshold, float pdf)
{
	if (!scene || (!lights && count)) return fail(ECHO_B200_ERR_INVALID, "null argument");
	scene->infiniteLights.assign(lights, lights + count);
	scene->infiniteThreshold = threshold;
	scene->infinitePdf = pdf;
	scene->committed = false;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_set_camera(EchoScene* scene, const EchoCamera* camera)
{
	if (!scene || !camera) return fail(ECHO_B200_ERR_INVALID, "null argument");
	scene->camera = *camera;
	if (scene->committed) scene->d.camera = *camera; // the camera travels by value with every launch
	for (EchoScene* replica : scene->replicas) echo_b200_scene_set_camera(replica, camera);
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_set_textures(EchoScene* scene, const EchoTexture* textures, uint32_t textureCount, const float* texels, uint64_t texelCount,
                                     const EchoMaterialTextures* materialTextures, uint32_t materialCount)
{
	if (!scene || (!textures && textureCount) || (!texels && texelCount) || (!materialTextures && textureCount)) return fail(ECHO_B200_ERR_INVALID, "null argument");

	for (uint32_t i = 0; i < textureCount; i++)
	{
		const EchoTexture& t = textures[i];
		if (t.width == 0 || t.height == 0 || (uint64_t)t.texelOffset + (uint64_t)t.width * t.height > texelCount) return fail(ECHO_B200_ERR_INVALID, "texture range out of bounds");
		if (t.filter > ECHO_FILTER_BILINEAR || t.wrapper > ECHO_WRAPPER_MIRROR) return fail(ECHO_B200_ERR_UNSUPPORTED, "unknown texture filter or wrapper");
	}

	for (uint32_t i = 0; textureCount && i < materialCount; i++)
	{
		const EchoMaterialTextures& m = materialTextures[i];
		for (uint32_t slot : { m.albedo, m.normal, m.roughness, m.paramA, m.paramB })
			if (slot != ECHO_TEXTURE_NONE && slot >= textureCount) return fail(ECHO_B200_ERR_INVALID, "material texture slot out of range");
	}

	scene->textures.assign(textures, textures + textureCount);
	scene->texels.assign(texels, texels + texelCount * 4);
	scene->materialTextures.assign(materialTextures, materialTextures + (textureCount ? materialCount : 0));
	scene->committed = false;
	return ECHO_B200_OK;
}

int32_t echo_b200_build_qbvh_instanced(int32_t device, const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
                                       const float* instanceBounds, uint32_t instanceCount, EchoQbvhNode* outNodes, uint32_t* outNodeCount, uint32_t* outMaxDepth)
{
	if ((!triangles && triangleCount) || (!spheres && sphereCount) || (!instanceBounds && instanceCount) || !outNodes || !outNodeCount || !outMaxDepth) return fail(ECHO_B200_ERR_INVALID, "null argument");
	int32_t count = 0;
	int32_t status = echo_b200_device_count(&count);
	if (status != ECHO_B200_OK) return status;
	if (device < 0 || device >= count) return fail(ECHO_B200_ERR_INVALID, "device index out of range");
	DeviceGuard guard(device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	return build_qbvh_device(triangles, triangleCount, spheres, sphereCount, instanceBounds, instanceCount, outNodes, outNodeCount, outMaxDepth) ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_build_qbvh(int32_t device, const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
                             EchoQbvhNode* outNodes, uint32_t* outNodeCount, uint32_t* outMaxDepth)
{
	return echo_b200_build_qbvh_instanced(device, triangles, triangleCount, spheres, sphereCount, nullptr, 0u, outNodes, outNodeCount, outMaxDepth);
}

int32_t echo_b200_build_light_tree(int32_t device, const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
                                   const EchoMaterial* materials, uint32_t materialCount, const EchoPointLight* points, uint32_t pointCount,
                                   const float* instanceLights, uint32_t instanceCount,
                                   EchoLightNode* outNodes, uint32_t nodeCapacity, uint32_t* outNodeCount,
                                   uint32_t* outTokens, uint64_t* outPaths, uint32_t emitterCapacity, uint32_t* outEmitterCount, float* outPower)
{
	if ((!triangles && triangleCount) || (!spheres && sphereCount) || (!materials && materialCount) || (!points && pointCount) || (!instanceLights && instanceCount)
		|| (!outNodes && nodeCapacity) || ((!outTokens || !outPaths) && emitterCapacity) || !outNodeCount || !outEmitterCount || !outPower) return fail(ECHO_B200_ERR_INVALID, "null argument");
	int32_t count = 0;
	int32_t status = echo_b200_device_count(&count);
	if (status != ECHO_B200_OK) return status;
	if (device < 0 || device >= count) return fail(ECHO_B200_ERR_INVALID, "device index out of range");
	DeviceGuard guard(device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;

	const lightbuild::Sources sources = { triangles, triangleCount, spheres, sphereCount, materials, materialCount, points, pointCount, instanceLights, instanceCount };
	std::vector<EchoLightNode> nodes;
	std::vector<uint32_t> tokens;
	std::vector<uint64_t> paths;
	bool refused = false;
	if (!build_light_tree_device(sources, nodes, tokens, paths, &refused)) return ECHO_B200_ERR_CUDA;
	if (refused) return fail(ECHO_B200_ERR_UNSUPPORTED, "light tree deeper than 63 levels (LightTree.cs:29)");

	*outNodeCount = (uint32_t)nodes.size();
	*outEmitterCount = (uint32_t)tokens.size();
	*outPower = nodes.empty() ? 0.0f : nodes[0].power;
	if (nodes.size() > nodeCapacity || tokens.size() > emitterCapacity) return fail(ECHO_B200_ERR_INVALID, "light tree output buffers too small (needed counts returned)");

	std::copy(nodes.begin(), nodes.end(), outNodes);
	std::copy(tokens.begin(), tokens.end(), outTokens);
	std::copy(paths.begin(), paths.end(), outPaths);
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_build_light_tree(EchoScene* scene, const EchoPointLight* points, uint32_t pointCount, uint32_t* outNodeCount, uint32_t* outEmitterCount, float* outPower)
{
	if (!scene || (!points && pointCount)) return fail(ECHO_B200_ERR_INVALID, "null argument");
	if (!scene->packs.empty()) return fail(ECHO_B200_ERR_UNSUPPORTED, "scene_build_light_tree builds the light tree of a scene without packs; build each pack with echo_b200_build_light_tree");
	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;

	const lightbuild::Sources sources = { scene->triangles.data(), (uint32_t)scene->triangles.size(), scene->spheres.data(), (uint32_t)scene->spheres.size(),
	                                      scene->materials.data(), (uint32_t)scene->materials.size(), points, pointCount, nullptr, 0u };
	std::vector<EchoLightNode> nodes;
	std::vector<uint32_t> tokens;
	std::vector<uint64_t> paths;
	bool refused = false;
	if (!build_light_tree_device(sources, nodes, tokens, paths, &refused)) return ECHO_B200_ERR_CUDA;
	if (refused) return fail(ECHO_B200_ERR_UNSUPPORTED, "light tree deeper than 63 levels (LightTree.cs:29)");

	if (outNodeCount) *outNodeCount = (uint32_t)nodes.size();
	if (outEmitterCount) *outEmitterCount = (uint32_t)tokens.size();
	if (outPower) *outPower = nodes.empty() ? 0.0f : nodes[0].power;

	scene->lightNodes.swap(nodes);
	scene->emitterTokens.swap(tokens);
	scene->emitterPaths.swap(paths);
	scene->pointLights.assign(points, points + pointCount);
	scene->committed = false;
	return ECHO_B200_OK;
}

int32_t echo_b200_build_packs(int32_t device, const EchoTriangle* triangles, uint32_t triangleCount, const EchoSphere* spheres, uint32_t sphereCount,
                              const EchoMaterial* materials, uint32_t materialCount, const EchoPointLight* points, uint32_t pointCount,
                              EchoPack* packs, uint32_t packCount, const EchoInstance* instances, uint32_t instanceCount,
                              EchoQbvhNode* outNodes, uint32_t nodeCapacity, uint32_t* outNodeCount,
                              EchoLightNode* outLightNodes, uint32_t lightNodeCapacity, uint32_t* outLightNodeCount,
                              uint32_t* outTokens, uint64_t* outPaths, uint32_t emitterCapacity, uint32_t* outEmitterCount, float* outPower)
{
	if ((!triangles && triangleCount) || (!spheres && sphereCount) || (!materials && materialCount) || (!points && pointCount) || !packs || (!instances && instanceCount)
		|| (!outNodes && nodeCapacity) || (!outLightNodes && lightNodeCapacity) || ((!outTokens || !outPaths) && emitterCapacity)
		|| !outNodeCount || !outLightNodeCount || !outEmitterCount || !outPower) return fail(ECHO_B200_ERR_INVALID, "null argument");
	int32_t count = 0;
	int32_t status = echo_b200_device_count(&count);
	if (status != ECHO_B200_OK) return status;
	if (device < 0 || device >= count) return fail(ECHO_B200_ERR_INVALID, "device index out of range");
	DeviceGuard guard(device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;

	const packbuild::Inputs inputs = { triangles, triangleCount, spheres, sphereCount, materials, materialCount, points, pointCount, packs, packCount, instances, instanceCount };
	packbuild::Output output;
	status = build_packs_device(inputs, output);
	if (status != ECHO_B200_OK) return status;

	std::string message;
	status = packbuild::deliver(output, packs, outNodes, nodeCapacity, outNodeCount, outLightNodes, lightNodeCapacity, outLightNodeCount, outTokens, outPaths, emitterCapacity,
	                            outEmitterCount, outPower, message);
	return status == ECHO_B200_OK ? status : fail(status, message.c_str());
}

int32_t echo_b200_scene_build_packs(EchoScene* scene, const EchoPointLight* points, uint32_t pointCount, uint32_t* outNodeCount, uint32_t* outLightNodeCount,
                                    uint32_t* outEmitterCount, float* outPower)
{
	if (!scene || (!points && pointCount)) return fail(ECHO_B200_ERR_INVALID, "null argument");
	if (scene->packs.empty()) return fail(ECHO_B200_ERR_INVALID, "scene_build_packs builds the packs declared with set_packs; a scene without packs uses scene_build_qbvh / scene_build_light_tree");
	DeviceGuard guard(scene->device); // a multi-device handle builds on its first device; commit replicates the staging
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;

	const packbuild::Inputs inputs = { scene->triangles.data(), (uint32_t)scene->triangles.size(), scene->spheres.data(), (uint32_t)scene->spheres.size(),
	                                   scene->materials.data(), (uint32_t)scene->materials.size(), points, pointCount, scene->packs.data(), (uint32_t)scene->packs.size(),
	                                   scene->instances.data(), (uint32_t)scene->instances.size() };
	packbuild::Output output;
	int32_t status = build_packs_device(inputs, output);
	if (status != ECHO_B200_OK) return status;

	uint32_t maxDepth = 0;
	for (const EchoPack& pack : output.packs) maxDepth = std::max(maxDepth, pack.maxDepth);
	if (outNodeCount) *outNodeCount = (uint32_t)output.nodes.size();
	if (outLightNodeCount) *outLightNodeCount = (uint32_t)output.lightNodes.size();
	if (outEmitterCount) *outEmitterCount = (uint32_t)output.emitterTokens.size();
	if (outPower) *outPower = output.power;

	scene->nodes.swap(output.nodes);
	scene->maxDepth = maxDepth;
	scene->packs.swap(output.packs);
	scene->lightNodes.swap(output.lightNodes);
	scene->emitterTokens.swap(output.emitterTokens);
	scene->emitterPaths.swap(output.emitterPaths);
	scene->pointLights.assign(points, points + pointCount);
	scene->committed = false;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_set_distributions(EchoScene* scene, const float* values, uint64_t count)
{
	if (!scene || (!values && count)) return fail(ECHO_B200_ERR_INVALID, "null argument");
	scene->distributions.assign(values, values + count);
	scene->committed = false;
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_set_bound_radius(EchoScene* scene, float radius)
{
	if (!scene) return fail(ECHO_B200_ERR_INVALID, "null argument");
	scene->boundRadius = radius;
	if (scene->committed) scene->d.boundRadius = radius; // travels by value with every launch, like the camera
	for (EchoScene* replica : scene->replicas) echo_b200_scene_set_bound_radius(replica, radius);
	return ECHO_B200_OK;
}

int32_t echo_b200_scene_set_packs(EchoScene* scene, const EchoPack* packs, uint32_t packCount, const EchoInstance* instances, uint32_t instanceCount)
{
	if (!scene || (!packs && packCount) || (!instances && instanceCount)) return fail(ECHO_B200_ERR_INVALID, "null argument");
	scene->packs.assign(packs, packs + packCount);
	scene->instances.assign(instances, instances + instanceCount);
	scene->committed = false;
	return ECHO_B200_OK;
}

namespace
{

// Traversal stack entries the deepest chain of packs needs from `pack` down: the reference stackallocs maxDepth * 3 + 1 per
// recursion (QuadBoundingVolumeHierarchy.cs:34,125); the device keeps all layers in one stack. Memoised per pack (a pack placed
// 1e5 times is walked once): `need[p]` entries and `height[p]` layers below p, `mark` = 1 while p is on the walk (a cycle), 2 when done.
// false = cyclic or deeper than TokenHierarchy.MaxLayer.
bool chain_stack(const EchoScene* scene, uint32_t pack, std::vector<uint32_t>& need, std::vector<uint32_t>& height, std::vector<uint8_t>& mark)
{
	if (mark[pack] == 2) return true;
	if (mark[pack] == 1) return false; // the pack contains itself
	mark[pack] = 1;

	const EchoPack& p = scene->packs[pack];
	uint32_t deepest = 0u, layers = 0u;

	for (uint32_t i = 0; i < p.instanceCount; i++)
	{
		uint32_t child = scene->instances[p.instanceOffset + i].pack;
		if (!chain_stack(scene, child, need, height, mark)) return false;
		deepest = std::max(deepest, need[child]);
		layers = std::max(layers, height[child] + 1u);
	}

	if (layers > ECHO_MAX_INSTANCE_LAYERS) return false;
	need[pack] = p.maxDepth * 3u + 1u + deepest;
	height[pack] = layers;
	mark[pack] = 2;
	return true;
}

} // namespace

static int32_t commit_device(EchoScene* scene);

// the host staging of a scene: what the set_* calls filled and commit reads
static void swap_staging(EchoScene* a, EchoScene* b)
{
	std::swap(a->nodes, b->nodes);
	std::swap(a->maxDepth, b->maxDepth);
	std::swap(a->triangles, b->triangles);
	std::swap(a->spheres, b->spheres);
	std::swap(a->materials, b->materials);
	std::swap(a->lightNodes, b->lightNodes);
	std::swap(a->emitterTokens, b->emitterTokens);
	std::swap(a->emitterPaths, b->emitterPaths);
	std::swap(a->pointLights, b->pointLights);
	std::swap(a->infiniteLights, b->infiniteLights);
	std::swap(a->infiniteThreshold, b->infiniteThreshold);
	std::swap(a->infinitePdf, b->infinitePdf);
	std::swap(a->camera, b->camera);
	std::swap(a->boundRadius, b->boundRadius);
	std::swap(a->distributions, b->distributions);
	std::swap(a->textures, b->textures);
	std::swap(a->texels, b->texels);
	std::swap(a->materialTextures, b->materialTextures);
	std::swap(a->packs, b->packs);
	std::swap(a->instances, b->instances);
}

int32_t echo_b200_scene_commit(EchoScene* scene)
{
	if (!scene) return fail(ECHO_B200_ERR_INVALID, "scene is null");
	int32_t status = commit_device(scene);

	// the same staging, uploaded to every other device of a multi-device scene (lent to the replica for the duration of its commit)
	for (size_t i = 0; status == ECHO_B200_OK && i < scene->replicas.size(); i++)
	{
		swap_staging(scene, scene->replicas[i]);
		status = commit_device(scene->replicas[i]);
		swap_staging(scene, scene->replicas[i]);
	}

	return status;
}

static int32_t commit_device(EchoScene* scene)
{
	if (scene->nodes.empty()) return fail(ECHO_B200_ERR_INVALID, "no QBVH was set");

	// the packs the arrays are divided into; a scene without set_packs is one pack
	std::vector<EchoPack> packs = scene->packs;

	if (packs.empty())
	{
		if (!scene->instances.empty()) return fail(ECHO_B200_ERR_INVALID, "instances without packs");
		EchoPack whole = {};
		whole.nodeCount = (uint32_t)scene->nodes.size();
		whole.maxDepth = scene->maxDepth;
		whole.triangleCount = (uint32_t)scene->triangles.size();
		whole.sphereCount = (uint32_t)scene->spheres.size();
		packs.push_back(whole);
	}

	for (const EchoPack& pack : packs)
	{
		if (pack.nodeCount == 0 || (uint64_t)pack.nodeOffset + pack.nodeCount > scene->nodes.size() || (uint64_t)pack.triangleOffset + pack.triangleCount > scene->triangles.size()
			|| (uint64_t)pack.sphereOffset + pack.sphereCount > scene->spheres.size() || (uint64_t)pack.instanceOffset + pack.instanceCount > scene->instances.size())
			return fail(ECHO_B200_ERR_INVALID, "pack range out of bounds");

		// every token in the pack's nodes must point at one of the pack's own primitives
		for (uint32_t n = 0; n < pack.nodeCount; n++)
		{
			for (uint32_t token : scene->nodes[pack.nodeOffset + n].token4)
			{
				if (token == ECHO_TOKEN_EMPTY) continue;
				uint32_t type = token >> ECHO_TOKEN_INDEX_BITS, index = token & ((1u << ECHO_TOKEN_INDEX_BITS) - 1u);
				bool ok = (type == ECHO_TOKEN_TYPE_NODE && index < pack.nodeCount) || (type == ECHO_TOKEN_TYPE_TRIANGLE && index < pack.triangleCount)
					|| (type == ECHO_TOKEN_TYPE_SPHERE && index < pack.sphereCount) || (type == ECHO_TOKEN_TYPE_INSTANCE && index < pack.instanceCount);
				if (!ok) return fail(ECHO_B200_ERR_INVALID, "QBVH token out of range");
			}
		}
	}

	for (const EchoInstance& instance : scene->instances)
		if (instance.pack >= packs.size() || instance.pack == 0u) return fail(ECHO_B200_ERR_INVALID, "instance refers to a pack that does not exist (pack 0 is the scene)");

	uint32_t stackDepth = scene->maxDepth;

	if (!scene->packs.empty())
	{
		std::vector<uint32_t> need(scene->packs.size(), 0u), height(scene->packs.size(), 0u);
		std::vector<uint8_t> mark(scene->packs.size(), 0);
		uint32_t entries = chain_stack(scene, 0u, need, height, mark) ? need[0] : 0u;
		if (entries == 0u) return fail(ECHO_B200_ERR_INVALID, "instancing deeper than TokenHierarchy.MaxLayer (5) or cyclic");
		stackDepth = (entries + 1u) / 3u; // smallest depth with depth * 3 + 1 >= entries
		if (stack_class(stackDepth) < 0) return fail(ECHO_B200_ERR_UNSUPPORTED, "the deepest chain of instanced packs needs more than 192 stack entries");
	}

	for (const EchoTriangle& t : scene->triangles)
		if (t.material >= scene->materials.size() && !scene->materials.empty()) return fail(ECHO_B200_ERR_INVALID, "triangle material index out of range");
	for (const EchoSphere& s : scene->spheres)
		if (s.material >= scene->materials.size() && !scene->materials.empty()) return fail(ECHO_B200_ERR_INVALID, "sphere material index out of range");

	// LightTree.map of every pack as a sorted array (binary-searched on the device)
	std::vector<uint32_t> emitterTokens(scene->emitterTokens.size());
	std::vector<uint64_t> emitterPaths(scene->emitterPaths.size());

	if (scene->packs.empty())
	{
		packs[0].lightNodeCount = (uint32_t)scene->lightNodes.size();
		packs[0].emitterCount = (uint32_t)scene->emitterTokens.size();
		packs[0].pointLightCount = (uint32_t)scene->pointLights.size();
	}

	for (const EchoPack& pack : packs)
	{
		if ((uint64_t)pack.lightNodeOffset + pack.lightNodeCount > scene->lightNodes.size() || (uint64_t)pack.emitterOffset + pack.emitterCount > scene->emitterTokens.size()
			|| (uint64_t)pack.pointLightOffset + pack.pointLightCount > scene->pointLights.size())
			return fail(ECHO_B200_ERR_INVALID, "pack light range out of bounds");

		std::vector<uint32_t> order(pack.emitterCount);
		std::iota(order.begin(), order.end(), 0u);
		const uint32_t* tokens = scene->emitterTokens.data() + pack.emitterOffset;
		std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return tokens[a] < tokens[b]; });

		for (uint32_t i = 0; i < pack.emitterCount; i++)
		{
			emitterTokens[pack.emitterOffset + i] = tokens[order[i]];
			emitterPaths[pack.emitterOffset + i] = scene->emitterPaths[pack.emitterOffset + order[i]];
		}
	}

	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	free_device(scene);

	DeviceScene& d = scene->d;
	d = DeviceScene{};

	// layout conversion (DESIGN.md "Data layout in HBM")
	std::vector<float4> triHot(scene->triangles.size() * 3), triShade(scene->triangles.size() * 3);

	for (size_t i = 0; i < scene->triangles.size(); i++)
	{
		const EchoTriangle& t = scene->triangles[i];
		float materialBits;
		std::memcpy(&materialBits, &t.material, 4);
		triHot[i * 3 + 0] = make_float4(t.vertex0[0], t.vertex0[1], t.vertex0[2], 0.0f);
		triHot[i * 3 + 1] = make_float4(t.edge1[0], t.edge1[1], t.edge1[2], 0.0f);
		triHot[i * 3 + 2] = make_float4(t.edge2[0], t.edge2[1], t.edge2[2], 0.0f);
		triShade[i * 3 + 0] = make_float4(t.normal0[0], t.normal0[1], t.normal0[2], materialBits);
		triShade[i * 3 + 1] = make_float4(t.normal1[0], t.normal1[1], t.normal1[2], 0.0f);
		triShade[i * 3 + 2] = make_float4(t.normal2[0], t.normal2[1], t.normal2[2], 0.0f);
	}

	for (const EchoInfiniteLight& light : scene->infiniteLights)
	{
		if (light.type > ECHO_INFINITE_CUBEMAP) return fail(ECHO_B200_ERR_UNSUPPORTED, "unknown infinite light type");
		if (light.type == ECHO_INFINITE_CUBEMAP && (uint64_t)light.texture + 6 > scene->textures.size()) return fail(ECHO_B200_ERR_INVALID, "cubemap needs six consecutive textures");
		if (light.type != ECHO_INFINITE_ENVIRONMENT) continue;
		if (light.texture >= scene->textures.size()) return fail(ECHO_B200_ERR_INVALID, "environment light texture out of range");
		const EchoTexture& t = scene->textures[light.texture];
		if ((uint64_t)light.distribution + (uint64_t)t.height * (t.width + 1ull) > scene->distributions.size()) return fail(ECHO_B200_ERR_INVALID, "environment light distribution out of range");
	}

	// texture coordinates are only read by textured scenes
	if (!scene->textures.empty() && scene->materialTextures.size() != scene->materials.size())
		return fail(ECHO_B200_ERR_INVALID, "set_textures needs one EchoMaterialTextures per material");

	std::vector<float4> triTexcoord(scene->textures.empty() ? 0 : scene->triangles.size() * 2);

	for (size_t i = 0; i < triTexcoord.size() / 2; i++)
	{
		const EchoTriangle& t = scene->triangles[i];
		triTexcoord[i * 2 + 0] = make_float4(t.texcoord0[0], t.texcoord0[1], t.texcoord1[0], t.texcoord1[1]);
		triTexcoord[i * 2 + 1] = make_float4(t.texcoord2[0], t.texcoord2[1], 0.0f, 0.0f);
	}

	std::vector<float4> spheres(scene->spheres.size());
	std::vector<uint32_t> sphereMaterial(scene->spheres.size());

	for (size_t i = 0; i < scene->spheres.size(); i++)
	{
		const EchoSphere& s = scene->spheres[i];
		spheres[i] = make_float4(s.position[0], s.position[1], s.position[2], s.radius);
		sphereMaterial[i] = s.material;
	}

	std::vector<float4> pointLights(scene->pointLights.size() * 2), infiniteLights(scene->infiniteLights.size() * 10);

	for (size_t i = 0; i < scene->pointLights.size(); i++)
	{
		const EchoPointLight& p = scene->pointLights[i];
		pointLights[i * 2] = make_float4(p.intensity[0], p.intensity[1], p.intensity[2], 0.0f);
		pointLights[i * 2 + 1] = make_float4(p.position[0], p.position[1], p.position[2], 0.0f);
	}

	static_assert(sizeof(EchoInfiniteLight) == 160, "POD layout");
	std::memcpy(infiniteLights.data(), scene->infiniteLights.data(), sizeof(EchoInfiniteLight) * scene->infiniteLights.size()); // 10 float4 each, verbatim

	static_assert(sizeof(EchoQbvhNode) == 128 && sizeof(EchoMaterial) == 64 && sizeof(EchoLightNode) == 64, "POD layout");
	static_assert(sizeof(EchoTriangle) == 100 && sizeof(EchoSphere) == 20 && sizeof(EchoRay) == 32 && sizeof(EchoHit) == 16, "POD layout");

	const EchoQbvhNode* nodes = nullptr;
	const EchoMaterial* materials = nullptr;
	const EchoLightNode* lightNodes = nullptr;
	const EchoPack* devicePacks = nullptr;
	const EchoInstance* deviceInstances = nullptr;
	const EchoTexture* deviceTextures = nullptr;
	const EchoMaterialTextures* deviceMaterialTextures = nullptr;
	const float* deviceTexels = nullptr;
	static_assert(sizeof(EchoTexture) == 32 && sizeof(EchoMaterialTextures) == 32, "POD layout");
	static_assert(sizeof(EchoPack) == 64 && sizeof(EchoInstance) == 128 && sizeof(EchoTokenHierarchy) == 24, "POD layout");

	bool ok = upload(scene, scene->packs, devicePacks) && upload(scene, scene->instances, deviceInstances) && upload(scene, scene->textures, deviceTextures)
		&& upload(scene, scene->materialTextures, deviceMaterialTextures) && upload(scene, scene->texels, deviceTexels) && upload(scene, triTexcoord, d.triTexcoord) && upload(scene, scene->distributions, d.distributions)
		&& upload(scene, scene->nodes, nodes) && upload(scene, triHot, d.triHot) && upload(scene, triShade, d.triShade)
		&& upload(scene, spheres, d.spheres) && upload(scene, sphereMaterial, d.sphereMaterial) && upload(scene, scene->materials, materials)
		&& upload(scene, scene->lightNodes, lightNodes) && upload(scene, emitterTokens, d.emitterTokens)
		&& upload(scene, emitterPaths, d.emitterPaths) && upload(scene, pointLights, d.pointLights) && upload(scene, infiniteLights, d.infiniteLights);

	if (!ok)
	{
		free_device(scene);
		return ECHO_B200_ERR_CUDA;
	}

	d.nodes = reinterpret_cast<const float4*>(nodes);
	d.materials = reinterpret_cast<const float4*>(materials);
	d.lightNodes = reinterpret_cast<const float4*>(lightNodes);
	d.nodeCount = (uint32_t)scene->nodes.size();
	d.triangleCount = (uint32_t)scene->triangles.size();
	d.sphereCount = (uint32_t)scene->spheres.size();
	d.materialCount = (uint32_t)scene->materials.size();
	d.lightNodeCount = (uint32_t)scene->lightNodes.size();
	d.emitterCount = (uint32_t)scene->emitterTokens.size();
	d.pointLightCount = (uint32_t)scene->pointLights.size();
	d.infiniteLightCount = (uint32_t)scene->infiniteLights.size();
	d.maxDepth = stackDepth;
	d.packs = reinterpret_cast<const uint4*>(devicePacks);
	d.instances = reinterpret_cast<const float4*>(deviceInstances);
	d.textures = reinterpret_cast<const uint4*>(deviceTextures);
	d.materialTextures = reinterpret_cast<const uint4*>(deviceMaterialTextures);
	d.texels = reinterpret_cast<const float4*>(deviceTexels);
	d.textureCount = (uint32_t)scene->textures.size();
	d.texelCount = (uint32_t)(scene->texels.size() / 4);
	d.distributionCount = (uint32_t)scene->distributions.size();

#ifdef ECHO_BOUNDS_CHECK
	{
		void* flag = nullptr;
		if (!check_cuda(cudaMalloc(&flag, sizeof(unsigned int)), "cudaMalloc(violations)") || !check_cuda(cudaMemset(flag, 0, sizeof(unsigned int)), "cudaMemset(violations)"))
		{
			free_device(scene);
			return ECHO_B200_ERR_CUDA;
		}
		scene->allocations.push_back(flag);
		d.violations = (unsigned int*)flag;
	}
#endif
	d.packCount = (uint32_t)scene->packs.size();
	d.instanceCount = (uint32_t)scene->instances.size();
	d.infiniteThreshold = scene->infiniteThreshold;
	d.infinitePdf = scene->infinitePdf;
	d.camera = scene->camera;
	d.boundRadius = scene->boundRadius;

	scene->committed = true;
	return ECHO_B200_OK;
}

int32_t echo_b200_trace_batch(EchoScene* scene, const EchoRay* rays, uint64_t n, EchoHit* hits)
{
	auto trace = [](EchoScene* target, const EchoRay* in, uint64_t count, EchoHit* out)
	{
		return batch_host<EchoHit>(target, in, count, out, [target](const EchoRay* chunk, uint64_t c, EchoHit* chunkOut, cudaStream_t stream)
		{
			return launch_trace(target->d, chunk, c, chunkOut, nullptr, stream);
		});
	};

	if (!scene || scene->replicas.empty() || !rays || !hits || n == 0) return trace(scene, rays, n, hits);

	const uint64_t devices = 1 + scene->replicas.size(); // one contiguous range of the batch per device
	return fan_out(scene, [&](EchoScene* target, size_t g)
	{
		uint64_t first = n * g / devices;
		return trace(target, rays + first, n * (g + 1) / devices - first, hits + first);
	});
}

int32_t echo_b200_occlude_batch(EchoScene* scene, const EchoRay* rays, uint64_t n, uint8_t* occluded)
{
	auto occlude = [](EchoScene* target, const EchoRay* in, uint64_t count, uint8_t* out)
	{
		return batch_host<uint8_t>(target, in, count, out, [target](const EchoRay* chunk, uint64_t c, uint8_t* chunkOut, cudaStream_t stream)
		{
			return launch_occlude(target->d, chunk, c, chunkOut, nullptr, stream);
		});
	};

	if (!scene || scene->replicas.empty() || !rays || !occluded || n == 0) return occlude(scene, rays, n, occluded);

	const uint64_t devices = 1 + scene->replicas.size();
	return fan_out(scene, [&](EchoScene* target, size_t g)
	{
		uint64_t first = n * g / devices;
		return occlude(target, rays + first, n * (g + 1) / devices - first, occluded + first);
	});
}

namespace
{

// Host-buffer hierarchy batch: one upload, one launch, one download (the instanced path is not the bandwidth-tuned one).
int32_t hierarchy_host(EchoScene* scene, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, EchoHit* hits, EchoTokenHierarchy* hitLayers, uint8_t* occluded)
{
	if (!require_committed(scene)) return ECHO_B200_ERR_INVALID;
	if (n == 0) return ECHO_B200_OK;
	if (!rays || (!hits && !occluded)) return fail(ECHO_B200_ERR_INVALID, "null buffer");
	if (scene->d.packCount == 0u) return fail(ECHO_B200_ERR_INVALID, "the scene has no packs: use the plain batch calls");

	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	std::lock_guard<std::mutex> turn(scene->compute);

	void *dRays = nullptr, *dIgnore = nullptr, *dOut = nullptr, *dLayers = nullptr;
	size_t outBytes = hits ? sizeof(EchoHit) * n : n;
	cudaStream_t stream = scene->stream;

	// grow-only device scratch, kept between calls
	auto scratch = [scene](int slot, size_t bytes, void*& pointer)
	{
		if (scene->hierarchyBytes[slot] < bytes)
		{
			if (scene->hierarchyScratch[slot]) cudaFree(scene->hierarchyScratch[slot]);
			scene->hierarchyScratch[slot] = nullptr;
			scene->hierarchyBytes[slot] = 0;
			if (!check_cuda(cudaMalloc(&scene->hierarchyScratch[slot], bytes), "cudaMalloc(hierarchy batch)")) return false;
			scene->hierarchyBytes[slot] = bytes;
		}

		pointer = scene->hierarchyScratch[slot];
		return true;
	};

	bool ok = scratch(0, sizeof(EchoRay) * n, dRays) && scratch(2, outBytes, dOut)
		&& (!ignore || scratch(1, sizeof(EchoTokenHierarchy) * n, dIgnore))
		&& (!hitLayers || scratch(3, sizeof(EchoTokenHierarchy) * n, dLayers))
		&& check_cuda(cudaMemcpyAsync(dRays, rays, sizeof(EchoRay) * n, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(rays)")
		&& (!ignore || check_cuda(cudaMemcpyAsync(dIgnore, ignore, sizeof(EchoTokenHierarchy) * n, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(ignore)"));

	if (ok)
	{
		ok = hits ? launch_trace_instanced(scene->d, (const EchoRay*)dRays, (const EchoTokenHierarchy*)dIgnore, n, (EchoHit*)dOut, (EchoTokenHierarchy*)dLayers, nullptr, stream)
		          : launch_occlude_instanced(scene->d, (const EchoRay*)dRays, (const EchoTokenHierarchy*)dIgnore, n, (uint8_t*)dOut, nullptr, stream);
	}

	ok = ok && check_cuda(cudaMemcpyAsync(hits ? (void*)hits : (void*)occluded, dOut, outBytes, cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(out)")
		&& (!hitLayers || check_cuda(cudaMemcpyAsync(hitLayers, dLayers, sizeof(EchoTokenHierarchy) * n, cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(layers)"))
		&& check_cuda(cudaStreamSynchronize(stream), "hierarchy batch");

	if (!ok) cudaStreamSynchronize(stream); // copies queued before the failure must not outlive the caller's buffers
	return ok ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

} // namespace

int32_t echo_b200_trace_batch_hierarchy(EchoScene* scene, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, EchoHit* hits, EchoTokenHierarchy* hitLayers)
{
	if (!hits && n != 0) return fail(ECHO_B200_ERR_INVALID, "null buffer");
	if (!scene || scene->replicas.empty() || !rays || n == 0) return hierarchy_host(scene, rays, ignore, n, hits, hitLayers, nullptr);

	const uint64_t devices = 1 + scene->replicas.size();
	return fan_out(scene, [&](EchoScene* target, size_t g)
	{
		uint64_t first = n * g / devices;
		return hierarchy_host(target, rays + first, ignore ? ignore + first : nullptr, n * (g + 1) / devices - first, hits + first, hitLayers ? hitLayers + first : nullptr, nullptr);
	});
}

int32_t echo_b200_occlude_batch_hierarchy(EchoScene* scene, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, uint8_t* occluded)
{
	if (!occluded && n != 0) return fail(ECHO_B200_ERR_INVALID, "null buffer");
	if (!scene || scene->replicas.empty() || !rays || n == 0) return hierarchy_host(scene, rays, ignore, n, nullptr, nullptr, occluded);

	const uint64_t devices = 1 + scene->replicas.size();
	return fan_out(scene, [&](EchoScene* target, size_t g)
	{
		uint64_t first = n * g / devices;
		return hierarchy_host(target, rays + first, ignore ? ignore + first : nullptr, n * (g + 1) / devices - first, nullptr, nullptr, occluded + first);
	});
}

int32_t echo_b200_trace_batch_device(EchoScene* scene, const EchoRay* rays, uint64_t n, EchoHit* hits, void* stream)
{
	if (!require_committed(scene) || !single_device(scene)) return ECHO_B200_ERR_INVALID;
	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	return launch_trace(scene->d, rays, n, hits, nullptr, (cudaStream_t)stream) ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_occlude_batch_device(EchoScene* scene, const EchoRay* rays, uint64_t n, uint8_t* occluded, void* stream)
{
	if (!require_committed(scene) || !single_device(scene)) return ECHO_B200_ERR_INVALID;
	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	return launch_occlude(scene->d, rays, n, occluded, nullptr, (cudaStream_t)stream) ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_trace_batch_device_counted(EchoScene* scene, const EchoRay* rays, uint64_t n, EchoHit* hits, uint64_t* counts, void* stream)
{
	if (!require_committed(scene) || !single_device(scene)) return ECHO_B200_ERR_INVALID;
	if (!counts) return fail(ECHO_B200_ERR_INVALID, "d_counts3 is null");
	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	return launch_trace(scene->d, rays, n, hits, (unsigned long long*)counts, (cudaStream_t)stream) ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_occlude_batch_device_counted(EchoScene* scene, const EchoRay* rays, uint64_t n, uint8_t* occluded, uint64_t* counts, void* stream)
{
	if (!require_committed(scene) || !single_device(scene)) return ECHO_B200_ERR_INVALID;
	if (!counts) return fail(ECHO_B200_ERR_INVALID, "d_counts3 is null");
	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	return launch_occlude(scene->d, rays, n, occluded, (unsigned long long*)counts, (cudaStream_t)stream) ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

// the scene's grow-only device buffer for tile-major output
static float4* tiles_out(EchoScene* scene, uint64_t bytes)
{
	if (scene->tilesOutBytes >= bytes) return (float4*)scene->tilesOut;
	if (scene->tilesOut) cudaFree(scene->tilesOut);
	scene->tilesOut = nullptr;
	scene->tilesOutBytes = 0;
	if (!check_cuda(cudaMalloc(&scene->tilesOut, bytes), "cudaMalloc(tiles)")) return nullptr;
	scene->tilesOutBytes = bytes;
	return (float4*)scene->tilesOut;
}

// the tiles [first, first + count) of the caller's sequence on one device: render, then download into the caller's tile-major buffer
static int32_t render_tiles_device(EchoScene* scene, const EchoRenderParams* params, const int32_t* tileXY, uint32_t tileCount, float* outRGBA, EchoStats* stats)
{
	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	std::lock_guard<std::mutex> turn(scene->compute);

	uint64_t pixels = (uint64_t)tileCount * params->tileSize * params->tileSize;
	float4* deviceOut = tiles_out(scene, sizeof(float4) * pixels);
	if (!deviceOut) return ECHO_B200_ERR_CUDA;

	bool ok = render_tiles(scene->render, scene->d, *params, tileXY, tileCount, deviceOut, nullptr, stats, scene->stream);
	ok = ok && check_cuda(cudaMemcpyAsync(outRGBA, deviceOut, sizeof(float4) * pixels, cudaMemcpyDeviceToHost, scene->stream), "cudaMemcpyAsync(tiles)");
	ok = check_cuda(cudaStreamSynchronize(scene->stream), "render_tiles") && ok;
	return ok ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_render_tiles(EchoScene* scene, const EchoRenderParams* params, const int32_t* tileXY, uint32_t tileCount, float* outRGBA, EchoStats* stats)
{
	if (!require_renderable(scene)) return ECHO_B200_ERR_INVALID;
	if (!params || (!tileXY && tileCount) || (!outRGBA && tileCount)) return fail(ECHO_B200_ERR_INVALID, "null argument");
	if (params->tileSize <= 0) return fail(ECHO_B200_ERR_INVALID, "invalid EchoRenderParams");
	if (stats) *stats = EchoStats{};
	if (tileCount == 0) return ECHO_B200_OK;
	if (scene->replicas.empty()) return render_tiles_device(scene, params, tileXY, tileCount, outRGBA, stats);

	// Several devices: blocks of kDealBlock consecutive tiles dealt round-robin; device g renders its blocks as one tile list and
	// its tiles go back block by block to their places in the caller's buffer. Disjoint tiles: nothing to reduce.
	const size_t devices = 1 + scene->replicas.size();
	const uint64_t tileFloats = (uint64_t)params->tileSize * params->tileSize * 4;
	const uint32_t blocks = (tileCount + kDealBlock - 1) / kDealBlock;
	std::vector<EchoStats> perDevice(devices, EchoStats{});

	int32_t status = fan_out(scene, [&](EchoScene* target, size_t g)
	{
		std::vector<int32_t> local;
		std::vector<uint32_t> blockOf; // the block each run of `local` came from

		for (uint32_t b = (uint32_t)g; b < blocks; b += (uint32_t)devices)
		{
			uint32_t first = b * kDealBlock, count = std::min(kDealBlock, tileCount - first);
			local.insert(local.end(), tileXY + (size_t)first * 2, tileXY + (size_t)(first + count) * 2);
			blockOf.push_back(b);
		}

		if (local.empty()) return (int32_t)ECHO_B200_OK;
		uint32_t localCount = (uint32_t)(local.size() / 2);

		DeviceGuard guard(target->device);
		if (!guard.ok) return (int32_t)ECHO_B200_ERR_NO_DEVICE;
		std::lock_guard<std::mutex> turn(target->compute);

		float4* deviceOut = tiles_out(target, sizeof(float) * tileFloats * localCount);
		if (!deviceOut) return (int32_t)ECHO_B200_ERR_CUDA;

		bool ok = render_tiles(target->render, target->d, *params, local.data(), localCount, deviceOut, nullptr, &perDevice[g], target->stream);
		uint32_t localFirst = 0;

		for (size_t k = 0; ok && k < blockOf.size(); k++)
		{
			uint32_t first = blockOf[k] * kDealBlock, count = std::min(kDealBlock, tileCount - first);
			ok = check_cuda(cudaMemcpyAsync(outRGBA + (uint64_t)first * tileFloats, reinterpret_cast<const float*>(deviceOut) + (uint64_t)localFirst * tileFloats,
			                                sizeof(float) * tileFloats * count, cudaMemcpyDeviceToHost, target->stream), "cudaMemcpyAsync(tiles)");
			localFirst += count;
		}

		ok = check_cuda(cudaStreamSynchronize(target->stream), "render_tiles") && ok;
		return (int32_t)(ok ? ECHO_B200_OK : ECHO_B200_ERR_CUDA);
	});

	if (stats)
	{
		uint64_t* total = reinterpret_cast<uint64_t*>(stats);
		for (const EchoStats& part : perDevice)
			for (size_t i = 0; i < sizeof(EchoStats) / sizeof(uint64_t); i++) total[i] += reinterpret_cast<const uint64_t*>(&part)[i];
	}

	return status;
}

int32_t echo_b200_render_frame_device(EchoScene* scene, const EchoRenderParams* params, const int32_t* tileXY, uint32_t tileCount, float* frame, EchoStats* stats, void* stream)
{
	if (!require_renderable(scene) || !single_device(scene)) return ECHO_B200_ERR_INVALID;
	if (!params || (!tileXY && tileCount) || !frame) return fail(ECHO_B200_ERR_INVALID, "null argument");
	if (stats) *stats = EchoStats{};
	if (tileCount == 0) return ECHO_B200_OK;

	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;

	cudaStream_t s = stream ? (cudaStream_t)stream : scene->stream;
	std::lock_guard<std::mutex> turn(scene->compute);
	return render_tiles(scene->render, scene->d, *params, tileXY, tileCount, nullptr, (float4*)frame, stats, s) ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_frame_resolve_device(EchoScene* scene, float* frame, int32_t width, int32_t height, void* stream)
{
	if (!scene || !frame || width <= 0 || height <= 0) return fail(ECHO_B200_ERR_INVALID, "invalid argument");
	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	cudaStream_t s = stream ? (cudaStream_t)stream : scene->stream;
	return launch_frame_resolve((float4*)frame, width, height, s) ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_debug_evaluate_samples(EchoScene* scene, const EchoRenderParams* params, const int32_t* pixelXY, const uint32_t* sampleIndex, uint64_t n, float* outRGB)
{
	if (!require_renderable(scene)) return ECHO_B200_ERR_INVALID;
	if (!params || !pixelXY || !sampleIndex || !outRGB) return fail(ECHO_B200_ERR_INVALID, "null argument");
	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	std::lock_guard<std::mutex> turn(scene->compute);
	return evaluate_sample_list(scene->render, scene->d, *params, 3, pixelXY, sampleIndex, n, outRGB, scene->stream) ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

// Bounds-check builds (-DECHO_BOUNDS_CHECK): the bit set of failed checks since commit (echo_scene.cuh CHECK_*); release builds
// report 0xFFFFFFFF = "not compiled in". Synchronises the device.
int32_t echo_b200_debug_bounds_violations(EchoScene* scene, uint32_t* out)
{
	if (!scene || !out) return fail(ECHO_B200_ERR_INVALID, "null argument");
	*out = 0xFFFFFFFFu;
#ifdef ECHO_BOUNDS_CHECK
	if (!scene->committed || !scene->d.violations) { *out = 0u; return ECHO_B200_OK; }
	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	if (!check_cuda(cudaDeviceSynchronize(), "bounds violations") || !check_cuda(cudaMemcpy(out, scene->d.violations, sizeof(uint32_t), cudaMemcpyDeviceToHost), "cudaMemcpy(violations)"))
		return ECHO_B200_ERR_CUDA;
#endif
	return ECHO_B200_OK;
}

int32_t echo_b200_debug_evaluate_samples4(EchoScene* scene, const EchoRenderParams* params, const int32_t* pixelXY, const uint32_t* sampleIndex, uint64_t n, float* outRGBA)
{
	if (!require_renderable(scene)) return ECHO_B200_ERR_INVALID;
	if (!params || !pixelXY || !sampleIndex || !outRGBA) return fail(ECHO_B200_ERR_INVALID, "null argument");
	DeviceGuard guard(scene->device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	std::lock_guard<std::mutex> turn(scene->compute);
	return evaluate_sample_list(scene->render, scene->d, *params, 4, pixelXY, sampleIndex, n, outRGBA, scene->stream) ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_debug_set_option(const char* name, int64_t value)
{
	if (!name) return fail(ECHO_B200_ERR_INVALID, "name is null");
	return set_render_option(name, (long long)value) || set_build_option(name, (long long)value) ? ECHO_B200_OK : fail(ECHO_B200_ERR_INVALID, "unknown option");
}

int32_t echo_b200_debug_last_build(float* out4)
{
	if (!out4) return fail(ECHO_B200_ERR_INVALID, "out4 is null");
	last_sweep_build(out4);
	return ECHO_B200_OK;
}

int32_t echo_b200_debug_last_light_build(float* out4)
{
	if (!out4) return fail(ECHO_B200_ERR_INVALID, "out4 is null");
	last_light_build(out4);
	return ECHO_B200_OK;
}

int32_t echo_b200_debug_last_pack_build(float* out8)
{
	if (!out8) return fail(ECHO_B200_ERR_INVALID, "out8 is null");
	last_pack_build(out8);
	return ECHO_B200_OK;
}

static int32_t debug_device(int32_t device)
{
	int32_t count = 0;
	int32_t status = echo_b200_device_count(&count);
	if (status != ECHO_B200_OK) return status;
	if (device < 0 || device >= count) return fail(ECHO_B200_ERR_INVALID, "device index out of range");
	return ECHO_B200_OK;
}

int32_t echo_b200_debug_measure_peaks(int32_t device, float* out3)
{
	if (!out3) return fail(ECHO_B200_ERR_INVALID, "out3 is null");
	int32_t status = debug_device(device);
	if (status != ECHO_B200_OK) return status;
	DeviceGuard guard(device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;
	return measure_peaks(out3) ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_debug_bxdf_batch(int32_t device, int32_t kind, const float* params, const float* outgoing, const float* samples, uint64_t n,
                                   float* sampled8, float* evaluated4, float* inverse4)
{
	int32_t status = debug_device(device);
	if (status != ECHO_B200_OK) return status;
	DeviceGuard guard(device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;

	float *dParams = nullptr, *dOutgoing = nullptr, *dSamples = nullptr, *dSampled = nullptr, *dEvaluated = nullptr, *dInverse = nullptr;
	bool ok = check_cuda(cudaMalloc((void**)&dParams, sizeof(float) * 11), "cudaMalloc") && check_cuda(cudaMalloc((void**)&dOutgoing, sizeof(float) * 3 * n), "cudaMalloc")
		&& check_cuda(cudaMalloc((void**)&dSamples, sizeof(float) * 2 * n), "cudaMalloc") && check_cuda(cudaMalloc((void**)&dSampled, sizeof(float) * 8 * n), "cudaMalloc")
		&& check_cuda(cudaMalloc((void**)&dEvaluated, sizeof(float) * 4 * n), "cudaMalloc") && check_cuda(cudaMalloc((void**)&dInverse, sizeof(float) * 4 * n), "cudaMalloc");

	ok = ok && check_cuda(cudaMemcpy(dParams, params, sizeof(float) * 11, cudaMemcpyHostToDevice), "cudaMemcpy")
		&& check_cuda(cudaMemcpy(dOutgoing, outgoing, sizeof(float) * 3 * n, cudaMemcpyHostToDevice), "cudaMemcpy")
		&& check_cuda(cudaMemcpy(dSamples, samples, sizeof(float) * 2 * n, cudaMemcpyHostToDevice), "cudaMemcpy");

	ok = ok && launch_debug_bxdf(kind, dParams, dOutgoing, dSamples, n, dSampled, dEvaluated, dInverse, nullptr);
	ok = ok && check_cuda(cudaDeviceSynchronize(), "debug_bxdf");
	ok = ok && check_cuda(cudaMemcpy(sampled8, dSampled, sizeof(float) * 8 * n, cudaMemcpyDeviceToHost), "cudaMemcpy")
		&& check_cuda(cudaMemcpy(evaluated4, dEvaluated, sizeof(float) * 4 * n, cudaMemcpyDeviceToHost), "cudaMemcpy")
		&& check_cuda(cudaMemcpy(inverse4, dInverse, sizeof(float) * 4 * n, cudaMemcpyDeviceToHost), "cudaMemcpy");

	for (float* p : { dParams, dOutgoing, dSamples, dSampled, dEvaluated, dInverse }) if (p) cudaFree(p);
	return ok ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

int32_t echo_b200_debug_math(int32_t device, int32_t op, const float* a, const float* b, const float* c, uint64_t n, float* out)
{
	int32_t status = debug_device(device);
	if (status != ECHO_B200_OK) return status;
	DeviceGuard guard(device);
	if (!guard.ok) return ECHO_B200_ERR_NO_DEVICE;

	float* buffers[4] = { nullptr, nullptr, nullptr, nullptr };
	const float* hosts[3] = { a, b, c };
	bool ok = true;

	for (int i = 0; i < 4 && ok; i++) ok = check_cuda(cudaMalloc((void**)&buffers[i], sizeof(float) * std::max<uint64_t>(n, 1)), "cudaMalloc");
	for (int i = 0; i < 3 && ok; i++) ok = check_cuda(cudaMemcpy(buffers[i], hosts[i], sizeof(float) * n, cudaMemcpyHostToDevice), "cudaMemcpy");

	ok = ok && launch_debug_math(op, buffers[0], buffers[1], buffers[2], n, buffers[3], nullptr);
	ok = ok && check_cuda(cudaDeviceSynchronize(), "debug_math");
	ok = ok && check_cuda(cudaMemcpy(out, buffers[3], sizeof(float) * n, cudaMemcpyDeviceToHost), "cudaMemcpy");

	for (float* p : buffers) if (p) cudaFree(p);
	return ok ? ECHO_B200_OK : ECHO_B200_ERR_CUDA;
}

} // extern "C"
