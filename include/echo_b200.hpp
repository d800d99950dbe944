// echo_b200.hpp — the host side above the C ABI (echo_b200.h) in a compiled language: a header-only C++17 mirror of the reference's
// interface for this path, with the reference's names, argument meaning and error behaviour, so that a host written against Echo's
// C# types ports line by line and so that the logic of INTEGRATION.md's C# `GpuEvaluationOperation` exists in a form this image can
// compile, run and test (tests/c_client/echo_host_client.cpp in the GPU suite). Nothing here computes: every call ends in libecho_b200.so.
//
//   reference (src/Echo.Core/...)                                        here
//   Aggregation/Preparation/PreparedScene.cs  Trace / Occlude            echo_b200::PreparedScene::Trace / Occlude (batched)
//   Processes/Evaluation/EvaluationProfile.cs:13-75  Validate            echo_b200::EvaluationProfile::Validate
//   Textures/Evaluation/RenderTexture.cs, EvaluationLayer.cs:16-121      echo_b200::RenderTexture (CreateTile / Apply folded into Apply)
//   Processes/Evaluation/ITilePattern.cs:20-36, 72-202                   echo_b200::OrderedPattern / HilbertCurvePattern
//   Common/Compute/IWorker.cs (Index, CheckSchedule)                     echo_b200::IWorker
//   Common/Compute/Operation.cs:164-177  Execute(IWorker)                echo_b200::EvaluationOperation::Execute(IWorker&)
//   Processes/Evaluation/EvaluationOperation.cs:21-177                   echo_b200::EvaluationOperation (+ Factory)
//   Processes/Composition/OidnDenoise.cs:201-206  ThrowOnNativeError     echo_b200::ThrowOnNativeError -> NativeException
#pragma once
#include <atomic>
#include <cstdint>
#include <cstdlib>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "echo_b200.h"

namespace echo_b200
{

class NativeException : public std::runtime_error // errors are pulled from the library and thrown on the host side, OidnDenoise.cs:201-206
{
public:
	NativeException(int32_t status, const std::string& message) : std::runtime_error(message), status(status) {}
	const int32_t status;
};

inline void ThrowOnNativeError(int32_t status, const char* call)
{
	if (status == ECHO_B200_OK) return;
	const char* pulled = echo_b200_last_error();
	throw NativeException(status, std::string(call) + " failed with " + std::to_string(status) + ": " + (pulled ? pulled : ""));
}

struct Int2
{
	int32_t X, Y;
};

struct Float4
{
	float X, Y, Z, W;
};

template<class T>
struct View // a span the library only reads during the call
{
	const T* data = nullptr;
	uint64_t count = 0;
};

// What ScenePreparer.Prepare produced (PreparedScene.cs:26-40), flattened as INTEGRATION.md section 2 describes.
struct SceneSource
{
	View<EchoQbvhNode> nodes; // ignored when buildAcceleratorOnDevice
	uint32_t maxDepth = 0;
	View<EchoTriangle> triangles;
	View<EchoSphere> spheres;
	View<EchoMaterial> materials;
	View<EchoLightNode> lightNodes;
	View<uint32_t> emitterTokens;
	View<uint64_t> emitterPaths;
	View<EchoPointLight> pointLights;
	View<EchoInfiniteLight> infiniteLights;
	float infiniteThreshold = 0.0f, infinitePdf = 0.0f;
	EchoCamera camera = {};
	float boundRadius = 0.0f;
	bool buildAcceleratorOnDevice = false; // echo_b200_scene_build_qbvh instead of set_qbvh: the SweepBuilder's tree, built by the library
	bool buildLightTreeOnDevice = false;   // echo_b200_scene_build_light_tree instead of set_light_tree: LightTree.Build, by the library (lightNodes / emitter* ignored)
};

// The prepared, flattened scene resident on the devices of `deviceMask` (bit d = CUDA device d): the device twin of Echo's PreparedScene.
class PreparedScene
{
public:
	explicit PreparedScene(const SceneSource& source, uint64_t deviceMask = 1)
	{
		ThrowOnNativeError(echo_b200_scene_create_multi(&handle, deviceMask), "echo_b200_scene_create_multi");

		try
		{
			ThrowOnNativeError(echo_b200_scene_set_triangles(handle, source.triangles.data, (uint32_t)source.triangles.count), "echo_b200_scene_set_triangles");
			ThrowOnNativeError(echo_b200_scene_set_spheres(handle, source.spheres.data, (uint32_t)source.spheres.count), "echo_b200_scene_set_spheres");
			if (source.buildAcceleratorOnDevice) ThrowOnNativeError(echo_b200_scene_build_qbvh(handle, nullptr, nullptr), "echo_b200_scene_build_qbvh");
			else ThrowOnNativeError(echo_b200_scene_set_qbvh(handle, source.nodes.data, (uint32_t)source.nodes.count, source.maxDepth), "echo_b200_scene_set_qbvh");
			ThrowOnNativeError(echo_b200_scene_set_materials(handle, source.materials.data, (uint32_t)source.materials.count), "echo_b200_scene_set_materials");
			if (source.buildLightTreeOnDevice)
				ThrowOnNativeError(echo_b200_scene_build_light_tree(handle, source.pointLights.data, (uint32_t)source.pointLights.count, nullptr, nullptr, nullptr), "echo_b200_scene_build_light_tree");
			else
				ThrowOnNativeError(echo_b200_scene_set_light_tree(handle, source.lightNodes.data, (uint32_t)source.lightNodes.count, source.emitterTokens.data, source.emitterPaths.data,
				                                                  (uint32_t)source.emitterTokens.count, source.pointLights.data, (uint32_t)source.pointLights.count), "echo_b200_scene_set_light_tree");
			ThrowOnNativeError(echo_b200_scene_set_infinite(handle, source.infiniteLights.data, (uint32_t)source.infiniteLights.count, source.infiniteThreshold, source.infinitePdf), "echo_b200_scene_set_infinite");
			ThrowOnNativeError(echo_b200_scene_set_camera(handle, &source.camera), "echo_b200_scene_set_camera");
			ThrowOnNativeError(echo_b200_scene_set_bound_radius(handle, source.boundRadius), "echo_b200_scene_set_bound_radius");
			ThrowOnNativeError(echo_b200_scene_commit(handle), "echo_b200_scene_commit");
		}
		catch (...)
		{
			echo_b200_scene_destroy(handle);
			throw;
		}
	}

	~PreparedScene() { echo_b200_scene_destroy(handle); }
	PreparedScene(const PreparedScene&) = delete;
	PreparedScene& operator=(const PreparedScene&) = delete;

	// PreparedScene.Trace / Occlude (PreparedScene.cs:66-93) for a whole batch: hits[i] answers rays[i]
	void Trace(const EchoRay* rays, uint64_t count, EchoHit* hits) const { ThrowOnNativeError(echo_b200_trace_batch(handle, rays, count, hits), "echo_b200_trace_batch"); }
	void Occlude(const EchoRay* rays, uint64_t count, uint8_t* occluded) const { ThrowOnNativeError(echo_b200_occlude_batch(handle, rays, count, occluded), "echo_b200_occlude_batch"); }

	int32_t GpuCount() const
	{
		int32_t count = 0;
		ThrowOnNativeError(echo_b200_scene_gpu_count(handle, &count), "echo_b200_scene_gpu_count");
		return count;
	}

	EchoScene* Handle() const { return handle; }

private:
	EchoScene* handle = nullptr;
};

struct PathTracedEvaluator // Evaluation/Evaluators/PathTracedEvaluator.cs:33,40
{
	int32_t BounceLimit = 128;
	float Survivability = 2.5f;
};

struct EvaluationProfile // Processes/Evaluation/EvaluationProfile.cs:13-75 (Distribution reduced to its Extend, a seed and its kind)
{
	int32_t Evaluator = ECHO_EVALUATOR_PATH_TRACED; // ECHO_EVALUATOR_* [| ECHO_EVALUATOR_DIVERGE_ONCE]; a negative value stands for a null Evaluator
	PathTracedEvaluator PathTraced;
	int32_t Extend = 16; // ContinuousDistribution.Extend
	int32_t MinEpoch = 1;
	int32_t MaxEpoch = 20;
	float NoiseThreshold = 0.045f;
	uint32_t Seed = 1;
	bool Stratified = false; // Distribution is a StratifiedDistribution (ECHO_DISTRIBUTION_STRATIFIED); Extend <= 2^23

	void Validate() const // :65-75
	{
		if (Evaluator < 0) throw std::invalid_argument("Evaluator is null");
		if (Extend <= 0 || (Stratified && Extend > ECHO_DISTRIBUTION_STRATIFIED_EXTEND_MAX)) throw std::invalid_argument("Distribution is null or its Extend is out of bounds");
		if (MinEpoch <= 0) throw std::invalid_argument("MinEpoch out of bounds");
		if (MaxEpoch < MinEpoch) throw std::invalid_argument("MaxEpoch out of bounds");
		if (NoiseThreshold < 0.0f) throw std::invalid_argument("NoiseThreshold out of bounds");
	}
};

// Tile-based destination, rows growing upward (Textures/Evaluation/RenderTexture.cs; IEvaluationLayer.CreateTile / Apply, EvaluationLayer.cs:96-121)
class RenderTexture
{
public:
	RenderTexture(Int2 size, int32_t tileSize = 16) : size(size), tileSize(tileSize)
	{
		if (size.X <= 0 || size.Y <= 0 || tileSize <= 0) throw std::invalid_argument("size out of bounds");
		pixels.assign((size_t)size.X * size.Y, Float4{ 0.0f, 0.0f, 0.0f, 0.0f });
	}

	const Int2 size;
	const int32_t tileSize;

	Int2 TileCount() const { return { (size.X + tileSize - 1) / tileSize, (size.Y + tileSize - 1) / tileSize }; } // size.CeiledDivide(tileSize)
	const Float4& operator[](Int2 position) const { return pixels[(size_t)position.Y * size.X + position.X]; }
	const std::vector<Float4>& Pixels() const { return pixels; }

	// CreateTile(tilePosition), tile[position] = value for every pixel of the tile inside the texture, Apply(tile). Tiles are disjoint, so
	// workers may apply different tiles at once.
	void Apply(Int2 tilePosition, const Float4* tile)
	{
		int32_t minX = tilePosition.X * tileSize, minY = tilePosition.Y * tileSize;
		int32_t maxX = minX + tileSize < size.X ? minX + tileSize : size.X, maxY = minY + tileSize < size.Y ? minY + tileSize : size.Y;
		for (int32_t y = minY; y < maxY; y++)
			for (int32_t x = minX; x < maxX; x++) pixels[(size_t)y * size.X + x] = tile[(size_t)(y - minY) * tileSize + (x - minX)];
	}

private:
	std::vector<Float4> pixels;
};

// ---- ITilePattern.cs ----

inline std::vector<Int2> OrderedPattern(Int2 size, bool horizontal = true) // :20-36
{
	std::vector<Int2> sequence;
	sequence.reserve((size_t)size.X * size.Y);
	if (horizontal) { for (int32_t y = 0; y < size.Y; y++) for (int32_t x = 0; x < size.X; x++) sequence.push_back({ x, y }); }
	else { for (int32_t x = 0; x < size.X; x++) for (int32_t y = 0; y < size.Y; y++) sequence.push_back({ x, y }); }
	return sequence;
}

namespace detail
{

inline int32_t Sign(int32_t v) { return (v > 0) - (v < 0); }
inline int32_t Abs(int32_t v) { return v < 0 ? -v : v; }

// the generalised Hilbert curve over an arbitrary rectangle, HilbertCurvePattern.Hilbert2D (:143-202); `/ 2` truncates toward zero as in C#
inline void Hilbert2D(Int2 position, Int2 rectA, Int2 rectB, std::vector<Int2>& out)
{
	int32_t width = Abs(rectA.X + rectA.Y), height = Abs(rectB.X + rectB.Y);
	Int2 da = { Sign(rectA.X), Sign(rectA.Y) }, db = { Sign(rectB.X), Sign(rectB.Y) };

	if (height == 1)
	{
		for (int32_t i = 0; i < width; i++) { out.push_back(position); position = { position.X + da.X, position.Y + da.Y }; }
		return;
	}

	if (width == 1)
	{
		for (int32_t i = 0; i < height; i++) { out.push_back(position); position = { position.X + db.X, position.Y + db.Y }; }
		return;
	}

	Int2 a2 = { rectA.X / 2, rectA.Y / 2 }, b2 = { rectB.X / 2, rectB.Y / 2 };
	int32_t width2 = Abs(a2.X + a2.Y), height2 = Abs(b2.X + b2.Y);

	if (width * 2 > height * 3)
	{
		if (width2 % 2 != 0 && width > 2) a2 = { a2.X + da.X, a2.Y + da.Y };
		Hilbert2D(position, a2, rectB, out);
		Hilbert2D({ position.X + a2.X, position.Y + a2.Y }, { rectA.X - a2.X, rectA.Y - a2.Y }, rectB, out);
	}
	else
	{
		if (height2 % 2 != 0 && height > 2) b2 = { b2.X + db.X, b2.Y + db.Y };
		Hilbert2D(position, b2, a2, out);
		Hilbert2D({ position.X + b2.X, position.Y + b2.Y }, rectA, { rectB.X - b2.X, rectB.Y - b2.Y }, out);
		Hilbert2D({ position.X + (rectA.X - da.X) + (b2.X - db.X), position.Y + (rectA.Y - da.Y) + (b2.Y - db.Y) },
		          { -b2.X, -b2.Y }, { -(rectA.X - a2.X), -(rectA.Y - a2.Y) }, out);
	}
}

inline std::vector<Int2> HilbertCorner(Int2 size)
{
	std::vector<Int2> out;
	if (size.X <= 0 || size.Y <= 0) return out;
	if (size.X > size.Y) Hilbert2D({ 0, 0 }, { size.X, 0 }, { 0, size.Y }, out);
	else Hilbert2D({ 0, 0 }, { 0, size.Y }, { size.X, 0 }, out);
	return out;
}

} // namespace detail

// HilbertCurvePattern.CreateSequence (:72-141), the default EvaluationProfile.Pattern: one generalised Hilbert curve per quadrant, mirrored so
// that all four start at the centre of the texture, interlaced one position at a time.
inline std::vector<Int2> HilbertCurvePattern(Int2 size)
{
	if (size.X == 1 && size.Y == 1) return { { 0, 0 } };

	int32_t floorX = size.X / 2, ceilX = (size.X + 1) / 2, floorY = size.Y / 2, ceilY = (size.Y + 1) / 2;
	Int2 topRightSize = { ceilX, floorY }, topLeftSize = { floorX, floorY }, bottomRightSize = { ceilX, ceilY }, bottomLeftSize = { floorX, ceilY };

	std::vector<Int2> corners[4] = { detail::HilbertCorner(topLeftSize), detail::HilbertCorner(topRightSize), detail::HilbertCorner(bottomLeftSize), detail::HilbertCorner(bottomRightSize) };
	for (Int2& p : corners[0]) p = { topLeftSize.X - p.X - 1, topLeftSize.Y - p.Y - 1 };
	for (Int2& p : corners[1]) p = { p.X + topLeftSize.X, topRightSize.Y - p.Y - 1 };
	for (Int2& p : corners[2]) p = { bottomLeftSize.X - p.X - 1, p.Y + topLeftSize.Y };
	for (Int2& p : corners[3]) p = { p.X + topLeftSize.X, p.Y + topLeftSize.Y };

	std::vector<Int2> result;
	result.reserve((size_t)size.X * size.Y);
	size_t cursors[4] = { 0, 0, 0, 0 };

	while (result.size() < (size_t)size.X * size.Y)
		for (int k = 0; k < 4; k++)
			if (cursors[k] < corners[k].size()) result.push_back(corners[k][cursors[k]++]);

	return result;
}

struct IWorker // Common/Compute/IWorker.cs: what an Operation sees of the thread that runs it
{
	virtual ~IWorker() = default;
	virtual uint32_t Index() const = 0; // 0 .. workerCount - 1
	virtual void CheckSchedule() = 0;   // blocks while paused, throws to abort (Worker.cs); called between tiles
};

// EvaluationOperation on the device. Same public surface as the reference's (tilePositions, destination, profile, TotalSamples); one procedure =
// one echo_b200_render_tiles call over up to TilesPerProcedure consecutive tiles of the sequence. Execute(worker) is entered concurrently by
// every worker, each claiming the next procedure with one atomic increment (Operation.cs:164-177); the library serialises calls on one scene
// handle itself, and one call keeps every device of the scene busy, so extra workers simply wait for their turn.
// the EchoRenderParams an EvaluationOperation renders `destination` with under `profile`
inline EchoRenderParams RenderParameters(const EvaluationProfile& profile, const RenderTexture& destination)
{
	EchoRenderParams parameters = {};
	parameters.width = destination.size.X;
	parameters.height = destination.size.Y;
	parameters.tileSize = destination.tileSize;
	parameters.extend = profile.Extend;
	parameters.minEpoch = profile.MinEpoch;
	parameters.maxEpoch = profile.MaxEpoch;
	parameters.noiseThreshold = profile.NoiseThreshold;
	parameters.bounceLimit = profile.PathTraced.BounceLimit;
	parameters.survivability = profile.PathTraced.Survivability;
	parameters.seed = profile.Seed;
	parameters.epochOffset = 0;
	parameters.evaluator = profile.Evaluator | (profile.Stratified ? ECHO_DISTRIBUTION_STRATIFIED : 0);
	return parameters;
}

class EvaluationOperation
{
public:
	static constexpr uint32_t TilesPerProcedure = 256;

	EvaluationOperation(uint32_t workerCount, std::vector<Int2> tilePositions, RenderTexture& destination, const EvaluationProfile& profile, PreparedScene* scene)
		: tilePositions(std::move(tilePositions)), destination(destination), profile(profile), scene(scene), workerCount(workerCount),
		  totalProcedureCount((uint32_t)((this->tilePositions.size() + TilesPerProcedure - 1) / TilesPerProcedure))
	{
		if (workerCount == 0) throw std::invalid_argument("an operation needs at least one worker");
		tileFloats = (size_t)destination.tileSize * destination.tileSize * 4;
		void* memory = nullptr; // page-locked, one slice of TilesPerProcedure tiles per worker (INTEGRATION.md "Host memory")
		ThrowOnNativeError(echo_b200_host_alloc(&memory, (uint64_t)workerCount * TilesPerProcedure * tileFloats * sizeof(float)), "echo_b200_host_alloc");
		pixelMemory = (float*)memory;
		statistics = {};
	}

	~EvaluationOperation() { echo_b200_host_free(pixelMemory); }
	EvaluationOperation(const EvaluationOperation&) = delete;
	EvaluationOperation& operator=(const EvaluationOperation&) = delete;

	const std::vector<Int2> tilePositions;
	RenderTexture& destination;
	const EvaluationProfile profile;

	uint32_t TotalProcedureCount() const { return totalProcedureCount; }
	uint32_t CompletedProcedureCount() const { return completedProcedures.load(); }
	bool IsCompleted() const { return completedProcedures.load() == totalProcedureCount; }

	uint64_t TotalSamples() const // the "Sample/Evaluated" row, EvaluationOperation.cs:73-81
	{
		std::lock_guard<std::mutex> lock(statisticsLock);
		return statistics.sampleEvaluated;
	}

	EchoStats Statistics() const // the EvaluatorStatistics rows summed over the procedures finished so far
	{
		std::lock_guard<std::mutex> lock(statisticsLock);
		return statistics;
	}

	// Operation.Execute(IWorker) (Operation.cs:164-177): joins the execution once; returns whether the worker should call again.
	bool Execute(IWorker& worker)
	{
		uint32_t index = nextProcedure.fetch_add(1u);
		if (index >= totalProcedureCount) return false;
		if (worker.Index() >= workerCount) throw std::invalid_argument("worker index out of range");

		if (scene != nullptr) Execute(index, worker); // "cannot do anything without a scene" (aborted preparation), EvaluationOperation.cs:89
		return completedProcedures.fetch_add(1u) + 1u < totalProcedureCount;
	}

	// IOperationFactory (EvaluationOperation.cs:153-176): validates the profile, lays out the tile sequence with the profile's pattern
	struct Factory
	{
		Factory(PreparedScene* scene, RenderTexture& renderTexture, const EvaluationProfile& profile, bool hilbert = true)
			: scene(scene), renderTexture(renderTexture), profile(profile), hilbert(hilbert) { profile.Validate(); }

		EvaluationOperation* CreateOperation(uint32_t workerCount) const
		{
			Int2 count = renderTexture.TileCount();
			return new EvaluationOperation(workerCount, hilbert ? HilbertCurvePattern(count) : OrderedPattern(count), renderTexture, profile, scene);
		}

		PreparedScene* scene;
		RenderTexture& renderTexture;
		EvaluationProfile profile;
		bool hilbert;
	};

private:
	void Execute(uint32_t procedure, IWorker& worker)
	{
		size_t first = (size_t)procedure * TilesPerProcedure;
		size_t count = tilePositions.size() - first < TilesPerProcedure ? tilePositions.size() - first : TilesPerProcedure;
		float* pixels = pixelMemory + (size_t)worker.Index() * TilesPerProcedure * tileFloats; // this worker's slice

		EchoRenderParams parameters = RenderParameters(profile, destination);
		EchoStats stats = {};
		static_assert(sizeof(Int2) == 2 * sizeof(int32_t), "Int2 is two packed 32-bit integers");
		ThrowOnNativeError(echo_b200_render_tiles(scene->Handle(), &parameters, &tilePositions[first].X, (uint32_t)count, pixels, &stats), "echo_b200_render_tiles");

		for (size_t i = 0; i < count; i++) // CreateTile / tile[position] = value / Apply, EvaluationOperation.cs:91,139,147
		{
			destination.Apply(tilePositions[first + i], reinterpret_cast<const Float4*>(pixels + i * tileFloats));
			worker.CheckSchedule(); // pause / abort still work between tiles (:143)
		}

		std::lock_guard<std::mutex> lock(statisticsLock);
		const uint64_t* source = reinterpret_cast<const uint64_t*>(&stats);
		uint64_t* target = reinterpret_cast<uint64_t*>(&statistics);
		for (size_t k = 0; k < sizeof(EchoStats) / sizeof(uint64_t); k++) target[k] += source[k]; // every row of EchoStats is a 64-bit count
	}

	PreparedScene* const scene;
	const uint32_t workerCount;
	const uint32_t totalProcedureCount;
	size_t tileFloats = 0;
	float* pixelMemory = nullptr;
	std::atomic<uint32_t> nextProcedure{ 0 };
	std::atomic<uint32_t> completedProcedures{ 0 };
	mutable std::mutex statisticsLock;
	EchoStats statistics;
};

} // namespace echo_b200
