// The validation rules of the batched PreparedScene queries (echorenderer_b200/csrc/echo_query_rules.h) compiled for the host on
// their own, over plain scene arrays: tests/query_rules_lib.py runs its table of edge inputs through them. TEST INFRASTRUCTURE ONLY.
#include "../../echorenderer_b200/csrc/echo_query_rules.h"

namespace
{

struct ArrayScene
{
	const EchoPack* packs;
	uint32_t packs_;
	const EchoInstance* instances;
	const EchoTriangle* triangles;
	uint32_t triangles_;
	const EchoSphere* spheres;
	uint32_t spheres_, points_, infinites_, materials_;

	uint32_t packCount() const { return packs_; }
	EchoPack pack(uint32_t p) const { return packs[p]; }
	void instance(uint32_t i, uint32_t& pack, uint32_t& materialOffset) const
	{
		pack = instances[i].pack;
		materialOffset = instances[i].materialOffset;
	}
	uint32_t triangleCount() const { return triangles_; }
	uint32_t sphereCount() const { return spheres_; }
	uint32_t pointLightCount() const { return points_; }
	uint32_t infiniteLightCount() const { return infinites_; }
	uint32_t materialCount() const { return materials_; }
	uint32_t triangleMaterial(uint32_t t) const { return triangles[t].material; }
	uint32_t sphereMaterial(uint32_t s) const { return spheres[s].material; }
};

} // namespace

extern "C"
{

// codes[i] = the reason query i of a contact call (interact: valueCount 0, scatter_sample: 2, scatter_evaluate: 3) is refused, 0 if accepted
void rules_contact(const EchoPack* packs, uint32_t packCount, const EchoInstance* instances, const EchoTriangle* triangles, uint32_t triangleCount,
                   const EchoSphere* spheres, uint32_t sphereCount, uint32_t pointLightCount, uint32_t infiniteLightCount, uint32_t materialCount,
                   const EchoRay* rays, const EchoHit* hits, const EchoTokenHierarchy* layers, const float* values, int valueCount, uint64_t n, uint32_t* codes)
{
	const ArrayScene scene = { packs, packCount, instances, triangles, triangleCount, spheres, sphereCount, pointLightCount, infiniteLightCount, materialCount };
	for (uint64_t i = 0; i < n; i++)
	{
		uint32_t layer = 0;
		codes[i] = echo::rules::check_contact(scene, layers ? layers + i : nullptr, rays[i], hits[i], valueCount ? values + i * valueCount : nullptr, valueCount, layer);
	}
}

// the same for the light calls (mass: valueCount 0, sample: 2, pdf: 3)
void rules_light(const EchoPack* packs, uint32_t packCount, const EchoInstance* instances, const EchoTriangle* triangles, uint32_t triangleCount,
                 const EchoSphere* spheres, uint32_t sphereCount, uint32_t pointLightCount, uint32_t infiniteLightCount, uint32_t materialCount,
                 const uint32_t* tokens, const EchoTokenHierarchy* layers, const EchoSurface* points, const float* values, int valueCount, uint64_t n, uint32_t* codes)
{
	const ArrayScene scene = { packs, packCount, instances, triangles, triangleCount, spheres, sphereCount, pointLightCount, infiniteLightCount, materialCount };
	for (uint64_t i = 0; i < n; i++)
	{
		uint32_t layer = 0;
		codes[i] = echo::rules::check_light_query(scene, layers ? layers + i : nullptr, tokens[i], points[i], valueCount ? values + i * valueCount : nullptr, valueCount, layer);
	}
}

const char* rules_reason(uint32_t code) { return echo::rules::reason_text(code); }

} // extern "C"
