// scene_query_oracle.cpp — TEST INFRASTRUCTURE ONLY: the oracle (oracle/api.cpp, compiled here unchanged) with one batch export per
// scene query of include/echo_b200_query.h, same arguments as the device call, each calling the oracle's own functions (interact,
// Contact::bsdf, Scene::pick / probability_mass, scene_sample_light, scene_light_pdf, evaluate_infinite). tests/scene_query_oracle.py
// builds it into a temporary directory and loads it beside liboracle.so.
#include "../../include/echo_b200_query.h"
#include "../../oracle/api.cpp"

static Layers query_layers(const EchoTokenHierarchy* layers, uint64_t i) { return make_layers(layers ? layers + i : nullptr); }
static GeometryPoint query_point(const EchoSurface& s) { return { f3(s.position), f3(s.normal) }; }
static void query_store(float* out, Float3 v) { out[0] = v.x; out[1] = v.y; out[2] = v.z; }
static void query_store_rgb(float* out, RGB v) { out[0] = v.r; out[1] = v.g; out[2] = v.b; }

// Interact + Material.Scatter of hit i; false on a miss
static bool query_contact(const OracleScene* s, const EchoRay* rays, const EchoHit* hits, const EchoTokenHierarchy* layers, uint64_t i, Contact& contact)
{
	if (hits[i].token == ECHO_TOKEN_EMPTY) return false;
	TraceQuery query = make_trace_query(rays[i]);
	query.token = hits[i].token;
	query.distance = hits[i].distance;
	query.uv = { hits[i].uv[0], hits[i].uv[1] };
	query.tokenLayers = query_layers(layers, i);
	interact(s->scene, query, contact);
	return true;
}

extern "C"
{

void oracle_interact_batch(const OracleScene* s, const EchoRay* rays, const EchoHit* hits, const EchoTokenHierarchy* hitLayers, uint64_t n, EchoContact* out)
{
	for (uint64_t i = 0; i < n; i++)
	{
		EchoContact o = {};
		o.material = ECHO_TOKEN_EMPTY;
		Contact contact;

		if (query_contact(s, rays, hits, hitLayers, i, contact))
		{
			query_store(o.position, contact.point.position);
			query_store(o.normal, contact.point.normal);
			query_store(o.shadeNormal, contact.shadeNormal);
			if (!s->scene.textures.empty()) // the texture coordinate is only computed where a texture can read it
			{
				o.texcoord[0] = contact.texcoord.x;
				o.texcoord[1] = contact.texcoord.y;
			}
			o.material = contact.material;
			const EchoMaterial& material = s->scene.materials[contact.material];
			bool emissive = material.type == ECHO_MATERIAL_EMISSIVE && positive(emissive_power(material)); // Path.contribute_emissive
			query_store_rgb(o.emission, emissive ? emissive_emit(material, contact.point, contact.outgoing) : kBlack);
			o.lobes = (uint32_t)contact.bsdf.count;
		}

		out[i] = o;
	}
}

void oracle_scatter_sample_batch(const OracleScene* s, const EchoRay* rays, const EchoHit* hits, const EchoTokenHierarchy* hitLayers, const float* samples2,
                                 uint64_t n, EchoScatter* out)
{
	for (uint64_t i = 0; i < n; i++)
	{
		EchoScatter o = {};
		Contact contact;

		if (query_contact(s, rays, hits, hitLayers, i, contact))
		{
			Float3 incident;
			const BxDF* selected;
			ProbableRGB sampled = contact.bsdf.sample(contact.outgoing, Float2{ sample1d(samples2[i * 2]), sample1d(samples2[i * 2 + 1]) }, incident, selected);
			query_store(o.incident, incident);
			o.pdf = sampled.pdf;
			query_store_rgb(o.value, sampled.content);
			o.specular = selected && type_any(selected->type, Specular) ? 1u : 0u;
		}

		out[i] = o;
	}
}

void oracle_scatter_evaluate_batch(const OracleScene* s, const EchoRay* rays, const EchoHit* hits, const EchoTokenHierarchy* hitLayers, const float* incident3,
                                   uint64_t n, float* outRGBA)
{
	for (uint64_t i = 0; i < n; i++)
	{
		float* o = outRGBA + i * 4;
		o[0] = o[1] = o[2] = o[3] = 0.0f;
		Contact contact;
		if (!query_contact(s, rays, hits, hitLayers, i, contact)) continue;

		Float3 incident = f3(incident3 + i * 3);
		query_store_rgb(o, contact.bsdf.evaluate(contact.outgoing, incident));
		o[3] = contact.bsdf.probability_density(contact.outgoing, incident);
	}
}

void oracle_light_pick_batch(const OracleScene* s, const EchoSurface* points, const float* samples1, uint64_t n, uint32_t* tokens, EchoTokenHierarchy* layers, float* pmf)
{
	for (uint64_t i = 0; i < n; i++)
	{
		Layers picked;
		tokens[i] = s->scene.pick(query_point(points[i]), sample1d(samples1[i]), pmf[i], &picked);
		if (!layers) continue;

		EchoTokenHierarchy h = {};
		h.instanceCount = picked.count;
		for (uint32_t k = 0; k < picked.count; k++) h.instances[k] = picked.instances[k];
		layers[i] = h;
	}
}

void oracle_light_mass_batch(const OracleScene* s, const uint32_t* tokens, const EchoTokenHierarchy* layers, const EchoSurface* points, uint64_t n, float* pmf)
{
	for (uint64_t i = 0; i < n; i++)
		pmf[i] = tokens[i] == ECHO_TOKEN_EMPTY ? 0.0f : s->scene.probability_mass(tokens[i], query_point(points[i]), query_layers(layers, i));
}

void oracle_light_sample_batch(const OracleScene* s, const uint32_t* tokens, const EchoTokenHierarchy* layers, const EchoSurface* points, const float* samples2,
                               uint64_t n, EchoLightSample* out)
{
	for (uint64_t i = 0; i < n; i++)
	{
		EchoLightSample o = {};

		if (tokens[i] != ECHO_TOKEN_EMPTY)
		{
			Float3 incident;
			float travel;
			ProbableRGB sampled = scene_sample_light(s->scene, tokens[i], query_layers(layers, i), query_point(points[i]),
			                                         Float2{ sample1d(samples2[i * 2]), sample1d(samples2[i * 2 + 1]) }, incident, travel);
			query_store_rgb(o.radiance, sampled.content);
			o.pdf = sampled.pdf;
			query_store(o.incident, incident);
			o.travel = travel;
		}

		out[i] = o;
	}
}

void oracle_light_pdf_batch(const OracleScene* s, const uint32_t* tokens, const EchoTokenHierarchy* layers, const EchoSurface* points, const float* incident3,
                            uint64_t n, float* pdf)
{
	for (uint64_t i = 0; i < n; i++)
		pdf[i] = tokens[i] == ECHO_TOKEN_EMPTY ? 0.0f : scene_light_pdf(s->scene, tokens[i], query_layers(layers, i), query_point(points[i]), f3(incident3 + i * 3));
}

void oracle_evaluate_infinite_batch(const OracleScene* s, const float* directions3, uint64_t n, int32_t direct, float* outRGB3)
{
	for (uint64_t i = 0; i < n; i++) query_store_rgb(outRGB3 + i * 3, evaluate_infinite(s->scene, f3(directions3 + i * 3), direct != 0));
}

} // extern "C"
