// debug.cu — device mirrors of the oracle's known-answer hooks (include/echo_b200_debug.h): single BxDF lobes and the
// FastMath shims, so tests can compare the device arithmetic with oracle/ bit for bit and replay the property checks of
// the reference's src/Echo.UnitTests/Evaluation/BxDFTests.cs and Common/FastMathTests.cs on the GPU.
#include "echo_internal.h"
#include "echo_shading.cuh"

namespace echo
{

// kinds: oracle/oracle.h ORACLE_BXDF_*
enum : int
{
	DBG_LAMBERTIAN_REFLECTION = 0, DBG_LAMBERTIAN, DBG_OREN_NAYAR, DBG_SPECULAR_REFLECTION_REAL, DBG_SPECULAR_REFLECTION_COMPLEX,
	DBG_SPECULAR_TRANSMISSION, DBG_SPECULAR_FRESNEL, DBG_GLOSSY_REFLECTION_REAL, DBG_GLOSSY_REFLECTION_COMPLEX, DBG_GLOSSY_TRANSMISSION, DBG_COATED_LAMBERTIAN
};

ECHO_DEVICE int debug_type(int kind)
{
	switch (kind)
	{
		case DBG_LAMBERTIAN_REFLECTION:
		case DBG_COATED_LAMBERTIAN:
		case DBG_OREN_NAYAR: return FT_REFLECTIVE | FT_DIFFUSE;
		case DBG_LAMBERTIAN: return FT_DIFFUSE | FT_REFLECTIVE | FT_TRANSMISSIVE;
		case DBG_SPECULAR_REFLECTION_REAL:
		case DBG_SPECULAR_REFLECTION_COMPLEX: return FT_SPECULAR | FT_REFLECTIVE;
		case DBG_SPECULAR_TRANSMISSION: return FT_SPECULAR | FT_TRANSMISSIVE;
		case DBG_SPECULAR_FRESNEL: return FT_SPECULAR | FT_REFLECTIVE | FT_TRANSMISSIVE;
		case DBG_GLOSSY_REFLECTION_REAL:
		case DBG_GLOSSY_REFLECTION_COMPLEX: return FT_GLOSSY | FT_REFLECTIVE;
		default: return FT_GLOSSY | FT_TRANSMISSIVE;
	}
}

ECHO_DEVICE Sampled debug_sample(int kind, const Bsdf& b, vec2 sample, vec3 outgoing, vec3& incident)
{
	switch (kind)
	{
		case DBG_LAMBERTIAN_REFLECTION: return lambert_reflection_sample<false>(b, sample, outgoing, incident);
		case DBG_LAMBERTIAN: return lambert_two_sided_sample(sample, outgoing, incident);
		case DBG_OREN_NAYAR: return lambert_reflection_sample<true>(b, sample, outgoing, incident);
		case DBG_SPECULAR_REFLECTION_REAL: return specular_reflection_sample<true>(b, outgoing, incident);
		case DBG_SPECULAR_REFLECTION_COMPLEX: return specular_reflection_sample<false>(b, outgoing, incident);
		case DBG_SPECULAR_TRANSMISSION: return specular_transmission_sample(b.etaAbove, b.etaBelow, outgoing, incident);
		case DBG_SPECULAR_FRESNEL: return specular_fresnel_sample(b, sample, outgoing, incident);
		case DBG_GLOSSY_REFLECTION_REAL: return glossy_reflection_sample<true>(b, sample, outgoing, incident);
		case DBG_GLOSSY_REFLECTION_COMPLEX: return glossy_reflection_sample<false>(b, sample, outgoing, incident);
		case DBG_COATED_LAMBERTIAN: return coated_lambert_sample(b, sample, outgoing, incident);
		default: return glossy_transmission_sample(b, sample, outgoing, incident);
	}
}

ECHO_DEVICE rgb debug_evaluate(int kind, const Bsdf& b, vec3 outgoing, vec3 incident)
{
	switch (kind)
	{
		case DBG_LAMBERTIAN_REFLECTION: return lambert_reflection_evaluate<false>(b, outgoing, incident);
		case DBG_LAMBERTIAN: return make_rgb(kTauR);
		case DBG_OREN_NAYAR: return lambert_reflection_evaluate<true>(b, outgoing, incident);
		case DBG_GLOSSY_REFLECTION_REAL: return glossy_reflection_evaluate<true>(b, outgoing, incident);
		case DBG_GLOSSY_REFLECTION_COMPLEX: return glossy_reflection_evaluate<false>(b, outgoing, incident);
		case DBG_GLOSSY_TRANSMISSION: return glossy_transmission_evaluate(b, outgoing, incident);
		case DBG_COATED_LAMBERTIAN: return coated_lambert_evaluate(b, outgoing, incident);
		default: return make_rgb(0.0f);
	}
}

ECHO_DEVICE float debug_pdf(int kind, const Bsdf& b, vec3 outgoing, vec3 incident)
{
	switch (kind)
	{
		case DBG_LAMBERTIAN_REFLECTION:
		case DBG_COATED_LAMBERTIAN:
		case DBG_OREN_NAYAR: return lambert_reflection_pdf(outgoing, incident);
		case DBG_LAMBERTIAN: return abs_bits(cosine_p(incident)) * kTauR;
		case DBG_GLOSSY_REFLECTION_REAL: return glossy_reflection_pdf<true>(b, outgoing, incident);
		case DBG_GLOSSY_REFLECTION_COMPLEX: return glossy_reflection_pdf<false>(b, outgoing, incident);
		case DBG_GLOSSY_TRANSMISSION: return glossy_transmission_pdf(b, outgoing, incident);
		default: return 0.0f;
	}
}

__global__ void debug_bxdf_kernel(int kind, const float* __restrict__ params, const float* __restrict__ outgoing3, const float* __restrict__ samples2,
                                  uint64_t n, float* __restrict__ sampled8, float* __restrict__ evaluated4, float* __restrict__ inverse4)
{
	uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;

	Bsdf b = {};
	b.alphaX = params[0];
	b.alphaY = params[1];
	b.etaAbove = params[2];
	b.etaBelow = params[3];

	if (kind == DBG_SPECULAR_REFLECTION_COMPLEX || kind == DBG_GLOSSY_REFLECTION_COMPLEX)
		complex_fresnel_setup({ params[2], params[3], params[4] }, { params[5], params[6], params[7] }, { params[8], params[9], params[10] }, b.eta2, b.etaK2);

	if (kind == DBG_COATED_LAMBERTIAN) coated_lambert_setup(b, { params[5], params[6], params[7] }, params[4]);

	if (kind == DBG_OREN_NAYAR)
	{
		b.orenA = rcp(fma_f(kPi / 2.0f - 2.0f / 3.0f, params[0], kPi));
		b.orenB = b.orenA * params[0];
	}

	vec3 outgoing = { outgoing3[i * 3], outgoing3[i * 3 + 1], outgoing3[i * 3 + 2] };
	vec2 sample = { sample1d(samples2[i * 2]), sample1d(samples2[i * 2 + 1]) };

	vec3 incident = { 0.0f, 0.0f, 0.0f };
	Sampled result = debug_sample(kind, b, sample, outgoing, incident);

	float* s8 = sampled8 + i * 8;
	s8[0] = result.content.r; s8[1] = result.content.g; s8[2] = result.content.b; s8[3] = result.pdf;
	s8[4] = incident.x; s8[5] = incident.y; s8[6] = incident.z; s8[7] = (float)debug_type(kind);

	rgb value = debug_evaluate(kind, b, outgoing, incident);
	float* e4 = evaluated4 + i * 4;
	e4[0] = value.r; e4[1] = value.g; e4[2] = value.b; e4[3] = debug_pdf(kind, b, outgoing, incident);

	value = debug_evaluate(kind, b, incident, outgoing);
	float* i4 = inverse4 + i * 4;
	i4[0] = value.r; i4[1] = value.g; i4[2] = value.b; i4[3] = debug_pdf(kind, b, incident, outgoing);
}

__global__ void debug_math_kernel(int op, const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c, uint64_t n, float* __restrict__ out)
{
	uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;

	float x = a[i], y = b[i], z = c[i], r;
	float s, co;

	switch (op)
	{
		case 0: r = max0(x); break;
		case 1: r = clamp01(x); break;
		case 2: r = clamp11(x); break;
		case 3: r = clamp_epsilon(x); break;
		case 4: r = abs_bits(x); break;
		case 5: r = sqrt0(x); break;
		case 6: r = sqrt_r0(x); break;
		case 7: r = one_minus2(x); break;
		case 8: r = identity(x); break;
		case 9: r = fma_f(x, y, z); break;
		case 10: r = positive(x) ? 1.0f : 0.0f; break;
		case 11: r = almost_zero(x) ? 1.0f : 0.0f; break;
		case 12: r = min_sse(x, y); break;
		case 13: r = max_sse(x, y); break;
		case 100: sincos_det(x, s, co); r = s; break;
		case 101: sincos_det(x, s, co); r = co; break;
		case 102: r = sample_value(sample_key(__float_as_uint(x), __float_as_uint(y), __float_as_uint(z)), 0u); break;
		default: r = __uint_as_float(0x7FC00000u); break;
	}

	out[i] = r;
}

// op 103: the stratified sequence's draw (ECHO_DISTRIBUTION_STRATIFIED), one per element pair (2i, 2i + 1), inputs as bits:
// a = {seed, pixel}, b = {sample index, extend}, c = {first dimension, 1 for a 2D draw}; out = {value, second value or 0}
__global__ void debug_stratified_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c, uint64_t pairs, float* __restrict__ out)
{
	uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= pairs) return;

	uint32_t seed = __float_as_uint(a[2 * i]), pixel = __float_as_uint(a[2 * i + 1]);
	uint32_t sample = __float_as_uint(b[2 * i]), extend = __float_as_uint(b[2 * i + 1]);
	uint32_t dimension = __float_as_uint(c[2 * i]);

	if (extend == 0u || extend > (uint32_t)ECHO_DISTRIBUTION_STRATIFIED_EXTEND_MAX)
	{
		out[2 * i] = out[2 * i + 1] = __uint_as_float(0x7FC00000u);
		return;
	}

	uint32_t series = stratified_series(seed, pixel, sample / extend);
	Strata strata = make_strata(extend, sample);
	vec2 value = __float_as_uint(c[2 * i + 1]) != 0u ? stratified_2d(series, dimension, strata) : vec2{ stratified_1d(series, dimension, strata), 0.0f };
	out[2 * i] = value.x;
	out[2 * i + 1] = value.y;
}

bool launch_debug_bxdf(int32_t kind, const float* params, const float* outgoing, const float* samples, uint64_t n,
                       float* sampled8, float* evaluated4, float* inverse4, cudaStream_t stream)
{
	if (kind < 0 || kind > DBG_COATED_LAMBERTIAN) { set_error("unknown BxDF kind"); return false; }
	if (n == 0) return true;
	debug_bxdf_kernel<<<(unsigned int)((n + 127) / 128), 128, 0, stream>>>(kind, params, outgoing, samples, n, sampled8, evaluated4, inverse4);
	return check_cuda(cudaGetLastError(), "debug_bxdf_kernel launch");
}

bool launch_debug_math(int32_t op, const float* a, const float* b, const float* c, uint64_t n, float* out, cudaStream_t stream)
{
	if (n == 0) return true;

	if (op == 103)
	{
		if (n % 2 != 0) { set_error("op 103 takes element pairs"); return false; }
		debug_stratified_kernel<<<(unsigned int)((n / 2 + 127) / 128), 128, 0, stream>>>(a, b, c, n / 2, out);
		return check_cuda(cudaGetLastError(), "debug_stratified_kernel launch");
	}

	debug_math_kernel<<<(unsigned int)((n + 127) / 128), 128, 0, stream>>>(op, a, b, c, n, out);
	return check_cuda(cudaGetLastError(), "debug_math_kernel launch");
}

} // namespace echo
