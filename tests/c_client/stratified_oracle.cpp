// stratified_oracle.cpp — TEST INFRASTRUCTURE ONLY: the oracle (oracle/api.cpp, compiled here unchanged) with the stratified sample
// sequence of ECHO_DISTRIBUTION_STRATIFIED in it, the CPU reference the device's stratified draws are compared with
// (tests/stratified_oracle.py builds it into a temporary directory and loads it in place of liboracle.so).
//
// The sequence is the reference's StratifiedDistribution (StratifiedDistribution.cs:34-50) without System.Random: every epoch of
// `extend` samples of a pixel is one series (BeginSeries), every dimension shuffles its strata with a keyed permutation (Kensler,
// "Correlated Multi-Jittered Sampling", Pixar technical memo 13-01) and jitters each sample inside its stratum; a 2D draw is correlated
// multi-jittered over an m x n grid (m the largest divisor of extend not above its root): one sample per cell and one per 1/extend stripe
// in either axis. Same constants and operations as csrc/echo_device_math.cuh; DESIGN.md §2 deviation 1.
//
// The oracle's evaluators draw through sample_key(seed, pixel, sample) and sample_value(key, dimension) in the reference's order; below,
// both names are bound to functions that return the series key and the stratified values when the call's EchoRenderParams carries the
// flag (the uniform sequence's values otherwise). A stratified draw needs to know whether its dimension belongs to a 2D draw: the pairing
// is the reference's (CameraSample.cs:19-23: 2D shift, 2D lens; PathTracedEvaluator.cs:60-66 per bounce: 2D bounce, 1D survival, 1D light
// pick, 2D light sample; the auxiliary and naive evaluators: one 2D draw per depth), the one SampleStream::next1d / next2d follow.
#include "../../oracle/math.hpp"
#include "../../include/echo_b200.h"

namespace oracle
{

inline uint32_t stratified_series(uint32_t seed, uint32_t pixel, uint32_t epoch) // BeginSeries: one key per pixel and epoch
{
	uint32_t h = hash32(seed ^ 0x3C6EF372u);
	h = hash32(h + pixel * 0x85EBCA6Bu + 0x165667B1u);
	h = hash32(h ^ (epoch * 0xC2B2AE35u + 0x27D4EB2Fu));
	return h;
}

inline uint32_t stratified_pattern(uint32_t series, uint32_t dimension) { return hash32(hash32(series + dimension * 0x9E3779B1u) ^ 0x5BD1E995u); }
inline uint32_t stratified_jitter(uint32_t pattern, uint32_t position) { return hash32(hash32(pattern ^ 0xB5297A4Du) + position * 0x68E31DA4u); }

// Kensler's permute: a keyed bijection of [0, length), hashing within the next power-of-two mask and cycle-walking
inline uint32_t stratified_permute(uint32_t i, uint32_t length, uint32_t p)
{
	uint32_t w = length - 1u;
	w |= w >> 1;
	w |= w >> 2;
	w |= w >> 4;
	w |= w >> 8;
	w |= w >> 16;

	do
	{
		i ^= p;
		i *= 0xE170893Du;
		i ^= p >> 16;
		i ^= (i & w) >> 4;
		i ^= p >> 8;
		i *= 0x0929EB3Fu;
		i ^= p >> 23;
		i ^= (i & w) >> 1;
		i *= 1u | p >> 27;
		i *= 0x6935FA69u;
		i ^= (i & w) >> 11;
		i *= 0x74DCB303u;
		i ^= (i & w) >> 2;
		i *= 0x9E501CC3u;
		i ^= (i & w) >> 2;
		i *= 0xC860A3DFu;
		i &= w;
		i ^= i >> 5;
	}
	while (i >= length);

	return (i + p) % length;
}

// (stratum + j) / extend with the jitter j an odd multiple of 2^-(24 - bits), bits = the width of extend - 1: the numerator and the
// denominator scaled by 2^(24 - bits) are exact floats below 2^24, and the one rounded division stays strictly inside the stratum
// (at least 2^-24 from either edge, more than half an ulp below 1). Up to extend = 2^23 every stratum keeps a bit of jitter.
inline float stratified_point(uint32_t stratum, uint32_t jitter, uint32_t extend)
{
	uint32_t bits = 0u;
	while ((1u << bits) < extend) bits++;
	uint32_t shift = 24u - bits;
	uint32_t numerator = (stratum << shift) | ((jitter >> 8 >> (bits + 1u)) << 1) | 1u;
	return sample1d((float)numerator / (float)(extend << shift));
}

inline float stratified_1d(uint32_t series, uint32_t dimension, uint32_t position, uint32_t extend)
{
	uint32_t p = stratified_pattern(series, dimension);
	return stratified_point(stratified_permute(position, extend, p), stratified_jitter(p, position), extend);
}

inline uint32_t stratified_columns(uint32_t extend) // m: the largest divisor of extend not above its square root
{
	uint32_t m = 1u;
	while ((uint64_t)(m + 1u) * (m + 1u) <= extend) m++;
	while (extend % m != 0u) m--;
	return m;
}

// dimensions (dimension, dimension + 1): u = (x + (sy + jx) / n) / m and v = (y + (sx + jy) / m) / n, each computed as one
// (stratum + j) / extend with stratum x * n + sy (y * m + sx)
inline Float2 stratified_2d(uint32_t series, uint32_t dimension, uint32_t position, uint32_t extend)
{
	uint32_t m = stratified_columns(extend), n = extend / m;
	uint32_t p = stratified_pattern(series, dimension);
	uint32_t px = hash32(p ^ 0xA511E9B3u), py = hash32(p ^ 0x63D83595u);
	uint32_t shuffled = stratified_permute(position, extend, p);
	uint32_t x = shuffled % m, y = shuffled / m;
	uint32_t sx = stratified_permute(x, m, px), sy = stratified_permute(y, n, py);
	return { stratified_point(x * n + sy, stratified_jitter(px, position), extend), stratified_point(y * m + sx, stratified_jitter(py, position), extend) };
}

// The sequence of the current call, set by the entry points below from its EchoRenderParams before any sample is drawn (calls on one
// library are not concurrent in the suite), and the position of the sample the calling worker thread is evaluating: sample_key is called
// at the start of each sample, on the thread that then draws all of its values.
struct SequenceOfCall
{
	bool stratified = false;
	uint32_t extend = 1u;
	int kind = ECHO_EVALUATOR_PATH_TRACED;
};

inline SequenceOfCall sequenceOfCall;
inline thread_local uint32_t samplePosition = 0u;

inline void begin_call(const EchoRenderParams* params)
{
	sequenceOfCall.stratified = (params->evaluator & ECHO_DISTRIBUTION_STRATIFIED) != 0 && params->extend > 0;
	sequenceOfCall.extend = sequenceOfCall.stratified ? (uint32_t)params->extend : 1u;
	sequenceOfCall.kind = params->evaluator & ECHO_EVALUATOR_KIND_MASK;
}

inline uint32_t sequence_key(uint32_t seed, uint32_t pixel, uint32_t sample)
{
	if (!sequenceOfCall.stratified) return sample_key(seed, pixel, sample);
	samplePosition = sample % sequenceOfCall.extend;
	return stratified_series(seed, pixel, sample / sequenceOfCall.extend);
}

inline float sequence_value(uint32_t key, uint32_t dimension)
{
	if (!sequenceOfCall.stratified) return sample_value(key, dimension);

	uint32_t first = dimension & ~1u; // the camera's two 2D draws, and the one 2D draw per depth of the other evaluators
	if (dimension >= 4u && sequenceOfCall.kind == ECHO_EVALUATOR_PATH_TRACED)
	{
		uint32_t slot = (dimension - 4u) % 6u; // 2D bounce, 1D survival, 1D light pick, 2D light sample
		if (slot == 2u || slot == 3u) return stratified_1d(key, dimension, samplePosition, sequenceOfCall.extend);
		first = dimension - (slot & 1u);
	}

	Float2 value = stratified_2d(key, first, samplePosition, sequenceOfCall.extend);
	return dimension == first ? value.x : value.y;
}

} // namespace oracle

#define sample_key sequence_key
#define sample_value sequence_value
#define oracle_render_tiles oracle_render_tiles_of_call
#define oracle_evaluate_samples oracle_evaluate_samples_of_call
#define oracle_evaluate_samples4 oracle_evaluate_samples4_of_call
#define oracle_spawn_rays oracle_spawn_rays_of_call
#include "../../oracle/api.cpp"
#undef oracle_render_tiles
#undef oracle_evaluate_samples
#undef oracle_evaluate_samples4
#undef oracle_spawn_rays

extern "C"
{

void oracle_render_tiles(const OracleScene* s, const EchoRenderParams* params, const int32_t* tileXY, uint32_t tileCount, float* outRGBA, EchoStats* outStats, int threads)
{
	begin_call(params);
	oracle_render_tiles_of_call(s, params, tileXY, tileCount, outRGBA, outStats, threads);
}

void oracle_evaluate_samples(const OracleScene* s, const EchoRenderParams* params, const int32_t* pixelXY, const uint32_t* sampleIndex, uint64_t n, float* outRGB, int threads)
{
	begin_call(params);
	oracle_evaluate_samples_of_call(s, params, pixelXY, sampleIndex, n, outRGB, threads);
}

void oracle_evaluate_samples4(const OracleScene* s, const EchoRenderParams* params, const int32_t* pixelXY, const uint32_t* sampleIndex, uint64_t n, float* out,
                              int channels, int threads)
{
	begin_call(params);
	oracle_evaluate_samples4_of_call(s, params, pixelXY, sampleIndex, n, out, channels, threads);
}

void oracle_spawn_rays(const OracleScene* s, const EchoRenderParams* params, const int32_t* pixelXY, const uint32_t* sampleIndex, uint64_t n, EchoRay* out)
{
	begin_call(params);
	oracle_spawn_rays_of_call(s, params, pixelXY, sampleIndex, n, out);
}

// the stratified sequence's draw at `dimension` of sample `sample` (epoch sample / extend) of a pixel: out[0], and out[1] for a 2D draw
void oracle_stratified_value(uint32_t seed, uint32_t pixel, uint32_t sample, uint32_t extend, uint32_t dimension, int32_t twoD, float* out)
{
	uint32_t series = stratified_series(seed, pixel, sample / extend);
	if (!twoD)
	{
		out[0] = stratified_1d(series, dimension, sample % extend, extend);
		return;
	}
	Float2 value = stratified_2d(series, dimension, sample % extend, extend);
	out[0] = value.x;
	out[1] = value.y;
}

} // extern "C"
