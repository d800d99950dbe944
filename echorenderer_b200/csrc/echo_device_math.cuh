// echo_device_math.cuh — device arithmetic with the bit behaviour of Echo's C#/x64 math.
//
// The whole library is compiled with -fmad=false (RyuJIT never contracts a*b+c); fused operations appear only where
// the reference calls FastMath.FMA / OneMinus2 / Float4.Lerp on an FMA3 host, written here as explicit __fmaf_rn.
// Divisions, reciprocals and square roots use the IEEE-rounded intrinsics, denormals are kept (no -ftz).
// Reference: src/Echo.Core/Common/Mathematics/FastMath.cs, Common/Packed/Float3.cs, Textures/Colors/RGB128.cs,
// Common/Mathematics/Primitives/OrthonormalTransform.cs, Evaluation/Sampling/Sample1D.cs + Sample2D.cs.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace echo
{

#define ECHO_DEVICE __device__ __forceinline__

// The shading kernels are long straight-line code (the dielectric class: 15 k SASS instructions, 6 k of them executed by every
// path) and stall on instruction fetch (ncu: stall_no_inst 49 % of samples, profiles/README.md). Helpers that are called from
// many sites with scalar arguments only are therefore compiled ONCE per kernel (noinline), so that their call sites reuse the
// same instruction-cache lines: level 1 = the microfacet helpers, level 2 = also Float3.Normalized and the glossy lobes'
// evaluate / pdf. -DECHO_SHARE_LEVEL=0 restores full inlining (A/B: variants/ab13.sh). The arithmetic is the same either way.
#ifndef ECHO_SHARE_LEVEL
#define ECHO_SHARE_LEVEL 2
#endif
#if ECHO_SHARE_LEVEL >= 1
#define ECHO_SHARED_CODE static __device__ __noinline__
#else
#define ECHO_SHARED_CODE ECHO_DEVICE
#endif
#if ECHO_SHARE_LEVEL >= 2
#define ECHO_SHARED_CODE_2 static __device__ __noinline__
#else
#define ECHO_SHARED_CODE_2 ECHO_DEVICE
#endif

constexpr float kInfinity = __builtin_huge_valf();
constexpr float kPi = 3.14159265358979323846f;     // Scalars.cs:15
constexpr float kPiR = 0.31830988618379067154f;    // Scalars.cs:20
constexpr float kTau = 6.28318530717958647692f;    // Scalars.cs:25
constexpr float kTauR = 0.15915494309189533577f;   // Scalars.cs:30
constexpr float kRoot2 = 1.41421356237309504880f;  // Scalars.cs:45
constexpr float kEpsilon = 8E-7f;                  // FastMath.cs:32
constexpr float kOneMinusEpsilon = 0.99999994f;    // FastMath.cs:37

// ---- scalar helpers (FastMath.cs) ----
ECHO_DEVICE float min_sse(float a, float b) { return a < b ? a : b; } // minss: second operand on NaN (:57-62)
ECHO_DEVICE float max_sse(float a, float b) { return a > b ? a : b; } // maxss (:69-74)
ECHO_DEVICE float max0(float v) { return max_sse(0.0f, v); }
ECHO_DEVICE float clamp01(float v) { return min_sse(1.0f, max_sse(0.0f, v)); }
ECHO_DEVICE float clamp11(float v) { return min_sse(1.0f, max_sse(-1.0f, v)); }
ECHO_DEVICE float clamp_epsilon(float v) { return min_sse(kOneMinusEpsilon, max_sse(0.0f, v)); }
ECHO_DEVICE float abs_bits(float v) { return __uint_as_float(__float_as_uint(v) & 0x7FFFFFFFu); }
ECHO_DEVICE float sqrt0(float v) { return v <= 0.0f ? 0.0f : __fsqrt_rn(v); }   // :134-140
ECHO_DEVICE float rcp(float v) { return __frcp_rn(v); }                        // IEEE 1f / v
ECHO_DEVICE float div(float a, float b) { return __fdiv_rn(a, b); }
ECHO_DEVICE float sqrt_r0(float v) { return rcp(sqrt0(v)); }                   // :148
ECHO_DEVICE float fma_f(float a, float b, float c) { return __fmaf_rn(a, b, c); } // :180-184
ECHO_DEVICE float one_minus2(float v) { return __fmaf_rn(-v, v, 1.0f); }       // :155-161
ECHO_DEVICE float identity(float v) { return sqrt0(one_minus2(v)); }          // :170
ECHO_DEVICE bool positive(float v) { return kEpsilon <= v; }                  // :204
ECHO_DEVICE bool positive(float v, float epsilon) { return epsilon <= v; }
ECHO_DEVICE bool almost_zero(float v) { return (__float_as_uint(v) << 1) < (__float_as_uint(kEpsilon) << 1); } // :210-217
ECHO_DEVICE float max_net(float a, float b) { return (a != a) ? a : ((b != b) ? b : (a > b ? a : b)); } // Math.Max (operands never both zero here)

// Deterministic sincos shared bit-for-bit with oracle/math.hpp::sincos_det; stands in for MathF.SinCos (FastMath.cs:190-198).
ECHO_DEVICE void sincos_det(float radians, float& sinOut, float& cosOut)
{
	float q = rintf(radians * 0.6366197466850281f);
	int quadrant = (int)q;

	float r = __fmaf_rn(q, -1.5707963705062866f, radians);
	r = __fmaf_rn(q, 4.371138828673793e-08f, r);
	r = __fmaf_rn(q, 1.7151245100058819e-15f, r);

	float r2 = r * r;

	float s = __fmaf_rn(r2, -1.9515295891e-4f, 8.3321608736e-3f);
	s = __fmaf_rn(s, r2, -1.6666654611e-1f);
	s = __fmaf_rn(s * r2, r, r);

	float c = __fmaf_rn(r2, 2.443315711809948e-5f, -1.388731625493765e-3f);
	c = __fmaf_rn(c, r2, 4.166664568298827e-2f);
	c = __fmaf_rn(c, r2, -0.5f);
	c = __fmaf_rn(c, r2, 1.0f);

	if (quadrant & 1)
	{
		float t = s;
		s = c;
		c = t;
	}

	if (quadrant & 2) s = -s;
	if ((quadrant + 1) & 2) c = -c;

	sinOut = s;
	cosOut = c;
}

// ---- Float3 (Common/Packed/Float3.cs) ----
struct vec3
{
	float x, y, z;
};

ECHO_DEVICE vec3 make_vec3(float x, float y, float z) { return vec3{ x, y, z }; }
ECHO_DEVICE vec3 operator+(vec3 a, vec3 b) { return { a.x + b.x, a.y + b.y, a.z + b.z }; }
ECHO_DEVICE vec3 operator-(vec3 a, vec3 b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
ECHO_DEVICE vec3 operator*(vec3 a, float b) { return { a.x * b, a.y * b, a.z * b }; }
ECHO_DEVICE vec3 operator*(float a, vec3 b) { return { a * b.x, a * b.y, a * b.z }; }
ECHO_DEVICE vec3 operator/(vec3 a, float b) { return { div(a.x, b), div(a.y, b), div(a.z, b) }; }
ECHO_DEVICE vec3 operator-(vec3 a) { return { -a.x, -a.y, -a.z }; }

ECHO_DEVICE float dot(vec3 a, vec3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; } // (x*x' + y*y') + z*z', Float3.cs:275
ECHO_DEVICE float squared_magnitude(vec3 a) { return a.x * a.x + a.y * a.y + a.z * a.z; }

// Float3.cs:268-273: fp64 products are exact, so fma(a, b, -(c*d)) rounds exactly like a*b - c*d
ECHO_DEVICE float cross_lane(float a, float b, float c, float d)
{
	return __double2float_rn(__fma_rn((double)a, (double)b, -__dmul_rn((double)c, (double)d)));
}

ECHO_DEVICE vec3 cross(vec3 a, vec3 b)
{
	return { cross_lane(a.y, b.z, a.z, b.y), cross_lane(a.z, b.x, a.x, b.z), cross_lane(a.x, b.y, a.y, b.x) };
}

ECHO_DEVICE double squared_magnitude_double(vec3 a) // Float3.cs:48-52: ((x*x) + (y*y)) + (z*z), products exact
{
	double x = a.x, y = a.y, z = a.z;
	return __dadd_rn(__fma_rn(y, y, __dmul_rn(x, x)), __dmul_rn(z, z));
}

ECHO_DEVICE float magnitude(vec3 a) { return __double2float_rn(__dsqrt_rn(squared_magnitude_double(a))); } // Float3.cs:30-40

ECHO_SHARED_CODE_2 vec3 normalized(vec3 a) // Float3.cs:171-181 + Scalars.cs:172-186
{
	double squared = squared_magnitude_double(a);
	if (squared == 0.0 || fabs(squared) < 1E-10 * 2.2250738585072014e-308) return { 0.0f, 0.0f, 0.0f };
	return rcp(__double2float_rn(__dsqrt_rn(squared))) * a;
}

ECHO_DEVICE vec3 reflect(vec3 value, vec3 normal) { return 2.0f * dot(value, normal) * normal - value; } // Float3.cs:340

// Float4x4.MultiplyDirection by the identity (root instance, PreparedScene.cs:100-101), kept literal for zero signs
ECHO_DEVICE vec3 identity_multiply_direction(vec3 d)
{
	return {
		1.0f * d.x + 0.0f * d.y + 0.0f * d.z,
		0.0f * d.x + 1.0f * d.y + 0.0f * d.z,
		0.0f * d.x + 0.0f * d.y + 1.0f * d.z
	};
}

// ---- RGB128 (Textures/Colors/RGB128.cs) ----
struct rgb
{
	float r, g, b;
};

constexpr float kWeightR = 0.212671f, kWeightG = 0.715160f, kWeightB = 0.072169f;

ECHO_DEVICE rgb make_rgb(float v) { return { v, v, v }; }
ECHO_DEVICE rgb operator+(rgb a, rgb b) { return { a.r + b.r, a.g + b.g, a.b + b.b }; }
ECHO_DEVICE rgb operator*(rgb a, rgb b) { return { a.r * b.r, a.g * b.g, a.b * b.b }; }
ECHO_DEVICE rgb operator*(rgb a, float b) { return { a.r * b, a.g * b, a.b * b }; }
ECHO_DEVICE rgb operator/(rgb a, float b) { return { div(a.r, b), div(a.g, b), div(a.b, b) }; }
ECHO_DEVICE float luminance(rgb c) { return (c.r * kWeightR + c.g * kWeightG) + (c.b * kWeightB + 0.0f * 0.0f); } // RGB128.cs:38, Float4.Sum
ECHO_DEVICE bool is_zero(rgb c) { return c.r < kEpsilon / kWeightR && c.g < kEpsilon / kWeightG && c.b < kEpsilon / kWeightB; } // :40-51
ECHO_DEVICE rgb max_epsilon(rgb c) { return { max_sse(c.r, kEpsilon / kWeightR), max_sse(c.g, kEpsilon / kWeightG), max_sse(c.b, kEpsilon / kWeightB) }; }

// ---- OrthonormalTransform.cs:12-66 ----
struct frame
{
	vec3 axisX, axisY, axisZ;
};

ECHO_DEVICE frame make_frame(vec3 z)
{
	frame f;
	f.axisZ = z;

	if (almost_zero(z.x) && almost_zero(z.y))
	{
		f.axisX = { 1.0f, 0.0f, 0.0f };
		f.axisY = z.z > 0.0f ? vec3{ 0.0f, 1.0f, 0.0f } : vec3{ 0.0f, -1.0f, 0.0f };
	}
	else
	{
		f.axisX = normalized(vec3{ z.y, -z.x, 0.0f });
		f.axisY = cross(z, f.axisX);
	}

	return f;
}

ECHO_DEVICE vec3 apply_forward(const frame& f, vec3 d)
{
	return {
		f.axisX.x * d.x + f.axisY.x * d.y + f.axisZ.x * d.z,
		f.axisX.y * d.x + f.axisY.y * d.y + f.axisZ.y * d.z,
		f.axisX.z * d.x + f.axisY.z * d.y + f.axisZ.z * d.z
	};
}

ECHO_DEVICE vec3 apply_inverse(const frame& f, vec3 d)
{
	return {
		f.axisX.x * d.x + f.axisX.y * d.y + f.axisX.z * d.z,
		f.axisY.x * d.x + f.axisY.y * d.y + f.axisY.z * d.z,
		f.axisZ.x * d.x + f.axisZ.y * d.y + f.axisZ.z * d.z
	};
}

// ---- Sample1D / Sample2D ----
struct vec2
{
	float x, y;
};

ECHO_DEVICE float sample1d(float u) { return clamp_epsilon(u); }                      // Sample1D.cs:13-17
ECHO_DEVICE int sample_range(float u, int max) { return (int)(u * (float)max); }      // Sample1D.cs:31-35

ECHO_DEVICE float sample_range(float u, int max, int& index)                          // Sample1D.cs:52-56
{
	index = sample_range(u, max);
	return sample1d(fma_f(u, (float)max, -(float)index));
}

ECHO_DEVICE float sample_stretch(float u, float lower, float upper) { return sample1d(div(u - lower, upper - lower)); } // Sample1D.cs:74-80

ECHO_DEVICE vec2 project_disk(float radius, float angle) // Sample2D.cs:160-166
{
	float s, c;
	sincos_det(angle, s, c);
	return { c * radius, s * radius };
}

ECHO_DEVICE vec3 project_sphere(float z, float u) // Sample2D.cs:153-158
{
	vec2 disk = project_disk(identity(z), kTau * u);
	return { disk.x, disk.y, z };
}

ECHO_DEVICE vec3 uniform_sphere(vec2 s) { return project_sphere(fma_f(s.x, -2.0f, 1.0f), s.y); } // Sample2D.cs:35

// MathF.Atan2 / Asin / Acos pinned to the Cephes single-precision algorithms, operation for operation as oracle/math.hpp
// (atan_det, atan2_det, asin_det, acos_det): only reached through textures.
ECHO_DEVICE float atan_det(float value)
{
	float sign = value < 0.0f ? -1.0f : 1.0f;
	float x = value < 0.0f ? -value : value;
	float y;

	if (x > 2.414213562373095f)
	{
		y = 1.5707963267948966f;
		x = -div(1.0f, x);
	}
	else if (x > 0.4142135623730950f)
	{
		y = 0.7853981633974483f;
		x = div(x - 1.0f, x + 1.0f);
	}
	else y = 0.0f;

	float z = x * x;
	float p = 8.05374449538e-2f * z - 1.38776856032e-1f;
	p = p * z + 1.99777106478e-1f;
	p = p * z - 3.33329491539e-1f;
	y = y + (p * z * x + x);
	return sign * y;
}

ECHO_DEVICE float atan2_det(float y, float x)
{
	if (x == 0.0f)
	{
		if (y == 0.0f) return 0.0f;
		return y > 0.0f ? 1.5707963267948966f : -1.5707963267948966f;
	}

	if (y == 0.0f) return x < 0.0f ? 3.14159265358979323846f : 0.0f;

	float w = x > 0.0f ? 0.0f : (y < 0.0f ? -3.14159265358979323846f : 3.14159265358979323846f);
	return w + atan_det(div(y, x));
}

ECHO_DEVICE float asin_det(float value)
{
	float sign = value < 0.0f ? -1.0f : 1.0f;
	float a = value < 0.0f ? -value : value;
	if (a < 1.0e-4f) return value;

	bool large = a > 0.5f;
	float z, x;

	if (large)
	{
		z = 0.5f * (1.0f - a);
		x = __fsqrt_rn(z);
	}
	else
	{
		x = a;
		z = x * x;
	}

	float p = 4.2163199048e-2f * z + 2.4181311049e-2f;
	p = p * z + 4.5470025998e-2f;
	p = p * z + 7.4953002686e-2f;
	p = p * z + 1.6666752422e-1f;
	float result = p * z * x + x;

	if (large) result = 1.5707963267948966f - (result + result);
	return sign * result;
}

ECHO_DEVICE float acos_det(float value) { return 1.5707963267948966f - asin_det(value); }

ECHO_DEVICE vec3 uniform_cone(vec2 s, float cosMaxP) { return project_sphere(fma_f(cosMaxP - 1.0f, s.x, 1.0f), s.y); } // Sample2D.cs:123-127

ECHO_DEVICE vec2 uniform_triangle(vec2 s) // Sample2D.cs:54-62
{
	float v = sqrt0(s.x);
	return { 1.0f - v, s.y * v };
}

ECHO_DEVICE vec2 concentric_disk(vec2 s) // Sample2D.cs:66-91
{
	float xValue = fma_f(s.x, 2.0f, -1.0f);
	float yValue = fma_f(s.y, 2.0f, -1.0f);

	if (almost_zero(xValue) && almost_zero(yValue)) return { 0.0f, 0.0f };

	float radius, angle;

	if (abs_bits(xValue) > abs_bits(yValue))
	{
		radius = xValue;
		angle = div(kPi / 4.0f * yValue, xValue);
	}
	else
	{
		radius = yValue;
		angle = fma_f(div(xValue, yValue), kPi / -4.0f, kPi / 2.0f);
	}

	return project_disk(radius, angle);
}

ECHO_DEVICE vec3 cosine_hemisphere(vec2 s) // Sample2D.cs:98-106
{
	vec2 disk = concentric_disk(s);
	float z = disk.x * disk.x + disk.y * disk.y;
	return { disk.x, disk.y, sqrt0(1.0f - z) };
}

constexpr float kUniformSpherePdf = kTauR / 2.0f;                                   // Sample2D.cs:108-110
ECHO_DEVICE float uniform_cone_pdf(float cosMaxP) { return div(kTauR, 1.0f - cosMaxP); } // Sample2D.cs:146

// ---- counter-based sample sequence (DESIGN.md "Sample sequence"); same constants as oracle/math.hpp ----
ECHO_DEVICE uint32_t hash32(uint32_t x)
{
	x ^= x >> 16;
	x *= 0x7FEB352Du;
	x ^= x >> 15;
	x *= 0x846CA68Bu;
	x ^= x >> 16;
	return x;
}

ECHO_DEVICE uint32_t sample_key(uint32_t seed, uint32_t pixel, uint32_t sample)
{
	uint32_t h = hash32(seed ^ 0x9E3779B9u);
	h = hash32(h + pixel * 0x85EBCA6Bu + 0x165667B1u);
	h = hash32(h ^ (sample * 0xC2B2AE35u + 0x27D4EB2Fu));
	return h;
}

ECHO_DEVICE float sample_value(uint32_t key, uint32_t dimension)
{
	uint32_t h = hash32(key + dimension * 0x9E3779B1u);
	h = hash32(h ^ 0x68E31DA4u);
	return sample1d((float)(h >> 8) * 5.9604644775390625e-8f);
}

// ---- the stratified sequence (ECHO_DISTRIBUTION_STRATIFIED); same constants and operations as its CPU reference, tests/c_client/stratified_oracle.cpp ----
ECHO_DEVICE uint32_t stratified_series(uint32_t seed, uint32_t pixel, uint32_t epoch)
{
	uint32_t h = hash32(seed ^ 0x3C6EF372u);
	h = hash32(h + pixel * 0x85EBCA6Bu + 0x165667B1u);
	h = hash32(h ^ (epoch * 0xC2B2AE35u + 0x27D4EB2Fu));
	return h;
}

ECHO_DEVICE uint32_t stratified_pattern(uint32_t series, uint32_t dimension) { return hash32(hash32(series + dimension * 0x9E3779B1u) ^ 0x5BD1E995u); }
ECHO_DEVICE uint32_t stratified_jitter(uint32_t pattern, uint32_t position) { return hash32(hash32(pattern ^ 0xB5297A4Du) + position * 0x68E31DA4u); }

ECHO_DEVICE uint32_t stratified_permute(uint32_t i, uint32_t length, uint32_t p) // Kensler's permute (CMJ, Pixar memo 13-01)
{
	uint32_t w = length - 1u; // the next power-of-two mask
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

// (stratum + j) / extend in one IEEE division of exact floats, strictly inside the stratum (stratified_point of tests/c_client/stratified_oracle.cpp)
ECHO_DEVICE float stratified_point(uint32_t stratum, uint32_t jitter, uint32_t extend)
{
	uint32_t bits = 32u - __clz(extend - 1u);
	uint32_t shift = 24u - bits;
	uint32_t numerator = (stratum << shift) | ((jitter >> 8 >> (bits + 1u)) << 1) | 1u;
	return sample1d(__fdiv_rn((float)numerator, (float)(extend << shift)));
}

// a sample's place in its epoch: the epoch's size, the columns m of its 2D grid (the largest divisor not above the root) and its position
struct Strata
{
	uint32_t extend, columns, position;
};

ECHO_DEVICE Strata make_strata(uint32_t extend, uint32_t sampleIndex)
{
	uint32_t m = (uint32_t)__fsqrt_rn((float)extend);
	while (m * m > extend) m--;
	while ((m + 1u) * (m + 1u) <= extend) m++;
	while (extend % m != 0u) m--;
	return { extend, m, sampleIndex % extend };
}

ECHO_DEVICE float stratified_1d(uint32_t series, uint32_t dimension, const Strata& s)
{
	uint32_t p = stratified_pattern(series, dimension);
	return stratified_point(stratified_permute(s.position, s.extend, p), stratified_jitter(p, s.position), s.extend);
}

ECHO_DEVICE vec2 stratified_2d(uint32_t series, uint32_t dimension, const Strata& s) // correlated multi-jittered over m x n
{
	uint32_t m = s.columns, n = s.extend / m;
	uint32_t p = stratified_pattern(series, dimension);
	uint32_t px = hash32(p ^ 0xA511E9B3u), py = hash32(p ^ 0x63D83595u);
	uint32_t shuffled = stratified_permute(s.position, s.extend, p);
	uint32_t x = shuffled % m, y = shuffled / m;
	uint32_t sx = stratified_permute(x, m, px), sy = stratified_permute(y, n, py);
	return { stratified_point(x * n + sy, stratified_jitter(px, s.position), s.extend), stratified_point(y * m + sx, stratified_jitter(py, s.position), s.extend) };
}

} // namespace echo
