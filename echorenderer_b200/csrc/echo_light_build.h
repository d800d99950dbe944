// echo_light_build.h — the reference's LightTree.Build (Aggregation/Selection/LightTree.cs:62-113) over LightBound / ConeBound
// (Aggregation/Bounds/LightBound.cs:10-28, ConeBound.cs:28-101) restated as a LEVEL-SYNCHRONOUS build that emits the reference's own
// tree — the same nodes in the same (pre-order) positions, the same emitter map — instead of some other light hierarchy. Unlike the QBVH,
// whose shape never changes a hit, the SHAPE of the light tree is the sampling distribution (LightTree.Pick descends it with the path's
// random number, :115-154), so only this tree keeps sample-level parity with a host-built one.
//
// The reference recurses: a node sorts its emitters by box centre along the major axis of their joint box, sweeps once from each end
// accumulating LightBound.Encapsulate (box union, CONE union, power sum) and LightBound.RelativeArea, cuts at the first position of
// lowest summed cost and recurses into both halves. The box union is exact and associative; the cone union (acos, a rotation, cos) and
// the float power sum are not — a sweep is a chain that has to be walked in order to reproduce its bits. What IS free: the two sweeps of
// a node do not depend on each other, and nothing couples two nodes of the same depth. So all nodes ("segments") of one depth are
// processed together over one array of emitter positions in which every segment is a contiguous range:
//   box     per position: six atomic min / max on the segment's joint box (integer images of the floats) -> BoxBound.MajorAxis
//   keys    per position: (segment begin << 32) | order-preserving image of the centre along that axis; ONE stable radix sort of the
//           whole level sorts every segment in place (finished positions keep theirs); the bounds are gathered in that order
//   sweeps  TWO threads per segment, one per direction, each walking its chain of Encapsulate and storing the bound before every cut
//   cost    per position: the two relative areas of its cut (they depend on nothing but the stored bounds, so they leave the chains) and
//           `costs[i] + area`; one 64-bit atomic min per cut over (image of the cost, cut index): the lowest cost, the FIRST cut among
//           equals (`cost < minCost`, :98)
//   split   per segment: the node's two children — the reference emits
//           nodes in pre-order, tail subtree first (`new Node(Build(bounds[minIndex..]), Build(bounds[..minIndex]))`), and a subtree over
//           L emitters holds 2 L - 1 nodes, so both child indices follow from the cut: parent + 1 and parent + 2 (L - minIndex)
//   assign  positions move to their child segment; a range of one emitter becomes a leaf and drops out
// then the branch bounds bottom-up (`bounds[child0].Encapsulate(bounds[child1])`, one pass per depth) and the emitter map
// (LightTree.AddToMap, :26-37: leaves in pre-order, bit `depth` of the path set on every child1 step).
//
// Transcendentals: the reference calls MathF.Acos / MathF.Cos (ConeBound), Math.Acos (Float3.Angle) and Math.Sin / Math.Cos cast to float
// (Versor(axis, angle)), whose bits belong to the platform's C runtime. They are pinned here (acos_pin / sincos_pin: the algorithms of
// oracle/math.hpp's acos_det / sincos_det, also for the Versor; acos_double_pin: the fdlibm rational approximation, < 1 ulp of binary64) so that g++ and nvcc produce the same bits: the host mirror (libecho_host.so), the CUDA
// backend (lightbuild.cu) and the CPU emulation the -m "not gpu" suite runs (tests/c_client/light_emulation.cpp) all compile THIS file.
// Byte identity is claimed for inputs on which the reference produces no NaN (x86 and the GPU encode a NaN's sign / payload differently).
//
// Every pass is a functor over an index; a Backend supplies for_each, the stable pair sort, the exclusive sum, memory and read-backs.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../include/echo_b200.h"

#if defined(__CUDACC__)
#define LIGHT_HD __host__ __device__ __forceinline__
#else
#define LIGHT_HD inline
#endif

namespace echo
{
namespace lightbuild
{

constexpr float kPi = 3.14159265358979323846f;
constexpr float kTau = 6.28318530717958647692f;
constexpr float kEpsilon = 8E-7f; // FastMath.Epsilon
constexpr uint32_t kNone = 0xFFFFFFFFu;
constexpr uint32_t kMaxLevels = 63u; // LightTree.cs:29: a path through the tree is 64 bits; depth 64 and deeper is refused

struct Vec3
{
	float x, y, z;
};

struct alignas(16) Bound // LightBound: BoxBound + ConeBound + power, 48 bytes (three 16-byte loads / stores)
{
	float lo[3], hi[3];
	float axis[3];
	float cosOffset, cosExtend;
	float power;
};

struct Segment // a branch under construction: positions [begin, begin + length) of the position array
{
	uint32_t begin, length, node, axis;
	uint32_t split, depth;
	unsigned long long path; // AddToMap's `branches` on the way to this node
	unsigned long long best; // (order-preserving image of the lowest cut cost << 32) | cut index; kNoCut until a cut has a finite cost
	int32_t lo[3], hi[3];    // the joint box of the segment's emitters as order-preserving integers (int order == float order, -0 < +0)
};

constexpr unsigned long long kNoCut = ~0ull;

// ---- bits ----

LIGHT_HD uint32_t float_bits(float value)
{
#if defined(__CUDA_ARCH__)
	return __float_as_uint(value);
#else
	uint32_t bits;
	memcpy(&bits, &value, 4);
	return bits;
#endif
}

LIGHT_HD double clear_low_word(double value)
{
#if defined(__CUDA_ARCH__)
	return __longlong_as_double(__double_as_longlong(value) & (long long)0xFFFFFFFF00000000ull);
#else
	uint64_t bits;
	memcpy(&bits, &value, 8);
	bits &= 0xFFFFFFFF00000000ull;
	memcpy(&value, &bits, 8);
	return value;
#endif
}

LIGHT_HD bool sign_bit(float value) { return (float_bits(value) >> 31) != 0u; }

LIGHT_HD float bits_float(uint32_t bits)
{
#if defined(__CUDA_ARCH__)
	return __uint_as_float(bits);
#else
	float value;
	memcpy(&value, &bits, 4);
	return value;
#endif
}

LIGHT_HD int32_t to_ordered(float value)
{
	int32_t bits = (int32_t)float_bits(value);
	return bits >= 0 ? bits : bits ^ 0x7FFFFFFF;
}

LIGHT_HD float from_ordered(int32_t value) { return bits_float((uint32_t)(value >= 0 ? value : value ^ 0x7FFFFFFF)); }

LIGHT_HD void atomic_min_i32(int32_t* address, int32_t value)
{
#if defined(__CUDA_ARCH__)
	atomicMin(address, value);
#else
	if (value < *address) *address = value;
#endif
}

LIGHT_HD void atomic_max_i32(int32_t* address, int32_t value)
{
#if defined(__CUDA_ARCH__)
	atomicMax(address, value);
#else
	if (value > *address) *address = value;
#endif
}

LIGHT_HD void atomic_min_u64(unsigned long long* address, unsigned long long value)
{
#if defined(__CUDA_ARCH__)
	atomicMin(address, value);
#else
	if (value < *address) *address = value;
#endif
}

LIGHT_HD float round_even(float value)
{
#if defined(__CUDA_ARCH__)
	return rintf(value);
#else
	return nearbyintf(value);
#endif
}

// ---- pinned transcendentals (see the header comment) ----

LIGHT_HD void sincos_pin(float radians, float& sinOut, float& cosOut) // == oracle/math.hpp sincos_det, |radians| <= 1024
{
	float q = round_even(radians * 0.6366197466850281f);
	int quadrant = (int)q;

	float r = fmaf(q, -1.5707963705062866f, radians);
	r = fmaf(q, 4.371138828673793e-08f, r);
	r = fmaf(q, 1.7151245100058819e-15f, r);

	float r2 = r * r;

	float s = fmaf(r2, -1.9515295891e-4f, 8.3321608736e-3f);
	s = fmaf(s, r2, -1.6666654611e-1f);
	s = fmaf(s * r2, r, r);

	float c = fmaf(r2, 2.443315711809948e-5f, -1.388731625493765e-3f);
	c = fmaf(c, r2, 4.166664568298827e-2f);
	c = fmaf(c, r2, -0.5f);
	c = fmaf(c, r2, 1.0f);

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

LIGHT_HD float cos_pin(float radians)
{
	float s, c;
	sincos_pin(radians, s, c);
	return c;
}

LIGHT_HD float asin_pin(float value) // == oracle/math.hpp asin_det (Cephes asinf), |value| <= 1
{
	float sign = value < 0.0f ? -1.0f : 1.0f;
	float a = value < 0.0f ? -value : value;
	if (a < 1.0e-4f) return value;

	bool large = a > 0.5f;
	float z, x;

	if (large)
	{
		z = 0.5f * (1.0f - a);
		x = sqrtf(z);
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

LIGHT_HD float acos_pin(float value) { return 1.5707963267948966f - asin_pin(value); }

// Math.Acos for Float3.Angle (binary64): the rational approximation of fdlibm's e_acos.c — R(z) = z P(z) / Q(z) ~ (asin(x) - x) / x^3 on
// z = x^2 <= 1/4, the half-angle identity beyond — every operation a separately rounded IEEE one (no contraction on either compiler).
LIGHT_HD double acos_rational(double z)
{
	double p = z * (1.66666666666666657415e-01 + z * (-3.25565818622400915405e-01 + z * (2.01212532134862925881e-01
		+ z * (-4.00555345006794114027e-02 + z * (7.91534994289814532176e-04 + z * 3.47933107596021167570e-05)))));
	double q = 1.0 + z * (-2.40339491173441421878e+00 + z * (2.02094576023350569471e+00 + z * (-6.88283971605453293030e-01 + z * 7.70381505559019352791e-02)));
	return p / q;
}

LIGHT_HD double acos_double_pin(double x)
{
	const double pio2Hi = 1.57079632679489655800e+00, pio2Lo = 6.12323399573676603587e-17, pi = 3.14159265358979311600e+00;
	double a = x < 0.0 ? -x : x;

	if (!(a < 1.0))
	{
		if (x == 1.0) return 0.0;
		if (x == -1.0) return pi + 2.0 * pio2Lo;
		return (x - x) / (x - x); // |x| > 1 or NaN
	}

	if (a < 0.5)
	{
		if (a < 6.938893903907228e-18) return pio2Hi + pio2Lo; // 2^-57
		double r = acos_rational(x * x);
		return pio2Hi - (x - (pio2Lo - x * r));
	}

	if (x < 0.0)
	{
		double z = (1.0 + x) * 0.5;
		double s = sqrt(z);
		double w = acos_rational(z) * s - pio2Lo;
		return pi - 2.0 * (s + w);
	}

	double z = (1.0 - x) * 0.5;
	double s = sqrt(z);
	double df = clear_low_word(s);
	double c = (z - df * df) / (s + df);
	double w = acos_rational(z) * s + c;
	return 2.0 * (df + w);
}

// ---- Float3 / FastMath ----

LIGHT_HD Vec3 load3(const float* p) { return { p[0], p[1], p[2] }; }

LIGHT_HD Vec3 cross(Vec3 a, Vec3 b) // Float3.Cross, Float3.cs:268-273 (products and difference in binary64)
{
	return {
		(float)((double)a.y * b.z - (double)a.z * b.y),
		(float)((double)a.z * b.x - (double)a.x * b.z),
		(float)((double)a.x * b.y - (double)a.y * b.x)
	};
}

LIGHT_HD double squared_double(Vec3 a) { return (double)a.x * a.x + (double)a.y * a.y + (double)a.z * a.z; }
LIGHT_HD float magnitude(Vec3 a) { return (float)sqrt(squared_double(a)); }

LIGHT_HD Vec3 normalized(Vec3 a) // Float3.Normalized, Float3.cs:171-181
{
	double squared = squared_double(a);
	if (squared == 0.0 || fabs(squared) < 1E-10 * 2.2250738585072014e-308) return { 0.0f, 0.0f, 0.0f };
	float scale = 1.0f / (float)sqrt(squared);
	return { a.x * scale, a.y * scale, a.z * scale };
}

LIGHT_HD float sse_min(float a, float b) { return a < b ? a : b; } // FastMath.Min / Max: Sse.MinScalar / MaxScalar
LIGHT_HD float sse_max(float a, float b) { return a > b ? a : b; }
LIGHT_HD float clamp11(float v) { return sse_min(1.0f, sse_max(-1.0f, v)); }

LIGHT_HD float identity(float v) // FastMath.Identity: sqrt(max(1 - v^2, 0)) with the square fused
{
	float s = fmaf(-v, v, 1.0f);
	return s <= 0.0f ? 0.0f : sqrtf(s);
}

// Math.Min / Math.Max (Float3.Min / Max, Float3.cs:301-302): a NaN wins (the first one), and -0 < +0. Written as selects over the
// order-preserving integer images — int order == float order with -0 below +0 — so that a chain step has no branches to resolve.
LIGHT_HD float math_min(float a, float b)
{
	float r = to_ordered(a) < to_ordered(b) ? a : b;
	r = b != b ? b : r;
	return a != a ? a : r;
}

LIGHT_HD float math_max(float a, float b)
{
	float r = to_ordered(a) > to_ordered(b) ? a : b;
	r = b != b ? b : r;
	return a != a ? a : r;
}

LIGHT_HD float angle_degrees(Vec3 a, Vec3 b) // Float3.Angle, Float3.cs:277-288 (DEGREES)
{
	double squared = squared_double(a) * squared_double(b);
	if (squared == 0.0) return 0.0f;
	double mag = sqrt(squared);
	if (mag == 0.0) return 0.0f;
	double d = (double)a.x * b.x + (double)a.y * b.y + (double)a.z * b.z;
	return (float)acos_double_pin(d / mag) * (float)(180.0 / 3.14159265358979323846);
}

LIGHT_HD Vec3 rotate_axis_angle(Vec3 axis, float angleDegrees, Vec3 v) // new Versor(axis, angle) * v, Versor.cs:37-55,173,223-240 ((float)Math.Sin / Cos there: pinned)
{
	float radians = (angleDegrees / 2.0f) * (float)(3.14159265358979323846 / 180.0);
	float s, c;
	sincos_pin(radians, s, c);
	float dx = axis.x * s, dy = axis.y * s, dz = axis.z * s, dw = c;

	float ddx = dx * dx, ddy = dy * dy, ddz = dz * dz, ddw = dw * dw;
	float dwx = dw * 2.0f * dx, dwy = dw * 2.0f * dy, dwz = dw * 2.0f * dz;
	float dzx = dz * 2.0f * dx, dzy = dz * 2.0f * dy;
	float dyx = dy * 2.0f * dx;

	return {
		ddw * v.x + ddx * v.x - dwz * v.y + dyx * v.y + dwy * v.z + dzx * v.z - ddz * v.x - ddy * v.x,
		dyx * v.x + dwz * v.x + ddy * v.y - ddz * v.y + dzy * v.z - dwx * v.z + ddw * v.y - ddx * v.y,
		dzx * v.x - dwy * v.x + dzy * v.y + dwx * v.y + ddz * v.z - ddy * v.z - ddx * v.z + ddw * v.z
	};
}

// ---- ConeBound / LightBound ----

struct Cone
{
	Vec3 axis;
	float cosOffset, cosExtend;
};

LIGHT_HD Cone cone_union(const Cone& value0, const Cone& value1) // ConeBound.Union, ConeBound.cs:76-101 (the degrees + radians sum is the reference's)
{
	float cosExtend = sse_min(value0.cosExtend, value1.cosExtend);
	Vec3 axis = value0.axis;

	// A cone that already is the whole sphere (offset0 == pi, the largest value acos gives) passes the early exit below whatever the angle
	// between the axes is — Min(max, pi) <= pi, also for a NaN max (Sse.Min hands back its second operand) — so neither arc cosine nor the
	// binary64 angle (a square root, a division, another arc cosine) is computed for it: the same result, and most of a long sweep over
	// emitters facing all ways is such steps. offset0 == pi exactly when the clamped cosine is -1: acos_pin stays below pi for every
	// other input (tests/test_light_build.py walks all of them next to -1).
	if (value0.cosOffset <= -1.0f) return { axis, value0.cosOffset, cosExtend };

	float offset0 = acos_pin(clamp11(value0.cosOffset));
	float offset1 = acos_pin(clamp11(value1.cosOffset));

	float max = angle_degrees(value0.axis, value1.axis) + offset1;

	if (sse_min(max, kPi) <= offset0) return { axis, value0.cosOffset, cosExtend };

	float offset = (offset0 + max) / 2.0f;
	if (offset >= kPi) return { { 0.0f, 1.0f, 0.0f }, -1.0f, cosExtend }; // CreateFullSphere

	Vec3 c = normalized(cross(axis, value1.axis));
	float rotation = offset - offset0;
	axis = rotate_axis_angle(c, rotation, axis);

	return { axis, cos_pin(offset), cosExtend };
}

LIGHT_HD Cone cone_encapsulate(const Cone& self, const Cone& other) // ConeBound.Encapsulate, ConeBound.cs:50-56
{
	return other.cosOffset > self.cosOffset ? cone_union(self, other) : cone_union(other, self);
}

LIGHT_HD float cone_relative_area(const Cone& cone) // ConeBound.RelativeArea, ConeBound.cs:28-46
{
	float offset = acos_pin(clamp11(cone.cosOffset));
	float extend = acos_pin(clamp11(cone.cosExtend));

	float angle = sse_min(offset + extend, kPi) * 2.0f;
	float sinOffset = identity(cone.cosOffset);

	return kTau * (1.0f - cone.cosOffset) + kPi / 2.0f * (angle * sinOffset - cos_pin(offset - angle) - 2.0f * offset * sinOffset + cone.cosOffset);
}

LIGHT_HD Cone cone_of(const Bound& b) { return { { b.axis[0], b.axis[1], b.axis[2] }, b.cosOffset, b.cosExtend }; }

LIGHT_HD float half_area(const Bound& b) // BoxBound.HalfArea, BoxBound.cs:80-87
{
	float x = b.hi[0] - b.lo[0], y = b.hi[1] - b.lo[1], z = b.hi[2] - b.lo[2];
	return x * (y + z) + y * z;
}

LIGHT_HD uint32_t major_axis(const float* lo, const float* hi) // BoxBound.MajorAxis (:92) + Float3.MaxIndex (Float3.cs:130-138)
{
	float x = hi[0] - lo[0], y = hi[1] - lo[1], z = hi[2] - lo[2];
	if (x > y) return x > z ? 0u : 2u;
	return y > z ? 1u : 2u;
}

LIGHT_HD float relative_area(const Bound& b) { return half_area(b) * cone_relative_area(cone_of(b)) * b.power; } // LightBound.RelativeArea, LightBound.cs:22

LIGHT_HD Bound encapsulate(const Bound& self, const Bound& other) // LightBound.Encapsulate, LightBound.cs:24-28
{
	Bound r;
	for (int k = 0; k < 3; k++) { r.lo[k] = math_min(self.lo[k], other.lo[k]); r.hi[k] = math_max(self.hi[k], other.hi[k]); } // BoxBound.Encapsulate, BoxBound.cs:128-132
	Cone cone = cone_encapsulate(cone_of(self), cone_of(other));
	r.axis[0] = cone.axis.x; r.axis[1] = cone.axis.y; r.axis[2] = cone.axis.z;
	r.cosOffset = cone.cosOffset;
	r.cosExtend = cone.cosExtend;
	r.power = self.power + other.power;
	return r;
}

LIGHT_HD float centre(const Bound& b, uint32_t axis) { return (b.hi[axis] + b.lo[axis]) * 0.5f; } // BoxBound.Center = (max + min) / 2

// The comparison of LightTree.cs:76-81 (`center0.CompareTo(center1)`; the sort is made stable, like the host mirror's) as a radix key:
// unsigned order == float order, and -0 == +0 as in the comparison.
LIGHT_HD uint32_t centre_key(float value) // also the image of a cut's cost
{
	if (value == 0.0f) value = 0.0f;
	uint32_t bits = float_bits(value);
	return (bits >> 31) ? ~bits : bits | 0x80000000u;
}

LIGHT_HD float luminance(const float* c) { return (c[0] * 0.212671f + c[1] * 0.715160f) + (c[2] * 0.072169f + 0.0f * 0.0f); } // RGB128.Luminance, RGB128.cs:30-38

LIGHT_HD void fill_node(EchoLightNode& node, const Bound& b)
{
	for (int k = 0; k < 3; k++) { node.boxMin[k] = b.lo[k]; node.boxMax[k] = b.hi[k]; node.coneAxis[k] = b.axis[k]; }
	node.cosOffset = b.cosOffset;
	node.cosExtend = b.cosExtend;
	node.power = b.power;
}

LIGHT_HD Bound bound_of(const EchoLightNode& node)
{
	Bound b;
	for (int k = 0; k < 3; k++) { b.lo[k] = node.boxMin[k]; b.hi[k] = node.boxMax[k]; b.axis[k] = node.coneAxis[k]; }
	b.cosOffset = node.cosOffset;
	b.cosExtend = node.cosExtend;
	b.power = node.power;
	return b;
}

// ---- LightCollection.CreateBounds (LightCollection.cs:91-137): the emitters, in the reference's order ----

struct Sources
{
	const EchoTriangle* triangles;
	uint32_t triangleCount;
	const EchoSphere* spheres;
	uint32_t sphereCount;
	const EchoMaterial* materials;
	uint32_t materialCount;
	const EchoPointLight* points;
	uint32_t pointCount;
	const float* instanceLights; // PreparedInstance.LightBound per placement: box min xyz, max xyz, cone axis xyz, cosOffset, cosExtend, power
	uint32_t instanceCount;

	LIGHT_HD uint32_t candidates() const { return pointCount + triangleCount + sphereCount + instanceCount; }
};

LIGHT_HD float geometry_power(const Sources& s, uint32_t material, float area) // LightCollection.GetGeometryPower (:221-222) over Emissive.Power (Emissive.cs:52-53)
{
	if (material >= s.materialCount || s.materials[material].type != ECHO_MATERIAL_EMISSIVE) return 0.0f;
	return luminance(s.materials[material].albedo) * kPi * area;
}

// candidate c: point lights, then triangles, spheres, placements. false = not an emitter (no emissive material, or power below epsilon)
LIGHT_HD bool emitter(const Sources& s, uint32_t c, Bound& bound, uint32_t& token)
{
	bound.axis[0] = 0.0f; bound.axis[1] = 1.0f; bound.axis[2] = 0.0f; // ConeBound.CreateFullSphere
	bound.cosOffset = -1.0f;
	bound.cosExtend = 0.0f;

	if (c < s.pointCount)
	{
		const EchoPointLight& light = s.points[c];
		for (int k = 0; k < 3; k++) bound.lo[k] = bound.hi[k] = light.position[k];
		bound.power = 4.0f * kPi * luminance(light.intensity); // PointLight.Power, PointLight.cs:31
		token = ECHO_LIGHT_TOKEN_MAKE(ECHO_LIGHT_TYPE_POINT, c);
		return true;
	}

	c -= s.pointCount;

	if (c < s.triangleCount)
	{
		const EchoTriangle& t = s.triangles[c];
		if (t.material >= s.materialCount || s.materials[t.material].type != ECHO_MATERIAL_EMISSIVE) return false;

		Vec3 normal = cross(load3(t.edge1), load3(t.edge2));
		float power = geometry_power(s, t.material, magnitude(normal) / 2.0f);
		if (!(kEpsilon <= power)) return false;

		for (int k = 0; k < 3; k++) // PreparedTriangle.BoxBound, TriangleEntity.cs:142
		{
			float v0 = t.vertex0[k], v1 = v0 + t.edge1[k], v2 = v0 + t.edge2[k];
			bound.lo[k] = sse_min(sse_min(v0, v1), v2);
			bound.hi[k] = sse_max(sse_max(v0, v1), v2);
		}

		Vec3 axis = normalized(normal); // ConeBound.CreateDirection
		bound.axis[0] = axis.x; bound.axis[1] = axis.y; bound.axis[2] = axis.z;
		bound.cosOffset = 1.0f;
		bound.power = power;
		token = ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_TRIANGLE, c);
		return true;
	}

	c -= s.triangleCount;

	if (c < s.sphereCount)
	{
		const EchoSphere& sphere = s.spheres[c];
		float power = geometry_power(s, sphere.material, 4.0f * kPi * sphere.radius * sphere.radius);
		if (!(kEpsilon <= power)) return false;

		for (int k = 0; k < 3; k++) { bound.lo[k] = sphere.position[k] - sphere.radius; bound.hi[k] = sphere.position[k] + sphere.radius; } // SphereEntity.cs:66
		bound.power = power;
		token = ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_SPHERE, c);
		return true;
	}

	c -= s.sphereCount;

	const float* v = s.instanceLights + (size_t)c * 12; // AddInstances, LightCollection.cs:123-135
	if (!(kEpsilon <= v[11])) return false;
	for (int k = 0; k < 3; k++) { bound.lo[k] = v[k]; bound.hi[k] = v[3 + k]; bound.axis[k] = v[6 + k]; }
	bound.cosOffset = v[9];
	bound.cosExtend = v[10];
	bound.power = v[11];
	token = ECHO_TOKEN_MAKE(ECHO_TOKEN_TYPE_INSTANCE, c);
	return true;
}

// ---- passes ----

// ---- a FOREST: the light trees of several packs in one run (the single-pack build is the forest of one tree) ----

struct LightPack // one tree: the pack's ranges of the shared arrays, and where its candidates, emitters and nodes start
{
	uint32_t triangleOffset, triangleCount, sphereOffset, sphereCount, instanceOffset, instanceCount;
	uint32_t materialOffset, materialCount; // the pack's own swatch (LightCollection.cs:145,151)
	uint32_t pointOffset, pointCount;
	uint32_t candidateBase;                 // candidates lie pack by pack, each pack's in LightCollection.CreateBounds order
	uint32_t emitterBase, emitterCount;     // filled by the driver once the emitters are counted
	uint32_t nodeBase;                      // 2 emitterCount - 1 nodes from here
	uint32_t rootSegment;                   // the pack's root segment, kNone for a pack of one emitter (a leaf) or none
	uint32_t pad;
};

LIGHT_HD uint32_t candidate_count(const LightPack& pack) { return pack.pointCount + pack.triangleCount + pack.sphereCount + pack.instanceCount; }

LIGHT_HD uint32_t light_pack_of(const LightPack* packs, uint32_t packCount, uint32_t candidate) // the last pack whose candidates begin at or before
{
	uint32_t low = 0u, high = packCount;
	while (high - low > 1u)
	{
		uint32_t middle = (low + high) / 2u;
		if (packs[middle].candidateBase <= candidate) low = middle;
		else high = middle;
	}
	return low;
}

struct Forest // the shared arrays (backend memory) and the packs
{
	const EchoTriangle* triangles;
	const EchoSphere* spheres;
	const EchoMaterial* materials;
	const EchoPointLight* points;
	const float* instanceLights; // 12 floats per placement
	const LightPack* packs;
	uint32_t packCount;

	LIGHT_HD Sources view(uint32_t p) const // what pack p's own LightCollection sees: its arrays from index 0, tokens relative to them
	{
		const LightPack& pack = packs[p];
		return { triangles + pack.triangleOffset, pack.triangleCount, spheres + pack.sphereOffset, pack.sphereCount, materials + pack.materialOffset, pack.materialCount,
		         points + pack.pointOffset, pack.pointCount, instanceLights + (size_t)pack.instanceOffset * 12, pack.instanceCount };
	}
};

struct FlagPass // 1 where candidate c is an emitter (c == the candidate count: 0, the end of the sum)
{
	Forest forest;
	uint32_t candidates;
	uint32_t* flags;

	LIGHT_HD void operator()(uint32_t c) const
	{
		Bound bound;
		uint32_t token;
		if (c >= candidates) { flags[c] = 0u; return; }
		uint32_t p = light_pack_of(forest.packs, forest.packCount, c);
		flags[c] = emitter(forest.view(p), c - forest.packs[p].candidateBase, bound, token) ? 1u : 0u;
	}
};

struct PackEmittersPass // the first emitter of every pack (and the total after the last): the exclusive sum at the pack's first candidate
{
	const LightPack* packs;
	uint32_t packCount, candidates;
	const uint32_t* slots;
	uint32_t* out;

	LIGHT_HD void operator()(uint32_t p) const { out[p] = slots[p < packCount ? packs[p].candidateBase : candidates]; }
};

struct EmitterPass // emitter k = the k-th flagged candidate; position k starts as emitter k, in the root segment of its pack
{
	Forest forest;
	const uint32_t* slots; // exclusive sum of the flags
	Bound* bounds;
	uint32_t* tokens;
	uint32_t* order;
	uint32_t* segmentOf;

	LIGHT_HD void operator()(uint32_t c) const
	{
		Bound bound;
		uint32_t token;
		uint32_t p = light_pack_of(forest.packs, forest.packCount, c);
		if (!emitter(forest.view(p), c - forest.packs[p].candidateBase, bound, token)) return;

		uint32_t k = slots[c];
		bounds[k] = bound;
		tokens[k] = token;
		order[k] = k;
		segmentOf[k] = forest.packs[p].rootSegment;
	}
};

struct LeafWriter // `new Node(bounds[0].content, bounds[0].token)`, LightTree.cs:64
{
	EchoLightNode* nodes;
	uint32_t* isLeaf;
	unsigned long long* pathOfNode;

	LIGHT_HD void operator()(uint32_t node, const Bound& bound, uint32_t token, unsigned long long path) const
	{
		fill_node(nodes[node], bound);
		nodes[node].child0 = ECHO_TOKEN_EMPTY;
		nodes[node].child1 = token;
		isLeaf[node] = 1u;
		pathOfNode[node] = path;
	}
};

LIGHT_HD Segment new_segment(uint32_t begin, uint32_t length, uint32_t node, uint32_t depth, unsigned long long path)
{
	Segment segment;
	segment.begin = begin; segment.length = length; segment.node = node; segment.axis = 0u;
	segment.split = 0u; segment.depth = depth;
	segment.path = path;
	segment.best = kNoCut;
	for (int k = 0; k < 3; k++) { segment.lo[k] = 0x7FFFFFFF; segment.hi[k] = (int32_t)0x80000000; }
	return segment;
}

struct RootPass // every pack's emitter list as one segment — or as one leaf, or nothing
{
	const LightPack* packs;
	const Bound* bounds;
	const uint32_t* tokens;
	Segment* segments;
	uint32_t* internalNodes;
	LeafWriter leaves;

	LIGHT_HD void operator()(uint32_t p) const
	{
		const LightPack& pack = packs[p];

		if (pack.emitterCount == 1u) leaves(pack.nodeBase, bounds[pack.emitterBase], tokens[pack.emitterBase], 0ull);
		else if (pack.emitterCount > 1u)
		{
			segments[pack.rootSegment] = new_segment(pack.emitterBase, pack.emitterCount, pack.nodeBase, 0u, 0ull);
			internalNodes[pack.rootSegment] = pack.nodeBase;
		}
	}
};

// LightTree.cs:68-74: the joint box of a segment's emitters. BoxBound.Encapsulate is Math.Min / Math.Max per component — exact, and on the
// integer images associative and commutative — so every position folds its emitter's box into its segment's with six atomics, in any order.
struct BoxPass
{
	const uint32_t* order;
	const uint32_t* segmentOf;
	const Bound* bounds;
	Segment* segments;

	LIGHT_HD void operator()(uint32_t p) const
	{
		uint32_t s = segmentOf[p];
		if (s == kNone) return;

		const Bound& b = bounds[order[p]];
		Segment& segment = segments[s];
		for (int k = 0; k < 3; k++) { atomic_min_i32(&segment.lo[k], to_ordered(b.lo[k])); atomic_max_i32(&segment.hi[k], to_ordered(b.hi[k])); }
	}
};

struct AxisPass // ... then its major axis
{
	Segment* segments;

	LIGHT_HD void operator()(uint32_t s) const
	{
		Segment& segment = segments[s];
		float lo[3], hi[3];
		for (int k = 0; k < 3; k++) { lo[k] = from_ordered(segment.lo[k]); hi[k] = from_ordered(segment.hi[k]); }
		segment.axis = major_axis(lo, hi);
	}
};

struct KeyPass
{
	const uint32_t* order;
	const uint32_t* segmentOf;
	const Segment* segments;
	const Bound* bounds;
	unsigned long long* keys;

	LIGHT_HD void operator()(uint32_t p) const
	{
		uint32_t s = segmentOf[p];

		if (s == kNone) keys[p] = (unsigned long long)p << 32; // a finished leaf stays where it is
		else
		{
			const Segment& segment = segments[s];
			keys[p] = (unsigned long long)segment.begin << 32 | centre_key(centre(bounds[order[p]], segment.axis));
		}
	}
};

struct GatherPass // the bounds in position order: the sweeps read them front to back (and back to front) instead of through `order`
{
	const uint32_t* order;
	const uint32_t* segmentOf;
	const Bound* bounds;
	Bound* sorted;

	LIGHT_HD void operator()(uint32_t p) const
	{
		if (segmentOf[p] != kNone) sorted[p] = bounds[order[p]];
	}
};

// LightTree.cs:83-104, the part that is a chain: one thread per (segment, direction) folds LightBound.Encapsulate over its segment and
// stores the bound BEFORE every step. Direction 0: from the last emitter backwards, tails[i] = the bound of emitters [i, length) for
// i = length - 1 .. 1; direction 1: from the first one forwards, heads[i] = that of [0, i) for i = 1 .. length - 1. What the reference
// evaluates inside the same loops — LightBound.RelativeArea of every one of those bounds, four transcendentals each — depends on nothing but
// its bound, so it leaves the chain for CostPass, one thread per cut. Threads [0, stride) walk backwards, [stride, 2 stride) forwards,
// stride a multiple of the warp size: the two chains of a segment run in different warps (at the root they ARE the level), each at the pace
// of its own branches. A chain is latency all the way — one thread, every step waiting for the last — so the emitter of the NEXT step is
// loaded before this step's arithmetic starts (keeping six in flight in a ring of registers, or asking lines into L1 a dozen steps ahead,
// changed nothing: the chain waits for its own arithmetic, not for memory).
struct SweepPass
{

	uint32_t live, stride;
	const Bound* __restrict__ sorted;
	const Segment* __restrict__ segments;
	Bound* __restrict__ tails;
	Bound* __restrict__ heads;

	LIGHT_HD void operator()(uint32_t t) const
	{
		const bool forward = t >= stride;
		const uint32_t s = forward ? t - stride : t;
		if (s >= live) return;

		const uint32_t begin = segments[s].begin, last = segments[s].length - 1u;
		Bound* __restrict__ out = forward ? heads : tails;

		// step k (1 .. last) folds in the emitter at begin + k (forwards) or begin + last - k (backwards)
		Bound bound = sorted[begin + (forward ? 0u : last)];
		Bound next = sorted[begin + (forward ? 1u : last - 1u)];

		for (uint32_t k = 1u; k <= last; k++)
		{
			const Bound current = next;
			if (k < last) next = sorted[begin + (forward ? k + 1u : last - k - 1u)];

			out[begin + (forward ? k : last + 1u - k)] = bound;
			bound = encapsulate(bound, current);
		}
	}
};

// LightTree.cs:85-104, the part that is not: per cut i the cost `costs[i] + lightBound.RelativeArea` = RelativeArea(tails[i]) +
// RelativeArea(heads[i]), and the first cut of lowest cost (`cost < minCost` from +inf: a NaN or infinite cost never wins) as one atomic
// min over (image of the cost, cut index): the lowest cost, and among equal costs the lowest index.
struct CostPass
{
	const uint32_t* segmentOf;
	const Bound* tails;
	const Bound* heads;
	Segment* segments;

	LIGHT_HD void operator()(uint32_t p) const
	{
		uint32_t s = segmentOf[p];
		if (s == kNone) return;

		Segment& segment = segments[s];
		uint32_t i = p - segment.begin;
		if (i == 0u) return;

		float cost = relative_area(tails[p]) + relative_area(heads[p]);
		if (cost < INFINITY) atomic_min_u64(&segment.best, (unsigned long long)centre_key(cost) << 32 | i);
	}
};

struct SplitPass // LightTree.cs:106-112: the branch and its children at the cut CostPass found (leaves are written, branches counted for the next level)
{
	const uint32_t* order;
	const Bound* bounds;
	const uint32_t* tokens;
	Segment* segments;
	EchoLightNode* nodes;
	uint32_t* counts; // [2 s] = the head half lives on, [2 s + 1] = the tail half does
	LeafWriter leaves;

	LIGHT_HD void operator()(uint32_t s) const
	{
		Segment& segment = segments[s];
		const uint32_t begin = segment.begin, length = segment.length;

		uint32_t minIndex = segment.best == kNoCut ? kNone : (uint32_t)(segment.best & 0xFFFFFFFFull);
		if (minIndex == kNone) minIndex = length / 2u; // every cost NaN / inf: the reference throws; the host mirror cuts in the middle
		segment.split = minIndex;

		// new Node(Build(bounds[minIndex..]), Build(bounds[..minIndex])): child0 = the tail, emitted right after its parent
		uint32_t tail = length - minIndex;
		uint32_t child0 = segment.node + 1u, child1 = segment.node + 2u * tail;
		nodes[segment.node].child0 = child0;
		nodes[segment.node].child1 = child1;

		if (tail == 1u) { uint32_t e = order[begin + minIndex]; leaves(child0, bounds[e], tokens[e], segment.path); }
		if (minIndex == 1u) { uint32_t e = order[begin]; leaves(child1, bounds[e], tokens[e], segment.path | 1ull << segment.depth); }

		counts[2u * s] = minIndex > 1u ? 1u : 0u;
		counts[2u * s + 1u] = tail > 1u ? 1u : 0u;
	}
};

struct ChildPass // the halves that live on become the next level's segments, in position order
{
	const Segment* segments;
	const uint32_t* slots; // exclusive sum of the counts
	Segment* next;
	uint32_t* internalNodes; // of the next level

	LIGHT_HD void operator()(uint32_t s) const
	{
		const Segment& segment = segments[s];
		uint32_t tail = segment.length - segment.split;

		if (segment.split > 1u)
		{
			uint32_t k = slots[2u * s];
			next[k] = new_segment(segment.begin, segment.split, segment.node + 2u * tail, segment.depth + 1u, segment.path | 1ull << segment.depth);
			internalNodes[k] = next[k].node;
		}

		if (tail > 1u)
		{
			uint32_t k = slots[2u * s + 1u];
			next[k] = new_segment(segment.begin + segment.split, tail, segment.node + 1u, segment.depth + 1u, segment.path);
			internalNodes[k] = next[k].node;
		}
	}
};

struct AssignPass // positions follow their half
{
	const Segment* segments;
	const uint32_t* slots;
	uint32_t* segmentOf;

	LIGHT_HD void operator()(uint32_t p) const
	{
		uint32_t s = segmentOf[p];
		if (s == kNone) return;

		const Segment& segment = segments[s];
		bool head = p < segment.begin + segment.split;
		uint32_t length = head ? segment.split : segment.length - segment.split;
		segmentOf[p] = length > 1u ? slots[2u * s + (head ? 0u : 1u)] : kNone;
	}
};

struct BranchPass // LightTree.Node's branch constructor (:160-165): child0.bound.Encapsulate(child1.bound), children first
{
	const uint32_t* internalNodes;
	EchoLightNode* nodes;

	LIGHT_HD void operator()(uint32_t i) const
	{
		EchoLightNode& node = nodes[internalNodes[i]];
		fill_node(node, encapsulate(bound_of(nodes[node.child0]), bound_of(nodes[node.child1])));
	}
};

struct RebasePass // child indices relative to the pack's first node, as every pack's own LightTree numbers them
{
	const LightPack* packs;
	uint32_t packCount;
	const uint32_t* isLeaf;
	EchoLightNode* nodes;

	LIGHT_HD void operator()(uint32_t node) const
	{
		if (isLeaf[node]) return;
		uint32_t low = 0u, high = packCount; // the last pack whose nodes begin at or before this one (a pack without nodes shares its base with the next)
		while (high - low > 1u)
		{
			uint32_t middle = (low + high) / 2u;
			if (packs[middle].nodeBase <= node) low = middle;
			else high = middle;
		}
		nodes[node].child0 -= packs[low].nodeBase;
		nodes[node].child1 -= packs[low].nodeBase;
	}
};

struct MapPass // LightTree.AddToMap (:26-37): the leaves in pre-order
{
	const EchoLightNode* nodes;
	const uint32_t* isLeaf;
	const uint32_t* slots; // exclusive sum of isLeaf
	const unsigned long long* pathOfNode;
	uint32_t* emitterTokens;
	unsigned long long* emitterPaths;

	LIGHT_HD void operator()(uint32_t node) const
	{
		if (!isLeaf[node]) return;
		emitterTokens[slots[node]] = nodes[node].child1;
		emitterPaths[slots[node]] = pathOfNode[node];
	}
};

// ---- driver ----

struct Arena
{
	char* base = nullptr;
	size_t used = 0;

	template<class T>
	T* take(size_t count)
	{
		size_t offset = (used + 255) & ~size_t(255);
		used = offset + sizeof(T) * (count ? count : 1);
		return base ? (T*)(base + offset) : nullptr;
	}
};

struct Result
{
	bool ok = false;          // false: a backend call failed
	bool unsupported = false; // some tree is deeper than a 64-bit path (LightTree.cs:29)
	uint32_t emitterCount = 0, nodeCount = 0, levels = 0; // all packs
	std::vector<LightPack> packs; // per pack: emitterBase / emitterCount, nodeBase (2 emitterCount - 1 nodes, or none)
	// backend memory, valid until the backend goes away
	EchoLightNode* nodes = nullptr;
	uint32_t* emitterTokens = nullptr;
	unsigned long long* emitterPaths = nullptr;
};

struct Working // everything sized by the emitter count
{
	Bound* bounds;
	Bound* sorted;
	uint32_t* tokens;
	uint32_t* order[2];
	unsigned long long* keys[2];
	uint32_t* segmentOf;
	Segment* segments[2];
	Bound* tails;
	Bound* heads;
	uint32_t* counts;
	uint32_t* slots;
	uint32_t* internalNodes;
	EchoLightNode* nodes;
	uint32_t* isLeaf;
	uint32_t* leafSlots;
	unsigned long long* pathOfNode;
	uint32_t* emitterTokens;
	unsigned long long* emitterPaths;

	void carve(Arena& arena, size_t n)
	{
		size_t nodeCount = 2 * n;
		bounds = arena.take<Bound>(n);
		sorted = arena.take<Bound>(n);
		tokens = arena.take<uint32_t>(n);
		for (int k = 0; k < 2; k++) { order[k] = arena.take<uint32_t>(n); keys[k] = arena.take<unsigned long long>(n); segments[k] = arena.take<Segment>(n / 2 + 1); }
		segmentOf = arena.take<uint32_t>(n);
		tails = arena.take<Bound>(n);
		heads = arena.take<Bound>(n);
		counts = arena.take<uint32_t>(n + 2);
		slots = arena.take<uint32_t>(n + 2);
		internalNodes = arena.take<uint32_t>(n);
		nodes = arena.take<EchoLightNode>(nodeCount);
		isLeaf = arena.take<uint32_t>(nodeCount + 1);
		leafSlots = arena.take<uint32_t>(nodeCount + 1);
		pathOfNode = arena.take<unsigned long long>(nodeCount);
		emitterTokens = arena.take<uint32_t>(n);
		emitterPaths = arena.take<unsigned long long>(n);
	}
};

// host -> backend: the backend's write(); a backend without one keeps its memory in the host's address space (the sequential CPU backends)
template<class Backend, class T>
auto write_to(Backend& backend, T* destination, const T* source, uint32_t n, int) -> decltype(backend.write(destination, source, n))
{
	return backend.write(destination, source, n);
}

template<class Backend, class T>
bool write_to(Backend&, T* destination, const T* source, uint32_t n, long)
{
	memcpy((void*)destination, (const void*)source, sizeof(T) * n);
	return true;
}

// Backend concept: allocate, for_each, sort_pairs, exclusive_sum, read, fill_zero as echo_sweep.h describes them; write where the
// backend's memory is not the host's.
//
// The light trees of `packCount` packs in one run: every pack's root is one more segment of the first level, so each level serves all
// packs and the run reads back as many levels as its deepest tree has. `forest` points into backend memory except `packs`, which is
// host memory (its ranges and materials; the driver fills in the rest): candidates, emitters and nodes lie pack by pack, and every
// pack's nodes, emitter tokens and bit paths are what its own single-pack build emits (child indices relative to the pack's first node).
template<class Backend>
Result build_forest(Backend& backend, const Forest& forest)
{
	Result result;
	const uint32_t packCount = forest.packCount;
	result.packs.assign(forest.packs, forest.packs + packCount);
	uint32_t candidates = 0u;
	for (LightPack& pack : result.packs) { pack.candidateBase = candidates; candidates += candidate_count(pack); pack.emitterBase = pack.emitterCount = pack.nodeBase = 0u; pack.rootSegment = kNone; }
	if (candidates == 0u) { result.ok = true; return result; }

	// the emitters: flag, rank, scatter
	Arena first;
	first.take<uint32_t>(candidates + 1);
	first.take<uint32_t>(candidates + 1);
	first.take<LightPack>(packCount);
	first.take<uint32_t>(packCount + 1);
	first.base = backend.allocate(first.used + 256);
	if (!first.base) return result;
	first.used = 0;
	uint32_t* flags = first.take<uint32_t>(candidates + 1);
	uint32_t* emitterSlots = first.take<uint32_t>(candidates + 1);
	LightPack* packs = first.take<LightPack>(packCount);
	uint32_t* bases = first.take<uint32_t>(packCount + 1);

	Forest device = forest;
	device.packs = packs;
	if (!write_to(backend, packs, result.packs.data(), packCount, 0)) return result;

	std::vector<uint32_t> emitterBases(packCount + 1);
	if (!backend.for_each(candidates + 1u, FlagPass{ device, candidates, flags })) return result;
	if (!backend.exclusive_sum(flags, emitterSlots, candidates + 1u)) return result;
	if (!backend.for_each(packCount + 1u, PackEmittersPass{ packs, packCount, candidates, emitterSlots, bases })) return result;
	if (!backend.read(bases, emitterBases.data(), packCount + 1u)) return result;
	const uint32_t count = emitterBases[packCount];
	if (count == 0u) { result.ok = true; return result; }

	// every pack's emitters, nodes and root segment
	uint32_t nodeCount = 0u, live = 0u;
	for (uint32_t p = 0; p < packCount; p++)
	{
		LightPack& pack = result.packs[p];
		pack.emitterBase = emitterBases[p];
		pack.emitterCount = emitterBases[p + 1u] - emitterBases[p];
		pack.nodeBase = nodeCount;
		if (pack.emitterCount != 0u) nodeCount += 2u * pack.emitterCount - 1u;
		if (pack.emitterCount > 1u) pack.rootSegment = live++;
	}
	if (!write_to(backend, packs, result.packs.data(), packCount, 0)) return result;

	Working w;
	Arena arena;
	w.carve(arena, count);
	arena.base = backend.allocate(arena.used + 256);
	if (!arena.base) return result;
	arena.used = 0;
	w.carve(arena, count);

	if (!backend.fill_zero(w.nodes, sizeof(EchoLightNode) * nodeCount) || !backend.fill_zero(w.isLeaf, sizeof(uint32_t) * (nodeCount + 1u))) return result;
	if (!backend.for_each(candidates, EmitterPass{ device, emitterSlots, w.bounds, w.tokens, w.order[0], w.segmentOf })) return result;

	LeafWriter leaves{ w.nodes, w.isLeaf, w.pathOfNode };
	if (!backend.for_each(packCount, RootPass{ packs, w.bounds, w.tokens, w.segments[0], w.internalNodes, leaves })) return result;

	std::vector<uint32_t> levelOffsets{ 0u }; // into internalNodes, one entry per depth + the end
	int side = 0;

	while (live != 0u)
	{
		if (result.levels == kMaxLevels) { result.ok = true; result.unsupported = true; return result; }

		Segment* segments = w.segments[side];
		uint32_t offset = levelOffsets.back();
		levelOffsets.push_back(offset + live);

		if (!backend.for_each(count, BoxPass{ w.order[side], w.segmentOf, w.bounds, segments })) return result;
		if (!backend.for_each(live, AxisPass{ segments })) return result;
		if (!backend.for_each(count, KeyPass{ w.order[side], w.segmentOf, segments, w.bounds, w.keys[0] })) return result;
		if (!backend.sort_pairs(w.keys[0], w.keys[1], w.order[side], w.order[side ^ 1], count, 64)) return result;
		const uint32_t* order = w.order[side ^ 1];

		const uint32_t stride = (live + 31u) & ~31u;
		if (!backend.for_each(count, GatherPass{ order, w.segmentOf, w.bounds, w.sorted })) return result;
		if (!backend.for_each(2u * stride, SweepPass{ live, stride, w.sorted, segments, w.tails, w.heads })) return result;
		if (!backend.for_each(count, CostPass{ w.segmentOf, w.tails, w.heads, segments })) return result;
		if (!backend.for_each(live, SplitPass{ order, w.bounds, w.tokens, segments, w.nodes, w.counts, leaves })) return result;
		if (!backend.fill_zero(w.counts + 2u * live, sizeof(uint32_t))) return result;
		if (!backend.exclusive_sum(w.counts, w.slots, 2u * live + 1u)) return result;
		if (!backend.for_each(live, ChildPass{ segments, w.slots, w.segments[side ^ 1], w.internalNodes + offset + live })) return result;
		if (!backend.for_each(count, AssignPass{ segments, w.slots, w.segmentOf })) return result;
		if (!backend.read(w.slots + 2u * live, &live, 1u)) return result;

		side ^= 1;
		++result.levels;
	}

	for (uint32_t level = result.levels; level-- > 0u;)
		if (!backend.for_each(levelOffsets[level + 1u] - levelOffsets[level], BranchPass{ w.internalNodes + levelOffsets[level], w.nodes })) return result;

	if (!backend.exclusive_sum(w.isLeaf, w.leafSlots, nodeCount + 1u)) return result;
	if (!backend.for_each(nodeCount, MapPass{ w.nodes, w.isLeaf, w.leafSlots, w.pathOfNode, w.emitterTokens, w.emitterPaths })) return result;
	if (packCount > 1u && !backend.for_each(nodeCount, RebasePass{ packs, packCount, w.isLeaf, w.nodes })) return result;

	result.ok = true;
	result.emitterCount = count;
	result.nodeCount = nodeCount;
	result.nodes = w.nodes;
	result.emitterTokens = w.emitterTokens;
	result.emitterPaths = w.emitterPaths;
	return result;
}

// one pack: LightCollection.CreateBounds + LightTree.Build of `sources` (backend memory)
template<class Backend>
Result build(Backend& backend, const Sources& sources)
{
	LightPack pack = {};
	pack.triangleCount = sources.triangleCount;
	pack.sphereCount = sources.sphereCount;
	pack.instanceCount = sources.instanceCount;
	pack.materialCount = sources.materialCount;
	pack.pointCount = sources.pointCount;
	const Forest forest = { sources.triangles, sources.spheres, sources.materials, sources.points, sources.instanceLights, &pack, 1u };
	return build_forest(backend, forest);
}

} // namespace lightbuild
} // namespace echo
