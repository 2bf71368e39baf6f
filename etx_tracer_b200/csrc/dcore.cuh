// dcore.cuh — device-side basics: vector algebra, sampler, spectral value type, complex numbers.
//
// Arithmetic contract: every expression keeps the operation ORDER of the reference's shared headers
// (sources/etx/render/shared/math.hxx, sampler.hxx, spectrum.hxx) so that the parity build
// (-fmad=false -DETXB_PARITY=1, transcendentals from portable_math.h) reproduces the CPU oracle bit for
// bit.  The fast build compiles the same source with FMA contraction and CUDA's own math functions.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "portable_math.h"

#define DEV __device__ __forceinline__
#define DEVN __device__ __noinline__
// experiment switches (default: out of line)
#if defined(ETXB_BSDF_INLINE)
#define DEVG_BSDF DEV
#else
#define DEVG_BSDF DEVN
#endif
#if defined(ETXB_MATH_INLINE)
#define DEVG_MATH DEV
#else
#define DEVG_MATH DEVN
#endif

namespace etxb {

// ---- constants (math.hxx:100-114) -------------------------------------------------------------------
constexpr float kQuarterPi = 0.78539816339744830961566084581988f;
constexpr float kHalfPi = 1.5707963267948966192313216916398f;
constexpr float kPi = 3.1415926535897932384626433832795f;
constexpr float kDoublePi = 6.283185307179586476925286766559f;
constexpr float kInvPi = 0.31830988618379067153776752674503f;
constexpr float kSqrtPi = 1.7724538509055160272981674833411f;
constexpr float kEpsilon = 1.192092896e-07f;
constexpr float kMaxFloat = 3.402823466e+38f;
constexpr float kMaxHalf = 65504.0f;
constexpr float kInvMaxHalf = 1.0f / kMaxHalf;
constexpr float kRayEpsilon = 15.0f / (kMaxHalf - 1.0f);
constexpr float kDeltaAlphaTreshold = 1.0e-4f;
constexpr uint32_t kInvalidIndex = ~0u;

// ---- transcendental switch ----------------------------------------------------------------------------
// Out of line where the body is large (the portable double-precision routines of the parity build; powf / inverse trig of the CUDA
// math library in the product build): these are called from dozens of inlined sites per kernel.
#if defined(ETXB_PARITY) && ETXB_PARITY
DEVN float m_sin(float x) { return pm::sinf_(x); }
DEVN float m_cos(float x) { return pm::cosf_(x); }
DEVN float m_exp(float x) { return pm::expf_(x); }
DEVN float m_log(float x) { return pm::logf_(x); }
DEVN float m_pow(float x, float y) { return pm::powf_(x, y); }
DEVN float m_acos(float x) { return pm::acosf_(x); }
DEVN float m_asin(float x) { return pm::asinf_(x); }
DEVN float m_atan(float x) { return pm::atanf_(x); }
DEVN float m_atan2(float y, float x) { return pm::atan2f_(y, x); }
DEVN float m_cosh(float x) { return pm::coshf_(x); }
DEVN float m_atanh(float x) { return pm::atanhf_(x); }
DEVN float m_sinh(float x) { return pm::sinhf_(x); }
DEVN float m_tanh(float x) { return pm::tanhf_(x); }
#else
// Product build: the special-function unit.  sin / cos / exp2 / log2 are single MUFU instructions (2^-21 absolute error on the reduced
// range); the library routines they replace are 40-150 instructions each and were inlined at ~100 sites of the BSDF code, which made the
// bounce and gather kernels instruction-fetch bound (profiles/r1b_c3_k_camera_merge_generic_batched.raw.csv: 31 no_instruction stalls per
// issue).  The estimators stay the reference's; only roundings move, and the product build is held to the statistical parity tests.
DEV float m_wrap_pi(float x) { return x - kDoublePi * rintf(x * (1.0f / kDoublePi)); }  // [-pi, pi]: where sin.approx / cos.approx are accurate
DEV float m_sin(float x) { return __sinf(m_wrap_pi(x)); }
DEV float m_cos(float x) { return __cosf(m_wrap_pi(x)); }
DEV float m_exp(float x) { return __expf(x); }
DEV float m_log(float x) { return __logf(x); }
DEV float m_pow(float x, float y) {
  // exp2(y * log2(x)) for x >= 0; pow(x, 0) = 1 and pow(0, y > 0) = 0 like powf (0 * -inf would be NaN)
  return (y == 0.0f) ? 1.0f : ((x <= 0.0f) ? ((y > 0.0f) ? 0.0f : kMaxFloat) : exp2f(y * __log2f(x)));
}
DEVG_MATH float m_acos(float x) { return acosf(x); }
DEVG_MATH float m_asin(float x) { return asinf(x); }
DEVG_MATH float m_atan(float x) { return atanf(x); }
DEVG_MATH float m_atan2(float y, float x) { return atan2f(y, x); }
DEV float m_cosh(float x) { float e = __expf(x); return 0.5f * (e + __fdividef(1.0f, e)); }
DEVG_MATH float m_atanh(float x) { return atanhf(x); }
DEV float m_sinh(float x) { float e = __expf(x); return 0.5f * (e - __fdividef(1.0f, e)); }
DEV float m_tanh(float x) { float e = __expf(2.0f * fminf(fmaxf(x, -40.0f), 40.0f)); return __fdividef(e - 1.0f, e + 1.0f); }
#endif

DEV float sqr(float t) { return t * t; }
DEV float saturatef(float v) { return v < 0.0f ? 0.0f : (v > 1.0f ? 1.0f : v); }  // clamp(val,0,1): (val<min)?min:(val>max?max:val)
DEV float lerpf(float a, float b, float t) { return a * (1.0f - t) + b * t; }       // math.hxx:691
DEV float tmin(float a, float b) { return a < b ? a : b; }                          // etx::min template (math.hxx:117)
DEV float tmax(float a, float b) { return a > b ? a : b; }                          // etx::max template (math.hxx:122)
DEV uint32_t umin(uint32_t a, uint32_t b) { return a < b ? a : b; }
DEV bool finitef(float v) { return (__float_as_uint(v) & 0x7f800000u) != 0x7f800000u; }
DEV bool valid_value(float t) { return (t >= 0.0f) && finitef(t); }  // math.hxx:841

// ---- float2 / float3 with the reference's per-component semantics --------------------------------------
struct V2 {
  float x, y;
};
struct V3 {
  float x, y, z;
};
DEV V3 v3(float x, float y, float z) { return V3{x, y, z}; }
DEV V3 v3(float a) { return V3{a, a, a}; }
DEV V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
DEV V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
DEV V3 operator*(V3 a, V3 b) { return {a.x * b.x, a.y * b.y, a.z * b.z}; }
DEV V3 operator/(V3 a, V3 b) { return {a.x / b.x, a.y / b.y, a.z / b.z}; }
DEV V3 operator*(V3 a, float b) { return {a.x * b, a.y * b, a.z * b}; }
DEV V3 operator*(float b, V3 a) { return {a.x * b, a.y * b, a.z * b}; }
DEV V3 operator/(V3 a, float b) { return {a.x / b, a.y / b, a.z / b}; }
DEV V3 operator/(float b, V3 a) { return {b / a.x, b / a.y, b / a.z}; }
DEV V3 operator+(V3 a, float b) { return {a.x + b, a.y + b, a.z + b}; }
DEV V3 operator-(V3 a, float b) { return {a.x - b, a.y - b, a.z - b}; }
DEV V3 operator-(float b, V3 a) { return {b - a.x, b - a.y, b - a.z}; }
DEV V3 operator-(V3 a) { return {-a.x, -a.y, -a.z}; }
DEV V3& operator+=(V3& a, V3 b) { a.x += b.x; a.y += b.y; a.z += b.z; return a; }
DEV V3& operator*=(V3& a, V3 b) { a.x *= b.x; a.y *= b.y; a.z *= b.z; return a; }
DEV V3& operator*=(V3& a, float b) { a.x *= b; a.y *= b; a.z *= b; return a; }
DEV V3& operator/=(V3& a, float b) { a.x /= b; a.y /= b; a.z /= b; return a; }
DEV V2 operator*(V2 a, float b) { return {a.x * b, a.y * b}; }
DEV V2 operator+(V2 a, V2 b) { return {a.x + b.x, a.y + b.y}; }
DEV V2 operator+(V2 a, float b) { return {a.x + b, a.y + b}; }
DEV V2 operator-(V2 a, float b) { return {a.x - b, a.y - b}; }

DEV float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }  // math.hxx:515
DEV float length(V3 v) { return sqrtf(dot(v, v)); }
DEV V3 normalize(V3 v) { return v / length(v); }
DEV V3 cross(V3 a, V3 b) { return {a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y}; }  // math.hxx:540
DEV V3 reflect(V3 v, V3 n) { return v - (2.0f * dot(v, n)) * n; }
DEV V3 lerp3(V3 a, V3 b, float t) {  // math.hxx:556
  float inv_t = 1.0f - t;
  return {a.x * inv_t + b.x * t, a.y * inv_t + b.y * t, a.z * inv_t + b.z * t};
}
DEV V3 vmin(V3 a, V3 b) { return {fminf(a.x, b.x), fminf(a.y, b.y), fminf(a.z, b.z)}; }
DEV V3 vmax(V3 a, V3 b) { return {fmaxf(a.x, b.x), fmaxf(a.y, b.y), fmaxf(a.z, b.z)}; }
DEV V3 vmaxs(V3 a, float b) { return {fmaxf(a.x, b), fmaxf(a.y, b), fmaxf(a.z, b)}; }
DEV V3 vfloor(V3 a) { return {floorf(a.x), floorf(a.y), floorf(a.z)}; }
DEV float luminance(V3 v) { return v.x * 0.212671f + v.y * 0.715160f + v.z * 0.072169f; }
DEV bool valid_value3(V3 v) { return valid_value(v.x) && valid_value(v.y) && valid_value(v.z); }

// math.hxx:737-746
struct Basis {
  V3 u, v;
};
DEV Basis orthonormal_basis(V3 n) {
  V3 a = normalize(((n.x != n.y) || (n.x != n.z)) ? V3{n.z - n.y, n.x - n.z, +n.y - n.x} : V3{n.z - n.y, n.x + n.z, -n.y - n.x});
  V3 b = normalize(cross(n, a));
  return {a, b};
}

// math.hxx:748-762
DEV V3 sample_cosine_local(V2 rnd, float exponent) {
  float cos_theta = m_pow(fmaxf(rnd.x, kEpsilon), 1.0f / (exponent + 1.0f));
  float sin_theta = sqrtf(1.0f - cos_theta * cos_theta);
  return {m_cos(rnd.y * kDoublePi) * sin_theta, m_sin(rnd.y * kDoublePi) * sin_theta, cos_theta};
}
DEV V3 sample_cosine_frame(V2 rnd, V3 n, V3 u, V3 v, float exponent) {
  V3 l = sample_cosine_local(rnd, exponent);
  return u * l.x + v * l.y + n * l.z;
}
DEV V3 sample_cosine_around(V2 rnd, V3 n, float exponent) {
  Basis b = orthonormal_basis(n);
  return sample_cosine_frame(rnd, n, b.u, b.v, exponent);
}
DEV V3 barycentrics_uv(float u, float v) { return {1.0f - u - v, u, v}; }  // math.hxx:764
DEV V3 random_barycentric(V2 rnd) {                                         // math.hxx:768
  float r1 = sqrtf(rnd.x);
  return {1.0f - r1, r1 * (1.0f - rnd.y), r1 * rnd.y};
}
DEV V2 sample_disk(V2 rnd) {  // math.hxx:773-789
  V2 offset = {2.0f * rnd.x - 1.0f, 2.0f * rnd.y - 1.0f};
  if ((offset.x == 0.0f) && (offset.y == 0.0f)) return {0.0f, 0.0f};
  float r, theta;
  if (fabsf(offset.x) > fabsf(offset.y)) {
    r = offset.x;
    theta = kQuarterPi * (offset.y / offset.x);
  } else {
    r = offset.y;
    theta = kHalfPi - kQuarterPi * (offset.x / offset.y);
  }
  return {r * m_cos(theta), r * m_sin(theta)};
}

// math.hxx:925-943 — integer-ULP ray origin nudging
DEV V3 offset_ray(V3 p, V3 n) {
  constexpr float int_scale = 256.0f;
  constexpr float float_scale = 1.0f / 65536.0f;
  constexpr float origin = 1.0f / 32.0f;
  int32_t of_i_x = static_cast<int32_t>(int_scale * n.x);
  int32_t of_i_y = static_cast<int32_t>(int_scale * n.y);
  int32_t of_i_z = static_cast<int32_t>(int_scale * n.z);
  float p_i_x = __int_as_float(__float_as_int(p.x) + ((p.x > 0.0f) ? of_i_x : -of_i_x));
  float p_i_y = __int_as_float(__float_as_int(p.y) + ((p.y > 0.0f) ? of_i_y : -of_i_y));
  float p_i_z = __int_as_float(__float_as_int(p.z) + ((p.z > 0.0f) ? of_i_z : -of_i_z));
  return {
    fabsf(p.x) < origin ? p.x + float_scale * n.x : p_i_x,
    fabsf(p.y) < origin ? p.y + float_scale * n.y : p_i_y,
    fabsf(p.z) < origin ? p.z + float_scale * n.z : p_i_z,
  };
}

// ---- sampler (sampler.hxx:7-78): TEA-16 seed, Wang-hash stream, three "fixed" slots -------------------
struct Smp {
  uint32_t seed;
  float fixed_u, fixed_v, fixed_w;

  DEV static uint32_t random_seed(uint32_t val0, uint32_t val1) {
    uint32_t v0 = val0, v1 = val1, s0 = 0u;
#pragma unroll
    for (uint32_t n = 0u; n < 16u; ++n) {
      s0 += 0x9e3779b9u;
      v0 += ((v1 << 4u) + 0xa341316cu) ^ (v1 + s0) ^ ((v1 >> 5u) + 0xc8013ea4u);
      v1 += ((v0 << 4u) + 0xad90777du) ^ (v0 + s0) ^ ((v0 >> 5u) + 0x7e95761eu);
    }
    return v0;
  }
  DEV void init(uint32_t a, uint32_t b) {
    seed = random_seed(a, b);
    fixed_u = fixed_v = fixed_w = 0.0f;
  }
  DEV float next() {
    seed = (seed ^ 61u) ^ (seed >> 16u);
    seed *= 9u;
    seed = seed ^ (seed >> 4u);
    seed *= 0x27d4eb2du;
    seed = seed ^ (seed >> 15u);
    return __uint_as_float((seed >> 9) | 0x3f800000u) - 1.0f;
  }
  DEV V2 next_2d() {
    float a = next();
    float b = next();
    return {a, b};
  }
  DEV void push_fixed(float u, float v, float w) {
    fixed_u = u;
    fixed_v = v;
    fixed_w = w;
  }
  DEV void pop_fixed() { fixed_u = fixed_v = fixed_w = 0.0f; }
  DEV bool has_fixed() const { return (sqr(fixed_u) + sqr(fixed_v) + sqr(fixed_w)) > kEpsilon; }
};

// ---- spectral value: one float in spectral mode, three in RGB mode (spectrum.hxx:242-374) --------------
// SpectralResponse keeps {value, integrated}; only `value` is observable in spectral mode and only
// `integrated` in RGB mode, so the device type stores exactly the observable part.
template <bool SP>
struct Spec;

template <>
struct Spec<true> {
  float v;
  DEV static Spec make(float a) { return {a}; }
  DEV static Spec make3(V3 c) { return {c.x}; }
  DEV float maximum() const { return v; }
  DEV float minimum() const { return v; }
  DEV float monochromatic() const { return v; }
  DEV float average() const { return v; }
  DEV float sum() const { return v; }
  DEV float component(uint32_t) const { return v; }
  DEV bool is_zero() const { return v <= kEpsilon; }
  DEV bool valid() const { return valid_value(v); }
  DEV V3 as_v3() const { return {v, v, v}; }
};
template <>
struct Spec<false> {
  float x, y, z;
  DEV static Spec make(float a) { return {a, a, a}; }
  DEV static Spec make3(V3 c) { return {c.x, c.y, c.z}; }
  DEV float maximum() const { return tmax(x, tmax(y, z)); }
  DEV float minimum() const { return tmin(x, tmin(y, z)); }
  DEV float monochromatic() const { return luminance({x, y, z}); }
  DEV float average() const { return (x + y + z) / 3.0f; }
  DEV float sum() const { return x + y + z; }
  DEV float component(uint32_t i) const { return i == 0 ? x : (i == 1 ? y : z); }
  DEV bool is_zero() const { return (x <= kEpsilon) && (y <= kEpsilon) && (z <= kEpsilon); }
  DEV bool valid() const { return valid_value(x) && valid_value(y) && valid_value(z); }
  DEV V3 as_v3() const { return {x, y, z}; }
};

#define SPEC_BIN(OP)                                                                                        \
  DEV Spec<true> operator OP(Spec<true> a, Spec<true> b) { return {a.v OP b.v}; }                           \
  DEV Spec<false> operator OP(Spec<false> a, Spec<false> b) { return {a.x OP b.x, a.y OP b.y, a.z OP b.z}; } \
  DEV Spec<true> operator OP(Spec<true> a, float b) { return {a.v OP b}; }                                  \
  DEV Spec<false> operator OP(Spec<false> a, float b) { return {a.x OP b, a.y OP b, a.z OP b}; }
SPEC_BIN(+)
SPEC_BIN(-)
SPEC_BIN(*)
SPEC_BIN(/)
#undef SPEC_BIN
DEV Spec<true> operator*(float b, Spec<true> a) { return {a.v * b}; }
DEV Spec<false> operator*(float b, Spec<false> a) { return {a.x * b, a.y * b, a.z * b}; }
DEV Spec<true> operator/(float b, Spec<true> a) { return {b / a.v}; }
DEV Spec<false> operator/(float b, Spec<false> a) { return {b / a.x, b / a.y, b / a.z}; }
DEV Spec<true> operator-(float b, Spec<true> a) { return {b - a.v}; }
DEV Spec<false> operator-(float b, Spec<false> a) { return {b - a.x, b - a.y, b - a.z}; }
template <bool SP>
DEV Spec<SP>& operator*=(Spec<SP>& a, Spec<SP> b) { a = a * b; return a; }
template <bool SP>
DEV Spec<SP>& operator*=(Spec<SP>& a, float b) { a = a * b; return a; }
template <bool SP>
DEV Spec<SP>& operator+=(Spec<SP>& a, Spec<SP> b) { a = a + b; return a; }
DEV Spec<true> operator-(Spec<true> a) { return {-a.v}; }
DEV Spec<false> operator-(Spec<false> a) { return {-a.x, -a.y, -a.z}; }
DEV Spec<true> spec_exp(Spec<true> a) { return {m_exp(a.v)}; }
DEV Spec<false> spec_exp(Spec<false> a) { return {m_exp(a.x), m_exp(a.y), m_exp(a.z)}; }
DEV Spec<true> spec_saturate(Spec<true> a) { return {saturatef(a.v)}; }
DEV Spec<false> spec_saturate(Spec<false> a) { return {saturatef(a.x), saturatef(a.y), saturatef(a.z)}; }

// spectrum.hxx:219-239
DEV float spectral_sampling_pdf(float wavelength) { return 0.0039398042f / sqr(m_cosh(0.0072f * (wavelength - 538.0f))); }
DEV float spectral_sample_wavelength(float rnd) {
  constexpr float offset = 0x1.35ce7a0000000p-5f;
  constexpr float scale = 1.0f - offset;
  return 538.0f - 138.888889f * m_atanh(0.85691062f - 1.82750197f * (rnd * scale + offset));
}
template <bool SP>
DEV float sampling_pdf(float wavelength) {
  if constexpr (SP) return spectral_sampling_pdf(wavelength);
  return 1.0f;
}

// spectrum.hxx:142-148
DEV V3 xyz_to_rgb(V3 xyz) {
  return {
    3.24045420f * xyz.x - 1.5371385f * xyz.y - 0.4985314f * xyz.z,
    -0.9692660f * xyz.x + 1.8760108f * xyz.y + 0.0415560f * xyz.z,
    0.05564340f * xyz.x - 0.2040259f * xyz.y + 1.0572252f * xyz.z,
  };
}
DEV V3 rgb_to_xyz(V3 rgb) {
  return {
    0.4124564f * rgb.x + 0.3575760f * rgb.y + 0.1804375f * rgb.z,
    0.2126729f * rgb.x + 0.7151521f * rgb.y + 0.0721750f * rgb.z,
    0.0193339f * rgb.x + 0.1191920f * rgb.y + 0.9503041f * rgb.z,
  };
}

// ---- complex<float> with libstdc++ / libgcc semantics (bsdf.hxx fresnel uses std::complex) -----------
struct Cx {
  float re, im;
};
DEV Cx cx(float re, float im = 0.0f) { return {re, im}; }
DEV Cx operator+(Cx a, Cx b) { return {a.re + b.re, a.im + b.im}; }
DEV Cx operator-(Cx a, Cx b) { return {a.re - b.re, a.im - b.im}; }
DEV Cx operator*(Cx a, Cx b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
DEV Cx operator*(Cx a, float b) { return {a.re * b, a.im * b}; }
DEV Cx operator*(float b, Cx a) { return {a.re * b, a.im * b}; }
DEV Cx operator/(Cx a, float b) { return {a.re / b, a.im / b}; }
DEV Cx operator-(float x, Cx a) { return {-a.re + x, -a.im}; }  // libstdc++: r = -y; r += x
DEV Cx operator+(float x, Cx a) { return {a.re + x, a.im}; }
DEV Cx operator/(Cx a, Cx b) {
#if defined(ETXB_PARITY) && ETXB_PARITY
  Cx r;
  pm::cdivf_(a.re, a.im, b.re, b.im, r.re, r.im);
  return r;
#else
  float denom = b.re * b.re + b.im * b.im;
  return {(a.re * b.re + a.im * b.im) / denom, (a.im * b.re - a.re * b.im) / denom};
#endif
}
DEV bool operator==(Cx a, Cx b) { return (a.re == b.re) && (a.im == b.im); }
DEV Cx cx_conj(Cx a) { return {a.re, -a.im}; }
DEV float cx_norm(Cx a) { return a.re * a.re + a.im * a.im; }
DEV Cx cx_sqrt(Cx a) {
  Cx r;
#if defined(ETXB_PARITY) && ETXB_PARITY
  pm::csqrtf_(a.re, a.im, r.re, r.im);
#else
  if (a.re == 0.0f && a.im == 0.0f) return {0.0f, a.im};
  float h = sqrtf(a.re * a.re + a.im * a.im);
  float t = sqrtf(0.5f * (fabsf(a.re) + h));
  if (a.re >= 0.0f) {
    r = {t, a.im / (2.0f * t)};
  } else {
    r = {fabsf(a.im) / (2.0f * t), copysignf(t, a.im)};
  }
#endif
  return r;
}
DEV Cx cx_exp(Cx a) {
  Cx r;
#if defined(ETXB_PARITY) && ETXB_PARITY
  pm::cexpf_(a.re, a.im, r.re, r.im);
#else
  float e = expf(a.re);
  float s, c;
  sincosf(a.im, &s, &c);
  r = {e * c, e * s};
#endif
  return r;
}
DEV float cx_abs(Cx a) {
#if defined(ETXB_PARITY) && ETXB_PARITY
  return pm::cabsf_(a.re, a.im);
#else
  return sqrtf(a.re * a.re + a.im * a.im);
#endif
}

}  // namespace etxb
