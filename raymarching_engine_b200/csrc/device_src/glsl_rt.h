// glsl_rt.h -- GLSL ES 3.00 vector/matrix types and built-in functions as C++, for
//   (1) scene code lowered from GLSL and compiled by NVRTC for sm_100a, and
//   (2) the host parity oracle (g++), which must evaluate bit-identical arithmetic.
//
// MULTI-INCLUDE HEADER.  Each inclusion defines one namespace:
//     #define GLSL_NS   xg        // namespace to create
//     #define GLSL_FAST 0         // 0 = "exact" policy, 1 = "fast" policy
//     #include "glsl_rt.h"
// exact policy: every float add/sub/mul/div/sqrt is a single correctly rounded IEEE-754
//   operation that the compiler may not contract into an FMA (device: __fmul_rn & co, which
//   ptxas never fuses; host: plain operators under -ffp-contract=off), transcendental
//   functions come from rm_math.h.  Device and host results are bit-identical.
// fast policy: plain operators (FMA contraction allowed) and CUDA fast intrinsics; device only.
//
// Default constructors are empty (values undefined, as in GLSL) so that the types can be
// __constant__ uniforms.
//
// Pinned choices for behaviour GLSL ES 3.00 leaves implementation-defined (SURVEY.md 8c):
//   dot(a,b) = fma(a.z,b.z, fma(a.y,b.y, a.x*b.x)) - the contraction GLSL permits (ES 3.00 4.5.2)
//     and GPU compilers perform; length(v) = sqrt(dot(v,v)) unscaled;
//   vector / scalar = vector * (1/scalar) with a correctly rounded reciprocal (within the 2.5 ULP
//     GLSL allows for division; GPU drivers lower division to reciprocal-multiply as well);
//     scalar / scalar and vector / vector are IEEE divisions;
//   mod(x,y) = fma(-y, floor(x * (1/y)), x);  mix(a,b,t) = fma(b, t, a*(1-t));
//   normalize(v) = v / length(v) (one reciprocal, three multiplies);
//   min/max drop NaN operands (IEEE minNum/maxNum, -0 < +0) like CUDA fminf/fmaxf;
//   round() rounds half away from zero;  mat*vec sums column contributions left to right;
//   every other a*b+c stays unfused (two roundings).
//
// Reference: the built-ins used by client/public/shader/raymarcher.frag and
// client/public/examples/*.glsl of radian628/raymarching-engine.
#include "rm_math.h"
#include "glsl_swizzle.inc"

#ifndef GLSL_NS
#error "define GLSL_NS before including glsl_rt.h"
#endif
#ifndef GLSL_FAST
#error "define GLSL_FAST (0 or 1) before including glsl_rt.h"
#endif

namespace GLSL_NS {

typedef unsigned int uint;

// ------------------------------------------------------------------ scalar op policy
#if GLSL_FAST
RM_HD float g_add(float a, float b) { return a + b; }
RM_HD float g_sub(float a, float b) { return a - b; }
RM_HD float g_mul(float a, float b) { return a * b; }
RM_HD float g_div(float a, float b) { return __fdividef(a, b); }
// single MUFU.SQRT / MUFU.RSQ (flush-to-zero forms: no denormal scaling code around them)
RM_HD float g_sqrt(float a) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a)); return r; }
RM_HD float g_rsqrt(float a) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a)); return r; }
// floor on the FP32 pipe: FRND issues on the 16-lane XU pipe and was the top stall of the exact
// flavour (profiles/r1_preview_exact_ncu_full.txt).  (a + 1.5*2^23) - 1.5*2^23 rounds to the nearest
// integer for |a| <= 2^22; one compare-and-subtract turns that into floor.  Larger |a| take FRND.
RM_HD float g_floor(float a) {
    const float M = 12582912.0f;
    const float t = __fadd_rn(__fadd_rn(a, M), -M);
    const float r = t > a ? __fadd_rn(t, -1.0f) : t;
    return fabsf(a) <= 4194304.0f ? r : floorf(a);
}
RM_HD float g_fma(float a, float b, float c) { return fmaf(a, b, c); }
// plain division (the fast flavour compiles with --prec-div=false): folds when the divisor is a
// compile-time constant, otherwise an approximate reciprocal
RM_HD float g_rcp(float a) { return 1.0f / a; }
#elif RM_DEVICE_CODE
RM_HD float g_add(float a, float b) { return __fadd_rn(a, b); }
RM_HD float g_sub(float a, float b) { return __fsub_rn(a, b); }
RM_HD float g_mul(float a, float b) { return __fmul_rn(a, b); }
RM_HD float g_div(float a, float b) { return __fdiv_rn(a, b); }
RM_HD float g_sqrt(float a) { return __fsqrt_rn(a); }
RM_HD float g_rsqrt(float a) { return __fdiv_rn(1.0f, __fsqrt_rn(a)); }
RM_HD float g_floor(float a) { return floorf(a); }
RM_HD float g_fma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
#if defined(RM_FLAVOUR_FAST) && RM_FLAVOUR_FAST
// inside a fast-flavour program (--prec-div=false) the exact namespace must not depend on flags
RM_HD float g_rcp(float a) { return __fdiv_rn(1.0f, a); }
#else
// written as a plain IEEE division (--prec-div=true) so that a constant divisor folds at compile time
RM_HD float g_rcp(float a) { return 1.0f / a; }
#endif
#else
RM_HD float g_add(float a, float b) { return a + b; }
RM_HD float g_sub(float a, float b) { return a - b; }
RM_HD float g_mul(float a, float b) { return a * b; }
RM_HD float g_div(float a, float b) { return a / b; }
RM_HD float g_sqrt(float a) { return __builtin_sqrtf(a); }
RM_HD float g_rsqrt(float a) { return 1.0f / __builtin_sqrtf(a); }
RM_HD float g_floor(float a) { return __builtin_floorf(a); }
RM_HD float g_fma(float a, float b, float c) { return __builtin_fmaf(a, b, c); }
RM_HD float g_rcp(float a) { return 1.0f / a; }
#endif

#if RM_DEVICE_CODE
// Blackwell packed FP32 (FFMA2 / FADD2 / FMUL2: two IEEE round-to-nearest operations per lane per issue
// slot, bit-identical to the scalar instructions).  The march loops are issue-bound, so the x and y
// components of the hot vector operations travel as one f32x2 value; z stays scalar.
#define GLSL_F32X2 1
// the CUDA 12.9 sm_100 builtins behind __ffma2_rn & co (crt/sm_100_rt.hpp), declared here because NVRTC
// sees no CUDA headers; unlike inline PTX the compiler understands them (broadcast / immediate operands)
extern "C" {      // (re-declared in every namespace this header creates; same C-linkage entities)
__device__ __device_builtin__ float2 __ffma2_rn_impl(float2 x, float2 y, float2 z);
__device__ __device_builtin__ float2 __fadd2_rn_impl(float2 x, float2 y);
__device__ __device_builtin__ float2 __fmul2_rn_impl(float2 x, float2 y);
__device__ __device_builtin__ float2 __fadd2_rd_impl(float2 x, float2 y);
}
typedef float2 f2_t;
RM_HD f2_t f2_pack(float a, float b) { return make_float2(a, b); }
RM_HD void f2_unpack(f2_t v, float& a, float& b) { a = v.x; b = v.y; }
RM_HD f2_t f2_fma(f2_t a, f2_t b, f2_t c) { return __ffma2_rn_impl(a, b, c); }
RM_HD f2_t f2_add(f2_t a, f2_t b) { return __fadd2_rn_impl(a, b); }
RM_HD f2_t f2_sub(f2_t a, f2_t b) { return __fadd2_rn_impl(a, make_float2(-b.x, -b.y)); }   // a + (-b) == a - b bit for bit
RM_HD f2_t f2_mul(f2_t a, f2_t b) { return __fmul2_rn_impl(a, b); }
RM_HD f2_t f2_add_rd(f2_t a, f2_t b) { return __fadd2_rd_impl(a, b); }                      // FADD2.RM: round towards -inf
#else
#define GLSL_F32X2 0
#endif

#if RM_DEVICE_CODE
RM_HD float g_min(float a, float b) { return fminf(a, b); }
RM_HD float g_max(float a, float b) { return fmaxf(a, b); }
RM_HD float g_abs(float a) { return fabsf(a); }
RM_HD float g_trunc(float a) { return truncf(a); }
RM_HD float g_ceil(float a) { return ceilf(a); }
RM_HD float g_rint(float a) { return rintf(a); }
#else
// PTX min/max.f32 semantics: a NaN operand is dropped, -0.0 orders below +0.0.
RM_HD float g_min(float a, float b) {
    if (rmx::f_isnan(a)) return b;
    if (rmx::f_isnan(b)) return a;
    if (a == b) return (rmx::f2i(a) < 0) ? a : b;
    return a < b ? a : b;
}
RM_HD float g_max(float a, float b) {
    if (rmx::f_isnan(a)) return b;
    if (rmx::f_isnan(b)) return a;
    if (a == b) return (rmx::f2i(a) < 0) ? b : a;
    return a > b ? a : b;
}
RM_HD float g_abs(float a) { return __builtin_fabsf(a); }
RM_HD float g_trunc(float a) { return __builtin_truncf(a); }
RM_HD float g_ceil(float a) { return __builtin_ceilf(a); }
RM_HD float g_rint(float a) { return __builtin_rintf(a); }
#endif

// ------------------------------------------------------------------ scalar built-ins
RM_HD float radians(float d) { return g_mul(d, 0.0174532925199432957692f); }
RM_HD float degrees(float r) { return g_mul(r, 57.2957795130823208768f); }
#if GLSL_FAST
RM_HD float sin(float x) { return __sinf(x); }
RM_HD float cos(float x) { return __cosf(x); }
RM_HD float tan(float x) { return __tanf(x); }
RM_HD float pow(float x, float y) { return __powf(x, y); }
RM_HD float exp(float x) { return __expf(x); }
RM_HD float log(float x) { return __logf(x); }
RM_HD float exp2(float x) { return exp2f(x); }
RM_HD float log2(float x) { return __log2f(x); }
// inverse trigonometry on the FP32 pipe (CUDA's single-precision routines: documented maximum error 2 ulp for
// asinf / acosf / atan2f, 1 ulp for atanf) instead of the exact flavour's binary64 evaluation: the Mandelbulb DE of
// BASELINE.json config 4 calls acos + atan once per iteration and was fp64-pipe bound in BOTH flavours
RM_HD float asin(float x) { return asinf(x); }
RM_HD float acos(float x) { return acosf(x); }
RM_HD float atan(float x) { return atanf(x); }
RM_HD float atan(float y, float x) { return atan2f(y, x); }
#else
RM_HD float sin(float x) { return rmx::sin_f(x); }
RM_HD float cos(float x) { return rmx::cos_f(x); }
RM_HD float tan(float x) { return rmx::tan_f(x); }
RM_HD float pow(float x, float y) { return rmx::pow_f(x, y); }
RM_HD float exp(float x) { return rmx::exp_f(x); }
RM_HD float log(float x) { return rmx::log_f(x); }
RM_HD float exp2(float x) { return rmx::exp2_f(x); }
RM_HD float log2(float x) { return rmx::log2_f(x); }
RM_HD float asin(float x) { return rmx::asin_f(x); }
RM_HD float acos(float x) { return rmx::acos_f(x); }
RM_HD float atan(float x) { return rmx::atan_f(x); }
RM_HD float atan(float y, float x) { return rmx::atan2_f(y, x); }
#endif
RM_HD float sinh(float x) { return rmx::sinh_f(x); }
RM_HD float cosh(float x) { return rmx::cosh_f(x); }
RM_HD float tanh(float x) { return rmx::tanh_f(x); }
RM_HD float asinh(float x) { return rmx::asinh_f(x); }
RM_HD float acosh(float x) { return rmx::acosh_f(x); }
RM_HD float atanh(float x) { return rmx::atanh_f(x); }
RM_HD float sqrt(float x) { return g_sqrt(x); }
RM_HD float inversesqrt(float x) { return g_rsqrt(x); }
RM_HD float abs(float x) { return g_abs(x); }
RM_HD float sign(float x) { return x > 0.0f ? 1.0f : (x < 0.0f ? -1.0f : 0.0f); }
RM_HD float floor(float x) { return g_floor(x); }
RM_HD float trunc(float x) { return g_trunc(x); }
RM_HD float ceil(float x) { return g_ceil(x); }
RM_HD float roundEven(float x) { return g_rint(x); }
RM_HD float round(float x) {
    float t = g_trunc(x);
    float d = g_abs(g_sub(x, t));
    if (d >= 0.5f) t = g_add(t, x < 0.0f ? -1.0f : 1.0f);
    return t;
}
RM_HD float fract(float x) { return g_sub(x, g_floor(x)); }
#if !GLSL_FAST && defined(RM_PIN_ALT) && RM_PIN_ALT
// second conforming implementation (RMB_FLAVOUR_EXACT_ALT, measurement aid): GLSL ES 3.00 8.3 as written
RM_HD float mod(float x, float y) { return g_sub(x, g_mul(y, g_floor(g_div(x, y)))); }
#else
RM_HD float mod(float x, float y) { return g_fma(-y, g_floor(g_mul(x, g_rcp(y))), x); }
#endif
// Domain repetition idiom `mod(x + h1, s) - h2` (and `mod(x, s) - h2`): the lowering
// (lower_glsl.cpp) hands the four operands to rm_rep / rm_rep0.  Exact policy: the expression as
// written.  Fast policy: when h2 == s/2 (a centred cell, the canonical opRep form) it is the centred
// remainder y - s*rint(y/s) of y = x + (h1 - h2): FFMA (y*(1/s) + 1.5*2^23), FADD, FFMA per component,
// no floor at all; operands that are compile-time constants in a baked program fold the test away.
#if GLSL_FAST
RM_HD float rm_rep1(float x, float h1, float s, float h2) {
    if (h2 == 0.5f * s && s > 0.0f && s < 1e30f) {
        const float M = 12582912.0f;
        const float y = (h1 == h2) ? x : x + (h1 - h2);
        const float r = __fadd_rn(__fmaf_rn(y, 1.0f / s, M), -M);
        return __fmaf_rn(-s, r, y);
    }
    return mod(x + h1, s) - h2;
}
#else
RM_HD float rm_rep1(float x, float h1, float s, float h2) { return g_sub(mod(g_add(x, h1), s), h2); }
#endif
RM_HD float rm_rep(float x, float h1, float s, float h2) { return rm_rep1(x, h1, s, h2); }
#if GLSL_FAST
RM_HD float rm_rep0(float x, float s, float h2) { return rm_rep1(x, 0.0f, s, h2); }
#else
RM_HD float rm_rep0(float x, float s, float h2) { return g_sub(mod(x, s), h2); }
#endif
RM_HD float min(float a, float b) { return g_min(a, b); }
RM_HD float max(float a, float b) { return g_max(a, b); }
RM_HD float clamp(float x, float lo, float hi) { return g_min(g_max(x, lo), hi); }
RM_HD float mix(float a, float b, float t) { return g_fma(b, t, g_mul(a, g_sub(1.0f, t))); }
RM_HD float mix(float a, float b, bool t) { return t ? b : a; }
RM_HD float step(float edge, float x) { return x < edge ? 0.0f : 1.0f; }
RM_HD float smoothstep(float e0, float e1, float x) {
    float t = clamp(g_div(g_sub(x, e0), g_sub(e1, e0)), 0.0f, 1.0f);
    return g_mul(g_mul(t, t), g_sub(3.0f, g_mul(2.0f, t)));
}
RM_HD bool isnan(float x) { return rmx::f_isnan(x); }
RM_HD bool isinf(float x) { return rmx::f_isinf(x); }
RM_HD int floatBitsToInt(float x) { return rmx::f2i(x); }
RM_HD uint floatBitsToUint(float x) { return (uint)rmx::f2i(x); }
RM_HD float intBitsToFloat(int x) { return rmx::i2f(x); }
RM_HD float uintBitsToFloat(uint x) { return rmx::i2f((int)x); }
RM_HD float length(float x) { return g_abs(x); }
RM_HD float distance(float a, float b) { return g_abs(g_sub(a, b)); }
RM_HD float dot(float a, float b) { return g_mul(a, b); }
RM_HD float normalize(float x) { return sign(x); }

RM_HD int abs(int x) { return x < 0 ? -x : x; }
RM_HD int sign(int x) { return x > 0 ? 1 : (x < 0 ? -1 : 0); }
RM_HD int min(int a, int b) { return a < b ? a : b; }
RM_HD int max(int a, int b) { return a > b ? a : b; }
RM_HD int clamp(int x, int lo, int hi) { return min(max(x, lo), hi); }
RM_HD uint min(uint a, uint b) { return a < b ? a : b; }
RM_HD uint max(uint a, uint b) { return a > b ? a : b; }
RM_HD uint clamp(uint x, uint lo, uint hi) { return min(max(x, lo), hi); }

// ------------------------------------------------------------------ vector types
struct vec2; struct vec3; struct vec4;
struct ivec2; struct ivec3; struct ivec4;
struct bvec2; struct bvec3; struct bvec4;
struct mat2; struct mat3; struct mat4;

// Swizzle proxies: views over the N floats of the owning vector.  They convert to the
// value type and support assignment, so `p.xy *= m;` and `c.rgb = v;` work as in GLSL.
template <int N, int A, int B> struct Sw2 {
    float v[N];
    RM_HD operator vec2() const;
    RM_HD Sw2& operator=(const vec2& o);
    RM_HD Sw2& operator=(const Sw2& o);
    RM_HD Sw2& operator+=(const vec2& o);
    RM_HD Sw2& operator-=(const vec2& o);
    RM_HD Sw2& operator*=(const vec2& o);
    RM_HD Sw2& operator/=(const vec2& o);
    RM_HD Sw2& operator+=(float o);
    RM_HD Sw2& operator-=(float o);
    RM_HD Sw2& operator*=(float o);
    RM_HD Sw2& operator/=(float o);
    RM_HD Sw2& operator*=(const mat2& m);
};
template <int N, int A, int B, int C> struct Sw3 {
    float v[N];
    RM_HD operator vec3() const;
    RM_HD Sw3& operator=(const vec3& o);
    RM_HD Sw3& operator=(const Sw3& o);
    RM_HD Sw3& operator+=(const vec3& o);
    RM_HD Sw3& operator-=(const vec3& o);
    RM_HD Sw3& operator*=(const vec3& o);
    RM_HD Sw3& operator/=(const vec3& o);
    RM_HD Sw3& operator+=(float o);
    RM_HD Sw3& operator-=(float o);
    RM_HD Sw3& operator*=(float o);
    RM_HD Sw3& operator/=(float o);
    RM_HD Sw3& operator*=(const mat3& m);
};
template <int N, int A, int B, int C, int D> struct Sw4 {
    float v[N];
    RM_HD operator vec4() const;
    RM_HD Sw4& operator=(const vec4& o);
    RM_HD Sw4& operator=(const Sw4& o);
    RM_HD Sw4& operator+=(const vec4& o);
    RM_HD Sw4& operator-=(const vec4& o);
    RM_HD Sw4& operator*=(const vec4& o);
    RM_HD Sw4& operator/=(const vec4& o);
    RM_HD Sw4& operator+=(float o);
    RM_HD Sw4& operator-=(float o);
    RM_HD Sw4& operator*=(float o);
    RM_HD Sw4& operator/=(float o);
    RM_HD Sw4& operator*=(const mat4& m);
};

struct vec2 {
    union {
        struct { float x, y; };
        struct { float r, g; };
        struct { float s, t; };
        GLSL_SWIZZLES_2
    };
    RM_HD vec2() {}
    RM_HD explicit vec2(float a) { x = a; y = a; }
    RM_HD vec2(float a, float b) { x = a; y = b; }
    RM_HD vec2(const vec2& o) { x = o.x; y = o.y; }
    RM_HD explicit vec2(const vec3& o);
    RM_HD explicit vec2(const vec4& o);
    RM_HD explicit vec2(const ivec2& o);
    RM_HD vec2& operator=(const vec2& o) { float a = o.x, b = o.y; x = a; y = b; return *this; }
    RM_HD float& operator[](int i) { return (&x)[i]; }
    RM_HD const float& operator[](int i) const { return (&x)[i]; }
};

struct vec3 {
    union {
        struct { float x, y, z; };
        struct { float r, g, b; };
        struct { float s, t, p; };
        GLSL_SWIZZLES_3
    };
    RM_HD vec3() {}
    RM_HD explicit vec3(float a) { x = a; y = a; z = a; }
    RM_HD vec3(float a, float b, float c) { x = a; y = b; z = c; }
    RM_HD vec3(const vec2& a, float c) { x = a.x; y = a.y; z = c; }
    RM_HD vec3(float a, const vec2& b) { x = a; y = b.x; z = b.y; }
    RM_HD vec3(const vec3& o) { x = o.x; y = o.y; z = o.z; }
    RM_HD explicit vec3(const vec4& o);
    RM_HD explicit vec3(const ivec3& o);
    RM_HD vec3& operator=(const vec3& o) { float a = o.x, b = o.y, c = o.z; x = a; y = b; z = c; return *this; }
    RM_HD float& operator[](int i) { return (&x)[i]; }
    RM_HD const float& operator[](int i) const { return (&x)[i]; }
};

struct vec4 {
    union {
        struct { float x, y, z, w; };
        struct { float r, g, b, a; };
        struct { float s, t, p, q; };
        GLSL_SWIZZLES_4
    };
    RM_HD vec4() {}
    RM_HD explicit vec4(float v) { x = v; y = v; z = v; w = v; }
    RM_HD vec4(float a_, float b_, float c_, float d_) { x = a_; y = b_; z = c_; w = d_; }
    RM_HD vec4(const vec3& v, float d_) { x = v.x; y = v.y; z = v.z; w = d_; }
    RM_HD vec4(float a_, const vec3& v) { x = a_; y = v.x; z = v.y; w = v.z; }
    RM_HD vec4(const vec2& u, const vec2& v) { x = u.x; y = u.y; z = v.x; w = v.y; }
    RM_HD vec4(const vec2& u, float c_, float d_) { x = u.x; y = u.y; z = c_; w = d_; }
    RM_HD vec4(float a_, const vec2& u, float d_) { x = a_; y = u.x; z = u.y; w = d_; }
    RM_HD vec4(float a_, float b_, const vec2& u) { x = a_; y = b_; z = u.x; w = u.y; }
    RM_HD vec4(const vec4& o) { x = o.x; y = o.y; z = o.z; w = o.w; }
    RM_HD explicit vec4(const ivec4& o);
    RM_HD vec4& operator=(const vec4& o) {
        float a_ = o.x, b_ = o.y, c_ = o.z, d_ = o.w; x = a_; y = b_; z = c_; w = d_; return *this;
    }
    RM_HD float& operator[](int i) { return (&x)[i]; }
    RM_HD const float& operator[](int i) const { return (&x)[i]; }
};

RM_HD vec2::vec2(const vec3& o) { x = o.x; y = o.y; }
RM_HD vec2::vec2(const vec4& o) { x = o.x; y = o.y; }
RM_HD vec3::vec3(const vec4& o) { x = o.x; y = o.y; z = o.z; }

// integer and boolean vectors (value types, no swizzle proxies: .x/.y/.z/.w only)
struct ivec2 { int x, y;
    RM_HD ivec2() {} RM_HD explicit ivec2(int a) : x(a), y(a) {} RM_HD ivec2(int a, int b) : x(a), y(b) {}
    RM_HD explicit ivec2(const vec2& v) : x((int)v.x), y((int)v.y) {}
    RM_HD int& operator[](int i) { return (&x)[i]; } RM_HD const int& operator[](int i) const { return (&x)[i]; } };
struct ivec3 { int x, y, z;
    RM_HD ivec3() {} RM_HD explicit ivec3(int a) : x(a), y(a), z(a) {} RM_HD ivec3(int a, int b, int c) : x(a), y(b), z(c) {}
    RM_HD explicit ivec3(const vec3& v) : x((int)v.x), y((int)v.y), z((int)v.z) {}
    RM_HD int& operator[](int i) { return (&x)[i]; } RM_HD const int& operator[](int i) const { return (&x)[i]; } };
struct ivec4 { int x, y, z, w;
    RM_HD ivec4() {} RM_HD explicit ivec4(int a) : x(a), y(a), z(a), w(a) {}
    RM_HD ivec4(int a, int b, int c, int d) : x(a), y(b), z(c), w(d) {}
    RM_HD explicit ivec4(const vec4& v) : x((int)v.x), y((int)v.y), z((int)v.z), w((int)v.w) {}
    RM_HD int& operator[](int i) { return (&x)[i]; } RM_HD const int& operator[](int i) const { return (&x)[i]; } };
struct uvec2 { uint x, y; RM_HD uvec2() {} RM_HD explicit uvec2(uint a) : x(a), y(a) {} RM_HD uvec2(uint a, uint b) : x(a), y(b) {} };
struct uvec3 { uint x, y, z; RM_HD uvec3() {} RM_HD explicit uvec3(uint a) : x(a), y(a), z(a) {} RM_HD uvec3(uint a, uint b, uint c) : x(a), y(b), z(c) {} };
struct uvec4 { uint x, y, z, w; RM_HD uvec4() {} RM_HD explicit uvec4(uint a) : x(a), y(a), z(a), w(a) {} RM_HD uvec4(uint a, uint b, uint c, uint d) : x(a), y(b), z(c), w(d) {} };
struct bvec2 { bool x, y; RM_HD bvec2() {} RM_HD bvec2(bool a, bool b) : x(a), y(b) {} };
struct bvec3 { bool x, y, z; RM_HD bvec3() {} RM_HD bvec3(bool a, bool b, bool c) : x(a), y(b), z(c) {} };
struct bvec4 { bool x, y, z, w; RM_HD bvec4() {} RM_HD bvec4(bool a, bool b, bool c, bool d) : x(a), y(b), z(c), w(d) {} };

RM_HD vec2::vec2(const ivec2& o) { x = (float)o.x; y = (float)o.y; }
RM_HD vec3::vec3(const ivec3& o) { x = (float)o.x; y = (float)o.y; z = (float)o.z; }
RM_HD vec4::vec4(const ivec4& o) { x = (float)o.x; y = (float)o.y; z = (float)o.z; w = (float)o.w; }

RM_HD ivec2 operator+(ivec2 a, ivec2 b) { return ivec2(a.x + b.x, a.y + b.y); }
RM_HD ivec2 operator-(ivec2 a, ivec2 b) { return ivec2(a.x - b.x, a.y - b.y); }
RM_HD ivec2 operator*(ivec2 a, ivec2 b) { return ivec2(a.x * b.x, a.y * b.y); }
RM_HD ivec2 operator*(ivec2 a, int b) { return ivec2(a.x * b, a.y * b); }
RM_HD ivec3 operator+(ivec3 a, ivec3 b) { return ivec3(a.x + b.x, a.y + b.y, a.z + b.z); }
RM_HD ivec3 operator-(ivec3 a, ivec3 b) { return ivec3(a.x - b.x, a.y - b.y, a.z - b.z); }
RM_HD ivec3 operator*(ivec3 a, ivec3 b) { return ivec3(a.x * b.x, a.y * b.y, a.z * b.z); }
RM_HD ivec3 operator*(ivec3 a, int b) { return ivec3(a.x * b, a.y * b, a.z * b); }
RM_HD ivec4 operator+(ivec4 a, ivec4 b) { return ivec4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
RM_HD ivec4 operator-(ivec4 a, ivec4 b) { return ivec4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
RM_HD ivec4 operator*(ivec4 a, int b) { return ivec4(a.x * b, a.y * b, a.z * b, a.w * b); }

RM_HD bool any(bvec2 v) { return v.x || v.y; }
RM_HD bool any(bvec3 v) { return v.x || v.y || v.z; }
RM_HD bool any(bvec4 v) { return v.x || v.y || v.z || v.w; }
RM_HD bool all(bvec2 v) { return v.x && v.y; }
RM_HD bool all(bvec3 v) { return v.x && v.y && v.z; }
RM_HD bool all(bvec4 v) { return v.x && v.y && v.z && v.w; }
// GLSL `not(bvec)` collides with the C++ alternative token; the lowering renames it to not_.
RM_HD bvec2 not_(bvec2 v) { return bvec2(!v.x, !v.y); }
RM_HD bvec3 not_(bvec3 v) { return bvec3(!v.x, !v.y, !v.z); }
RM_HD bvec4 not_(bvec4 v) { return bvec4(!v.x, !v.y, !v.z, !v.w); }

// ------------------------------------------------------------------ component-wise operators
#define GLSL_BINOP(op, fn) GLSL_BINOP2(op, fn, fn)
#define GLSL_BINOP2(op, fn, fns)                                                                    \
    RM_HD vec2 operator op(const vec2& a, const vec2& b) { return vec2(fn(a.x, b.x), fn(a.y, b.y)); } \
    RM_HD vec2 operator op(const vec2& a, float b) { return vec2(fns(a.x, b), fns(a.y, b)); }        \
    RM_HD vec2 operator op(float a, const vec2& b) { return vec2(fn(a, b.x), fn(a, b.y)); }          \
    RM_HD vec3 operator op(const vec3& a, const vec3& b) { return vec3(fn(a.x, b.x), fn(a.y, b.y), fn(a.z, b.z)); } \
    RM_HD vec3 operator op(const vec3& a, float b) { return vec3(fns(a.x, b), fns(a.y, b), fns(a.z, b)); } \
    RM_HD vec3 operator op(float a, const vec3& b) { return vec3(fn(a, b.x), fn(a, b.y), fn(a, b.z)); } \
    RM_HD vec4 operator op(const vec4& a, const vec4& b) { return vec4(fn(a.x, b.x), fn(a.y, b.y), fn(a.z, b.z), fn(a.w, b.w)); } \
    RM_HD vec4 operator op(const vec4& a, float b) { return vec4(fns(a.x, b), fns(a.y, b), fns(a.z, b), fns(a.w, b)); } \
    RM_HD vec4 operator op(float a, const vec4& b) { return vec4(fn(a, b.x), fn(a, b.y), fn(a, b.z), fn(a, b.w)); } \
    RM_HD vec2& operator op##=(vec2& a, const vec2& b) { a = a op b; return a; }                     \
    RM_HD vec2& operator op##=(vec2& a, float b) { a = a op b; return a; }                           \
    RM_HD vec3& operator op##=(vec3& a, const vec3& b) { a = a op b; return a; }                     \
    RM_HD vec3& operator op##=(vec3& a, float b) { a = a op b; return a; }                           \
    RM_HD vec4& operator op##=(vec4& a, const vec4& b) { a = a op b; return a; }                     \
    RM_HD vec4& operator op##=(vec4& a, float b) { a = a op b; return a; }
GLSL_BINOP(+, g_add)
GLSL_BINOP(-, g_sub)
GLSL_BINOP(*, g_mul)
// vector / scalar multiplies by the (correctly rounded) reciprocal of the scalar
RM_HD float g_div_by_scalar(float a, float b) { return g_mul(a, g_rcp(b)); }
GLSL_BINOP2(/, g_div, g_div_by_scalar)
#undef GLSL_BINOP
#undef GLSL_BINOP2
// fused multiply-add of vectors: a*b + c with one rounding per component (used by the pipeline
// for `rayPosition + rayDirection * sdfNow`, which GLSL compilers contract)
RM_HD vec2 fmaV(const vec2& a, float b, const vec2& c) { return vec2(g_fma(a.x, b, c.x), g_fma(a.y, b, c.y)); }
RM_HD vec3 fmaV(const vec3& a, float b, const vec3& c) { return vec3(g_fma(a.x, b, c.x), g_fma(a.y, b, c.y), g_fma(a.z, b, c.z)); }
RM_HD vec4 fmaV(const vec4& a, float b, const vec4& c) { return vec4(g_fma(a.x, b, c.x), g_fma(a.y, b, c.y), g_fma(a.z, b, c.z), g_fma(a.w, b, c.w)); }

RM_HD vec2 operator-(const vec2& a) { return vec2(-a.x, -a.y); }
RM_HD vec3 operator-(const vec3& a) { return vec3(-a.x, -a.y, -a.z); }
RM_HD vec4 operator-(const vec4& a) { return vec4(-a.x, -a.y, -a.z, -a.w); }
RM_HD vec2 operator+(const vec2& a) { return a; }
RM_HD vec3 operator+(const vec3& a) { return a; }
RM_HD vec4 operator+(const vec4& a) { return a; }
RM_HD bool operator==(const vec2& a, const vec2& b) { return a.x == b.x && a.y == b.y; }
RM_HD bool operator==(const vec3& a, const vec3& b) { return a.x == b.x && a.y == b.y && a.z == b.z; }
RM_HD bool operator==(const vec4& a, const vec4& b) { return a.x == b.x && a.y == b.y && a.z == b.z && a.w == b.w; }
RM_HD bool operator!=(const vec2& a, const vec2& b) { return !(a == b); }
RM_HD bool operator!=(const vec3& a, const vec3& b) { return !(a == b); }
RM_HD bool operator!=(const vec4& a, const vec4& b) { return !(a == b); }
// GLSL `v++` / `v--` on vectors are rare; provided for completeness.
RM_HD vec2& operator++(vec2& a) { a = a + 1.0f; return a; }
RM_HD vec3& operator++(vec3& a) { a = a + 1.0f; return a; }
RM_HD vec4& operator++(vec4& a) { a = a + 1.0f; return a; }

// ------------------------------------------------------------------ component-wise functions
#define GLSL_MAP1(name)                                                              \
    RM_HD vec2 name(const vec2& a) { return vec2(name(a.x), name(a.y)); }            \
    RM_HD vec3 name(const vec3& a) { return vec3(name(a.x), name(a.y), name(a.z)); } \
    RM_HD vec4 name(const vec4& a) { return vec4(name(a.x), name(a.y), name(a.z), name(a.w)); }
#define GLSL_MAP2(name)                                                                                  \
    RM_HD vec2 name(const vec2& a, const vec2& b) { return vec2(name(a.x, b.x), name(a.y, b.y)); }       \
    RM_HD vec3 name(const vec3& a, const vec3& b) { return vec3(name(a.x, b.x), name(a.y, b.y), name(a.z, b.z)); } \
    RM_HD vec4 name(const vec4& a, const vec4& b) { return vec4(name(a.x, b.x), name(a.y, b.y), name(a.z, b.z), name(a.w, b.w)); }
#define GLSL_MAP2S(name) /* second argument scalar */                                          \
    RM_HD vec2 name(const vec2& a, float b) { return vec2(name(a.x, b), name(a.y, b)); }       \
    RM_HD vec3 name(const vec3& a, float b) { return vec3(name(a.x, b), name(a.y, b), name(a.z, b)); } \
    RM_HD vec4 name(const vec4& a, float b) { return vec4(name(a.x, b), name(a.y, b), name(a.z, b), name(a.w, b)); }
GLSL_MAP1(radians) GLSL_MAP1(degrees) GLSL_MAP1(sin) GLSL_MAP1(cos) GLSL_MAP1(tan)
GLSL_MAP1(asin) GLSL_MAP1(acos) GLSL_MAP1(atan) GLSL_MAP1(sinh) GLSL_MAP1(cosh) GLSL_MAP1(tanh)
GLSL_MAP1(asinh) GLSL_MAP1(acosh) GLSL_MAP1(atanh)
GLSL_MAP1(exp) GLSL_MAP1(log) GLSL_MAP1(exp2) GLSL_MAP1(log2) GLSL_MAP1(sqrt) GLSL_MAP1(inversesqrt)
GLSL_MAP1(abs) GLSL_MAP1(sign) GLSL_MAP1(floor) GLSL_MAP1(trunc) GLSL_MAP1(round) GLSL_MAP1(roundEven)
GLSL_MAP1(ceil) GLSL_MAP1(fract)
GLSL_MAP2(atan) GLSL_MAP2(pow) GLSL_MAP2(mod) GLSL_MAP2(min) GLSL_MAP2(max)
GLSL_MAP2S(min) GLSL_MAP2S(max) GLSL_MAP2S(mod)
#undef GLSL_MAP1
#undef GLSL_MAP2
#undef GLSL_MAP2S

// component access for "float or vector" operands of the repetition idiom
RM_HD float rm_c(float a, int) { return a; }
RM_HD float rm_c(const vec2& a, int i) { return a[i]; }
RM_HD float rm_c(const vec3& a, int i) { return a[i]; }
RM_HD float rm_c(const vec4& a, int i) { return a[i]; }
template <class H1, class S, class H2> RM_HD vec2 rm_rep(const vec2& x, const H1& h1, const S& s, const H2& h2) {
    return vec2(rm_rep1(x.x, rm_c(h1, 0), rm_c(s, 0), rm_c(h2, 0)), rm_rep1(x.y, rm_c(h1, 1), rm_c(s, 1), rm_c(h2, 1)));
}
#if !GLSL_FAST && GLSL_F32X2 && !(defined(RM_PIN_ALT) && RM_PIN_ALT)
// exact policy, packed: the same operations as rm_rep1 on every component - add, multiply by the
// correctly rounded reciprocal, floor, fused multiply-add, subtract - with x and y sharing FADD2 /
// FMUL2 / FFMA2 instructions (IEEE round-to-nearest per element, so the bits are those of rm_rep1)
template <class H1, class S, class H2> RM_HD vec3 rm_rep(const vec3& x, const H1& h1, const S& s, const H2& h2) {
    const float sx = rm_c(s, 0), sy = rm_c(s, 1), sz = rm_c(s, 2);
    const float rx = g_rcp(sx), ry = g_rcp(sy), rz = g_rcp(sz);
    const f2_t A = f2_add(f2_pack(x.x, x.y), f2_pack(rm_c(h1, 0), rm_c(h1, 1)));
    const f2_t Q = f2_mul(A, f2_pack(rx, ry));
    float qx, qy;
    f2_unpack(Q, qx, qy);
    const f2_t F = f2_pack(g_floor(qx), g_floor(qy));
    const f2_t Mxy = f2_fma(f2_pack(-sx, -sy), F, A);
    const f2_t E = f2_sub(Mxy, f2_pack(rm_c(h2, 0), rm_c(h2, 1)));
    vec3 out;
    f2_unpack(E, out.x, out.y);
    out.z = rm_rep1(x.z, rm_c(h1, 2), sz, rm_c(h2, 2));
    (void)rz;
    return out;
}
#elif GLSL_FAST && GLSL_F32X2
// packed (x, y) + scalar z version of the centred remainder
template <class H1, class S, class H2> RM_HD vec3 rm_rep(const vec3& x, const H1& h1, const S& s, const H2& h2) {
    const float s0 = rm_c(s, 0), a0 = rm_c(h1, 0), b0 = rm_c(h2, 0);
    const bool uniform = s0 == rm_c(s, 1) && s0 == rm_c(s, 2) && a0 == rm_c(h1, 1) && a0 == rm_c(h1, 2) && b0 == rm_c(h2, 1) && b0 == rm_c(h2, 2);
    if (uniform && a0 == b0 && b0 == 0.5f * s0 && s0 > 0.0f && s0 < 1e30f) {
        const float M = 12582912.0f, rs = 1.0f / s0;
        const f2_t Y = f2_pack(x.x, x.y);
        const f2_t R = f2_add(f2_fma(Y, f2_pack(rs, rs), f2_pack(M, M)), f2_pack(-M, -M));
        const f2_t Q = f2_fma(f2_pack(-s0, -s0), R, Y);
        vec3 out;
        f2_unpack(Q, out.x, out.y);
        const float rz = __fadd_rn(__fmaf_rn(x.z, rs, M), -M);
        out.z = __fmaf_rn(-s0, rz, x.z);
        return out;
    }
    return vec3(rm_rep1(x.x, rm_c(h1, 0), rm_c(s, 0), rm_c(h2, 0)), rm_rep1(x.y, rm_c(h1, 1), rm_c(s, 1), rm_c(h2, 1)),
                rm_rep1(x.z, rm_c(h1, 2), rm_c(s, 2), rm_c(h2, 2)));
}
#else
template <class H1, class S, class H2> RM_HD vec3 rm_rep(const vec3& x, const H1& h1, const S& s, const H2& h2) {
    return vec3(rm_rep1(x.x, rm_c(h1, 0), rm_c(s, 0), rm_c(h2, 0)), rm_rep1(x.y, rm_c(h1, 1), rm_c(s, 1), rm_c(h2, 1)),
                rm_rep1(x.z, rm_c(h1, 2), rm_c(s, 2), rm_c(h2, 2)));
}
#endif
template <class H1, class S, class H2> RM_HD vec4 rm_rep(const vec4& x, const H1& h1, const S& s, const H2& h2) {
    return vec4(rm_rep1(x.x, rm_c(h1, 0), rm_c(s, 0), rm_c(h2, 0)), rm_rep1(x.y, rm_c(h1, 1), rm_c(s, 1), rm_c(h2, 1)),
                rm_rep1(x.z, rm_c(h1, 2), rm_c(s, 2), rm_c(h2, 2)), rm_rep1(x.w, rm_c(h1, 3), rm_c(s, 3), rm_c(h2, 3)));
}
template <class S, class H2> RM_HD vec2 rm_rep0(const vec2& x, const S& s, const H2& h2) {
    return vec2(rm_rep0(x.x, rm_c(s, 0), rm_c(h2, 0)), rm_rep0(x.y, rm_c(s, 1), rm_c(h2, 1)));
}
template <class S, class H2> RM_HD vec3 rm_rep0(const vec3& x, const S& s, const H2& h2) {
    return vec3(rm_rep0(x.x, rm_c(s, 0), rm_c(h2, 0)), rm_rep0(x.y, rm_c(s, 1), rm_c(h2, 1)), rm_rep0(x.z, rm_c(s, 2), rm_c(h2, 2)));
}
template <class S, class H2> RM_HD vec4 rm_rep0(const vec4& x, const S& s, const H2& h2) {
    return vec4(rm_rep0(x.x, rm_c(s, 0), rm_c(h2, 0)), rm_rep0(x.y, rm_c(s, 1), rm_c(h2, 1)), rm_rep0(x.z, rm_c(s, 2), rm_c(h2, 2)),
                rm_rep0(x.w, rm_c(s, 3), rm_c(h2, 3)));
}

// ---- bounded-floor sites (lower_glsl.cpp pass 2) ------------------------------------------------
// rm_rep_b / rm_rep0_b are rm_rep / rm_rep0 at call sites whose operand is sdf()'s position parameter itself and
// whose H1, S do not depend on the position.  Here - host, oracle-side test harness, every guarded evaluation -
// they ARE rm_rep / rm_rep0.  The march kernels' fragment type overrides them with rm_rep_nf below.
// rm_plim_site(acc, ..) lowers acc to the largest |coordinate| for which the site's floor() argument
// q = (x + h1) * (1/s) is certainly within 2^22:  |q| <= (|x| + |h1|) / |s| * (1 + 2^-22), so
// |x| <= 0.999 * 2^22 * |s| - |h1| suffices; a limit that is not a number (s or h1 NaN) becomes -1: never fast.
template <class X, class H1, class S, class H2> RM_HD X rm_rep_b(const X& x, const H1& h1, const S& s, const H2& h2) { return rm_rep(x, h1, s, h2); }
template <class X, class S, class H2> RM_HD X rm_rep0_b(const X& x, const S& s, const H2& h2) { return rm_rep0(x, s, h2); }
RM_HD int rm_ncomp(float) { return 1; }
RM_HD int rm_ncomp(const vec2&) { return 2; }
RM_HD int rm_ncomp(const vec3&) { return 3; }
RM_HD int rm_ncomp(const vec4&) { return 4; }
RM_HD void rm_plim_lower(float& acc, float h1, float s) {
    const float lim = g_sub(g_mul(4190109.0f, g_abs(s)), g_abs(h1));       // 0.999 * 2^22
    if (!(lim == lim)) acc = -1.0f;
    else if (lim < acc) acc = lim;
}
template <class X, class H1, class S, class H2> RM_HD X rm_plim_site(float& acc, const X& x, const H1& h1, const S& s, const H2&) {
    for (int c = 0; c < rm_ncomp(x); c++) rm_plim_lower(acc, rm_c(h1, c), rm_c(s, c));
    return X(0.0f);
}
template <class X, class S, class H2> RM_HD X rm_plim_site0(float& acc, const X& x, const S& s, const H2&) {
    for (int c = 0; c < rm_ncomp(x); c++) rm_plim_lower(acc, 0.0f, rm_c(s, c));
    return X(0.0f);
}
#if !GLSL_FAST && RM_DEVICE_CODE && !(defined(RM_PIN_ALT) && RM_PIN_ALT)
// floor(q) on the FP32 pipe for |q| <= 2^22, +-inf and NaN (the caller has checked the range, see above):
// round-DOWN add of 1.5 * 2^23 (ulp 1 there, so the sum is floor(q) + M exactly), subtract M.  The only
// input whose result differs from floorf is -0 (gives +0); the mod() built on it then yields -0 instead of
// +0 for x + h1 == -0, which the `- h2` that follows erases unless h2 is zero - so the sign is only
// restored (LOP3) when h2 == 0 or NaN; with baked uniforms that test folds at compile time.
RM_HD float g_floor_nf(float q, float h2) {
    const float M = 12582912.0f;
    float r = __fadd_rn(__fadd_rd(q, M), -M);
    if (!(h2 != 0.0f) || !(h2 == h2)) r = __uint_as_float(__float_as_uint(r) | (__float_as_uint(q) & 0x80000000u));
    return r;
}
RM_HD float rm_rep1_nf(float x, float h1, float s, float h2) {
    const float a = g_add(x, h1);
    return g_sub(g_fma(-s, g_floor_nf(g_mul(a, g_rcp(s)), h2), a), h2);
}
// the packed rm_rep (above) with that floor: FADD2 / FMUL2 / FADD2.RM / FADD2 / FFMA2 / FADD2 for x and y
template <class H1, class S, class H2> RM_HD vec3 rm_rep_nf(const vec3& x, const H1& h1, const S& s, const H2& h2) {
    const float M = 12582912.0f;
    const float sx = rm_c(s, 0), sy = rm_c(s, 1), sz = rm_c(s, 2);
    const float h2x = rm_c(h2, 0), h2y = rm_c(h2, 1);
    const f2_t A = f2_add(f2_pack(x.x, x.y), f2_pack(rm_c(h1, 0), rm_c(h1, 1)));
    const f2_t Q = f2_mul(A, f2_pack(g_rcp(sx), g_rcp(sy)));
    f2_t F = f2_add(f2_add_rd(Q, f2_pack(M, M)), f2_pack(-M, -M));
    if (!(h2x != 0.0f) || !(h2x == h2x)) F.x = __uint_as_float(__float_as_uint(F.x) | (__float_as_uint(Q.x) & 0x80000000u));
    if (!(h2y != 0.0f) || !(h2y == h2y)) F.y = __uint_as_float(__float_as_uint(F.y) | (__float_as_uint(Q.y) & 0x80000000u));
    const f2_t E = f2_sub(f2_fma(f2_pack(-sx, -sy), F, A), f2_pack(h2x, h2y));
    vec3 out;
    f2_unpack(E, out.x, out.y);
    out.z = rm_rep1_nf(x.z, rm_c(h1, 2), sz, rm_c(h2, 2));
    return out;
}
#endif

RM_HD vec2 clamp(const vec2& v, float lo, float hi) { return vec2(clamp(v.x, lo, hi), clamp(v.y, lo, hi)); }
RM_HD vec3 clamp(const vec3& v, float lo, float hi) { return vec3(clamp(v.x, lo, hi), clamp(v.y, lo, hi), clamp(v.z, lo, hi)); }
RM_HD vec4 clamp(const vec4& v, float lo, float hi) { return vec4(clamp(v.x, lo, hi), clamp(v.y, lo, hi), clamp(v.z, lo, hi), clamp(v.w, lo, hi)); }
RM_HD vec2 clamp(const vec2& v, const vec2& lo, const vec2& hi) { return vec2(clamp(v.x, lo.x, hi.x), clamp(v.y, lo.y, hi.y)); }
RM_HD vec3 clamp(const vec3& v, const vec3& lo, const vec3& hi) { return vec3(clamp(v.x, lo.x, hi.x), clamp(v.y, lo.y, hi.y), clamp(v.z, lo.z, hi.z)); }
RM_HD vec4 clamp(const vec4& v, const vec4& lo, const vec4& hi) { return vec4(clamp(v.x, lo.x, hi.x), clamp(v.y, lo.y, hi.y), clamp(v.z, lo.z, hi.z), clamp(v.w, lo.w, hi.w)); }
RM_HD vec2 mix(const vec2& a, const vec2& b, float t) { return vec2(mix(a.x, b.x, t), mix(a.y, b.y, t)); }
RM_HD vec3 mix(const vec3& a, const vec3& b, float t) { return vec3(mix(a.x, b.x, t), mix(a.y, b.y, t), mix(a.z, b.z, t)); }
RM_HD vec4 mix(const vec4& a, const vec4& b, float t) { return vec4(mix(a.x, b.x, t), mix(a.y, b.y, t), mix(a.z, b.z, t), mix(a.w, b.w, t)); }
RM_HD vec2 mix(const vec2& a, const vec2& b, const vec2& t) { return vec2(mix(a.x, b.x, t.x), mix(a.y, b.y, t.y)); }
RM_HD vec3 mix(const vec3& a, const vec3& b, const vec3& t) { return vec3(mix(a.x, b.x, t.x), mix(a.y, b.y, t.y), mix(a.z, b.z, t.z)); }
RM_HD vec4 mix(const vec4& a, const vec4& b, const vec4& t) { return vec4(mix(a.x, b.x, t.x), mix(a.y, b.y, t.y), mix(a.z, b.z, t.z), mix(a.w, b.w, t.w)); }
RM_HD vec2 step(float e, const vec2& v) { return vec2(step(e, v.x), step(e, v.y)); }
RM_HD vec3 step(float e, const vec3& v) { return vec3(step(e, v.x), step(e, v.y), step(e, v.z)); }
RM_HD vec4 step(float e, const vec4& v) { return vec4(step(e, v.x), step(e, v.y), step(e, v.z), step(e, v.w)); }
RM_HD vec2 step(const vec2& e, const vec2& v) { return vec2(step(e.x, v.x), step(e.y, v.y)); }
RM_HD vec3 step(const vec3& e, const vec3& v) { return vec3(step(e.x, v.x), step(e.y, v.y), step(e.z, v.z)); }
RM_HD vec4 step(const vec4& e, const vec4& v) { return vec4(step(e.x, v.x), step(e.y, v.y), step(e.z, v.z), step(e.w, v.w)); }
RM_HD vec2 smoothstep(float a, float b, const vec2& v) { return vec2(smoothstep(a, b, v.x), smoothstep(a, b, v.y)); }
RM_HD vec3 smoothstep(float a, float b, const vec3& v) { return vec3(smoothstep(a, b, v.x), smoothstep(a, b, v.y), smoothstep(a, b, v.z)); }
RM_HD vec4 smoothstep(float a, float b, const vec4& v) { return vec4(smoothstep(a, b, v.x), smoothstep(a, b, v.y), smoothstep(a, b, v.z), smoothstep(a, b, v.w)); }
RM_HD vec2 smoothstep(const vec2& a, const vec2& b, const vec2& v) { return vec2(smoothstep(a.x, b.x, v.x), smoothstep(a.y, b.y, v.y)); }
RM_HD vec3 smoothstep(const vec3& a, const vec3& b, const vec3& v) { return vec3(smoothstep(a.x, b.x, v.x), smoothstep(a.y, b.y, v.y), smoothstep(a.z, b.z, v.z)); }
RM_HD vec4 smoothstep(const vec4& a, const vec4& b, const vec4& v) { return vec4(smoothstep(a.x, b.x, v.x), smoothstep(a.y, b.y, v.y), smoothstep(a.z, b.z, v.z), smoothstep(a.w, b.w, v.w)); }

RM_HD bvec2 isnan(const vec2& v) { return bvec2(isnan(v.x), isnan(v.y)); }
RM_HD bvec3 isnan(const vec3& v) { return bvec3(isnan(v.x), isnan(v.y), isnan(v.z)); }
RM_HD bvec4 isnan(const vec4& v) { return bvec4(isnan(v.x), isnan(v.y), isnan(v.z), isnan(v.w)); }
RM_HD bvec2 isinf(const vec2& v) { return bvec2(isinf(v.x), isinf(v.y)); }
RM_HD bvec3 isinf(const vec3& v) { return bvec3(isinf(v.x), isinf(v.y), isinf(v.z)); }
RM_HD bvec4 isinf(const vec4& v) { return bvec4(isinf(v.x), isinf(v.y), isinf(v.z), isinf(v.w)); }
#define GLSL_CMP(name, op)                                                                              \
    RM_HD bvec2 name(const vec2& a, const vec2& b) { return bvec2(a.x op b.x, a.y op b.y); }            \
    RM_HD bvec3 name(const vec3& a, const vec3& b) { return bvec3(a.x op b.x, a.y op b.y, a.z op b.z); } \
    RM_HD bvec4 name(const vec4& a, const vec4& b) { return bvec4(a.x op b.x, a.y op b.y, a.z op b.z, a.w op b.w); }
GLSL_CMP(lessThan, <) GLSL_CMP(lessThanEqual, <=) GLSL_CMP(greaterThan, >) GLSL_CMP(greaterThanEqual, >=)
GLSL_CMP(equal, ==) GLSL_CMP(notEqual, !=)
#undef GLSL_CMP

// ------------------------------------------------------------------ geometric functions
RM_HD float dot(const vec2& a, const vec2& b) { return g_fma(a.y, b.y, g_mul(a.x, b.x)); }
RM_HD float dot(const vec3& a, const vec3& b) { return g_fma(a.z, b.z, g_fma(a.y, b.y, g_mul(a.x, b.x))); }
RM_HD float dot(const vec4& a, const vec4& b) { return g_fma(a.w, b.w, g_fma(a.z, b.z, g_fma(a.y, b.y, g_mul(a.x, b.x)))); }
RM_HD float length(const vec2& a) { return g_sqrt(dot(a, a)); }
RM_HD float length(const vec3& a) { return g_sqrt(dot(a, a)); }
RM_HD float length(const vec4& a) { return g_sqrt(dot(a, a)); }
RM_HD float distance(const vec2& a, const vec2& b) { return length(a - b); }
RM_HD float distance(const vec3& a, const vec3& b) { return length(a - b); }
RM_HD float distance(const vec4& a, const vec4& b) { return length(a - b); }
#if GLSL_FAST
RM_HD vec2 normalize(const vec2& a) { return a * g_rsqrt(dot(a, a)); }
RM_HD vec3 normalize(const vec3& a) { return a * g_rsqrt(dot(a, a)); }
RM_HD vec4 normalize(const vec4& a) { return a * g_rsqrt(dot(a, a)); }
#else
RM_HD vec2 normalize(const vec2& a) { return a / length(a); }
RM_HD vec3 normalize(const vec3& a) { return a / length(a); }
RM_HD vec4 normalize(const vec4& a) { return a / length(a); }
#endif
RM_HD vec3 cross(const vec3& a, const vec3& b) {
    return vec3(g_sub(g_mul(a.y, b.z), g_mul(b.y, a.z)),
                g_sub(g_mul(a.z, b.x), g_mul(b.z, a.x)),
                g_sub(g_mul(a.x, b.y), g_mul(b.x, a.y)));
}
RM_HD vec2 reflect(const vec2& i, const vec2& n) { return i - g_mul(2.0f, dot(n, i)) * n; }
RM_HD vec3 reflect(const vec3& i, const vec3& n) { return i - g_mul(2.0f, dot(n, i)) * n; }
RM_HD vec4 reflect(const vec4& i, const vec4& n) { return i - g_mul(2.0f, dot(n, i)) * n; }
RM_HD vec3 refract(const vec3& i, const vec3& n, float eta) {
    float d = dot(n, i);
    float k = g_sub(1.0f, g_mul(g_mul(eta, eta), g_sub(1.0f, g_mul(d, d))));
    if (k < 0.0f) return vec3(0.0f);
    return eta * i - g_add(g_mul(eta, d), g_sqrt(k)) * n;
}
RM_HD vec2 refract(const vec2& i, const vec2& n, float eta) {
    float d = dot(n, i);
    float k = g_sub(1.0f, g_mul(g_mul(eta, eta), g_sub(1.0f, g_mul(d, d))));
    if (k < 0.0f) return vec2(0.0f);
    return eta * i - g_add(g_mul(eta, d), g_sqrt(k)) * n;
}
RM_HD vec3 faceforward(const vec3& n, const vec3& i, const vec3& nref) { return dot(nref, i) < 0.0f ? n : -n; }

// ------------------------------------------------------------------ matrices (column-major)
struct mat2 {
    vec2 c[2];
    RM_HD mat2() {}
    RM_HD explicit mat2(float d) { c[0] = vec2(d, 0.0f); c[1] = vec2(0.0f, d); }
    RM_HD mat2(float a, float b, float c_, float d) { c[0] = vec2(a, b); c[1] = vec2(c_, d); }
    RM_HD mat2(const vec2& a, const vec2& b) { c[0] = a; c[1] = b; }
    RM_HD vec2& operator[](int i) { return c[i]; }
    RM_HD const vec2& operator[](int i) const { return c[i]; }
};
struct mat3 {
    vec3 c[3];
    RM_HD mat3() {}
    RM_HD explicit mat3(float d) { c[0] = vec3(d, 0.0f, 0.0f); c[1] = vec3(0.0f, d, 0.0f); c[2] = vec3(0.0f, 0.0f, d); }
    RM_HD mat3(float a0, float a1, float a2, float b0, float b1, float b2, float c0, float c1, float c2) {
        c[0] = vec3(a0, a1, a2); c[1] = vec3(b0, b1, b2); c[2] = vec3(c0, c1, c2);
    }
    RM_HD mat3(const vec3& a, const vec3& b, const vec3& d) { c[0] = a; c[1] = b; c[2] = d; }
    RM_HD explicit mat3(const mat4& m);
    RM_HD vec3& operator[](int i) { return c[i]; }
    RM_HD const vec3& operator[](int i) const { return c[i]; }
};
struct mat4 {
    vec4 c[4];
    RM_HD mat4() {}
    RM_HD explicit mat4(float d) {
        c[0] = vec4(d, 0.0f, 0.0f, 0.0f); c[1] = vec4(0.0f, d, 0.0f, 0.0f);
        c[2] = vec4(0.0f, 0.0f, d, 0.0f); c[3] = vec4(0.0f, 0.0f, 0.0f, d);
    }
    RM_HD mat4(float a0, float a1, float a2, float a3, float b0, float b1, float b2, float b3,
               float c0, float c1, float c2, float c3, float d0, float d1, float d2, float d3) {
        c[0] = vec4(a0, a1, a2, a3); c[1] = vec4(b0, b1, b2, b3); c[2] = vec4(c0, c1, c2, c3); c[3] = vec4(d0, d1, d2, d3);
    }
    RM_HD mat4(const vec4& a, const vec4& b, const vec4& d, const vec4& e) { c[0] = a; c[1] = b; c[2] = d; c[3] = e; }
    RM_HD vec4& operator[](int i) { return c[i]; }
    RM_HD const vec4& operator[](int i) const { return c[i]; }
};
RM_HD mat3::mat3(const mat4& m) { c[0] = vec3(m.c[0]); c[1] = vec3(m.c[1]); c[2] = vec3(m.c[2]); }

// M * v: linear combination of columns, summed left to right.  v * M: dot with each column.
RM_HD vec2 operator*(const mat2& m, const vec2& v) { return m.c[0] * v.x + m.c[1] * v.y; }
RM_HD vec3 operator*(const mat3& m, const vec3& v) { return m.c[0] * v.x + m.c[1] * v.y + m.c[2] * v.z; }
RM_HD vec4 operator*(const mat4& m, const vec4& v) { return m.c[0] * v.x + m.c[1] * v.y + m.c[2] * v.z + m.c[3] * v.w; }
RM_HD vec2 operator*(const vec2& v, const mat2& m) { return vec2(dot(v, m.c[0]), dot(v, m.c[1])); }
RM_HD vec3 operator*(const vec3& v, const mat3& m) { return vec3(dot(v, m.c[0]), dot(v, m.c[1]), dot(v, m.c[2])); }
RM_HD vec4 operator*(const vec4& v, const mat4& m) { return vec4(dot(v, m.c[0]), dot(v, m.c[1]), dot(v, m.c[2]), dot(v, m.c[3])); }
RM_HD mat2 operator*(const mat2& a, const mat2& b) { return mat2(a * b.c[0], a * b.c[1]); }
RM_HD mat3 operator*(const mat3& a, const mat3& b) { return mat3(a * b.c[0], a * b.c[1], a * b.c[2]); }
RM_HD mat4 operator*(const mat4& a, const mat4& b) { return mat4(a * b.c[0], a * b.c[1], a * b.c[2], a * b.c[3]); }
RM_HD mat2 operator*(const mat2& a, float s) { return mat2(a.c[0] * s, a.c[1] * s); }
RM_HD mat3 operator*(const mat3& a, float s) { return mat3(a.c[0] * s, a.c[1] * s, a.c[2] * s); }
RM_HD mat4 operator*(const mat4& a, float s) { return mat4(a.c[0] * s, a.c[1] * s, a.c[2] * s, a.c[3] * s); }
RM_HD mat2 operator*(float s, const mat2& a) { return a * s; }
RM_HD mat3 operator*(float s, const mat3& a) { return a * s; }
RM_HD mat4 operator*(float s, const mat4& a) { return a * s; }
RM_HD mat2 operator+(const mat2& a, const mat2& b) { return mat2(a.c[0] + b.c[0], a.c[1] + b.c[1]); }
RM_HD mat3 operator+(const mat3& a, const mat3& b) { return mat3(a.c[0] + b.c[0], a.c[1] + b.c[1], a.c[2] + b.c[2]); }
RM_HD mat4 operator+(const mat4& a, const mat4& b) { return mat4(a.c[0] + b.c[0], a.c[1] + b.c[1], a.c[2] + b.c[2], a.c[3] + b.c[3]); }
RM_HD mat2 operator-(const mat2& a, const mat2& b) { return mat2(a.c[0] - b.c[0], a.c[1] - b.c[1]); }
RM_HD mat3 operator-(const mat3& a, const mat3& b) { return mat3(a.c[0] - b.c[0], a.c[1] - b.c[1], a.c[2] - b.c[2]); }
RM_HD mat4 operator-(const mat4& a, const mat4& b) { return mat4(a.c[0] - b.c[0], a.c[1] - b.c[1], a.c[2] - b.c[2], a.c[3] - b.c[3]); }
RM_HD vec2& operator*=(vec2& v, const mat2& m) { v = v * m; return v; }
RM_HD vec3& operator*=(vec3& v, const mat3& m) { v = v * m; return v; }
RM_HD vec4& operator*=(vec4& v, const mat4& m) { v = v * m; return v; }
RM_HD mat2& operator*=(mat2& a, const mat2& b) { a = a * b; return a; }
RM_HD mat3& operator*=(mat3& a, const mat3& b) { a = a * b; return a; }
RM_HD mat4& operator*=(mat4& a, const mat4& b) { a = a * b; return a; }
RM_HD mat2 transpose(const mat2& m) { return mat2(m.c[0].x, m.c[1].x, m.c[0].y, m.c[1].y); }
RM_HD mat3 transpose(const mat3& m) {
    return mat3(m.c[0].x, m.c[1].x, m.c[2].x, m.c[0].y, m.c[1].y, m.c[2].y, m.c[0].z, m.c[1].z, m.c[2].z);
}
RM_HD mat4 transpose(const mat4& m) {
    return mat4(m.c[0].x, m.c[1].x, m.c[2].x, m.c[3].x, m.c[0].y, m.c[1].y, m.c[2].y, m.c[3].y,
                m.c[0].z, m.c[1].z, m.c[2].z, m.c[3].z, m.c[0].w, m.c[1].w, m.c[2].w, m.c[3].w);
}
RM_HD mat2 matrixCompMult(const mat2& a, const mat2& b) { return mat2(a.c[0] * b.c[0], a.c[1] * b.c[1]); }
RM_HD mat3 matrixCompMult(const mat3& a, const mat3& b) { return mat3(a.c[0] * b.c[0], a.c[1] * b.c[1], a.c[2] * b.c[2]); }
RM_HD float determinant(const mat2& m) { return g_sub(g_mul(m.c[0].x, m.c[1].y), g_mul(m.c[1].x, m.c[0].y)); }
RM_HD float determinant(const mat3& m) { return dot(m.c[0], cross(m.c[1], m.c[2])); }
RM_HD mat2 inverse(const mat2& m) {
    float d = determinant(m);
    return mat2(g_div(m.c[1].y, d), g_div(-m.c[0].y, d), g_div(-m.c[1].x, d), g_div(m.c[0].x, d));
}
RM_HD mat3 inverse(const mat3& m) {
    vec3 r0 = cross(m.c[1], m.c[2]), r1 = cross(m.c[2], m.c[0]), r2 = cross(m.c[0], m.c[1]);
    float d = dot(m.c[0], r0);
    return transpose(mat3(r0 / d, r1 / d, r2 / d));
}

// ------------------------------------------------------------------ swizzle proxy bodies
#define GLSL_SW_OPS(SW, TPL, VEC, MAT, LOAD, STORE)                                           \
    TPL RM_HD SW::operator VEC() const { return LOAD; }                                       \
    TPL RM_HD SW& SW::operator=(const VEC& o) { VEC t(o); STORE; return *this; }              \
    TPL RM_HD SW& SW::operator=(const SW& o) { VEC t = (VEC)o; STORE; return *this; }         \
    TPL RM_HD SW& SW::operator+=(const VEC& o) { VEC t = (VEC)(*this) + o; STORE; return *this; } \
    TPL RM_HD SW& SW::operator-=(const VEC& o) { VEC t = (VEC)(*this) - o; STORE; return *this; } \
    TPL RM_HD SW& SW::operator*=(const VEC& o) { VEC t = (VEC)(*this) * o; STORE; return *this; } \
    TPL RM_HD SW& SW::operator/=(const VEC& o) { VEC t = (VEC)(*this) / o; STORE; return *this; } \
    TPL RM_HD SW& SW::operator+=(float o) { VEC t = (VEC)(*this) + o; STORE; return *this; }  \
    TPL RM_HD SW& SW::operator-=(float o) { VEC t = (VEC)(*this) - o; STORE; return *this; }  \
    TPL RM_HD SW& SW::operator*=(float o) { VEC t = (VEC)(*this) * o; STORE; return *this; }  \
    TPL RM_HD SW& SW::operator/=(float o) { VEC t = (VEC)(*this) / o; STORE; return *this; }  \
    TPL RM_HD SW& SW::operator*=(const MAT& m) { VEC t = (VEC)(*this) * m; STORE; return *this; }
#define GLSL_TPL2 template <int N, int A, int B>
#define GLSL_TPL3 template <int N, int A, int B, int C>
#define GLSL_TPL4 template <int N, int A, int B, int C, int D>
#define GLSL_SW2 Sw2<N, A, B>
#define GLSL_SW3 Sw3<N, A, B, C>
#define GLSL_SW4 Sw4<N, A, B, C, D>
GLSL_SW_OPS(GLSL_SW2, GLSL_TPL2, vec2, mat2, vec2(v[A], v[B]), (v[A] = t.x, v[B] = t.y))
GLSL_SW_OPS(GLSL_SW3, GLSL_TPL3, vec3, mat3, vec3(v[A], v[B], v[C]), (v[A] = t.x, v[B] = t.y, v[C] = t.z))
GLSL_SW_OPS(GLSL_SW4, GLSL_TPL4, vec4, mat4, vec4(v[A], v[B], v[C], v[D]), (v[A] = t.x, v[B] = t.y, v[C] = t.z, v[D] = t.w))
#undef GLSL_SW_OPS
#undef GLSL_TPL2
#undef GLSL_TPL3
#undef GLSL_TPL4
#undef GLSL_SW2
#undef GLSL_SW3
#undef GLSL_SW4

}  // namespace GLSL_NS

#undef GLSL_NS
#undef GLSL_FAST
