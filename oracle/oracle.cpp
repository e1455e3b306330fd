// oracle.cpp -- CPU restatement of the raymarching-engine hot path.  TEST INFRASTRUCTURE ONLY.
//
// PARITY UNPINNED: the reference (radian628/raymarching-engine) ships no tests, golden images
// or known-answer vectors for this path, and it cannot be executed in this environment (its
// arithmetic runs inside a browser's WebGL2 stack; no browser/GL/Node here - SURVEY.md 8c).
// This file is therefore a line-by-line restatement of the reference GLSL, pinned only by the
// known-answer values derivable from the source (tests/test_oracle_kat.py) and by an independent
// numpy cross-check (tests/test_oracle_numpy.py).
//
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
// load this library.  The product (raymarching_engine_b200/) never links, imports or calls it.
//
// What is restated (paths relative to /root/reference/client):
//   public/shader/raymarcher.vert:8-11      texcoord of a pixel centre
//   public/shader/raymarcher.frag:44-49     gold_noise
//   public/shader/raymarcher.frag:61-65     rodrigues
//   public/shader/raymarcher.frag:78-101    boxMullerTransform / uniformSample / sphereSample
//   public/shader/raymarcher.frag:108-112   sdBox
//   public/shader/raymarcher.frag:148-175   invExpDist / sceneNormal / castRay / schlick
//   public/shader/raymarcher.frag:178-387   main(): camera models, preview branch, path tracer
//   public/shader/blit.frag:14-18           prev := curr (in-place accumulation is equivalent)
//   public/shader/display.frag:20-61        present pass (DoF blur, brightness, gamma) -> RGBA8
//   src/util/Halton.tsx:1-19                Halton sequence
//   src/renderer/LoadRenderJobContext.tsx:43-124  RGBA32F + 2x RGBA16F, NEAREST, REPEAT
//   src/settings/shader-editor/Validate.tsx:18-51 default material functions
//   public/examples/*.glsl, dist/examples/sphere-grid.glsl, src/index.tsx:365-389  scenes
//
// Arithmetic: scalar fp32, no compiler FMA contraction (-ffp-contract=off); the only fused
// operations are the ones pinned explicitly (glsl_rt.h header: dot/length, mod, mix, and the march
// advance p + d*s / depth += deltaZ*s below - contractions GLSL ES 3.00 4.5.2 permits and GPU
// compilers perform).  GLSL built-ins come from the shared deterministic math layer (glsl_rt.h /
// rm_math.h, exact policy) so that the CUDA kernel can be compared bit for bit (SURVEY.md H1).  Scenes are hand-translated here, independently of
// the product's GLSL->CUDA lowering, so the lowering itself is under test.
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <atomic>
#include <string>
#include <thread>
#include <vector>

#define GLSL_NS xg
#define GLSL_FAST 0
#include "../raymarching_engine_b200/csrc/device_src/glsl_rt.h"

using namespace xg;

// ------------------------------------------------------------------------------------------
// Built-in uniform block (names follow raymarcher.frag:6-42).  Plain C layout for ctypes.
// ------------------------------------------------------------------------------------------
extern "C" {
struct OrcUniforms {
    float blendWithPreviousFactor;
    float randNoise[2];
    float position[3];
    float rotation[16];  // column-major, as uploaded by uniformMatrix4fv(transpose=false)
    float dofAmount;
    float dofFocalPlaneDistance;
    int cameraMode;      // 0 perspective, 1 orthographic, 2 panoramic
    float fov;
    float reflections;
    float aspect;
    float fogDensity;
    float exposure;
    float raymarchingStepCountsArray[10];
    int blendMode;       // 1 additive, 0 mix
    int renderMode;      // 1 preview, 0 full
    float lightPositions[30];
    float lightColors[30];
    float lightSizes[10];
    int lightCount;
    int showDofFocalPlane;
};
}

// ------------------------------------------------------------------------------------------
// half-float storage for the two RGBA16F accumulators (LoadRenderJobContext.tsx:77-111).
// Round-to-nearest-even, IEEE binary16 with denormals, overflow to infinity.
// ------------------------------------------------------------------------------------------
static inline uint16_t f32_to_f16(float f) {
    uint32_t x; memcpy(&x, &f, 4);
    uint32_t sign = (x >> 16) & 0x8000u;
    uint32_t ax = x & 0x7fffffffu;
    if (ax > 0x7f800000u) return (uint16_t)(sign | 0x7e00u);            // NaN
    if (ax >= 0x477ff000u) return (uint16_t)(sign | 0x7c00u);           // >= 65520 -> inf
    if (ax < 0x33000001u) return (uint16_t)sign;                        // <= 2^-25 -> 0
    if (ax < 0x38800000u) {                                             // denormal half
        uint32_t mant = (ax & 0x007fffffu) | 0x00800000u;
        int shift = 126 - (int)(ax >> 23);                              // 14..24
        uint32_t h = mant >> shift;
        uint32_t rem = mant & ((1u << shift) - 1u);
        uint32_t half = 1u << (shift - 1);
        if (rem > half || (rem == half && (h & 1u))) h++;
        return (uint16_t)(sign | h);
    }
    uint32_t h = ((ax - 0x38000000u) >> 13);
    uint32_t rem = ax & 0x1fffu;
    if (rem > 0x1000u || (rem == 0x1000u && (h & 1u))) h++;
    return (uint16_t)(sign | h);
}
static inline float f16_to_f32(uint16_t h) {
    uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
    uint32_t e = (h >> 10) & 0x1fu, m = h & 0x3ffu, x;
    if (e == 0) {
        if (m == 0) x = sign;
        else { int s = 0; while (!(m & 0x400u)) { m <<= 1; s++; } x = sign | ((uint32_t)(113 - s) << 23) | ((m & 0x3ffu) << 13); }
    } else if (e == 31) x = sign | 0x7f800000u | (m << 13);
    else x = sign | ((e + 112u) << 23) | (m << 13);
    float f; memcpy(&f, &x, 4); return f;
}

// ------------------------------------------------------------------------------------------
// Scenes.  Each scene is a struct with the custom uniforms as members, sdf() and the seven
// material functions; `load(const float*, int)` fills the uniforms from a flat float array in
// declaration order.  Defaults follow Validate.tsx:18-51.
// ------------------------------------------------------------------------------------------
static inline float sdBox(vec3 p, vec3 b) {                         // raymarcher.frag:108-112
    vec3 q = abs(p) - b;
    return length(max(q, 0.0f)) + min(max(q.x, max(q.y, q.z)), 0.0f);
}

struct DefaultMaterials {                                           // Validate.tsx:18-51
    vec3 sceneDiffuseColor(vec3 position) {
        if (length(position) > 35.0f) return vec3(0.0f);
        return vec3(0.6f);
    }
    vec3 sceneSpecularColor(vec3 position) {
        if (length(position) > 35.0f) return vec3(0.0f);
        return vec3(0.6f);
    }
    float sceneSpecularRoughness(vec3) { return 0.2f; }
    float sceneSubsurfaceScattering(vec3) { return 11111115.0f; }
    vec3 sceneSubsurfaceScatteringColor(vec3 position) {
        if (length(position) > 30.0f) return vec3(1.0f);
        return vec3(1.0f);
    }
    float sceneIOR(vec3) { return 100.0f; }
    vec3 sceneEmission(vec3 position) {
        float d = max(normalize(position).y, 0.2f);
        vec3 brightColor = vec3(0.7f, 0.8f, 1.0f) * d * 1.0f;
        return (length(position) > 36.0f) ? (brightColor * 2.00f) : vec3(0.0f);
    }
};

// The sphere-grid fractal shared by guide.glsl:91-102 and fractal1.glsl:23-34.
static inline float sphereGridFractal(vec3 position, float fractalIterations, float gridScaleFactor,
                                      vec3 bigSphereCenter, float bigSphereSize) {
    float minDist = 9999.9f;
    for (float i = -1.0f; i < fractalIterations; i++) {
        float sf = pow(gridScaleFactor, i);
        vec3 d = abs(mod(position + vec3(0.5f * sf), sf) - vec3(sf / 2.0f)) - vec3(sf / 3.0f);
        float dist = length(d) - 0.21f * sf;
        minDist = min(dist, minDist);
    }
    minDist = max(length(position - bigSphereCenter) - bigSphereSize, -minDist);
    return minDist;
}

struct SceneGuide : DefaultMaterials {                              // examples/guide.glsl
    float bigSphereSize = 4.0f; vec3 fractalColor = vec3(0.5f, 0.5f, 0.5f); float fractalIterations = 8.0f;
    float gridScaleFactor = 0.33333333333f; vec3 bigSphereCenter = vec3(0.0f, 0.0f, 10.0f);
    static constexpr int NU = 9;
    void load(const float* u) {
        bigSphereSize = u[0]; fractalColor = vec3(u[1], u[2], u[3]); fractalIterations = u[4];
        gridScaleFactor = u[5]; bigSphereCenter = vec3(u[6], u[7], u[8]);
    }
    vec3 sceneDiffuseColor(vec3 position) {                         // guide.glsl:51-54
        if (length(position) > 35.0f) return vec3(0.0f);
        return vec3(fractalColor);
    }
    // specular, roughness, subsurface, IOR, emission at guide.glsl:57-88 equal the defaults
    float sdf(vec3 position) { return sphereGridFractal(position, fractalIterations, gridScaleFactor, bigSphereCenter, bigSphereSize); }
};

struct SceneFractal1 : DefaultMaterials {                           // examples/fractal1.glsl
    float bigSphereSize = 4.0f; float fractalIterations = 8.0f; float gridScaleFactor = 0.33333333333f;
    vec3 bigSphereCenter = vec3(0.0f, 0.0f, 10.0f);
    static constexpr int NU = 6;
    void load(const float* u) { bigSphereSize = u[0]; fractalIterations = u[1]; gridScaleFactor = u[2]; bigSphereCenter = vec3(u[3], u[4], u[5]); }
    float sdf(vec3 position) { return sphereGridFractal(position, fractalIterations, gridScaleFactor, bigSphereCenter, bigSphereSize); }
};

struct SceneMenger : DefaultMaterials {                             // examples/menger-sponge.glsl:6-23
    float fractalIterations = 8.0f;
    static constexpr int NU = 1;
    void load(const float* u) { fractalIterations = u[0]; }
    float sdf(vec3 position) {
        float minDist = sdBox(position + vec3(0.5f), vec3(0.5f));
        for (float i = 1.0f; i < fractalIterations; i++) {
            float sf = pow(0.33333333333333f, i);
            vec3 gridPosition = mod(position, sf * 3.0f) - sf * 1.5f;
            minDist = max(minDist,
                          -min(min(sdBox(gridPosition, vec3(sf * 1.51f, sf * 0.5f, sf * 0.5f)),
                                   sdBox(gridPosition, vec3(sf * 0.5f, sf * 1.51f, sf * 0.5f))),
                               sdBox(gridPosition, vec3(sf * 0.5f, sf * 0.5f, sf * 1.51f))));
        }
        return minDist;
    }
};

// GLSL `v.ab *= mat2(c, -s, s, c)`: row vector times column-major matrix (SURVEY.md H4):
// columns c0 = (c, -s), c1 = (s, c);  (a,b)*M = (dot((a,b),c0), dot((a,b),c1)), with the pinned
// (fused) dot of glsl_rt.h.
static inline void rotPair(float& a, float& b, float ang) {
    float c = cos(ang), s = sin(ang);
    vec2 v(a, b);
    float na = dot(v, vec2(c, -s));
    float nb = dot(v, vec2(s, c));
    a = na; b = nb;
}

struct SceneTree : DefaultMaterials {                               // examples/tree.glsl:16-36
    float fractalIterations = 8.0f, scaleFactor = 0.7f; vec3 angles = vec3(2.9f, -0.8f, 0.4f); float offset = 1.2f;
    static constexpr int NU = 6;
    void load(const float* u) { fractalIterations = u[0]; scaleFactor = u[1]; angles = vec3(u[2], u[3], u[4]); offset = u[5]; }
    float sdf(vec3 position) {
        vec3 transformedPos = position;
        float minDist = 9999.0f;
        for (float i = 0.0f; i < fractalIterations; i++) {
            float combinedScaleFactor = pow(scaleFactor, i);
            vec3 tpos2 = transformedPos * combinedScaleFactor;
            minDist = min(minDist, sdBox(tpos2, vec3(1.0f, 0.1f, 0.1f) * (combinedScaleFactor)));
            transformedPos /= scaleFactor;
            transformedPos = abs(transformedPos) - vec3(1.0f, 0.1f, 0.1f) * vec3(offset);
            rotPair(transformedPos.x, transformedPos.y, angles.x);
            rotPair(transformedPos.y, transformedPos.z, angles.y);
            rotPair(transformedPos.x, transformedPos.z, angles.z);
        }
        return minDist;
    }
};

struct SceneSmoothTree : DefaultMaterials {                         // examples/smooth-tree.glsl:20-56
    float fractalIterations = 14.0f, scaleFactor = 0.7f; vec3 angles = vec3(2.9f, -0.8f, 0.4f); float offset = 1.2f; int smoothen = 1;
    static constexpr int NU = 7;
    void load(const float* u) { fractalIterations = u[0]; scaleFactor = u[1]; angles = vec3(u[2], u[3], u[4]); offset = u[5]; smoothen = (int)u[6]; }
    float opSmoothUnion(float d1, float d2, float k) {
        float h = clamp(0.5f + 0.5f * (d2 - d1) / k, 0.0f, 1.0f);
        return mix(d2, d1, h) - k * h * (1.0f - h);
    }
    float generalUnion(float d1, float d2, float k) {
        if (smoothen == 1) return opSmoothUnion(d1, d2, k);
        return min(d1, d2);
    }
    float sdf(vec3 position) {
        vec3 transformedPos = position;
        float minDist = 9999.0f;
        for (float i = 0.0f; i < fractalIterations; i++) {
            float combinedScaleFactor = pow(scaleFactor, i);
            vec3 tpos2 = transformedPos * combinedScaleFactor;
            minDist = generalUnion(minDist, sdBox(tpos2, vec3(1.0f, 0.1f, 0.1f) * (combinedScaleFactor)), combinedScaleFactor * 0.25f);
            transformedPos /= scaleFactor;
            transformedPos = abs(transformedPos) - vec3(1.0f, 0.1f, 0.1f) * vec3(offset);
            rotPair(transformedPos.x, transformedPos.y, angles.x);
            rotPair(transformedPos.y, transformedPos.z, angles.y);
            rotPair(transformedPos.x, transformedPos.z, angles.z);
        }
        return minDist;
    }
};

struct SceneRotationFractal : DefaultMaterials {                    // examples/rotation-fractal.glsl:16-35
    float fractalIterations = 14.0f, scaleFactor = 0.5f; vec3 angles = vec3(0.4f, 0.4f, 0.4f); float offset = 1.2f;
    static constexpr int NU = 6;
    void load(const float* u) { fractalIterations = u[0]; scaleFactor = u[1]; angles = vec3(u[2], u[3], u[4]); offset = u[5]; }
    float sdf(vec3 position) {
        vec3 transformedPos = position;
        for (float i = 0.0f; i < fractalIterations; i++) {
            transformedPos /= scaleFactor;
            transformedPos = abs(transformedPos) - vec3(offset);
            rotPair(transformedPos.x, transformedPos.y, angles.x);
            rotPair(transformedPos.y, transformedPos.z, angles.y);
            rotPair(transformedPos.x, transformedPos.z, angles.z);
        }
        float combinedScaleFactor = pow(scaleFactor, round(fractalIterations));
        transformedPos *= combinedScaleFactor;
        return sdBox(transformedPos, vec3(combinedScaleFactor));
    }
};

struct SceneSphereGrid : DefaultMaterials {                         // dist/examples/sphere-grid.glsl
    static constexpr int NU = 0;
    void load(const float*) {}
    vec3 sceneDiffuseColor(vec3 position) { if (length(position) > 35.0f) return vec3(0.0f); return vec3(0.5f); }
    vec3 sceneSpecularColor(vec3 position) { if (length(position) > 35.0f) return vec3(0.0f); return vec3(0.9f); }
    float sceneSpecularRoughness(vec3) { return 0.01f; }
    vec3 sceneEmission(vec3 position) {                             // sphere-grid.glsl:36-40 (.x, floor 0.0)
        float d = max(normalize(position).x, 0.0f);
        vec3 brightColor = vec3(0.7f, 0.8f, 1.0f) * d * 1.0f;
        return (length(position) > 36.0f) ? (brightColor * 2.00f) : vec3(0.0f);
    }
    float sd_sphere(vec3 p, float radius, vec3 position) { return length(p - position) - radius; }
    float sdf(vec3 p) {
        vec3 repeat = mod(p + 1.0f, vec3(2.0f)) - 1.0f;
        return sd_sphere(repeat, 0.4f, vec3(0.0f));
    }
};

struct SceneInlineDefault : DefaultMaterials {                      // src/index.tsx:374-388 (placeholder scene)
    static constexpr int NU = 0;
    void load(const float*) {}
    float sdf(vec3 position) {
        float minDist = 9999.9f;
        for (float i = -1.0f; i < 10.0f; i++) {
            float sf = pow(0.3333333333333f, i);
            vec3 d = abs(mod(position + vec3(0.5f * sf), sf) - vec3(sf / 2.0f)) - vec3(sf / 3.0f);
            float dist = length(d) - 0.21f * sf;
            minDist = min(dist, minDist);
        }
        minDist = max(length(position) - 5.0f, -minDist);
        return minDist;
    }
};

// Synthetic divergence-stress scene of BASELINE.json config 4 (NOT in the reference): power-8
// Mandelbulb distance estimator with in-DE bailout.  Mirrors scenes/mandelbulb.glsl.
// g_de_iterations: trips of the DE loop on this thread (workload analysis only - bench.py prices an SDF evaluation of
// config 4 by the iterations it runs; read with orc_de_iterations_reset)
static thread_local unsigned long long g_de_iterations = 0;
struct SceneMandelbulb : DefaultMaterials {
    float power = 8.0f, bailout = 2.0f, maxIterations = 12.0f;
    static constexpr int NU = 3;
    void load(const float* u) { power = u[0]; bailout = u[1]; maxIterations = u[2]; }
    float sdf(vec3 position) {
        vec3 z = position;
        float dr = 1.0f;
        float r = 0.0f;
        for (float i = 0.0f; i < maxIterations; i++) {
            r = length(z);
            if (r > bailout) break;
            g_de_iterations++;
            float theta = acos(z.z / r);
            float phi = atan(z.y, z.x);
            dr = pow(r, power - 1.0f) * power * dr + 1.0f;
            float zr = pow(r, power);
            theta = theta * power;
            phi = phi * power;
            z = zr * vec3(sin(theta) * cos(phi), sin(phi) * sin(theta), cos(theta));
            z += position;
        }
        return 0.5f * log(r) * r / dr;
    }
};

// ------------------------------------------------------------------------------------------
// The fragment shader, one invocation per pixel-sample.
// ------------------------------------------------------------------------------------------
struct Accum {            // one pixel of the three accumulators + the fp32 depth plane
    vec4 color;           // RGBA32F
    vec4 normalAndDofRadius;  // RGBA16F (stored as half)
    vec4 albedoAndDepth;      // RGBA16F (stored as half)
};

template <class Scene>
struct Frag {
    const OrcUniforms& U;
    Scene& S;
    vec2 texcoord;
    int W, H;
    float seed = 0.0f;                                              // raymarcher.frag:78
    unsigned long long sdfEvals = 0;

    // outputs (H6: outputs a branch does not write are 0 -> "keep previous" is NOT implied;
    // the caller stores whatever main() leaves here)
    vec4 fragColor, normalAndDofRadius, albedoAndDepth;
    bool wroteAux = false;
    float hitDepth = 0.0f;                                          // fp32 depth before fp16 storage (H5)
    // trace of the last main() call, for the numpy cross-check (tests/test_oracle_numpy.py)
    vec3 trOrigin, trDir, trEnd;
    float trDeltaZ = 0.0f, trStepsTaken = 0.0f, trJitterX = 0.0f, trJitterY = 0.0f;

    // event log of the full branch, for the float64 numpy restatement (tests/test_oracle_numpy_full.py):
    // records [tag, v0, v1, ...] per event; tags are listed at orc_trace_full_pixel
    std::vector<float>* trace = nullptr;
    void tr(float tag, std::initializer_list<float> v) {
        if (!trace) return;
        trace->push_back(tag);
        for (float x : v) trace->push_back(x);
    }
    void tr3(float tag, const vec3& a) { tr(tag, {a.x, a.y, a.z}); }

    Frag(const OrcUniforms& u, Scene& s, int w, int h) : U(u), S(s), W(w), H(h) {}

    const float PHI = 1.61803398874989484820459f;                   // raymarcher.frag:44
    const float PI = 3.141592f;                                     // raymarcher.frag:79

    float sdf(vec3 p) { sdfEvals++; return S.sdf(p); }
    float trSdf(vec3 p) { const float v = sdf(p); tr(13.0f, {v, p.x, p.y, p.z}); return v; }

    float gold_noise(vec2 xy, float sd) {                           // raymarcher.frag:46-49
        return fract(tan(distance(xy * PHI, xy) * sd) * xy.x);
    }
    vec2 boxMullerTransform() {                                     // raymarcher.frag:80-89
        seed += 0.123123213f;
        float u1 = gold_noise(texcoord * 1000.0f, fract(U.randNoise[0] + seed));
        seed += 0.123123213f;
        float u2 = gold_noise(texcoord * 1000.0f, fract(U.randNoise[1] + seed));
        float twoPiU2 = 2.0f * PI * u2;
        float c = cos(twoPiU2);
        float s = sin(twoPiU2);
        tr(2.0f, {u1, u2});
        return sqrt(-2.0f * log(u1)) * vec2(c, s);
    }
    float uniformSample() {                                         // raymarcher.frag:91-94
        seed += 0.131223f;
        const float v = gold_noise(texcoord * 1000.0f, fract(U.randNoise[0] + seed));
        tr(1.0f, {v});
        return v;
    }
    vec3 sphereSample() {                                           // raymarcher.frag:96-101 (args left to right)
        vec2 a = boxMullerTransform();
        float b = boxMullerTransform().x;
        return normalize(vec3(a, b));
    }
    vec3 rodrigues(vec3 v, vec3 k, float theta) {                   // raymarcher.frag:61-65
        float cosTheta = cos(theta);
        float sinTheta = sqrt(1.0f - cosTheta * cosTheta);
        return v * cosTheta + cross(k, v) * sinTheta + k * dot(k, v) * (1.0f - cosTheta);
    }
    float invExpDist(float x, float lambda) { return -log(1.0f - x) / lambda; }   // :148-150
    vec3 sceneNormal(vec3 position, float delta) {                  // raymarcher.frag:153-160
        float sdfAtPos = sdf(position);
        float nx = sdf(position + vec3(delta, 0, 0)) - sdfAtPos;
        float ny = sdf(position + vec3(0, delta, 0)) - sdfAtPos;
        float nz = sdf(position + vec3(0, 0, delta)) - sdfAtPos;
        return normalize(vec3(nx, ny, nz));
    }
    vec3 castRay(vec3 rayPosition, vec3 rayDirection, float steps) {  // raymarcher.frag:163-170
        for (float i = 0.0f; i < steps; i++) {
            float sdfNow = sdf(rayPosition);
            rayPosition = fmaV(rayDirection, sdfNow, rayPosition);   // p + d*s contracted to one fma per component (pinned)
        }
        return rayPosition;
    }
    float schlick(float cosTheta, float n1, float n2) {             // raymarcher.frag:172-175
        float r0 = pow((n1 - n2) / (n1 + n2), 2.0f);
        return r0 + (1.0f - r0) * pow(1.0f - cosTheta, 5.0f);
    }

    mat4 rotationMatrix() const {
        const float* r = U.rotation;
        return mat4(r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7], r[8], r[9], r[10], r[11], r[12], r[13], r[14], r[15]);
    }

    // `prev` = this pixel's texels of the three previous-sample textures (NEAREST at own centre)
    void main(const Accum& prev) {                                  // raymarcher.frag:178-387
        const vec3 position(U.position[0], U.position[1], U.position[2]);
        const mat4 rotation = rotationMatrix();
        vec3 rayDirection(0.0f), rayPosition(0.0f);   // an unknown cameraMode leaves them undefined in GLSL
        float r0 = uniformSample();
        float r1 = uniformSample();
        vec2 randomDirectionOffset = vec2(r0, r1) / vec2((float)W, (float)H) * 1.0f;     // :182-183
        vec2 texcoord2 = texcoord + randomDirectionOffset;
        float deltaZ = 1.0f;
        if (U.cameraMode == 0) {                                    // :186-193
            vec3 dofOffset = sphereSample() * U.dofAmount;
            rayPosition = position + dofOffset;
            vec2 projectionPlanePosition = (texcoord2.xy * 2.0f - 1.0f) * vec2(U.aspect, 1.0f) * tan(U.fov / 2.0f);
            vec3 rayDirectionNotNormalized = (rotation * vec4(projectionPlanePosition + randomDirectionOffset, 1.0f, 0.0f)).xyz;
            vec3 rayDirectionGoal = rayDirectionNotNormalized * U.dofFocalPlaneDistance;
            deltaZ = 1.0f / length(vec3(projectionPlanePosition, 1.0f));
            rayDirection = normalize(rayDirectionGoal - dofOffset);
        } else if (U.cameraMode == 1) {                             // :194-196
            rayDirection = normalize(vec3((rotation * vec4(0.0f, 0.0f, 1.0f, 0.0f)).xyz));
            rayPosition = position + vec3((rotation * vec4((texcoord2.xy - vec2(0.5f)) * vec2(U.aspect, 1.0f) * U.fov, 0.0f, 0.0f)).xyz);
        } else if (U.cameraMode == 2) {                             // :197-205
            vec2 angles = (texcoord2 - vec2(0.5f, 0.5f)) * vec2(2.0f * PI, PI);
            float cx = cos(angles.x), cy = cos(angles.y), sy = sin(angles.y), sx = sin(angles.x);
            rayDirection = vec3((rotation * vec4(cx * cy, sy, sx * cy, 0.0f)).xyz);
            rayPosition = position;
        }

        trOrigin = rayPosition; trDir = rayDirection; trDeltaZ = deltaZ;
        tr(3.0f, {rayPosition.x, rayPosition.y, rayPosition.z, rayDirection.x, rayDirection.y, rayDirection.z});
        trJitterX = randomDirectionOffset.x; trJitterY = randomDirectionOffset.y;
        if (U.renderMode == 1) {                                    // preview branch :207-244
            float stepsTaken = 0.0f;
            float depth = 0.0f;
            const float n = U.raymarchingStepCountsArray[0];
            for (float i = 0.0f; i < n; i++) {
                float sdfNow = sdf(rayPosition);
                if (sdfNow < 100000000000.0f) {
                    rayPosition = fmaV(rayDirection, sdfNow, rayPosition);   // contracted (pinned)
                    depth = g_fma(deltaZ, sdfNow, depth);
                }
                if (sdfNow > 0.0001f) stepsTaken = i;
            }
            vec3 outColor = (S.sceneDiffuseColor(rayPosition) + S.sceneSpecularColor(rayPosition)) * (1.0f - stepsTaken / n)
                            + S.sceneEmission(rayPosition);
            vec4 col;
            if (U.blendMode == 0) col = mix(vec4(outColor, 1.0f), prev.color, U.blendWithPreviousFactor);
            else col = prev.color + vec4(outColor, 0.0f) * U.exposure;
            if (U.showDofFocalPlane != 0) {                         // :233-242
                float focusAmount = abs(depth - U.dofFocalPlaneDistance) / depth;
                if (focusAmount < U.dofFocalPlaneDistance * 0.005f)
                    fragColor = vec4(1.0f, mod(vec2(col.yz) + vec2(0.5f), vec2(1.0f)), 1.0f);
                else fragColor = col;
            } else fragColor = col;
            hitDepth = depth;
            trEnd = rayPosition; trStepsTaken = stepsTaken;
            return;                                                 // attachments 1,2 unwritten (H6)
        }

        vec3 currentAlbedo = vec3(1.0f);                            // :247-249
        vec3 currentLight = vec3(0.0f);
        float probabilityFactor = 1.0f;

        for (float i = 0.0f; i < U.reflections; i++) {              // :252
            vec3 oldRayPosition = rayPosition;
            tr(10.0f, {i, oldRayPosition.x, oldRayPosition.y, oldRayPosition.z, rayDirection.x, rayDirection.y, rayDirection.z});
            rayPosition = castRay(rayPosition, rayDirection, U.raymarchingStepCountsArray[(int)i]);
            tr3(11.0f, rayPosition);
            float pathLength = invExpDist(uniformSample(), U.fogDensity);
            currentLight += currentAlbedo * S.sceneEmission(rayPosition);
            vec3 normal = sceneNormal(rayPosition, 0.00001f);
            tr3(12.0f, normal);
            float sss = S.sceneSubsurfaceScattering(rayPosition);
            float subsurfVolumetricSample = -1.0f / sss * log(1.0f - uniformSample());      // :266
            vec3 subsurfScatterDirection = normalize(mix(rayDirection, normalize(sphereSample()), 1.0f));
            subsurfScatterDirection *= -sign(dot(subsurfScatterDirection, normal));
            vec3 subsurfScatterFinalPos = rayPosition + subsurfScatterDirection * subsurfVolumetricSample;

            vec3 prevAlbedo = currentAlbedo;
            vec3 diffuseCol = S.sceneDiffuseColor(rayPosition);
            vec3 specularCol = S.sceneSpecularColor(rayPosition);
            vec3 prevRayDirection = rayDirection;

            if (distance(oldRayPosition, rayPosition) > pathLength || any(isinf(rayPosition)) || any(isnan(rayPosition))) {  // :278
                rayPosition = oldRayPosition + min(pathLength, 1000000.0f) * rayDirection;
                rayDirection = sphereSample();
                diffuseCol = vec3(1.0f);
                specularCol = vec3(1.0f);
                prevRayDirection = rayDirection;
            } else if (trSdf(subsurfScatterFinalPos) > 0.001f) {    // :284-288
                currentAlbedo *= S.sceneSubsurfaceScatteringColor(rayPosition);
                rayPosition = subsurfScatterFinalPos;
                rayDirection = normalize(mix(rayDirection, sphereSample(), 1.0f));
            } else {
                float diffuseBrightness = length(diffuseCol);       // :293-297
                float specularBrightness = length(specularCol);
                float probFactor = (diffuseBrightness > specularBrightness)
                                       ? (1.0f - specularBrightness / diffuseBrightness / 2.0f)
                                       : (diffuseBrightness / specularBrightness / 2.0f);
                if (uniformSample() < probFactor) {                 // diffuse :300-319
                    probabilityFactor *= 1.0f - probFactor;
                    currentAlbedo *= diffuseCol;
                    vec3 newDir = sphereSample();
                    rayDirection = sign(dot(normal, newDir)) * newDir;
                } else {                                            // specular :322-330
                    probabilityFactor *= probFactor;
                    currentAlbedo *= specularCol * clamp(schlick(-dot(rayDirection, normal), 1.0f, S.sceneIOR(rayPosition)), 0.0f, 1.0f);
                    vec3 randVec = sphereSample();
                    rayDirection = reflect(rayDirection, normal);
                    vec3 axis = normalize(cross(randVec, rayDirection));
                    float rough = S.sceneSpecularRoughness(rayPosition);
                    float us = uniformSample();
                    rayDirection = rodrigues(rayDirection, axis, rough * us);
                }
            }
            rayPosition += rayDirection * 0.001f;                   // :334
            tr(14.0f, {rayPosition.x, rayPosition.y, rayPosition.z, rayDirection.x, rayDirection.y, rayDirection.z,
                       currentAlbedo.x, currentAlbedo.y, currentAlbedo.z, currentLight.x, currentLight.y, currentLight.z});

            if (i == 0.0f) {                                        // :336-352
                float depth = clamp(distance(rayPosition, position), 0.00001f, 100000000.0f);
                if (isinf(normal.r) || isnan(normal.r)) normal.r = 0.0f;
                if (isinf(normal.g) || isnan(normal.g)) normal.g = 0.0f;
                if (isinf(normal.b) || isnan(normal.b)) normal.b = 0.0f;
                float dofRadius = clamp(U.dofAmount * abs(depth - U.dofFocalPlaneDistance) / depth, 0.0f, 1.0f);
                if (isinf(dofRadius) || isnan(dofRadius)) dofRadius = 0.0f;
                normalAndDofRadius = vec4(normal, dofRadius) + prev.normalAndDofRadius;
                albedoAndDepth = vec4(currentAlbedo, depth) + prev.albedoAndDepth;
                wroteAux = true;
                hitDepth = depth;
                tr(15.0f, {normalAndDofRadius.x, normalAndDofRadius.y, normalAndDofRadius.z, normalAndDofRadius.w,
                           albedoAndDepth.x, albedoAndDepth.y, albedoAndDepth.z, albedoAndDepth.w});
            }

            for (int j = 0; j < U.lightCount; j++) {                // :354-373
                vec3 lightPosition(U.lightPositions[3 * j], U.lightPositions[3 * j + 1], U.lightPositions[3 * j + 2]);
                vec3 lightColor(U.lightColors[3 * j], U.lightColors[3 * j + 1], U.lightColors[3 * j + 2]);
                float lightSize = U.lightSizes[j];
                vec3 adjustedLightPosition = lightPosition + sphereSample() * lightSize;
                vec3 directionToLight = normalize(adjustedLightPosition - rayPosition);
                vec3 result = castRay(rayPosition, directionToLight, U.raymarchingStepCountsArray[(int)i]);
                tr(16.0f, {(float)j, result.x, result.y, result.z});
                if (distance(result, adjustedLightPosition) >= distance(rayPosition, adjustedLightPosition)) {
                    float r = max(0.0f, dot(directionToLight, reflect(prevRayDirection, normal)));
                    float roughness = S.sceneSpecularRoughness(rayPosition);
                    currentLight += prevAlbedo * diffuseCol * lightColor * max(0.0f, dot(directionToLight, normal))
                                    + prevAlbedo * specularCol * lightColor * roughness * roughness
                                          / (3.14159265f * pow(r * r * (roughness * roughness - 1.0f) + 1.0f, 2.0f));
                }
                tr3(17.0f, currentLight);
            }
        }
        (void)probabilityFactor;   // computed by the reference, never read (SURVEY.md a7)

        if (U.blendMode == 0) fragColor = mix(vec4(currentLight * U.exposure, 1.0f), prev.color, U.blendWithPreviousFactor);   // :379-387
        else fragColor = vec4(currentLight * U.exposure, 1.0f) + prev.color;
        tr(18.0f, {fragColor.x, fragColor.y, fragColor.z, fragColor.w});
    }
};

// ------------------------------------------------------------------------------------------
// Drivers
// ------------------------------------------------------------------------------------------
static std::atomic<unsigned long long> g_sdf_evals{0};

template <class Scene>
static int render_sample_t(const float* custom, int ncustom, const OrcUniforms* U, int W, int H,
                           int sx, int sy, int sw, int sh, float* color, uint16_t* nd, uint16_t* ad,
                           float* depth, int nthreads) {
    if (ncustom != 0 && ncustom != Scene::NU) return -2;
    // GL scissor box (x, y, width, height), clipped to the framebuffer.  The reference passes
    // (x1, y1, x2, y2) to gl.scissor (RenderJobExecutor.tsx:182); callers reproduce that quirk.
    long long x0 = sx, y0 = sy, x1 = (long long)sx + sw, y1 = (long long)sy + sh;
    if (x0 < 0) x0 = 0; if (y0 < 0) y0 = 0; if (x1 > W) x1 = W; if (y1 > H) y1 = H;
    if (nthreads < 1) nthreads = 1;
    std::atomic<int> nextRow{(int)y0};
    auto worker = [&]() {
        Scene S;
        if (ncustom) S.load(custom);
        unsigned long long evals = 0;
        for (;;) {
            int py = nextRow.fetch_add(1);
            if (py >= y1) break;
            for (int px = (int)x0; px < x1; px++) {
                size_t idx = (size_t)py * W + px;
                Frag<Scene> f(*U, S, W, H);
                f.texcoord = vec2(((float)px + 0.5f) / (float)W, ((float)py + 0.5f) / (float)H);   // raymarcher.vert:10
                Accum prev;
                prev.color = vec4(color[4 * idx], color[4 * idx + 1], color[4 * idx + 2], color[4 * idx + 3]);
                prev.normalAndDofRadius = vec4(f16_to_f32(nd[4 * idx]), f16_to_f32(nd[4 * idx + 1]), f16_to_f32(nd[4 * idx + 2]), f16_to_f32(nd[4 * idx + 3]));
                prev.albedoAndDepth = vec4(f16_to_f32(ad[4 * idx]), f16_to_f32(ad[4 * idx + 1]), f16_to_f32(ad[4 * idx + 2]), f16_to_f32(ad[4 * idx + 3]));
                f.main(prev);
                evals += f.sdfEvals;
                for (int c = 0; c < 4; c++) color[4 * idx + c] = f.fragColor[c];
                // H6: an attachment the shader did not write becomes 0 (draw writes all three
                // attachments; the blit then copies curr -> prev).
                for (int c = 0; c < 4; c++) {
                    nd[4 * idx + c] = f.wroteAux ? f32_to_f16(f.normalAndDofRadius[c]) : 0;
                    ad[4 * idx + c] = f.wroteAux ? f32_to_f16(f.albedoAndDepth[c]) : 0;
                }
                if (depth) depth[idx] = f.hitDepth;
            }
        }
        g_sdf_evals += evals;
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nthreads; t++) th.emplace_back(worker);
    worker();
    for (auto& t : th) t.join();
    return 0;
}

template <class Scene>
static float sdf_t(const float* custom, int ncustom, float x, float y, float z) {
    Scene S;
    if (ncustom == Scene::NU && ncustom) S.load(custom);
    return S.sdf(vec3(x, y, z));
}

template <class Scene>
static void materials_t(const float* custom, int ncustom, float x, float y, float z, float* out17) {
    Scene S;
    if (ncustom == Scene::NU && ncustom) S.load(custom);
    vec3 p(x, y, z);
    vec3 a = S.sceneDiffuseColor(p), b = S.sceneSpecularColor(p), c = S.sceneSubsurfaceScatteringColor(p), e = S.sceneEmission(p);
    float o[17] = {a.x, a.y, a.z, b.x, b.y, b.z, S.sceneSpecularRoughness(p), S.sceneSubsurfaceScattering(p), c.x, c.y, c.z, S.sceneIOR(p), e.x, e.y, e.z, S.sdf(p), 0.0f};
    memcpy(out17, o, sizeof(o));
}

// Analysis helper (kernel design, DESIGN.md): for every pixel of a preview-mode sample, the first
// march iteration after which the ray state is a fixed point (p + d*s == p bitwise, or the
// s >= 1e11 freeze of raymarcher.frag:212) - i.e. the number of SDF evaluations a bit-exact
// early-out kernel has to execute.  out[W*H] int32.
template <class Scene>
static void exit_steps_t(const float* custom, int ncustom, const OrcUniforms* U, int W, int H, int* out) {
    Scene S;
    if (ncustom == Scene::NU && ncustom) S.load(custom);
    for (int py = 0; py < H; py++) for (int px = 0; px < W; px++) {
        Frag<Scene> f(*U, S, W, H);
        f.texcoord = vec2(((float)px + 0.5f) / (float)W, ((float)py + 0.5f) / (float)H);
        // camera set-up only: run main() with zero steps by copying the uniforms
        OrcUniforms U0 = *U; U0.raymarchingStepCountsArray[0] = 0.0f; U0.renderMode = 1;
        Frag<Scene> g(U0, S, W, H);
        g.texcoord = f.texcoord;
        // replicate the set-up of main() for cameraMode 0 (the analysis is only used for that mode)
        float r0 = g.uniformSample(), r1 = g.uniformSample();
        vec2 rdo = vec2(r0, r1) / vec2((float)W, (float)H) * 1.0f;
        vec2 tc2 = g.texcoord + rdo;
        vec3 position(U->position[0], U->position[1], U->position[2]);
        vec3 dofOffset = g.sphereSample() * U->dofAmount;
        vec3 p = position + dofOffset;
        vec2 ppp = (vec2(tc2.xy) * 2.0f - 1.0f) * vec2(U->aspect, 1.0f) * tan(U->fov / 2.0f);
        vec3 dn = vec3((g.rotationMatrix() * vec4(ppp + rdo, 1.0f, 0.0f)).xyz);
        vec3 d = normalize(dn * U->dofFocalPlaneDistance - dofOffset);
        int n = (int)U->raymarchingStepCountsArray[0], e = n;
        for (int i = 0; i < n; i++) {
            float s = S.sdf(p);
            if (!(s < 100000000000.0f)) { e = i + 1; break; }
            vec3 q = fmaV(d, s, p);
            if (rmx::f2i(q.x) == rmx::f2i(p.x) && rmx::f2i(q.y) == rmx::f2i(p.y) && rmx::f2i(q.z) == rmx::f2i(p.z)) { e = i + 1; break; }
            p = q;
        }
        out[(size_t)py * W + px] = e;
    }
}

// Trace of one preview-mode pixel for the independent numpy cross-check: out[17] = origin xyz,
// direction xyz, deltaZ, jitter xy, end position xyz, stepsTaken, depth, rgb of the new sample.
template <class Scene>
static void trace_pixel_t(const float* custom, int ncustom, const OrcUniforms* U, int W, int H, int px, int py, float* out) {
    Scene S;
    if (ncustom == Scene::NU && ncustom) S.load(custom);
    Frag<Scene> f(*U, S, W, H);
    f.texcoord = vec2(((float)px + 0.5f) / (float)W, ((float)py + 0.5f) / (float)H);
    Accum prev;
    prev.color = vec4(0.0f); prev.normalAndDofRadius = vec4(0.0f); prev.albedoAndDepth = vec4(0.0f);
    f.main(prev);
    float o[17] = {f.trOrigin.x, f.trOrigin.y, f.trOrigin.z, f.trDir.x, f.trDir.y, f.trDir.z, f.trDeltaZ, f.trJitterX, f.trJitterY,
                   f.trEnd.x, f.trEnd.y, f.trEnd.z, f.trStepsTaken, f.hitDepth, f.fragColor.x, f.fragColor.y, f.fragColor.z};
    memcpy(out, o, sizeof(o));
}
#define ORC_SCENES(X)                      \
    X("guide", SceneGuide)                 \
    X("fractal1", SceneFractal1)           \
    X("menger-sponge", SceneMenger)        \
    X("tree", SceneTree)                   \
    X("smooth-tree", SceneSmoothTree)      \
    X("rotation-fractal", SceneRotationFractal) \
    X("sphere-grid", SceneSphereGrid)      \
    X("inline-default", SceneInlineDefault) \
    X("mandelbulb", SceneMandelbulb)

// Event log of one full-mode (renderMode 0) invocation on zeroed previous texels, for the float64 numpy
// restatement of the path tracer.  Events are [tag, payload...]:
//   1 uniformSample() -> v            2 boxMullerTransform() inputs -> u1, u2      3 camera ray: origin, direction
//  10 bounce i starts: i, oldRayPosition, rayDirection        11 castRay result           12 sceneNormal
//  13 subsurface probe: sdf value, position                   14 after :334: rayPosition, rayDirection, currentAlbedo, currentLight
//  15 bounce-0 attachments: normalAndDofRadius, albedoAndDepth
//  16 light j: j, shadow castRay result                      17 currentLight after light j
//  18 fragColor
// Returns the number of floats the log holds (the first min(n, cap) are written to out).
template <class Scene>
static int trace_full_t(const float* custom, int ncustom, const OrcUniforms* U, int W, int H, int px, int py, float* out, int cap) {
    Scene S;
    if (ncustom == Scene::NU && ncustom) S.load(custom);
    Frag<Scene> f(*U, S, W, H);
    std::vector<float> log;
    f.trace = &log;
    f.texcoord = vec2(((float)px + 0.5f) / (float)W, ((float)py + 0.5f) / (float)H);
    Accum prev;
    prev.color = vec4(0.0f); prev.normalAndDofRadius = vec4(0.0f); prev.albedoAndDepth = vec4(0.0f);
    f.main(prev);
    for (size_t i = 0; i < log.size() && (int)i < cap; i++) out[i] = log[i];
    return (int)log.size();
}
extern "C" {

int orc_abi_version() { return 1; }
int orc_uniforms_size() { return (int)sizeof(OrcUniforms); }

int orc_scene_count() {
    int n = 0;
#define X(name, T) n++;
    ORC_SCENES(X)
#undef X
    return n;
}
const char* orc_scene_name(int i) {
    int n = 0;
#define X(name, T) if (n++ == i) return name;
    ORC_SCENES(X)
#undef X
    return nullptr;
}
int orc_scene_num_uniform_floats(const char* scene) {
#define X(name, T) if (!strcmp(scene, name)) return T::NU;
    ORC_SCENES(X)
#undef X
    return -1;
}

// One raymarch "draw" + blit of the reference (RenderJobExecutor.tsx:299-326) over the GL
// scissor box (sx, sy, sw, sh).  color: W*H*4 fp32, nd/ad: W*H*4 binary16 bit patterns, depth:
// optional W*H fp32 (this repo's extension: fp32 hit depth of the latest sample, SURVEY.md H5).
// Row 0 is the bottom row (GL convention).  Returns 0, -1 unknown scene, -2 bad uniform count.
int orc_render_sample(const char* scene, const float* custom, int ncustom, const OrcUniforms* U, int W, int H,
                      int sx, int sy, int sw, int sh, float* color, uint16_t* nd, uint16_t* ad, float* depth,
                      int nthreads) {
#define X(name, T) if (!strcmp(scene, name)) return render_sample_t<T>(custom, ncustom, U, W, H, sx, sy, sw, sh, color, nd, ad, depth, nthreads);
    ORC_SCENES(X)
#undef X
    return -1;
}

float orc_sdf(const char* scene, const float* custom, int ncustom, float x, float y, float z) {
#define X(name, T) if (!strcmp(scene, name)) return sdf_t<T>(custom, ncustom, x, y, z);
    ORC_SCENES(X)
#undef X
    return rmx::f_nan();
}

// out17 = diffuse rgb, specular rgb, roughness, subsurface, subsurfaceColor rgb, IOR, emission rgb, sdf, 0
int orc_materials(const char* scene, const float* custom, int ncustom, float x, float y, float z, float* out17) {
#define X(name, T) if (!strcmp(scene, name)) { materials_t<T>(custom, ncustom, x, y, z, out17); return 0; }
    ORC_SCENES(X)
#undef X
    return -1;
}

// orc_materials at n points: xyz = n * 3 floats, out = n * 17 floats
int orc_materials_n(const char* scene, const float* custom, int ncustom, const float* xyz, int n, float* out) {
    for (int i = 0; i < n; i++) {
        const int st = orc_materials(scene, custom, ncustom, xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], out + 17 * (size_t)i);
        if (st != 0) return st;
    }
    return 0;
}

unsigned long long orc_sdf_evals_reset() { return g_sdf_evals.exchange(0); }

float orc_sdbox(float px, float py, float pz, float bx, float by, float bz) { return sdBox(vec3(px, py, pz), vec3(bx, by, bz)); }

float orc_gold_noise(float x, float y, float sd) {
    OrcUniforms U{};
    SceneSphereGrid S;
    Frag<SceneSphereGrid> f(U, S, 1, 1);
    return f.gold_noise(vec2(x, y), sd);
}

// seed sequence probe: returns the first n uniformSample() values of a pixel
void orc_uniform_samples(float rnx, float rny, int px, int py, int W, int H, int n, float* out) {
    OrcUniforms U{};
    U.randNoise[0] = rnx; U.randNoise[1] = rny;
    SceneSphereGrid S;
    Frag<SceneSphereGrid> f(U, S, W, H);
    f.texcoord = vec2(((float)px + 0.5f) / (float)W, ((float)py + 0.5f) / (float)H);
    for (int i = 0; i < n; i++) out[i] = f.uniformSample();
}

// Halton sequence, Halton.tsx:1-19 (double arithmetic like JavaScript numbers).
void orc_halton(int b, int n, double* out) {
    double nn = 0, d = 1;
    for (int k = 0; k < n; k++) {
        double x = d - nn;
        if (x == 1) { nn = 1; d *= b; }
        else { double y = d; while (x <= y) y /= b; nn = (b + 1) * y - x; }
        out[k] = nn / d;
    }
}

// DE-loop trips of the Mandelbulb scene executed on the calling thread since the last call (orc_preview_exit_steps runs
// on the calling thread: evaluations = sum of its output, iterations = this counter)
unsigned long long orc_de_iterations_reset() { unsigned long long v = g_de_iterations; g_de_iterations = 0; return v; }

int orc_preview_exit_steps(const char* scene, const float* custom, int ncustom, const OrcUniforms* U, int W, int H, int* out) {
#define X(name, T) if (!strcmp(scene, name)) { exit_steps_t<T>(custom, ncustom, U, W, H, out); return 0; }
    ORC_SCENES(X)
#undef X
    return -1;
}

int orc_trace_full_pixel(const char* scene, const float* custom, int ncustom, const OrcUniforms* U, int W, int H, int px, int py, float* out, int cap) {
#define X(name, T) if (!strcmp(scene, name)) return trace_full_t<T>(custom, ncustom, U, W, H, px, py, out, cap);
    ORC_SCENES(X)
#undef X
    return -1;
}

int orc_trace_pixel(const char* scene, const float* custom, int ncustom, const OrcUniforms* U, int W, int H, int px, int py, float* out17) {
#define X(name, T) if (!strcmp(scene, name)) { trace_pixel_t<T>(custom, ncustom, U, W, H, px, py, out17); return 0; }
    ORC_SCENES(X)
#undef X
    return -1;
}

// GLSL built-in probe used by the device-vs-host consistency test: op id -> f(a, b)
float orc_builtin(int op, float a, float b) {
    switch (op) {
        case 0: return sin(a); case 1: return cos(a); case 2: return tan(a); case 3: return pow(a, b);
        case 4: return exp(a); case 5: return log(a); case 6: return exp2(a); case 7: return log2(a);
        case 8: return sqrt(a); case 9: return inversesqrt(a); case 10: return mod(a, b); case 11: return fract(a);
        case 12: return floor(a); case 13: return round(a); case 14: return min(a, b); case 15: return max(a, b);
        case 16: return atan(a, b); case 17: return asin(a); case 18: return acos(a); case 19: return atan(a);
        case 20: return a / b; case 21: return sinh(a); case 22: return cosh(a); case 23: return tanh(a);
        case 24: return sign(a); case 25: return ceil(a); case 26: return trunc(a); case 27: return roundEven(a);
        case 28: return smoothstep(0.0f, b, a); case 29: return mix(a, b, 0.3f);
        case 30: return asinh(a); case 31: return acosh(a); case 32: return atanh(a);
        default: return rmx::f_nan();
    }
}

uint16_t orc_f32_to_f16(float f) { return f32_to_f16(f); }
float orc_f16_to_f32(uint16_t h) { return f16_to_f32(h); }

// Present pass, display.frag:20-61 driven as index.tsx:25-59 (full-frame scissor).
// color: W*H*4 fp32; nd: W*H*4 binary16; out: W*H*4 bytes RGBA8, row 0 = bottom.
int orc_display(const float* color, const uint16_t* nd, int W, int H, float brightness, uint8_t* rgba, int nthreads) {
    if (nthreads < 1) nthreads = 1;
    std::atomic<int> nextRow{0};
    auto texel = [&](vec2 uv) -> vec4 {     // NEAREST + REPEAT (LoadRenderJobContext.tsx:43-48)
        float u = uv.x * (float)W, v = uv.y * (float)H;
        long long i = (long long)floor(u), j = (long long)floor(v);
        i %= W; if (i < 0) i += W;
        j %= H; if (j < 0) j += H;
        const float* c = color + 4 * ((size_t)j * W + (size_t)i);
        return vec4(c[0], c[1], c[2], c[3]);
    };
    auto worker = [&]() {
        const float PI_D = 3.1415926535f;                          // display.frag:9
        for (;;) {
            int py = nextRow.fetch_add(1);
            if (py >= H) break;
            for (int px = 0; px < W; px++) {
                size_t idx = (size_t)py * W + px;
                vec2 texcoord(((float)px + 0.5f) / (float)W, ((float)py + 0.5f) / (float)H);
                float ndw = f16_to_f32(nd[4 * idx + 3]) * brightness;             // display.frag:18
                float kernelSize = clamp(ndw * 200.0f, 0.0f, 16.0f);              // :20
                vec4 avgColorSample = vec4(0.0f);
                float sampleCount = 0.0f;
                for (float y = -kernelSize; y <= kernelSize; y++) {               // :42-50
                    for (float x = -kernelSize; x <= kernelSize; x++) {
                        vec2 offset = vec2(x, y);
                        vec2 texOffset = offset / vec2((float)W, (float)H);
                        float sigma = max(kernelSize, 1.0f) * 0.3f;
                        float factor = 1.0f / (2.0f * PI_D * sigma * sigma) * exp(-(dot(offset, offset) / (2.0f * sigma * sigma)));   // :11-13
                        sampleCount += factor;
                        avgColorSample += texel(texcoord + texOffset) * factor;
                    }
                }
                avgColorSample /= sampleCount;
                vec4 frag = pow(vec4(vec3(vec3(avgColorSample.xyz) * brightness), 1.0f), vec4(1.0f / 2.2f));   // :54
                for (int c = 0; c < 4; c++) {
                    float v = frag[c];
                    if (rmx::f_isnan(v)) v = 0.0f;
                    v = clamp(v, 0.0f, 1.0f);
                    rgba[4 * idx + c] = (uint8_t)(int)floor(v * 255.0f + 0.5f);   // unorm8 conversion
                }
            }
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nthreads; t++) th.emplace_back(worker);
    worker();
    for (auto& t : th) t.join();
    return 0;
}

}  // extern "C"
