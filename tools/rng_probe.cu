// Device side of the RNG fast-path checks (rm_math.h tan_ft_fast, sincos_ft_fast, log_ft_fast).
//
// As a program (nvcc -gencode arch=compute_100a,code=sm_100a, tests/test_rng_fast_paths_gpu.py builds it with
// --fmad=false and --fmad=true, the flags of the exact and the fast flavour): every float of each fast path's domain,
// plus specials, subnormals and binade edges of all signs and exponents, fast result against pinned result, bit for
// bit, on the GPU.  Prints one JSON line per function; exits 1 on any mismatch.
//
// The probe_* kernels are one call each, for the per-call SASS counts of tools/rng_sweep.py --sass.
#include <cstdint>
#include <cstdio>
#include <vector>

#include <cuda_runtime.h>

#include "rm_math.h"

extern "C" __global__ void probe_copy(const float* in, float* out) { out[threadIdx.x] = in[threadIdx.x]; }
extern "C" __global__ void probe_tan_pinned(const float* in, float* out) { out[threadIdx.x] = rmx::tan_ft(in[threadIdx.x]); }
extern "C" __global__ void probe_tan_fast(const float* in, float* out) { out[threadIdx.x] = rmx::tan_ft_fast(in[threadIdx.x]); }
extern "C" __global__ void probe_log_pinned(const float* in, float* out) { out[threadIdx.x] = rmx::log_ft(in[threadIdx.x]); }
extern "C" __global__ void probe_log_fast(const float* in, float* out) { out[threadIdx.x] = rmx::log_ft_fast(in[threadIdx.x]); }
extern "C" __global__ void probe_sincos_pinned(const float* in, float* out) {
    float s, c;
    rmx::sincos_ft(in[threadIdx.x], &s, &c);
    out[threadIdx.x] = s;
    out[threadIdx.x + 32] = c;
}
extern "C" __global__ void probe_sincos_fast(const float* in, float* out) {
    float s, c;
    rmx::sincos_ft_fast(in[threadIdx.x], &s, &c);
    out[threadIdx.x] = s;
    out[threadIdx.x + 32] = c;
}

__device__ __forceinline__ bool sameResult(int fn, float x) {
    if (fn == 1) {
        float s0, c0, s1, c1;
        rmx::sincos_ft(x, &s0, &c0);
        rmx::sincos_ft_fast(x, &s1, &c1);
        return __float_as_uint(s0) == __float_as_uint(s1) && __float_as_uint(c0) == __float_as_uint(c1);
    }
    const float want = fn == 0 ? rmx::tan_ft(x) : rmx::log_ft(x);
    const float got = fn == 0 ? rmx::tan_ft_fast(x) : rmx::log_ft_fast(x);
    return __float_as_uint(want) == __float_as_uint(got);
}

// floats lo .. hi-1 (bit patterns), or the n listed ones
__global__ void sweepKernel(int fn, uint32_t lo, uint32_t hi, const uint32_t* list, uint32_t n,
                            unsigned long long* mismatches, uint32_t* first) {
    const uint64_t count = list ? n : (uint64_t)hi - lo;
    unsigned long long bad = 0;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t b = list ? list[i] : (uint32_t)(lo + i);
        if (!sameResult(fn, __uint_as_float(b))) {
            bad++;
            atomicMin(first, b);
        }
    }
    if (bad) atomicAdd(mismatches, bad);
}

#define CK(x)                                                                     \
    do {                                                                          \
        cudaError_t e_ = (x);                                                     \
        if (e_ != cudaSuccess) {                                                  \
            std::fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e_));         \
            return 2;                                                             \
        }                                                                         \
    } while (0)

int main() {
    const char* names[3] = {"tan", "sincos", "log"};
    // fast domains as float bit ranges [lo, hi): tan [2^-126, 1024), sincos [+0, 8), log [2^-126, 1] (tools/rng_sweep.cpp)
    const uint32_t LO[3] = {0x00800000u, 0x00000000u, 0x00800000u};
    const uint32_t HI[3] = {0x44800000u, 0x41000000u, 0x3f800001u};
    std::vector<uint32_t> edges = {0x7fc00000u, 0xffc00000u, 0x7fffffffu, 0xffffffffu, 0x7f800001u, 0x7fa00000u};
    for (uint32_t sign = 0; sign < 2; sign++)
        for (uint32_t e = 0; e < 256; e++)
            for (uint32_t d : {0u, 1u, 2u, 3u, 0x400000u, 0x7ffffdu, 0x7ffffeu, 0x7fffffu}) edges.push_back((sign << 31 | e << 23) + d);
    uint32_t* dEdges;
    unsigned long long* dBad;
    uint32_t* dFirst;
    CK(cudaMalloc(&dEdges, edges.size() * 4));
    CK(cudaMalloc(&dBad, 8));
    CK(cudaMalloc(&dFirst, 4));
    CK(cudaMemcpy(dEdges, edges.data(), edges.size() * 4, cudaMemcpyHostToDevice));
    int bad = 0;
    for (int fn = 0; fn < 3; fn++)
        for (int pass = 0; pass < 2; pass++) {
            const unsigned long long zero = 0;
            const uint32_t none = 0xffffffffu;
            CK(cudaMemcpy(dBad, &zero, 8, cudaMemcpyHostToDevice));
            CK(cudaMemcpy(dFirst, &none, 4, cudaMemcpyHostToDevice));
            cudaEvent_t t0, t1;
            CK(cudaEventCreate(&t0));
            CK(cudaEventCreate(&t1));
            CK(cudaEventRecord(t0));
            if (pass == 0) sweepKernel<<<148 * 16, 256>>>(fn, LO[fn], HI[fn], nullptr, 0, dBad, dFirst);
            else sweepKernel<<<16, 256>>>(fn, 0, 0, dEdges, (uint32_t)edges.size(), dBad, dFirst);
            CK(cudaGetLastError());
            CK(cudaEventRecord(t1));
            CK(cudaEventSynchronize(t1));
            float ms = 0.0f;
            CK(cudaEventElapsedTime(&ms, t0, t1));
            unsigned long long nBad;
            uint32_t first;
            CK(cudaMemcpy(&nBad, dBad, 8, cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(&first, dFirst, 4, cudaMemcpyDeviceToHost));
            const unsigned long long n = pass == 0 ? (unsigned long long)HI[fn] - LO[fn] : edges.size();
            std::printf("{\"fn\": \"%s\", \"set\": \"%s\", \"checked\": %llu, \"mismatches\": %llu, \"first_mismatch\": \"0x%08x\", \"ms\": %.1f}\n",
                        names[fn], pass == 0 ? "domain" : "edges", n, nBad, first, ms);
            bad |= nBad != 0;
        }
    return bad;
}
