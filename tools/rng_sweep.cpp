// Host check of the RNG fast paths of rm_math.h (tan_ft_fast, sincos_ft_fast, log_ft_fast) against the pinned
// functions, built with the oracle's flags (g++ -O2 -ffp-contract=off -mfma) - the same binary64 operations the
// device runs.  tools/rng_sweep.py builds and drives it; tests/test_rng_fast_paths_cpu.py runs a strided subset.
//
//   rng_sweep tan|sincos|log STRIDE THREADS   every STRIDE-th float of the function's fast domain
//   rng_sweep edges                           specials, subnormals, binade edges of all signs and exponents
//
// Prints one JSON line: floats checked, results that differ from the pinned function (must be 0), fast-path
// fallbacks, and the largest |F - P| in ulps of P (F: the fast path's binary64 value, P: the pinned one).
#include <cinttypes>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "rm_math.h"

using namespace rmx;

namespace {

struct Stats {
    uint64_t checked = 0, mismatches = 0, fallbacks = 0;
    double maxUlps = 0.0;
    uint32_t firstMismatch = 0xffffffffu;
    void add(const Stats& o) {
        checked += o.checked;
        mismatches += o.mismatches;
        fallbacks += o.fallbacks;
        if (o.maxUlps > maxUlps) maxUlps = o.maxUlps;
        if (o.firstMismatch < firstMismatch) firstMismatch = o.firstMismatch;
    }
};

uint32_t fbits(float x) { uint32_t u; std::memcpy(&u, &x, 4); return u; }
float bitsf(uint32_t u) { float x; std::memcpy(&x, &u, 4); return x; }

// the binary64 values the pinned functions convert to float (tan_k and log_ft, term for term)
double tan_P(float x) {
    int q;
    const double r = trig_reduce<TrigTab>((double)x, &q);
    const double s = ksin<TrigTab>(r), c = kcos<TrigTab>(r);
    return (q & 1) ? -c / s : s / c;
}
double log_P(float x) { return dlog2_pos_k<LeTab>((double)x) * LeTab::at(14); }

double ulps(double F, double P) {
    if (F == P) return 0.0;
    const double ulp = ll2d(d2ll(P) & 0x7ff0000000000000LL) * 0x1p-52;
    return dabs(F - P) / ulp;
}

// one float: fast result against pinned result, bit for bit; in the fast domain also F against P
void check(int fn, uint32_t b, bool inDomain, Stats& st) {
    const float x = bitsf(b);
    bool same;
    if (fn == 1) {
        float s0, c0, s1, c1;
        sincos_ft(x, &s0, &c0);
        sincos_ft_fast(x, &s1, &c1);
        same = fbits(s0) == fbits(s1) && fbits(c0) == fbits(c1);
    } else {
        const float want = fn == 0 ? tan_ft(x) : log_ft(x);
        const float got = fn == 0 ? tan_ft_fast(x) : log_ft_fast(x);
        same = fbits(want) == fbits(got);
        if (inDomain) {
            const double F = fn == 0 ? tan_ft_fast_value(x) : log_ft_fast_value(x);
            const double P = fn == 0 ? tan_P(x) : log_P(x);
            const double u = ulps(F, P);
            if (u > st.maxUlps) st.maxUlps = u;
            if (!rounds_clear(F, fn == 0 ? RM_TAN_FAST_D : RM_LOG_FAST_D)) st.fallbacks++;
        }
    }
    st.checked++;
    if (!same) {
        st.mismatches++;
        if (b < st.firstMismatch) st.firstMismatch = b;
    }
}

const char* NAMES[3] = {"tan", "sincos", "log"};
// fast domains as float bit ranges [lo, hi): tan [2^-126, 1024), sincos [+0, 8), log [2^-126, 1]
const uint32_t LO[3] = {0x00800000u, 0x00000000u, 0x00800000u};
const uint32_t HI[3] = {0x44800000u, 0x41000000u, 0x3f800001u};
const unsigned BOUND[3] = {RM_TAN_FAST_D, 0, RM_LOG_FAST_D};

void print(const char* name, const char* what, const Stats& st, unsigned D) {
    std::printf("{\"fn\": \"%s\", \"set\": \"%s\", \"checked\": %" PRIu64 ", \"mismatches\": %" PRIu64
                ", \"fallbacks\": %" PRIu64 ", \"fallback_rate\": %.3g, \"max_ulps\": %.4g, \"bound_ulps\": %u",
                name, what, st.checked, st.mismatches, st.fallbacks,
                st.checked ? (double)st.fallbacks / (double)st.checked : 0.0, st.maxUlps, D);
    if (st.mismatches) std::printf(", \"first_mismatch\": \"0x%08x\"", st.firstMismatch);
    std::printf("}\n");
}

int sweep(int fn, uint64_t stride, unsigned nThreads) {
    const uint64_t lo = LO[fn], hi = HI[fn];
    const uint64_t n = (hi - lo + stride - 1) / stride;
    std::vector<Stats> part(nThreads);
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nThreads; t++)
        th.emplace_back([&, t] {
            for (uint64_t i = n * t / nThreads; i < n * (t + 1) / nThreads; i++) check(fn, (uint32_t)(lo + i * stride), true, part[t]);
        });
    Stats all;
    for (unsigned t = 0; t < nThreads; t++) {
        th[t].join();
        all.add(part[t]);
    }
    // the last float of the domain, whatever the stride
    if ((hi - 1 - lo) % stride) check(fn, (uint32_t)(hi - 1), true, all);
    char what[64];
    std::snprintf(what, sizeof what, "domain/%" PRIu64, stride);
    print(NAMES[fn], what, all, BOUND[fn]);
    return all.mismatches ? 1 : 0;
}

int edges() {
    std::vector<uint32_t> v = {0x7fc00000u, 0xffc00000u, 0x7fffffffu, 0xffffffffu, 0x7f800001u, 0x7fa00000u};
    for (uint32_t sign = 0; sign < 2; sign++)
        for (uint32_t e = 0; e < 256; e++) {
            const uint32_t base = sign << 31 | e << 23;
            for (uint32_t d : {0u, 1u, 2u, 3u, 0x400000u, 0x7ffffdu, 0x7ffffeu, 0x7fffffu}) v.push_back(base + d);
        }
    for (int fn = 0; fn < 3; fn++)
        for (uint32_t b : {LO[fn], HI[fn]}) {
            v.push_back(b - 1);
            v.push_back(b);
            v.push_back(b + 1);
        }
    int bad = 0;
    for (int fn = 0; fn < 3; fn++) {
        Stats st;
        for (uint32_t b : v) check(fn, b, b >= LO[fn] && b < HI[fn], st);
        print(NAMES[fn], "edges", st, BOUND[fn]);
        bad |= st.mismatches != 0;
    }
    return bad;
}

}  // namespace

int main(int argc, char** argv) {
    if (argc == 2 && !std::strcmp(argv[1], "edges")) return edges();
    if (argc != 4) {
        std::fprintf(stderr, "usage: rng_sweep tan|sincos|log STRIDE THREADS | rng_sweep edges\n");
        return 2;
    }
    for (int fn = 0; fn < 3; fn++)
        if (!std::strcmp(argv[1], NAMES[fn])) return sweep(fn, std::strtoull(argv[2], nullptr, 10), (unsigned)std::atoi(argv[3]));
    std::fprintf(stderr, "unknown function %s\n", argv[1]);
    return 2;
}
