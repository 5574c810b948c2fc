// Host build of cimba_b200/csrc/glibc_exp.cuh for tests/test_awacs_math.py (device intrinsics -> IEEE meanings).
// Build: g++ -std=c++17 -O2 -ffp-contract=off glibc_exp_harness.cpp -o harness
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

static inline long long __double_as_longlong(double d) { long long i; std::memcpy(&i, &d, 8); return i; }
static inline double __longlong_as_double(long long i) { double d; std::memcpy(&d, &i, 8); return d; }
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __dsub_rn(double a, double b) { return a - b; }
static inline double __fma_rn(double a, double b, double c) { return std::fma(a, b, c); }

#include "../cimba_b200/csrc/glibc_exp.cuh"

static uint64_t state = 88172645463325252ull;
static inline uint64_t next64() { state ^= state << 13; state ^= state >> 7; state ^= state << 17; return state; }

int main(int argc, char **argv)
{
    const long n = argc > 1 ? std::atol(argv[1]) : 2000000;
    unsigned long bad = 0;
    for (long i = 0; i < n; i++) {
        const double scale = (i & 3) == 0 ? 760.0 : ((i & 3) == 1 ? 40.0 : ((i & 3) == 2 ? 8.0 : 1.0e-3));
        const double x = (double)(int64_t)next64() / 9.3e18 * scale;
        const double a = std::exp(x), b = cimba_b200::glibc_exp(x);
        if (std::memcmp(&a, &b, 8) != 0) bad++;
    }
    std::printf("{\"n\": %ld, \"exp\": %lu}\n", n, bad);
    return 0;
}
