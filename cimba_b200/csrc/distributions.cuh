// distributions.cuh - the rest of cmb_random on the device.
//
// Reference: include/cmb_random.h:189-940 and src/cmb_random.c:299-313, 465-766.  Every
// function is a thin layer over sfc64 and the two ziggurats (rng.cuh), in the reference's
// draw order, so a stream seeded like the reference's yields the same variates:
//   * bit-exact by construction (sqrt and division are IEEE-exact on both sides):
//     triangular, cauchy, hypo/hyperexponential, rayleigh, flip, binomial, poisson,
//     loaded_dice, alias_sample;
//   * bit-exact in practice - log() only feeds the accept/reject comparison of the
//     Marsaglia-Tsang squeeze, so a last-place difference between CUDA's and glibc's log
//     matters only if the two sides of that comparison agree to ~1e-16:
//     std_gamma, gamma (shape >= 1), beta, PERT, chisquared (k >= 2), F, t;
//   * bit-exact because the only libm call is exp(), restated from glibc (glibc_exp.cuh): lognormal
//     (the ziggurat wedge tests in rng.cuh use the same routine);
//   * within the accuracy of CUDA's log / pow (<= 2 ulp) of the reference's glibc result,
//     because the transcendental IS the variate: logistic, weibull, pareto, gamma with
//     shape < 1 (and what builds on it); geometric / negative_binomial apply ceil() to such a
//     value and can differ by one on a measure-zero set.  glibc's log and pow tables were
//     chosen by search and cannot be recomputed from first principles, so they stay CUDA's.
// Where the reference itself is undefined, nothing can match it and nothing is promised:
//   * geometric with p = 0, or with p so small that the count exceeds 2^32 (and negative_binomial / pascal on it): an
//     out-of-range double converted to unsigned is undefined in C - x86 wraps, sm_100 saturates;
//   * hyper-exponential and loaded dice whose probabilities sum to less than 1: the reference indexes past its table.
// tests/test_random_edges.py and tests/test_gpu_random_edges.py hold every other edge (p = 0 and 1, lo == hi, a shape of
// exactly 1, one degree of freedom, overflow to inf, subnormal results) to the reference's draws.
// Compiled with -fmad=false: the expressions keep the reference's operation order.
#pragma once

#include <cmath>
#include <cstdint>

#include "rng.cuh"

namespace cimba_b200 {

// Out-of-line draws for the general-path kernels.  rng.cuh's members inline their ziggurat slow
// paths (exp(), alias tables, rejection loops: 400-600 instructions) into every call site, which is
// right for the small hot kernels and wrong for code that draws in dozens of places: the harbor
// kernel was 40 % inlined generator code and stalled on the instruction cache.
__device__ __noinline__ double gp_std_normal(Sfc64 &r, const ZigHot &hot)
{
    return r.std_normal(hot);
}

__device__ __noinline__ double gp_exponential(Sfc64 &r, const ZigHot &hot, double mean)
{
    return r.exponential(hot, mean);
}

__device__ __noinline__ double gp_uniform01(Sfc64 &r)
{
    return r.uniform01();
}

// src/cmb_random.c:500-520
__device__ inline double rnd_triangular(Sfc64 &r, double min, double mode, double max)
{
    const double u = gp_uniform01(r);
    if (u < (mode - min) / (max - min)) {
        return min + sqrt(u * (max - min) * (mode - min));
    }
    return max - sqrt((1.0 - u) * (max - min) * (max - mode));
}

// include/cmb_random.h:249-257
__device__ inline double rnd_lognormal(Sfc64 &r, const ZigHot &hot, double m, double s)
{
    return glibc_exp((m + s * gp_std_normal(r, hot)));      // the variate IS an exp: glibc's bits (glibc_exp.cuh)
}

// :267-273
__device__ inline double rnd_logistic(Sfc64 &r, double m, double s)
{
    const double x = gp_uniform01(r);
    return m + s * log(x / (1.0 - x));
}

// :290-299
__device__ inline double rnd_cauchy(Sfc64 &r, const ZigHot &hot, double mode, double scale)
{
    const double x = gp_std_normal(r, hot);
    double y;
    while ((y = gp_std_normal(r, hot)) == 0.0) {}
    return mode + scale * x / y;
}

// :394-408
__device__ inline double rnd_hypoexponential(Sfc64 &r, const ZigHot &hot, unsigned n, const double *ma)
{
    double x = 0.0;
    for (unsigned i = 0u; i < n; i++) {
        x += gp_exponential(r, hot, ma[i]);
    }
    return x;
}

// src/cmb_random.c:644-662
__device__ inline unsigned rnd_loaded_dice(Sfc64 &r, unsigned n, const double *pa)
{
    const double x = gp_uniform01(r);
    double q = 0.0;
    unsigned ui;
    for (ui = 0u; ui < n; ui++) {
        q += pa[ui];
        if (x < q) {
            break;
        }
    }
    return ui;
}

// :299-313
__device__ inline double rnd_hyperexponential(Sfc64 &r, const ZigHot &hot, unsigned n,
                                              const double *ma, const double *pa)
{
    const unsigned ui = rnd_loaded_dice(r, n, pa);
    return gp_exponential(r, hot, ma[ui]);
}

// Marsaglia & Tsang, src/cmb_random.c:465-497.  Out of line on purpose (it carries a full normal draw,
// slow path included): callers are the cold, code-heavy general-path kernels.
__device__ __noinline__ double rnd_std_gamma(Sfc64 &r, const ZigHot &hot, double shape)
{
    const double d = shape - 1.0 / 3.0;
    const double c = 1.0 / sqrt(9.0 * d);
    double x, v;
    for (;;) {
        do {
            x = gp_std_normal(r, hot);
            v = 1.0 + c * x;
        } while (v <= 0.0);
        const double w = v * v * v;
        const double u = gp_uniform01(r);
        if ((u < 1.0 - 0.331 * (x * x) * (x * x))
            || (log(u) < (0.5 * x * x) + (d * (1.0 - w + log(w))))) {
            return d * w;
        }
    }
}

// include/cmb_random.h:451-463.  For shape < 1 the reference writes
// cmb_random_std_gamma(shape + 1) * pow(cmb_random(), 1 / shape): C leaves the evaluation order of the two operands
// unspecified; gcc 13 (-O2/-O3, x86-64) - the build the oracle and the golden vectors come from - draws std_gamma
// first, and so does this.  A different compiler could legitimately produce the other stream.
__device__ inline double rnd_gamma(Sfc64 &r, const ZigHot &hot, double shape, double scale)
{
    if (shape >= 1.0) {
        return scale * rnd_std_gamma(r, hot, shape);
    }
    const double g = rnd_std_gamma(r, hot, shape + 1.0);
    const double u = gp_uniform01(r);
    return scale * (g * pow(u, 1.0 / shape));
}

// :476-487
__device__ inline double rnd_std_beta(Sfc64 &r, const ZigHot &hot, double a, double b)
{
    const double x = rnd_std_gamma(r, hot, a);
    const double y = rnd_std_gamma(r, hot, b);
    return x / (x + y);
}

// :500-512
__device__ inline double rnd_beta(Sfc64 &r, const ZigHot &hot, double a, double b, double min, double max)
{
    return min + (max - min) * rnd_std_beta(r, hot, a, b);
}

// src/cmb_random.c:523-538; cmb_random_PERT (include/cmb_random.h:541-553) is lambda = 4
__device__ inline double rnd_PERT_mod(Sfc64 &r, const ZigHot &hot, double min, double mode, double max, double lambda)
{
    const double rng = max - min;
    const double a = 1.0 + lambda * (mode - min) / rng;
    const double b = 1.0 + lambda * (max - mode) / rng;
    return min + rng * rnd_std_beta(r, hot, a, b);
}

// :571-582
__device__ inline double rnd_weibull(Sfc64 &r, const ZigHot &hot, double shape, double scale)
{
    const double u = gp_exponential(r, hot, 1.0);
    return scale * pow(u, 1.0 / shape);
}

// :595-605
__device__ inline double rnd_pareto(Sfc64 &r, double shape, double mode)
{
    return mode / pow(gp_uniform01(r), 1.0 / shape);
}

// :618-626
__device__ inline double rnd_chisquared(Sfc64 &r, const ZigHot &hot, double k)
{
    return rnd_gamma(r, hot, k / 2.0, 2.0);
}

// :639-653
__device__ inline double rnd_F_dist(Sfc64 &r, const ZigHot &hot, double a, double b)
{
    const double x = rnd_chisquared(r, hot, a) / a;
    double y;
    while ((y = rnd_chisquared(r, hot, b) / b) == 0.0) {}
    return x / y;
}

// :668-679
__device__ inline double rnd_std_t_dist(Sfc64 &r, const ZigHot &hot, double v)
{
    const double x = gp_std_normal(r, hot);
    double y;
    while ((y = rnd_chisquared(r, hot, v)) == 0.0) {}
    return x / sqrt(y / v);
}

// :693-702
__device__ inline double rnd_t_dist(Sfc64 &r, const ZigHot &hot, double m, double s, double v)
{
    return m + s * rnd_std_t_dist(r, hot, v);
}

// :714-725
__device__ inline double rnd_rayleigh(Sfc64 &r, const ZigHot &hot, double s)
{
    const double x = (0.0 + s * gp_std_normal(r, hot));
    const double y = (0.0 + s * gp_std_normal(r, hot));
    return sqrt(x * x + y * y);
}

// cmb_random_flip, src/cmb_random.c:541-552: 64 coin flips per sfc64 word, most significant
// bit first.  The reference keeps the cache in thread-local statics; here it is part of
// the trial's generator state.
struct FlipCache {
    uint64_t bits;
    uint32_t pos;
};

__device__ inline int rnd_flip(Sfc64 &r, FlipCache &f)
{
    if (f.pos == 0u) {
        f.bits = r.next();
        f.pos = 64u;
    }
    return (int)((f.bits >> --f.pos) & 1u);
}

// :558-573
__device__ inline unsigned rnd_geometric(Sfc64 &r, const ZigHot &hot, double p)
{
    const double denom = -log(1.0 - p);
    return (unsigned)ceil(gp_exponential(r, hot, 1.0) / denom);
}

// :576-588
__device__ inline unsigned rnd_binomial(Sfc64 &r, unsigned n, double p)
{
    unsigned s = 0u;
    for (unsigned i = 0u; i < n; i++) {
        s += r.bernoulli(p);
    }
    return s;
}

// :594-606; cmb_random_pascal (include/cmb_random.h:812-815) is the same function
__device__ inline unsigned rnd_negative_binomial(Sfc64 &r, const ZigHot &hot, unsigned m, double p)
{
    unsigned f = 0u;
    for (unsigned i = 0u; i < m; i++) {
        f += rnd_geometric(r, hot, p) - 1u;
    }
    return f;
}

// :612-632
__device__ inline unsigned rnd_poisson(Sfc64 &r, const ZigHot &hot, double rate)
{
    const double m = 1.0 / rate;
    double t = 0.0;
    unsigned ctr = 0u;
    for (;;) {
        t += gp_exponential(r, hot, m);
        if (t <= 1.0) {
            ctr++;
        }
        else {
            break;
        }
    }
    return ctr;
}

// cmb_random_alias_sample, include/cmb_random.h:922-933 (tables from cimba_b200_alias_create)
__device__ inline unsigned rnd_alias_sample(Sfc64 &r, unsigned n, const uint64_t *uprob, const uint32_t *alias)
{
    const unsigned idx = (unsigned)floor((double)n * gp_uniform01(r));
    const bool c = r.next() >= uprob[idx];
    return c ? alias[idx] : idx;
}

}  // namespace cimba_b200
