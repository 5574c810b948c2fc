// tests/sampler_model.cuh - TEST INFRASTRUCTURE: one process that holds num_objects times for CMB_PROCESS_HOLD_SAMPLED(0), so that
// every hold's duration is one run of the model's sampler and the pop trace is the running sum of the sampled durations.
// params[0] picks the sampler (the SAMPLER_* numbers below, mirrored in tests/sampler_cases.py), params[1..] are its parameters.
// The samplers are the cmb_random_* calls of the authoring surface, some of them inside a rejection loop (the truncated ones),
// and the hold takes fabs() of the variate (exact), so that negative variates are fine.
// A template over the engine, like cimba_b200/models/*.cuh: SamplerT<cmb::Sim> and SamplerT<cmb::StaticSim<1, 0>>; built for the
// device by tests/test_gpu_random_edges.py and for the CPU by tests/sampler_host.cpp.
#pragma once
#include "../cimba_b200/csrc/cmb_kernel.cuh"
#include "../cimba_b200/csrc/cmb_static.cuh"

namespace cimba_b200 {
namespace tests {

enum : int {
    SAMPLER_EXP_BELOW = 0,          // exponential(p0) redrawn while > p1 * p0
    SAMPLER_NORMAL_ABOVE = 1,       // normal(p0, p1) redrawn while < p2
    SAMPLER_EXP_ABOVE = 2,          // exponential(p0) redrawn while < p1
    SAMPLER_EXPONENTIAL = 3,        // exponential(p0)
    SAMPLER_NORMAL = 4,             // normal(p0, p1)
    SAMPLER_ERLANG = 5,             // erlang(p0, p1)
    SAMPLER_GAMMA = 6,              // gamma(p0, p1)
    SAMPLER_BETA = 7,               // beta(p0, p1, p2, p3)
    SAMPLER_PERT = 8,               // PERT(p0, p1, p2)
    SAMPLER_LOGNORMAL = 9,          // lognormal(p0, p1)
    SAMPLER_POISSON = 10,           // poisson(p0)
    SAMPLER_TRIANGULAR = 11,        // triangular(p0, p1, p2)
    SAMPLER_RAYLEIGH = 12,          // rayleigh(p0)
    SAMPLER_UNIFORM = 13,           // uniform(p0, p1)
    SAMPLER_DICE = 14,              // dice(p0, p1)
    SAMPLER_BERNOULLI = 15,         // bernoulli(p0)
    SAMPLER_COMPOSITE = 16,         // exponential(p0) + gamma(2, p1)
};

template <class S>
struct SamplerT {
    uint32_t holder;
    int      which;
    double   p[8];
    uint64_t num_objects, held;
    static CMB_FN constexpr uint32_t static_kind(uint32_t) { return 0u; }

    CMB_FN void holderfunc(S &sim, uint32_t me, int64_t sig)
    {
        SamplerT &m = *this;
        CMB_PROCESS_BEGIN
        for (held = 0u; held < num_objects; held++) {
            CMB_PROCESS_HOLD_SAMPLED(0);
        }
        CMB_PROCESS_END
    }

    CMB_FN double sample(S &sim, uint32_t)
    {
        double v = 0.0;
        switch (which) {
        case SAMPLER_EXP_BELOW:
            do {
                v = cmb_random_exponential(p[0]);
            } while (v > p[1] * p[0]);
            break;
        case SAMPLER_NORMAL_ABOVE:
            do {
                v = cmb_random_normal(p[0], p[1]);
            } while (v < p[2]);
            break;
        case SAMPLER_EXP_ABOVE:
            do {
                v = cmb_random_exponential(p[0]);
            } while (v < p[1]);
            break;
        case SAMPLER_EXPONENTIAL: v = cmb_random_exponential(p[0]); break;
        case SAMPLER_NORMAL:      v = cmb_random_normal(p[0], p[1]); break;
        case SAMPLER_ERLANG:      v = cmb_random_erlang((unsigned)p[0], p[1]); break;
        case SAMPLER_GAMMA:       v = cmb_random_gamma(p[0], p[1]); break;
        case SAMPLER_BETA:        v = cmb_random_beta(p[0], p[1], p[2], p[3]); break;
        case SAMPLER_PERT:        v = cmb_random_PERT(p[0], p[1], p[2]); break;
        case SAMPLER_LOGNORMAL:   v = cmb_random_lognormal(p[0], p[1]); break;
        case SAMPLER_POISSON:     v = (double)cmb_random_poisson(p[0]); break;
        case SAMPLER_TRIANGULAR:  v = cmb_random_triangular(p[0], p[1], p[2]); break;
        case SAMPLER_RAYLEIGH:    v = cmb_random_rayleigh(p[0]); break;
        case SAMPLER_UNIFORM:     v = cmb_random_uniform(p[0], p[1]); break;
        case SAMPLER_DICE:        v = (double)cmb_random_dice((long long)p[0], (long long)p[1]); break;
        case SAMPLER_BERNOULLI:   v = (double)cmb_random_bernoulli(p[0]); break;
        case SAMPLER_COMPOSITE: {
            const double e = cmb_random_exponential(p[0]);       // the rectangles first ...
            v = __dadd_rn(e, cmb_random_gamma(2.0, p[1]));       // ... then a draw with its slow paths inline
            break;
        }
        default: return -1.0;                                    // an unknown sampler: TRIAL_ERR_NEGATIVE_HOLD
        }
        return fabs(v);
    }

    CMB_FN void run_trial(S &sim, const cmb::TrialIn &in)
    {
        which = in.num_params > 0u ? (int)in.params[0] : -1;
        for (int k = 0; k < 8; k++) p[k] = (uint32_t)(k + 1) < in.num_params ? in.params[k + 1] : 0.0;
        num_objects = in.num_objects;
        held = 0u;
        holder = cmb_process_create(0u, 0, 0u);
        cmb_process_start(holder);
    }

    CMB_FN void process(S &sim, uint32_t me, uint32_t, int64_t sig) { holderfunc(sim, me, sig); }
    CMB_FN void event(S &, uint32_t, uint32_t, int64_t) {}
    CMB_FN bool demand(S &, uint32_t, uint32_t, int32_t) { return false; }

    CMB_FN void finish(S &, cmb::TrialOut &out)
    {
        out.objects = held;
        out.sum_wait = 0.0;
    }
};

}  // namespace tests
}  // namespace cimba_b200
