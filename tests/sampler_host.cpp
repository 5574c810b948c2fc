// tests/sampler_host.cpp - TEST INFRASTRUCTURE: tests/sampler_model.cuh compiled for the CPU on both engines, with the CUDA
// vocabulary and the trial runners of tests/cmb_engine_host.cpp.  The static tier's host build tries each sampler with the
// ziggurats' rectangles only and repeats it after a rewind, as the device does (static_run_trial_host).
// Not a product path: built by tests/sampler_cases.py.
//
// Build: g++ -std=c++17 -O2 -ffp-contract=off -shared -fPIC sampler_host.cpp -o libsampler_host.so
#include "cmb_engine_host.cpp"
#include "sampler_model.cuh"

// engine 0 = the general engine (cmb::Sim), 1 = the static tier (cmb::StaticSim<1, 0>); params[0] = the sampler
extern "C" int host_sampler_run_trials(int engine, uint64_t master_seed, uint64_t first, uint64_t count, uint64_t num_objects,
                                       const double *params, uint32_t num_params, uint64_t trace_cap, uint64_t *trace_key,
                                       double *trace_time, HostResult *out)
{
    static ZigHot hot;
    for (int i = 0; i < 256; i++) {
        hot.exp_x[i] = zig::zig_exp_x[i];
        hot.nor_x[i] = zig::zig_nor_x[i];
    }
    const uint64_t arena_bytes = 1u << 16;
    std::vector<unsigned char> mem(arena_bytes + 256);
    for (uint64_t i = 0; i < count; i++) {
        unsigned long long cursor = 0;
        cmb::Arena arena{mem.data(), &cursor, arena_bytes};
        cmb::TrialIn in{};
        in.num_objects = num_objects;
        in.servers = 1;
        in.num_params = num_params;
        for (uint32_t k = 0; k < num_params && k < 16u; k++) in.params[k] = params[k];
        in.trial = first + i;
        const uint64_t seed = fmix64(master_seed, first + i);
        uint64_t *tk = trace_cap ? trace_key + i * trace_cap : nullptr;
        double *tt = trace_cap ? trace_time + i * trace_cap : nullptr;
        if (engine == 0) run_model<tests::SamplerT<cmb::Sim>>(seed, in, arena, hot, out[i], trace_cap, tk, tt);
        else if (engine == 1) run_static<tests::SamplerT, 1, 0>(seed, in, hot, out[i], 1u, trace_cap, tk, tt);
        else return -1;
    }
    return 0;
}
