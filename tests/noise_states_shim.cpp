// tests/noise_states_shim.cpp -- C entry points over dfb::fill_noise_states (csrc/stepplan.cpp) and noise_step_state (csrc/noise.cuh)
// for tests/test_attached_host.py: the noise positions a host-driven step takes, and the per-array function the advance kernel of an
// attached step evaluates on the device, compiled here for the host against no CUDA library.
#include <cstdio>
#include "plan.hpp"
#include "noise.cuh"

using namespace dfb;

extern "C" {

// For the plan of `cfg` with `nplanes` planes: the arrays' field, kind and pairs per step ([6] each), the host's states and increments
// [P][6] for `step`, and the device function's states [P][6].  Returns the number of arrays, or -1 on error (err = "code msg").
int ns_states(const dfb_config* cfg, int nplanes, unsigned long long seed, int plane_id, long long step, int* field, int* kind,
              unsigned long long* npairs, unsigned long long* host_state, unsigned long long* host_inc, unsigned long long* dev_state,
              char* err, int errlen) {
    try {
        Plan plan;
        build_plan(*cfg, plan);
        const StepPlan S = plan_step(plan, nplanes, DeviceLimits{148, 232448}, Overrides{});
        NoiseParams np = S.np;
        uint64_t pairs[6] = {};
        for (int n = 0; n < np.n_arrays; ++n) {
            pairs[n] = S.noise[n].npairs;
            field[n] = np.a[n].field; kind[n] = np.a[n].kind; npairs[n] = pairs[n];
        }
        fill_noise_states(np, pairs, seed, plane_id, nplanes, step);
        for (int p = 0; p < nplanes; ++p)
            for (int n = 0; n < np.n_arrays; ++n) {
                host_state[p * 6 + n] = np.pstate[p][n];
                host_inc[p * 6 + n] = np.pinc[p][n];
                dev_state[p * 6 + n] = noise_step_state(seed, np.pinc[p][n], step, pairs[n]);
            }
        return np.n_arrays;
    } catch (const Error& e) {
        std::snprintf(err, (size_t)errlen, "%d %s", e.code, e.msg.c_str());
        return -1;
    }
}

}  // extern "C"
