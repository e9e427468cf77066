// tests/filter_shape_shim.cpp -- C entry points over the host code of the filter shape for tests/test_filter_shape_host.py: the
// coefficient table (csrc/setup.cpp) and the step's plan of a plane of either shape (csrc/stepplan.cpp), read through the accessors of
// tests/step_plan_shim.cpp.  Linked against no CUDA library.
#include "step_plan_shim.cpp"

extern "C" {

// b[2N+1] of half-width N in filter shape `shape`
void fs_coefficients(int N, int shape, double* b) { coefficients(N, shape, b); }

// sp_plan with the plan's coefficient table rebuilt for `shape`, as dfb_set_filter_shape rebuilds it
void* fs_plan(const dfb_config* cfg, int shape, int nplanes, int sms, long long smem_optin, const int* ovr, int set, char* err, int errlen) {
    Result* r = new Result;
    try {
        build_plan(*cfg, r->plan);
        r->plan.filter_shape = shape;
        build_coef_table(r->plan);
        Overrides o;
        std::optional<int>* slot[5] = {&o.y_mode, &o.y_tk, &o.y_colgroup, &o.zk, &o.z_mode};
        for (int i = 0; i < 5; ++i)
            if ((set >> i) & 1) *slot[i] = ovr[i];
        r->S = plan_step(r->plan, nplanes, DeviceLimits{sms, (size_t)smem_optin}, o);
        return r;
    } catch (const Error& e) {
        std::snprintf(err, (size_t)errlen, "%d %s", e.code, e.msg.c_str());
        delete r;
        return nullptr;
    }
}

// the plan's coefficient row of half-width N (2N+1 values); 0 when N does not occur
int fs_plan_coef(void* h, int N, double* b) {
    const Plan& P = static_cast<Result*>(h)->plan;
    if (N < 0 || N > P.coef.Nmax || P.coef.ptr[N] < 0) return 0;
    std::memcpy(b, P.coef.vals.data() + P.coef.ptr[N], sizeof(double) * (2 * N + 1));
    return 1;
}

}  // extern "C"
