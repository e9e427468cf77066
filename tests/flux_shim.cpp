// tests/flux_shim.cpp -- C entry points over the host tables of the inflow mass-flux correction for tests/test_flux_host.py:
// flux_tables (csrc/fluxtables.cpp) on the plan dfb_create would build from cfg.  Linked with csrc/setup.cpp and csrc/fluxtables.cpp
// alone, against no CUDA library.  A refusal returns its code with err = "code msg".  fx_fma is C's correctly rounded fma, elementwise,
// for the GPU tests' bit-for-bit restatement of the correction (numpy has no fma).
#include <cmath>
#include <cstdio>
#include <cstring>
#include "plan.hpp"

using namespace dfb;

namespace {

int failed(const Error& e, char* err, int errlen) {
    std::snprintf(err, (size_t)errlen, "%d %s", e.code, e.msg.c_str());
    return e.code;
}

}  // namespace

extern "C" {

int fx_dims(const dfb_config* cfg, int* Ny, int* NzG, char* err, int errlen) {
    try {
        Plan P;
        build_plan(*cfg, P);
        *Ny = P.Ny;
        *NzG = P.NzG;
        return 0;
    } catch (const Error& e) {
        return failed(e, err, errlen);
    }
}

// rows [8][Ny], vert_y [Ny+1], vert_z [NzG+1] of the plan; wy, rc0 [Ny], hz [NzG], D and the mean flux of flux_tables(plan, mode)
int fx_tables(const dfb_config* cfg, int mode, double* rows, double* vert_y, double* vert_z, double* wy, double* rc0, double* hz, double* D,
              double* mean, char* err, int errlen) {
    try {
        Plan P;
        build_plan(*cfg, P);
        const FluxTables T = flux_tables(P, mode);
        std::memcpy(rows, P.rows.data(), P.rows.size() * sizeof(double));
        std::memcpy(vert_y, P.vert_y.data(), P.vert_y.size() * sizeof(double));
        std::memcpy(vert_z, P.vert_z.data(), P.vert_z.size() * sizeof(double));
        std::memcpy(wy, T.wy.data(), T.wy.size() * sizeof(double));
        std::memcpy(rc0, T.rc0.data(), T.rc0.size() * sizeof(double));
        std::memcpy(hz, T.hz.data(), T.hz.size() * sizeof(double));
        *D = T.D;
        *mean = T.mean;
        return 0;
    } catch (const Error& e) {
        return failed(e, err, errlen);
    }
}

void fx_fma(long long n, const double* a, const double* b, const double* c, double* out) {
    for (long long i = 0; i < n; ++i) out[i] = std::fma(a[i], b[i], c[i]);
}

}  // extern "C"
