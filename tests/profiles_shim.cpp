// tests/profiles_shim.cpp -- C entry points over the host side of the per-cell profiles for tests/test_profiles_host.py: profile_consts
// (csrc/profiles.cpp), the row constants of plan_step (csrc/stepplan.cpp), the restart fingerprint (csrc/restart.cpp) and the flux
// correction's tables (csrc/fluxtables.cpp), on the plan dfb_create would build from cfg.  Linked against no CUDA library.  A refusal
// returns its code with err = "code msg".
#include <cstdio>
#include <cstring>
#include "plan.hpp"
#include "restart.hpp"

using namespace dfb;

namespace {

int failed(const Error& e, char* err, int errlen) {
    std::snprintf(err, (size_t)errlen, "%d %s", e.code, e.msg.c_str());
    return e.code;
}

// the plan of cfg with the profiles of `cells` ([8][Ny][NzG]) set as dfb_set_profiles sets them; cells == nullptr: none
Plan plan_with(const dfb_config* cfg, const double* cells) {
    Plan P;
    build_plan(*cfg, P);
    if (cells) {
        profile_consts(P, cells);
        P.cells = std::make_shared<const std::vector<double>>(profile_columns(P, cells));
        P.cells_hash = rst::hash_f64(cells, (size_t)8 * P.Ny * P.NzG);
    }
    return P;
}

}  // namespace

extern "C" {

// Ny, NzG, k0, k1 of the plan; rows [8][Ny], vert_y [Ny+1], vert_z [NzG+1] (any may be NULL)
int pr_plane(const dfb_config* cfg, int* dims, double* rows, double* vert_y, double* vert_z, char* err, int errlen) {
    try {
        Plan P;
        build_plan(*cfg, P);
        dims[0] = P.Ny; dims[1] = P.NzG; dims[2] = P.k0; dims[3] = P.k1;
        if (rows) std::memcpy(rows, P.rows.data(), P.rows.size() * sizeof(double));
        if (vert_y) std::memcpy(vert_y, P.vert_y.data(), P.vert_y.size() * sizeof(double));
        if (vert_z) std::memcpy(vert_z, P.vert_z.data(), P.vert_z.size() * sizeof(double));
        return 0;
    } catch (const Error& e) {
        return failed(e, err, errlen);
    }
}

// profile_consts of cells [8][Ny][NzG] -> out [7][Ny][W]; the row constants of plan_step -> rowc [Ny][ROWC]
int pr_consts(const dfb_config* cfg, const double* cells, double* out, double* rowc, char* err, int errlen) {
    try {
        Plan P;
        build_plan(*cfg, P);
        const std::vector<double> pc = profile_consts(P, cells);
        std::memcpy(out, pc.data(), pc.size() * sizeof(double));
        const StepPlan S = plan_step(P, 1, DeviceLimits{148, 232448}, Overrides{});
        std::memcpy(rowc, S.rowc.data(), S.rowc.size() * sizeof(double));
        return 0;
    } catch (const Error& e) {
        return failed(e, err, errlen);
    }
}

// the restart fingerprint with the profiles of cells (NULL: none)
int pr_fingerprint(const dfb_config* cfg, const double* cells, uint64_t* fp, char* err, int errlen) {
    try {
        *fp = rst::fingerprint(plan_with(cfg, cells));
        return 0;
    } catch (const Error& e) {
        return failed(e, err, errlen);
    }
}

// flux_tables(plan with the profiles of cells, mode): wy [Ny], hz [NzG], wz [Ny][NzG] (cells only), D, mean
int pr_flux(const dfb_config* cfg, const double* cells, int mode, double* wy, double* hz, double* wz, double* D, double* mean, char* err,
            int errlen) {
    try {
        const FluxTables T = flux_tables(plan_with(cfg, cells), mode);
        std::memcpy(wy, T.wy.data(), T.wy.size() * sizeof(double));
        std::memcpy(hz, T.hz.data(), T.hz.size() * sizeof(double));
        if (wz) std::memcpy(wz, T.wz.data(), T.wz.size() * sizeof(double));
        *D = T.D;
        *mean = T.mean;
        return 0;
    } catch (const Error& e) {
        return failed(e, err, errlen);
    }
}

}  // extern "C"
