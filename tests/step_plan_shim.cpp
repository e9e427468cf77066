// tests/step_plan_shim.cpp -- C entry points over dfb::plan_step (csrc/stepplan.cpp) for tests/test_step_plan.py.  Linked with the
// planner and csrc/setup.cpp alone, against no CUDA library: that it links at all shows the planner makes no CUDA call.
#include <cstdio>
#include <cstring>
#include <string>
#include "plan.hpp"

using namespace dfb;

namespace {
struct Result { Plan plan; StepPlan S; };
}

extern "C" {

// ovr[5] = DFB_Y_MODE, DFB_Y_TK, DFB_Y_COLGROUP, DFB_ZK, DFB_Z_MODE; bit i of `set`: ovr[i] is given.  nullptr on error (err = "code msg").
void* sp_plan(const dfb_config* cfg, int nplanes, int sms, long long smem_optin, const int* ovr, int set, char* err, int errlen) {
    Result* r = new Result;
    try {
        build_plan(*cfg, r->plan);
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

void sp_free(void* h) { delete static_cast<Result*>(h); }

// scalar `name`; i = field (layout, half-widths) or noise array (n_seg, kind, field, npairs)
long long sp_scalar(void* h, const char* name, int i) {
    const Result& r = *static_cast<Result*>(h);
    const StepPlan& S = r.S;
    const std::string n(name);
    const FieldDev& F = S.D.f[i < 3 ? i : 0];
    const long long v[] = {
        S.tuned, S.y_form, S.n_tiles_dense, S.n_tiles_rec, S.yp.n_rtiles, S.yp.tk, S.yp.r_wrows, S.yp.r_nbuf, S.yp.r_smem, S.yp.r_grid,
        S.zp.zk, S.zp.zmode, S.zp.n_items, S.zp.n_uv, S.zp.box_lines, S.zp.smem_bytes, S.np.max_np, S.np.chunks, S.np.n_arrays,
        S.D.Ny, S.D.W, S.D.NzG, S.D.k0, r.plan.k1, r.plan.periodic, F.We, F.xk0, F.rows_y, F.Ny_max, F.Nz_max,
        (long long)ysweep_run_smem(0, 0), NOISE_THREADS, NOISE_PAIRS, YR_C, YR_BOX, Y_RC, Y_G, Y_TK, YJ};
    const char* names[] = {
        "tuned", "y_form", "n_tiles_dense", "n_tiles_rec", "n_rtiles", "tk", "r_wrows", "r_nbuf", "r_smem", "r_grid",
        "zk", "zmode", "n_items", "n_uv", "box_lines", "z_smem", "max_np", "chunks", "n_arrays",
        "Ny", "W", "NzG", "k0", "k1", "periodic", "We", "xk0", "rows_y", "Ny_max", "Nz_max",
        "run_smem_ctl", "NOISE_THREADS", "NOISE_PAIRS", "YR_C", "YR_BOX", "Y_RC", "Y_G", "Y_TK", "YJ"};
    static_assert(sizeof(v) / sizeof(v[0]) == sizeof(names) / sizeof(names[0]), "one name per value");
    for (size_t k = 0; k < sizeof(names) / sizeof(names[0]); ++k)
        if (n == names[k]) return v[k];
    if (i < S.np.n_arrays) {
        if (n == "n_seg") return S.np.a[i].n_seg;
        if (n == "kind") return S.np.a[i].kind;
        if (n == "field") return S.np.a[i].field;
        if (n == "npairs") return (long long)S.noise[i].npairs;
    }
    return -1;
}

// array `name` (i = field for N_y_row / N_z_row, noise array for jump / off / np / win): bytes and element size; nullptr if unknown
const void* sp_array(void* h, const char* name, int i, long long* bytes, int* elem) {
    const Result& r = *static_cast<Result*>(h);
    const StepPlan& S = r.S;
    const std::string n(name);
    auto out = [&](const auto& vec) -> const void* {
        *bytes = (long long)(vec.size() * sizeof(vec[0]));
        *elem = (int)sizeof(vec[0]);
        return vec.data();
    };
    if (n == "rowc") return out(S.rowc);
    if (n == "groups") return out(S.groups);
    if (n == "tiles") return out(S.tiles);
    if (n == "cmat") return out(S.cmat);
    if (n == "yrec") return out(S.yrec);
    if (n == "ygc") return out(S.ygc);
    if (n == "rgroups") return out(S.rgroups);
    if (n == "rtiles") return out(S.rtiles);
    if (n == "coef_pad") return out(S.coef_pad);
    if (n == "coef_pad_ptr") return out(S.coef_pad_ptr);
    if (n == "units") return out(S.units);
    if (n == "unit_par") return out(S.unit_par);
    if (n == "slot_jump") return out(S.slot_jump);
    if (n == "N_y_row") return out(r.plan.f[i].N_y_row);
    if (n == "N_z_row") return out(r.plan.f[i].N_z_row);
    if (i < (int)S.noise.size()) {
        if (n == "jump") return out(S.noise[i].jump);
        if (n == "off") return out(S.noise[i].off);
        if (n == "np") return out(S.noise[i].np);
        if (n == "win") return out(S.noise[i].win);
    }
    return nullptr;
}

}  // extern "C"
