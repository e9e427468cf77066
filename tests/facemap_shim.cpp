// tests/facemap_shim.cpp -- C entry points over dfb::build_face_map (csrc/facemap.cpp) for tests/test_facemap_host.py.  Linked with
// csrc/setup.cpp alone, against no CUDA library: that it links at all shows the maps are built without a CUDA call.
#include <cstdio>
#include <cstring>
#include "facemap.hpp"

using namespace dfb;

namespace {
struct Result { Plan plan; FaceMap map; };
}

extern "C" {

// nullptr on error (err = "code msg")
void* fm_build(const dfb_config* cfg, int kind, int n, const double* yf, const double* zf, const double* hy, const double* hz, int own0,
               int own1, int flags, char* err, int errlen) {
    Result* r = new Result;
    try {
        build_plan(*cfg, r->plan);
        r->map = build_face_map(r->plan, kind, n, yf, zf, hy, hz, own0, own1, flags);
        return r;
    } catch (const Error& e) {
        std::snprintf(err, (size_t)errlen, "%d %s", e.code, e.msg.c_str());
        delete r;
        return nullptr;
    }
}

void fm_free(void* h) { delete static_cast<Result*>(h); }

// {Ny, NzG, k0, k1, periodic, n, n_served, taps}
void fm_sizes(void* h, long long* out) {
    const Result& r = *static_cast<Result*>(h);
    const long long v[8] = {r.plan.Ny, r.plan.NzG, r.plan.k0, r.plan.k1, r.plan.periodic, r.map.n, r.map.n_served, (long long)r.map.w.size()};
    std::memcpy(out, v, sizeof(v));
}

// served [n], ptr [n+1] (AREA; ignored for POINT), idx and w [taps]
void fm_arrays(void* h, int* served, int* ptr, int* idx, double* w) {
    const FaceMap& m = static_cast<Result*>(h)->map;
    std::memcpy(served, m.served.data(), m.served.size() * sizeof(int));
    if (ptr) std::memcpy(ptr, m.ptr.data(), m.ptr.size() * sizeof(int));
    std::memcpy(idx, m.idx.data(), m.idx.size() * sizeof(int));
    std::memcpy(w, m.w.data(), m.w.size() * sizeof(double));
}

// 0 csv_yc [Ny], 1 csv_zc [NzG], 2 vert_y [Ny+1], 3 vert_z [NzG+1]
void fm_geom(void* h, int which, double* out) {
    const Plan& P = static_cast<Result*>(h)->plan;
    const std::vector<double>* t[4] = {&P.csv_yc, &P.csv_zc, &P.vert_y, &P.vert_z};
    std::memcpy(out, t[which]->data(), t[which]->size() * sizeof(double));
}

}  // extern "C"
