// tests/time_scales_shim.cpp -- C entry points over the host code of the per-row time scales for tests/test_time_scales_host.py:
// check_time_scales and time_scales_from_lengths (csrc/setup.cpp) and the restart fingerprint with and without rows (csrc/restart.cpp).
// Linked with those two files alone, against no CUDA library.  Every call builds the plan dfb_create would build from cfg; a refusal
// returns its code with err = "code msg".
#include <cstdio>
#include <cstring>
#include "restart.hpp"

using namespace dfb;

namespace {

int failed(const Error& e, char* err, int errlen) {
    std::snprintf(err, (size_t)errlen, "%d %s", e.code, e.msg.c_str());
    return e.code;
}

}  // namespace

extern "C" {

// Ny after the trim, d_i, and the rows the formula reads: y_j (dfb_get_table 8) and Us (dfb_get_table 4), [Ny] each (cap >= Ny)
int ts_plan(const dfb_config* cfg, int* Ny, double* d_i, double* yc, double* Us, int cap, char* err, int errlen) {
    try {
        Plan P;
        build_plan(*cfg, P);
        *Ny = P.Ny;
        *d_i = P.d_i;
        if (cap >= P.Ny) {
            std::memcpy(yc, P.yc_row.data(), sizeof(double) * P.Ny);
            std::memcpy(Us, P.rows.data() + (size_t)4 * P.Ny, sizeof(double) * P.Ny);
        }
        return 0;
    } catch (const Error& e) {
        return failed(e, err, errlen);
    }
}

int ts_from_lengths(const dfb_config* cfg, const double* Ix, double u_min, double* Lt_rows, char* err, int errlen) {
    try {
        Plan P;
        build_plan(*cfg, P);
        time_scales_from_lengths(P, Ix, u_min, Lt_rows);
        return 0;
    } catch (const Error& e) {
        return failed(e, err, errlen);
    }
}

// fingerprint of the plan with Lt_rows [3][Ny] set as dfb_set_time_scales sets them (NULL: none)
int ts_fingerprint(const dfb_config* cfg, const double* Lt_rows, uint64_t* fp, char* err, int errlen) {
    try {
        Plan P;
        build_plan(*cfg, P);
        if (Lt_rows) {
            check_time_scales(P, Lt_rows);
            P.Lt_rows.assign(Lt_rows, Lt_rows + (size_t)3 * P.Ny);
        }
        *fp = rst::fingerprint(P);
        return 0;
    } catch (const Error& e) {
        return failed(e, err, errlen);
    }
}

}  // extern "C"
