// csrc/plan.hpp -- host-side description of one inflow plane: everything the constructor of the
// reference computes once (df.cpp:4-66) in the shape the device wants it.
#pragma once
#include <cstdint>
#include <string>
#include <vector>
#include "dfb200.h"

namespace dfb {

struct Error {
    int code;
    std::string msg;
};

// Coefficients depend on the half-width N alone (df.cpp:168-177): one row per distinct N,
// CSR-style: vals[ptr[N] + i + N], i = -N..N.  ptr[N] < 0 -> N does not occur.
struct CoefTable {
    int Nmax = 0;
    std::vector<int64_t> ptr;
    std::vector<double> vals;
    const double* centre(int N) const { return vals.data() + ptr[N] + N; }
};

struct FieldPlan {
    double Iz_inn = 0, Iz_out = 0, Lt = 0;       // df.hpp:32
    int Ny_max = 0, Nz_max = 0;                  // df.hpp:33 (max over the WHOLE plane, not the slab)
    bool row_uniform = true;                     // N_y, N_z constant along k in every row
    std::vector<int> N_y_row, N_z_row;           // [Ny]     (valid when row_uniform)
    std::vector<int> N_y, N_z;                   // [Ny*NzG] (always filled unless huge && row_uniform)
};

struct Plan {
    int Ny = 0, NzG = 0;                         // trimmed rows, global spanwise width
    int k0 = 0, k1 = 0;                          // slab owned by this handle
    bool periodic = false;                       // dfb_config.periodic_z: the z filter wraps around the plane (Nz_max <= NzG)
    double d_i = 0, d_v = 0, U_e = 0, rho_e = 0, mu = 0, gcon = 287.0;
    double u_tau = 0, tau_w = 0;
    std::vector<double> yc_row, dy_row;          // first column of the geometry (ydline*d_i, df.cpp:115-116)
    std::vector<double> csv_yc, csv_zc;          // cell-centre coordinates as write_csv prints them (df.cpp:785-786): [Ny], [NzG]
    std::vector<double> vert_y, vert_z;          // vertex coordinates y[j*(Nz+1)+k], z[...] of df.cpp:99-100 (uniform in the other index): [Ny+1], [NzG+1]
    std::vector<double> rows;                    // [8][Ny] R11,R21,R22,R33,Us,Ts,rhos,Ms
    FieldPlan f[3];
    CoefTable coef;
    int64_t taps_per_step = 0;                   // sum over fields and LOCAL cells of (2Ny+1)+(2Nz+1)
    int Nz() const { return k1 - k0; }
};

// Builds the plan from the config; throws dfb::Error.
void build_plan(const dfb_config& cfg, Plan& plan);

// pieces, exposed for unit tests through the C ABI
void coefficients(int N, double* b /* 2N+1 */);
std::vector<double> linear_interpolate(const std::vector<double>& y_data, const std::vector<double>& f_data,
                                       const std::vector<double>& y_new);

}  // namespace dfb
