// csrc/plan.hpp -- host-side description of one inflow plane: everything the constructor of the
// reference computes once (df.cpp:4-66) in the shape the device wants it.
#pragma once
#include <cmath>
#include <cstdint>
#include <memory>
#include <optional>
#include <string>
#include <vector>
#include "dfb200.h"
#include "device.cuh"

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
    int kernel_variant = 0;                      // dfb_config.kernel_variant: != 0 forces the one-thread-per-cell kernels
    int filter_shape = DFB_FILTER_EXPONENTIAL;   // dfb_set_filter_shape: the kernel of the spatial filters (coef)
    double d_i = 0, d_v = 0, U_e = 0, rho_e = 0, mu = 0, gcon = 287.0;
    double u_tau = 0, tau_w = 0;
    std::vector<double> yc_row, dy_row;          // first column of the geometry (ydline*d_i, df.cpp:115-116)
    std::vector<double> csv_yc, csv_zc;          // cell-centre coordinates as write_csv prints them (df.cpp:785-786): [Ny], [NzG]
    std::vector<double> vert_y, vert_z;          // vertex coordinates y[j*(Nz+1)+k], z[...] of df.cpp:99-100 (uniform in the other index): [Ny+1], [NzG+1]
    std::vector<double> rows;                    // [8][Ny] R11,R21,R22,R33,Us,Ts,rhos,Ms
    FieldPlan f[3];
    CoefTable coef;
    int64_t taps_per_step = 0;                   // sum over fields and LOCAL cells of (2Ny+1)+(2Nz+1)
    std::vector<double> Lt_rows;                 // [3][Ny] per-row time scales (dfb_set_time_scales); empty: f[].Lt for every row
    // per-cell profiles (dfb_set_profiles): the eight quantities of `rows` for the cells of this handle's columns, [8][Ny][Nz()], and the
    // hash of the whole-plane table they came from (restart fingerprint).  Null: `rows` for every column.
    std::shared_ptr<const std::vector<double>> cells;
    uint64_t cells_hash = 0;
    int Nz() const { return k1 - k0; }
};

// Builds the plan from the config (exponential filter shape); throws dfb::Error.
void build_plan(const dfb_config& cfg, Plan& plan);
// (Re)builds plan.coef for plan.filter_shape: one row per half-width that occurs in the plane.
void build_coef_table(Plan& plan);

struct DeviceLimits { int sms; size_t smem_optin; };   // multiprocessors, shared memory one block may opt in to (bytes)

// Development switches, read from the environment once by the caller; unset = the planner decides: DFB_Y_MODE (0 dense, 1 chunk-
// recursive, 2 run-recursive y-sweep), DFB_Y_TK (64-column dense tiles), DFB_Y_COLGROUP, DFB_ZK (8 or 16), DFB_Z_MODE (0 direct, 1 recursive)
struct Overrides { std::optional<int> y_mode, y_tk, y_colgroup, zk, z_mode; };

struct NoiseTable {                              // segments of one logical array of the noise contract (include/dfb_rng_spec.h)
    uint64_t npairs;                             // pairs one step draws from the array's stream
    std::vector<Jump> jump;
    std::vector<int> off, np;                    // r_ys: extended column of a segment's first pair (its first column, or one less); halo: 0
    std::vector<int4> win;                       // periodic_z, extended rows that wrap: {padded row, first, end extended column} per piece
};

// What a handle's step needs that follows from the plan and the device's limits alone, as host values: the layout, the work of
// the tuned sweeps (tuned only) and the noise tables.  The pointers in D, yp, zp and np are null: the caller uploads.
struct StepPlan {
    bool tuned = false;                          // row-uniform half-widths whose z window fits: the tuned sweeps (else the one-thread-per-cell kernels)
    PlaneDev D{};
    std::vector<double> rowc;                    // [Ny][ROWC]
    int y_form = 0;                              // dfb_info 10: 0 dense band matrices, 1 chunk-recursive, 2 run-recursive, 3 run + dense
    int n_tiles_dense = 0, n_tiles_rec = 0;      // band-matrix tiles: dense first, then recursive
    YParams yp{};                                // tk, n_rtiles, r_smem, r_wrows, r_nbuf, r_grid
    std::vector<YGroup> groups; std::vector<YTile> tiles;
    std::vector<double> cmat, yrec, ygc;
    std::vector<YRGroup> rgroups; std::vector<YRTile> rtiles;   // y_form >= 2
    ZParams zp{};                                // zk, zmode, n_items, n_uv, box_lines, box_bytes, unit_bytes, rc_off, fo_off, smem_bytes
    std::vector<double> coef_pad, unit_par;      // unit_par: zmode 1 only
    std::vector<long long> coef_pad_ptr; std::vector<ZUnit> units;
    std::vector<NoiseTable> noise; std::vector<Jump> slot_jump;   // noise: the arrays drawn, in the order of np.a
    NoiseParams np{};                            // n_arrays, each array's n_seg, kind, field; max_np, stride, chunks
};

// No CUDA call, no environment; throws dfb::Error.
StepPlan plan_step(const Plan& plan, int nplanes, const DeviceLimits& dev, const Overrides& ovr);

// np.pstate / np.pinc of every array np draws and every plane of the handle: pcg32 state at the first draw of step `step` (plane p of a
// batch draws from stream group plane_id + p).  The advance kernel of attached steps computes the same states with noise_step_state.
void fill_noise_states(NoiseParams& np, const uint64_t* npairs, uint64_t seed, int plane_id, int nplanes, int64_t step);

// The epilogue's constants (df.cpp:425-438, 474) of one row or cell from its eight profile values q = R11, R21, R22, R33, Us, Ts, rhos,
// Ms: rc = sqrt(R11), b, sqrt(R22 - b^2), sqrt(R33), -0.2 Ms^2 / Us, Ts, rhos.  The row tables (plan_step) and the per-cell profiles
// (profile_consts) both use it, so that a cell whose values equal a row's gets that row's constants bit for bit.
inline void epilogue_consts(const double q[8], double rc[7]) {
    const double b = (q[0] < 1e-10) ? 0.0 : q[1] / std::sqrt(q[0]);
    rc[0] = std::sqrt(q[0]);
    rc[1] = b;
    rc[2] = std::sqrt(q[2] - b * b);
    rc[3] = std::sqrt(q[3]);
    rc[4] = -0.5 * (1.4 - 1) * q[7] * q[7] / q[4];
    rc[5] = q[5];
    rc[6] = q[6];
}
constexpr int PROFILE_CONSTS = 7;                // epilogue_consts per cell

// dfb_set_profiles (profiles.cpp): checks a whole-plane table [8][Ny][NzG] and returns the epilogue constants of the cells of the plan's
// columns, [PROFILE_CONSTS][Ny][Nz()].  Throws DFB_ERR_ARG naming the quantity, row and column of the first value that is not finite
// or whose constant is not (R11 < 0, R22 < b^2, Us = 0, ...).
std::vector<double> profile_consts(const Plan& plan, const double* cells);
// the plan's columns of a whole-plane table: [8][Ny][Nz()]
std::vector<double> profile_columns(const Plan& plan, const double* cells);

// Per-row time scales [3][Ny]: throws DFB_ERR_ARG naming the first entry that is not finite or not > 0.
void check_time_scales(const Plan& plan, const double* Lt_rows);
// dfb_time_scales_from_lengths: Lt_f(j) = Ix_f(y_j) / max(Us_j, u_min), Ix_f blended from Ix[2f] to Ix[2f+1] like Iz.  Throws dfb::Error.
void time_scales_from_lengths(const Plan& plan, const double Ix[6], double u_min, double* Lt_rows);

// Inflow mass-flux correction (dfb_set_flux_correction, fluxtables.cpp): per plane and step c = m' / D with m' = sum_j wy_j sum_k hz_k u'_jk,
// and u' <- u' - c rc0_j.  wy_j = g_j hy_j, g_j = rhos_j (1 + 0.2 Ms_j^2) (DFB_FLUX_MASS) or 1 (DFB_FLUX_VOLUME); rc0_j = sqrt(R11_j);
// D = sum_jk hy_j hz_k g_j rc0_j; mean = sum_jk hy_j hz_k rhos_j Us_j (mass) or hy_j hz_k Us_j (volume).
// With per-cell profiles (plan.cells) g, rc0 and the mean flux are per cell: m' = sum_j wy_j sum_k wz_jk u'_jk with wy_j = hy_j and
// wz_jk = g_jk hz_k, u' <- u' - c rc0_jk, D = sum_j hy_j sum_k wz_jk rc0_jk.
struct FluxTables {
    int mode = 0;
    std::vector<double> wy, rc0;                 // [Ny]; rc0 empty with per-cell profiles
    std::vector<double> hz;                      // [NzG]
    std::vector<double> wz;                      // [Ny][NzG] per-cell profiles only, else empty
    double D = 0, mean = 0;
};
// Throws DFB_ERR_ARG for a mode other than DFB_FLUX_MASS / DFB_FLUX_VOLUME, a slab plan, or D = 0.
FluxTables flux_tables(const Plan& plan, int mode);

// pieces, exposed for unit tests through the C ABI
void coefficients(int N, int shape /* DFB_FILTER_* */, double* b /* 2N+1 */);
std::vector<double> linear_interpolate(const std::vector<double>& y_data, const std::vector<double>& f_data,
                                       const std::vector<double>& y_new);

}  // namespace dfb
