// csrc/setup.cpp -- one-time host setup: the part of DIGITAL_FILTER::DIGITAL_FILTER (df.cpp:4-66) that
// runs before the first sweep.  It is executed once per handle, on the host, with the host's libm
// (exp / tanh / sqrt), exactly like the reference, so that no device transcendental ever enters
// the parity gate (SURVEY 8c "third-party arithmetic").  Expression order follows the cited lines:
// the resulting tables are bit-identical to the reference object's (tests/test_gpu_parity.py::
// test_G2_default_plane_against_reference_object_code compares rows, half-widths, coefficients and Lt
// with the running reference object; tests/test_oracle_vs_ref.py pins the restatement they are checked with).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <algorithm>
#include "plan.hpp"

namespace dfb {

namespace {

constexpr double pi_c = -2.0 * 3.14159265358979323846;   // df.hpp:16

std::string cstr(const char* p, int len) {
    if (!p) return std::string();
    if (len < 0) return std::string(p);
    std::string s(p, p + len);
    while (!s.empty() && (s.back() == ' ' || s.back() == '\0')) s.pop_back();   // Fortran blank padding
    return s;
}

// One VARIABLES line, one "ZONE ... i=N" line, then rows of whitespace-separated numbers
// (df.cpp:231-278 and 498-537 parse both files this way).
std::vector<std::vector<double>> read_zone_file(const std::string& path, int& n_rows) {
    std::ifstream fin(path);
    if (!fin) throw Error{DFB_ERR_IO, "cannot open input file '" + path + "' (df.cpp:225/492)"};
    std::string line;
    std::getline(fin, line);
    std::getline(fin, line);
    double n_in = 0;
    size_t pos = line.find("i=");
    if (pos == std::string::npos) throw Error{DFB_ERR_IO, "no 'i=' count on line 2 of '" + path + "'"};
    {
        std::istringstream iss(line.substr(pos + 2));
        iss >> n_in;
    }
    n_rows = (int)n_in;
    if (n_rows < 2) throw Error{DFB_ERR_INTERP, "Need at least two data points to interpolate. (" + path + ")"};
    std::vector<std::vector<double>> rows;
    while (std::getline(fin, line)) {
        if (line.empty()) continue;
        std::istringstream iss(line);
        std::vector<double> v;
        double x;
        while (iss >> x) v.push_back(x);
        if (v.empty()) continue;
        if ((int)rows.size() < n_rows) rows.push_back(std::move(v));
    }
    if ((int)rows.size() < n_rows)
        throw Error{DFB_ERR_IO, "'" + path + "' announces more rows than it holds"};
    return rows;
}

}  // namespace

// Clamped piecewise-linear resampling of a tabulated profile onto new abscissae (the job of df.cpp:805-848).
// The table is ascending, so the bracketing interval is found by bisection; the reference walks the table
// from the start for every point, which lands on the same interval.  Only the interpolation expression
// itself is kept in the reference's operand order, because the row tables must come out bit-identical.
std::vector<double> linear_interpolate(const std::vector<double>& xs, const std::vector<double>& fs,
                                       const std::vector<double>& at) {
    const size_t n = xs.size();
    if (fs.size() != n) throw Error{DFB_ERR_INTERP, "interpolation table: abscissae and values differ in length"};
    if (n < 2) throw Error{DFB_ERR_INTERP, "interpolation table needs at least two points"};
    std::vector<double> out;
    out.reserve(at.size());
    for (double q : at) {
        if (q <= xs[0]) { out.push_back(fs[0]); continue; }           // below the table: first value
        if (q >= xs[n - 1]) { out.push_back(fs[n - 1]); continue; }   // above the table: last value
        const size_t hi = (size_t)(std::lower_bound(xs.begin() + 1, xs.end(), q) - xs.begin());   // first knot >= q
        const size_t lo = hi - 1;
        const double w = (q - xs[lo]) / (xs[hi] - xs[lo]);
        out.push_back(fs[lo] + (fs[hi] - fs[lo]) * w);
    }
    return out;
}

// Filter coefficients of half-width N (df.cpp:166-177 == 202-216), normalised to unit energy.  DFB_FILTER_EXPONENTIAL: the
// reference's two-sided exponential exp(-2 pi |i| / N).  DFB_FILTER_GAUSSIAN: Klein, Sadiki & Janicka's exp(-pi i^2 / (2 n^2)) with
// n = N / 2, i.e. exp(-2 pi i^2 / N^2), whose correlation exp(-pi d^2 / (4 n^2)) has an integral scale of n cells.  One side is
// evaluated and mirrored; the energy is accumulated from the centre outwards in the reference's order (t_0^2, then 2 t_i^2) so that
// the exponential table is bit-identical to its by / bz.  N = 0: [1] in either shape.
void coefficients(int N, int shape, double* b) {
    if (N == 0) { b[0] = 1.0; return; }
    double* mid = b + N;
    double energy = 0.0;
    for (int i = 0; i <= N; ++i) {
        const double t = shape == DFB_FILTER_GAUSSIAN ? std::exp(pi_c * ((double)i * i) / ((double)N * N)) : std::exp(pi_c * i / N);
        mid[i] = t;
        energy += (i ? 2.0 : 1.0) * t * t;
    }
    const double norm = std::sqrt(energy);
    for (int i = 0; i <= N; ++i) mid[i] /= norm;
    for (int i = 1; i <= N; ++i) mid[-i] = mid[i];
}

void build_coef_table(Plan& P) {
    int Nmax = 0;
    for (int f = 0; f < 3; ++f) Nmax = std::max({Nmax, P.f[f].Ny_max, P.f[f].Nz_max});
    std::vector<char> present(Nmax + 1, 0);
    for (int f = 0; f < 3; ++f) {
        const FieldPlan& F = P.f[f];
        if (F.row_uniform) { for (int j = 0; j < P.Ny; ++j) { present[F.N_y_row[j]] = 1; present[F.N_z_row[j]] = 1; } }
        else { for (int v : F.N_y) present[v] = 1; for (int v : F.N_z) present[v] = 1; }
    }
    P.coef.Nmax = Nmax;
    P.coef.ptr.assign(Nmax + 1, -1);
    int64_t total = 0;
    for (int N = 0; N <= Nmax; ++N) if (present[N]) { P.coef.ptr[N] = total; total += 2 * N + 1; }
    P.coef.vals.assign(total, 0.0);
    for (int N = 0; N <= Nmax; ++N)
        if (present[N]) coefficients(N, P.filter_shape, P.coef.vals.data() + P.coef.ptr[N]);   // N = 0 only through explicit N arrays
}

void build_plan(const dfb_config& cfg, Plan& P) {
    // ---- flow constants: df.cpp:7-16 (the C++ reference ignores DFConfig); df.f90:80-87 honours it
    if (cfg.honor_flow_config) {
        if (!(cfg.d_i > 0) || !(cfg.U_e > 0)) throw Error{DFB_ERR_ARG, "honor_flow_config needs d_i > 0 and U_e > 0"};
        P.d_i = cfg.d_i; P.rho_e = cfg.rho_e; P.U_e = cfg.U_e; P.mu = cfg.mu_e;
    } else {
        P.d_i = 0.0013; P.rho_e = 0.044; P.U_e = 869.1; P.mu = 7.1212e-6;
    }
    P.gcon = 287.0;
    const double d_i = P.d_i;

    // ---- geometry: read_grid, df.cpp:71-118 ----
    const bool default_grid = (cfg.Ny == 0 && cfg.Nz == 0);
    int Ny, NzG;
    bool per_row;
    std::vector<double> yc, dy, dz;   // per row or per cell
    if (default_grid) {
        Ny = 560; NzG = 400; per_row = true;                     // df.cpp:73-74
        std::vector<double> y(Ny + 1);
        double y_max = 3 * d_i, a = 2.0;                          // df.cpp:92-94
        for (int j = Ny; j >= 0; --j) {
            double eta = ((j) * y_max / (Ny + 1)) / y_max;        // df.cpp:98
            y[std::abs(j - Ny)] = y_max * (1 - std::tanh(a * eta) / std::tanh(a));   // df.cpp:99
        }
        yc.resize(Ny); dy.resize(Ny); dz.assign(Ny, 0.000133);    // df.cpp:108
        for (int j = 0; j < Ny; ++j) {
            dy[j] = y[j + 1] - y[j];                              // df.cpp:107
            yc[j] = 0.25 * (y[j] + y[j + 1] + y[j] + y[j + 1]);   // df.cpp:109-112 (grid is z-independent)
        }
    } else {
        if (cfg.Ny <= 0 || cfg.Nz <= 0) throw Error{DFB_ERR_ARG, "Ny and Nz must both be positive (or both 0)"};
        Ny = cfg.Ny; NzG = cfg.Nz; per_row = cfg.geom_per_row != 0;
        const bool explicit_N = cfg.N_y && cfg.N_z;
        if (!explicit_N && (!cfg.yc || !cfg.dy || !cfg.dz))
            throw Error{DFB_ERR_ARG, "explicit plane needs yc/dy/dz or N_y/N_z"};
        size_t n = per_row ? (size_t)Ny : (size_t)Ny * NzG;
        if (cfg.yc) yc.assign(cfg.yc, cfg.yc + n);
        if (cfg.dy) dy.assign(cfg.dy, cfg.dy + n);
        if (cfg.dz) dz.assign(cfg.dz, cfg.dz + n);
        if (!cfg.rows && yc.empty()) throw Error{DFB_ERR_ARG, "interpolating the row tables from files needs yc"};
    }
    const size_t gstride = per_row ? 1 : (size_t)NzG;   // index of (j, k=0) = j*gstride
    const int Ny_in = Ny;                                // rows as the caller laid its arrays out (the DNS-range trim below may shorten Ny)
    for (double v : dy) if (!(v > 0)) throw Error{DFB_ERR_ARG, "cell heights dy must be positive"};
    for (double v : dz) if (!(v > 0)) throw Error{DFB_ERR_ARG, "cell widths dz must be positive"};

    // ---- row tables: get_RST_in df.cpp:220-330, read_line_file df.cpp:487-553 ----
    if (cfg.rows) {
        P.rows.assign(cfg.rows, cfg.rows + (size_t)8 * Ny);
    } else {
        std::string rst_path = cstr(cfg.vel_fluc_file, cfg.vel_fluc_file_len);
        if (rst_path.empty()) rst_path = "../files/RST.dat";      // df.cpp:224
        std::string line_path = cstr(cfg.line_file, cfg.line_file_len);
        if (line_path.empty()) line_path = "../line.dat";          // df.cpp:16
        int N_in = 0;
        std::vector<double> yin_d, urms, vrms, wrms, uv;
        if (cfg.vel_file_offset > 0) {
            // The DNS statistics file itself (M6Tw025_Stat.dat layout), as the Fortran caller configures it
            // (fortran-main.f90:17-19: vel_file_offset = 142 header lines, vel_file_N_values = 330 rows).  Column
            // choice as in the reference's preprocessor RST.cpp:43-50: y/delta = col 1, urms = 8, "v" (wall-normal)
            // = col 10, "w" = col 9, u'v' = col 15.
            std::ifstream fin(rst_path);
            if (!fin) throw Error{DFB_ERR_IO, "cannot open input file '" + rst_path + "' (df.f90:327-330)"};
            std::string line;
            for (int i = 0; i < cfg.vel_file_offset; ++i) std::getline(fin, line);
            while (std::getline(fin, line)) {
                if (line.empty()) continue;
                std::istringstream iss(line);
                std::vector<double> v;
                double x;
                while (iss >> x) v.push_back(x);
                if (v.size() > 15) {
                    yin_d.push_back(v[1]); urms.push_back(v[8]); vrms.push_back(v[10]); wrms.push_back(v[9]); uv.push_back(v[15]);
                    if (cfg.vel_file_N_values > 0 && (int)yin_d.size() >= cfg.vel_file_N_values) break;
                }
            }
            N_in = (int)yin_d.size();
            if (N_in < 2) throw Error{DFB_ERR_INTERP, "Need at least two data points to interpolate. (" + rst_path + ")"};
        } else {
            auto rst = read_zone_file(rst_path, N_in);
            yin_d.resize(N_in); urms.resize(N_in); vrms.resize(N_in); wrms.resize(N_in); uv.resize(N_in);
            for (int i = 0; i < N_in; ++i) {
                if (rst[i].size() < 6) throw Error{DFB_ERR_IO, "'" + rst_path + "': fewer than 6 columns"};
                yin_d[i] = rst[i][1]; urms[i] = rst[i][2]; vrms[i] = rst[i][3]; wrms[i] = rst[i][4]; uv[i] = rst[i][5];   // :270-275
            }
        }
        // trim Ny to the rows inside the DNS data, df.cpp:282-288
        int new_Ny = 0;
        while (new_Ny < Ny && yc[(size_t)new_Ny * gstride] / d_i <= yin_d[N_in - 1]) new_Ny++;
        if (new_Ny < 2) throw Error{DFB_ERR_ARG, "fewer than 2 rows lie inside the fluctuation file's y/delta range"};
        if (new_Ny != Ny) {
            Ny = new_Ny;
            size_t n = per_row ? (size_t)Ny : (size_t)Ny * NzG;
            yc.resize(n); dy.resize(n); if (dz.size() > n) dz.resize(n);
        }
        std::vector<double> yline(Ny), ydline(Ny);
        for (int j = 0; j < Ny; ++j) { yline[j] = yc[(size_t)j * gstride]; ydline[j] = yline[j] / d_i; }   // :113-116

        int N_line = 0;
        auto ln = read_zone_file(line_path, N_line);
        std::vector<double> y_file(N_line), rho_file(N_line), u_file(N_line), T_file(N_line);
        for (int i = 0; i < N_line; ++i) {
            if (ln[i].size() < 10) throw Error{DFB_ERR_IO, "'" + line_path + "': fewer than 10 columns"};
            y_file[i] = ln[i][1]; rho_file[i] = ln[i][4]; u_file[i] = ln[i][5]; T_file[i] = ln[i][8];   // :530-534
        }
        auto Us = linear_interpolate(y_file, u_file, yline);       // :539
        auto Ts = linear_interpolate(y_file, T_file, yline);       // :541
        auto rhos = linear_interpolate(y_file, rho_file, yline);   // :542
        std::vector<double> Ms(Ny);
        for (int j = 0; j < Ny; ++j) Ms[j] = Us[j] / std::sqrt(1.4 * P.gcon * Ts[j]);   // :544
        double dyf = y_file[1] - y_file[0];                        // :547 (SURVEY quirk 10)
        double du = Us[1] - Us[0];
        P.tau_w = P.mu * du / dyf;
        P.u_tau = std::sqrt(P.tau_w / rhos[0]);
        const double u_tau = P.u_tau;
        std::vector<double> R11_in(N_in), R22_in(N_in), R33_in(N_in), R21_in(N_in);
        for (int j = 0; j < N_in; ++j) {                           // :312-317
            R11_in[j] = urms[j] * urms[j] * u_tau * u_tau;
            R22_in[j] = vrms[j] * vrms[j] * u_tau * u_tau;
            R33_in[j] = wrms[j] * wrms[j] * u_tau * u_tau;
            R21_in[j] = uv[j] * u_tau * u_tau;
        }
        auto R11 = linear_interpolate(yin_d, R11_in, ydline);      // :320-323
        auto R22 = linear_interpolate(yin_d, R22_in, ydline);
        auto R21 = linear_interpolate(yin_d, R21_in, ydline);
        auto R33 = linear_interpolate(yin_d, R33_in, ydline);
        P.rows.resize((size_t)8 * Ny);
        const std::vector<double>* src[8] = {&R11, &R21, &R22, &R33, &Us, &Ts, &rhos, &Ms};
        for (int t = 0; t < 8; ++t) std::copy(src[t]->begin(), src[t]->end(), P.rows.begin() + (size_t)t * Ny);
    }
    P.Ny = Ny; P.NzG = NzG;
    P.d_v = d_i / 4500;                                            // df.cpp:326
    P.yc_row.resize(Ny); P.dy_row.resize(Ny);
    for (int j = 0; j < Ny; ++j) {
        P.yc_row[j] = yc.empty() ? 0.0 : yc[(size_t)j * gstride];
        P.dy_row[j] = dy.empty() ? 0.0 : dy[(size_t)j * gstride];
    }

    // ---- coordinates for the opt-in writers: vertices (write_tecplot / plot_rms print y[], z[], df.cpp:99-100) and the
    //      cell centres write_csv derives from them (df.cpp:776-786) ----
    P.vert_y.resize(Ny + 1); P.vert_z.resize(NzG + 1);
    P.csv_yc.resize(Ny); P.csv_zc.resize(NzG);
    if (default_grid) {
        // the reference's vertex grid: y = the tanh stretching, z = k * 0.000133 (df.cpp:92-100); cell centre = mean of the four corners
        const int Ny0 = 560;
        const double y_max = 3 * d_i, a = 2.0;
        std::vector<double> yv(Ny0 + 1);
        for (int j = Ny0; j >= 0; --j) {
            const double eta = ((j) * y_max / (Ny0 + 1)) / y_max;
            yv[std::abs(j - Ny0)] = y_max * (1 - std::tanh(a * eta) / std::tanh(a));
        }
        for (int j = 0; j <= Ny; ++j) P.vert_y[j] = yv[j];
        for (int k = 0; k <= NzG; ++k) P.vert_z[k] = k * 0.000133;
        for (int j = 0; j < Ny; ++j) P.csv_yc[j] = 0.25 * (yv[j] + yv[j] + yv[j + 1] + yv[j + 1]);        // df.cpp:785 (n00,n01,n10,n11)
        for (int k = 0; k < NzG; ++k) P.csv_zc[k] = 0.25 * (k * 0.000133 + (k + 1) * 0.000133 + k * 0.000133 + (k + 1) * 0.000133);   // df.cpp:786
    } else {
        // caller-supplied geometry: vertices from the centres and cell sizes of the first column / first row
        for (int j = 0; j < Ny; ++j) {
            const double c = yc.empty() ? (double)j + 0.5 : yc[(size_t)j * gstride];
            const double hgt = dy.empty() ? 1.0 : dy[(size_t)j * gstride];
            P.csv_yc[j] = yc.empty() ? 0.0 : c;
            P.vert_y[j] = c - 0.5 * hgt;
            if (j == Ny - 1) P.vert_y[Ny] = c + 0.5 * hgt;
        }
        double zacc = 0.0;
        for (int k = 0; k < NzG; ++k) {
            const double w = dz.empty() ? 1.0 : (per_row ? dz[0] : dz[k]);
            P.vert_z[k] = zacc;
            P.csv_zc[k] = zacc + 0.5 * w; zacc += w;
        }
        P.vert_z[NzG] = zacc;
    }

    // ---- slab ----
    if (cfg.k_begin == 0 && cfg.k_end == 0) { P.k0 = 0; P.k1 = NzG; }
    else {
        if (cfg.k_begin < 0 || cfg.k_end > NzG || cfg.k_begin >= cfg.k_end)
            throw Error{DFB_ERR_ARG, "slab [k_begin,k_end) must lie inside [0,Nz)"};
        P.k0 = cfg.k_begin; P.k1 = cfg.k_end;
    }

    // ---- integral scales, df.cpp:35-45 ----
    if (cfg.scales) {
        for (int f = 0; f < 3; ++f) { P.f[f].Iz_inn = cfg.scales[3 * f]; P.f[f].Iz_out = cfg.scales[3 * f + 1]; P.f[f].Lt = cfg.scales[3 * f + 2]; }
    } else {
        P.f[0].Iz_out = 0.4 * d_i; P.f[0].Iz_inn = 150 * P.d_v; P.f[0].Lt = 0.8 * d_i / P.U_e;
        P.f[1].Iz_out = 0.3 * d_i; P.f[1].Iz_inn = 75 * P.d_v;  P.f[1].Lt = 0.3 * d_i / P.U_e;
        P.f[2].Iz_out = 0.4 * d_i; P.f[2].Iz_inn = 150 * P.d_v; P.f[2].Lt = 0.3 * d_i / P.U_e;
    }
    for (int f = 0; f < 3; ++f)
        if (!(P.f[f].Lt > 0)) throw Error{DFB_ERR_ARG, "Lagrangian time scale Lt must be positive"};

    // ---- half-widths: calculate_filter_properties, df.cpp:144-154 and 186-195 ----
    const size_t ncol = per_row ? 1 : (size_t)NzG;
    for (int f = 0; f < 3; ++f) {
        FieldPlan& F = P.f[f];
        std::vector<int> Ny_arr((size_t)Ny * ncol), Nz_arr((size_t)Ny * ncol);
        if (cfg.N_y && cfg.N_z) {
            const int* sy = cfg.N_y + (size_t)f * Ny_in * ncol;      // caller's layout: [3][Ny_in * ncol], untrimmed
            const int* sz = cfg.N_z + (size_t)f * Ny_in * ncol;
            for (size_t i = 0; i < Ny_arr.size(); ++i) {
                if (sy[i] < 0 || sz[i] < 0) throw Error{DFB_ERR_ARG, "half-widths must be >= 0"};
                Ny_arr[i] = sy[i]; Nz_arr[i] = sz[i];
            }
        } else {
            for (size_t idx = 0; idx < Ny_arr.size(); ++idx) {
                double Iz = F.Iz_inn + (F.Iz_out - F.Iz_inn) * 0.5 * (1 + std::tanh((yc[idx] / d_i - 0.2) / 0.03));   // :146
                double n_int = std::max(1.0, Iz / dz[idx]);        // :147
                Nz_arr[idx] = 2 * static_cast<int>(n_int);         // :148
                double Iy = 0.67 * Iz;                             // :187
                n_int = std::max(1.0, Iy / dy[idx]);               // :188
                Ny_arr[idx] = 2 * static_cast<int>(n_int);         // :189
            }
        }
        F.Ny_max = *std::max_element(Ny_arr.begin(), Ny_arr.end());   // :153,194 (over the whole plane)
        F.Nz_max = *std::max_element(Nz_arr.begin(), Nz_arr.end());
        F.row_uniform = true;
        F.N_y_row.resize(Ny); F.N_z_row.resize(Ny);
        for (int j = 0; j < Ny; ++j) {
            F.N_y_row[j] = Ny_arr[(size_t)j * ncol]; F.N_z_row[j] = Nz_arr[(size_t)j * ncol];
            for (size_t k = 1; k < ncol && F.row_uniform; ++k)
                if (Ny_arr[(size_t)j * ncol + k] != F.N_y_row[j] || Nz_arr[(size_t)j * ncol + k] != F.N_z_row[j])
                    F.row_uniform = false;
        }
        if (!F.row_uniform) { F.N_y = std::move(Ny_arr); F.N_z = std::move(Nz_arr); }
    }

    // ---- spanwise-periodic plane: a window may wrap at most once around the plane ----
    if (cfg.periodic_z != 0 && cfg.periodic_z != 1) throw Error{DFB_ERR_ARG, "periodic_z must be 0 or 1"};
    P.periodic = cfg.periodic_z == 1;
    P.kernel_variant = cfg.kernel_variant;
    if (P.periodic)
        for (int f = 0; f < 3; ++f)
            if (P.f[f].Nz_max > NzG)
                throw Error{DFB_ERR_ARG, std::string("periodic_z: field ") + "uvw"[f] + " has Nz_max = " + std::to_string(P.f[f].Nz_max) +
                                             " > Nz = " + std::to_string(NzG) + " (a z window may wrap around the plane at most once)"};

    // ---- coefficient table keyed by N ----
    P.filter_shape = DFB_FILTER_EXPONENTIAL;
    build_coef_table(P);

    // ---- algorithmic work of one step on the local slab (SURVEY 8d: F_alg = 2 * taps) ----
    P.taps_per_step = 0;
    for (int f = 0; f < 3; ++f) {
        const FieldPlan& F = P.f[f];
        for (int j = 0; j < Ny; ++j) {
            if (F.row_uniform) P.taps_per_step += (int64_t)(P.k1 - P.k0) * ((2 * F.N_y_row[j] + 1) + (2 * F.N_z_row[j] + 1));
            else for (int k = P.k0; k < P.k1; ++k)
                P.taps_per_step += (2 * F.N_y[(size_t)j * NzG + k] + 1) + (2 * F.N_z[(size_t)j * NzG + k] + 1);
        }
    }
}

void check_time_scales(const Plan& P, const double* Lt_rows) {
    static const char* const name[3] = {"u", "v", "w"};
    for (int f = 0; f < 3; ++f)
        for (int j = 0; j < P.Ny; ++j) {
            const double v = Lt_rows[(size_t)f * P.Ny + j];
            if (std::isfinite(v) && v > 0.0) continue;
            char buf[160];
            std::snprintf(buf, sizeof(buf), "time scale of field %d (%s), row %d is %g: every entry must be finite and > 0", f, name[f], j, v);
            throw Error{DFB_ERR_ARG, buf};
        }
}

void time_scales_from_lengths(const Plan& P, const double Ix[6], double u_min, double* Lt_rows) {
    if (!(std::isfinite(u_min) && u_min > 0.0)) throw Error{DFB_ERR_ARG, "u_min must be finite and > 0"};
    for (int i = 0; i < 6; ++i)
        if (!(std::isfinite(Ix[i]) && Ix[i] > 0.0)) throw Error{DFB_ERR_ARG, "the lengths Ix must be finite and > 0"};
    const double* Us = P.rows.data() + (size_t)4 * P.Ny;
    for (int f = 0; f < 3; ++f) {
        const double inn = Ix[2 * f], out = Ix[2 * f + 1];
        for (int j = 0; j < P.Ny; ++j) {
            const double Ixj = inn + (out - inn) * 0.5 * (1 + std::tanh((P.yc_row[j] / P.d_i - 0.2) / 0.03));   // the Iz blend, df.cpp:146
            Lt_rows[(size_t)f * P.Ny + j] = Ixj / std::max(Us[j], u_min);
        }
    }
}

}  // namespace dfb
