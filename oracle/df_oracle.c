/* oracle/df_oracle.c -- TEST INFRASTRUCTURE ONLY (tests/, __graft_entry__.smoke(), bench.py's CPU legs).
 *
 * Plain-C restatement of the reference's per-timestep hot path DIGITAL_FILTER::filter(dt)
 * (digital-filtering-c++/df/df.cpp:449-468) and of the numeric part of the one-time setup that feeds
 * it (df.cpp:71-118, 130-218, 805-848).  Every function cites the lines it follows.
 *
 * Arithmetic is kept in the reference's order (sequential fp64 accumulation, taps ascending, no
 * FMA: built with -ffp-contract=off like the reference's x86-64 -O2 build), so that this file is
 * BIT-IDENTICAL to the reference object code in oracle/_ref/libdfref.so; tests/test_oracle_vs_ref.py
 * pins that on the default plane and on synthetic shapes.  The only structural difference is the
 * coefficient storage: keyed by the half-width N (coefficients depend on N alone, df.cpp:168-177)
 * instead of the reference's per-cell ragged copy, so that the 4096x8192 plane, which overflows the
 * reference's `int` offsets (SURVEY quirk 7), still has a CPU oracle.
 *
 * Layouts are the reference's: fields row-major idx = j*Nz + k (df.cpp:106); r_ys is
 * (Ny + 2*Ny_max) x Nz (df.cpp:197); r_zs is Ny x (Nz + 2*Nz_max) (df.cpp:157).
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include "df_oracle.h"

/* df.hpp:16 */
static const double pi_c = -2.0 * 3.14159265358979323846;

/* ---- setup ------------------------------------------------------------------------------------ */

/* read_grid, df.cpp:92-117: the made-up tanh-stretched grid.  y_vert has Ny+1 entries (the grid is
 * identical for every k), yc/dy have Ny entries.  Ny is the UNTRIMMED row count (560 by default). */
void orc_default_grid(int Ny, double d_i, double* y_vert, double* yc, double* dy) {
    double y_max = 3 * d_i, a = 2.0;
    for (int j = Ny; j >= 0; --j) {
        double eta = ((j) * y_max / (Ny + 1)) / y_max;                 /* df.cpp:98 */
        y_vert[abs(j - Ny)] = y_max * (1 - tanh(a * eta) / tanh(a));   /* df.cpp:99 */
    }
    for (int j = 0; j < Ny; ++j) {
        dy[j] = y_vert[j + 1] - y_vert[j];                             /* df.cpp:107 */
        yc[j] = 0.25 * (y_vert[j] + y_vert[j + 1] + y_vert[j] + y_vert[j + 1]); /* df.cpp:109-112 */
    }
}

/* linear_interpolate, df.cpp:805-848: clamped, linear scan */
void orc_linear_interpolate(int n, const double* y_data, const double* f_data, int m, const double* y_new,
                            double* f_new) {
    for (int j = 0; j < m; ++j) {
        double y = y_new[j];
        if (y <= y_data[0]) { f_new[j] = f_data[0]; continue; }
        if (y >= y_data[n - 1]) { f_new[j] = f_data[n - 1]; continue; }
        int i = 0;
        while (i + 1 < n && y > y_data[i + 1]) ++i;
        double x0 = y_data[i], x1 = y_data[i + 1], f0 = f_data[i], f1 = f_data[i + 1];
        f_new[j] = f0 + (f1 - f0) * ((y - x0) / (x1 - x0));
    }
}

/* calculate_filter_properties, df.cpp:144-154 and 186-195: half-widths of every cell.
 * Returns Nz_max / Ny_max through the pointers. */
void orc_half_widths(int Ny, int Nz, const double* yc, const double* dy, const double* dz, double d_i,
                     double Iz_inn, double Iz_out, int* N_y, int* N_z, int* Ny_max, int* Nz_max) {
    long n = (long)Ny * Nz;
    *Ny_max = 0; *Nz_max = 0;
    for (long idx = 0; idx < n; ++idx) {
        double Iz = Iz_inn + (Iz_out - Iz_inn) * 0.5 * (1 + tanh((yc[idx] / d_i - 0.2) / 0.03)); /* :146 */
        double n_int = fmax(1.0, Iz / dz[idx]);            /* :147 */
        int n_val = 2 * (int)n_int;                        /* :148 */
        N_z[idx] = n_val;
        if (n_val > *Nz_max) *Nz_max = n_val;
        double Iy = 0.67 * Iz;                             /* :187 */
        n_int = fmax(1.0, Iy / dy[idx]);                   /* :188 */
        n_val = 2 * (int)n_int;                            /* :189 */
        N_y[idx] = n_val;
        if (n_val > *Ny_max) *Ny_max = n_val;
    }
}

/* the 2N+1 coefficients of half-width N, df.cpp:166-177 (identically :202-216): b[N + i], i=-N..N.
 * N = 0 only comes from explicit half-width arrays (the reference's geometry gives N >= 2, :148,189), where its expression is
 * exp(0/0): the one tap of the limit N -> 0+, b_0 = 1, as the library's setup defines it. */
void orc_coeffs(int N, double* b) {
    if (N == 0) { b[0] = 1.0; return; }
    double* temp = (double*)malloc(sizeof(double) * (size_t)(N + 1));
    double sum = 0.0;
    for (int i = 0; i <= N; ++i) {
        temp[i] = exp(pi_c * abs(i) / N);
        sum += (i == 0 ? 1.0 : 2.0) * temp[i] * temp[i];
    }
    sum = sqrt(sum);
    for (int i = -N; i <= N; ++i) b[N + i] = temp[abs(i)] / sum;
    free(temp);
}

/* coefficient table keyed by N for every half-width present in N_y/N_z */
typedef struct { int Nmax; double** b; } coef_tab;
static void tab_init(coef_tab* t, int Nmax) { t->Nmax = Nmax; t->b = (double**)calloc((size_t)Nmax + 1, sizeof(double*)); }
static const double* tab_get(coef_tab* t, int N) {
    if (!t->b[N]) { t->b[N] = (double*)malloc(sizeof(double) * (size_t)(2 * N + 1)); orc_coeffs(N, t->b[N]); }
    return t->b[N] + N;   /* centre pointer, like by[offset] (df.cpp:369,374) */
}
static void tab_free(coef_tab* t) { for (int i = 0; i <= t->Nmax; ++i) free(t->b[i]); free(t->b); }

/* ---- hot path ----------------------------------------------------------------------------------- */

/* filtering_sweeps, y part: df.cpp:360-383.  r_ys -> interior of r_zs. */
void orc_sweep_y(int Ny, int Nz, int Ny_max, int Nz_max, const int* N_y, const double* r_ys, double* r_zs) {
    coef_tab tab; tab_init(&tab, Ny_max);
    for (int j = 0; j < Ny; ++j) for (int k = 0; k < Nz; ++k) tab_get(&tab, N_y[(long)j * Nz + k]);
    #pragma omp parallel for schedule(dynamic, 4)
    for (int j = 0; j < Ny; ++j) {
        long r_idy = (long)(j + Ny_max) * Nz;
        long r_idz = (long)j * (Nz + 2 * Nz_max) + Nz_max;
        long idx = (long)j * Nz;
        for (int k = 0; k < Nz; ++k) {
            int N = N_y[idx];
            const double* b = tab.b[N] + N;
            double sum = 0.0;
            for (int i = -N; i <= N; ++i) sum += b[i] * r_ys[r_idy + (long)i * Nz];   /* df.cpp:373-375 */
            r_zs[r_idz] = sum;
            r_idy++; r_idz++; idx++;
        }
    }
    tab_free(&tab);
}

/* filtering_sweeps, z part: df.cpp:386-405.  r_zs (interior = y-filtered, halo columns = raw noise,
 * SURVEY quirk 1) -> filt. */
void orc_sweep_z(int Ny, int Nz, int Nz_max, const int* N_z, const double* r_zs, double* filt) {
    coef_tab tab; tab_init(&tab, Nz_max);
    for (int j = 0; j < Ny; ++j) for (int k = 0; k < Nz; ++k) tab_get(&tab, N_z[(long)j * Nz + k]);
    #pragma omp parallel for schedule(dynamic, 4)
    for (int j = 0; j < Ny; ++j) {
        long r_idz = (long)j * (Nz + 2 * Nz_max) + Nz_max;
        long idx = (long)j * Nz;
        for (int k = 0; k < Nz; ++k) {
            int N = N_z[idx];
            const double* b = tab.b[N] + N;
            double sum = 0.0;
            for (int i = -N; i <= N; ++i) sum += b[i] * r_zs[r_idz + i];   /* df.cpp:397-399 */
            filt[idx] = sum;
            r_idz++; idx++;
        }
    }
    tab_free(&tab);
}

/* correlate_fields, df.cpp:408-417 -- NB the truncated literal pi (SURVEY quirk 2) */
void orc_correlate(long n_cells, const double* filt_old, double* filt, double dt, double Lt) {
    double pi = 3.141592654;
    double alpha = exp(-pi * dt / Lt);
    for (long idx = 0; idx < n_cells; ++idx)
        filt[idx] = filt_old[idx] * sqrt(alpha) + filt[idx] * sqrt(1.0 - alpha);
}

/* apply_RST_scaling, df.cpp:419-447 (Lund / Cholesky with R31 = R32 = 0); filt_old <- filt */
void orc_rst_scaling(int Ny, int Nz, const double* R11, const double* R21, const double* R22, const double* R33,
                     const double* ufilt, const double* vfilt, const double* wfilt,
                     double* ufluc, double* vfluc, double* wfluc,
                     double* ufilt_old, double* vfilt_old, double* wfilt_old) {
    for (int j = 0; j < Ny; ++j) {
        double b;
        if (R11[j] < 1e-10) b = 0.0; else b = R21[j] / sqrt(R11[j]);
        long idx = (long)j * Nz;
        for (int k = 0; k < Nz; ++k) {
            ufluc[idx] = sqrt(R11[j]) * ufilt[idx];
            vfluc[idx] = b * ufilt[idx] + sqrt(R22[j] - b * b) * vfilt[idx];
            wfluc[idx] = sqrt(R33[j]) * wfilt[idx];
            ufilt_old[idx] = ufilt[idx]; vfilt_old[idx] = vfilt[idx]; wfilt_old[idx] = wfilt[idx];
            idx++;
        }
    }
}

/* get_rho_T_fluc, df.cpp:470-485 (Strong Reynolds Analogy; the code's 0.5 factor, not the README's) */
void orc_sra(int Ny, int Nz, const double* Ms, const double* Us, const double* Ts, const double* rhos,
             const double* ufluc, double* T_fluc, double* rho_fluc) {
    for (int j = 0; j < Ny; ++j) {
        double temp1 = -0.5 * (1.4 - 1) * Ms[j] * Ms[j] / Us[j];
        for (int k = 0; k < Nz; ++k) {
            double temp2 = temp1 * ufluc[(long)j * Nz + k];
            T_fluc[(long)j * Nz + k] = temp2 * Ts[j];
            rho_fluc[(long)j * Nz + k] = -temp2 * rhos[j];
        }
    }
}

/* filter(dt), df.cpp:449-461, with the noise already in r_ys / r_zs-halos (H1 is replaced by the
 * counter-based generator or by injection).  first_step != 0 follows the constructor instead
 * (df.cpp:57-62: no blend, no SRA; SURVEY quirk 3).
 *   N_y,N_z    [3][Ny*Nz]          Ny_max,Nz_max [3]         Lt [3]
 *   r_ys[f]    (Ny+2*Ny_max[f]) x Nz                         r_zs[f]  Ny x (Nz+2*Nz_max[f])  (interior overwritten)
 *   rows       [8][Ny] = R11,R21,R22,R33,Us,Ts,rhos,Ms
 *   filt_old   [3][Ny*Nz] in/out   filt, fluc [3][Ny*Nz] out     T_fluc, rho_fluc [Ny*Nz] out */
void orc_step(int Ny, int Nz, const int* const* N_y, const int* const* N_z, const int* Ny_max, const int* Nz_max,
              const double* Lt, const double* rows, double dt, int first_step,
              const double* const* r_ys, double* const* r_zs,
              double* const* filt_old, double* const* filt, double* const* fluc,
              double* T_fluc, double* rho_fluc) {
    long n = (long)Ny * Nz;
    for (int f = 0; f < 3; ++f) {
        orc_sweep_y(Ny, Nz, Ny_max[f], Nz_max[f], N_y[f], r_ys[f], r_zs[f]);
        orc_sweep_z(Ny, Nz, Nz_max[f], N_z[f], r_zs[f], filt[f]);
        if (!first_step) orc_correlate(n, filt_old[f], filt[f], dt, Lt[f]);
    }
    orc_rst_scaling(Ny, Nz, rows + 0 * Ny, rows + 1 * Ny, rows + 2 * Ny, rows + 3 * Ny,
                    filt[0], filt[1], filt[2], fluc[0], fluc[1], fluc[2],
                    filt_old[0], filt_old[1], filt_old[2]);
    if (!first_step)
        orc_sra(Ny, Nz, rows + 7 * Ny, rows + 4 * Ny, rows + 5 * Ny, rows + 6 * Ny, fluc[0], T_fluc, rho_fluc);
}
