// csrc/fluxtables.cpp -- host tables of the inflow mass-flux correction (dfb_set_flux_correction).  No CUDA call, no environment.
#include <cmath>
#include <string>
#include "plan.hpp"

namespace dfb {

// The cells are those of the area face maps: [vert_y[j], vert_y[j+1]) x [vert_z[k], vert_z[k+1]), area hy_j hz_k.  The mass flux of a
// cell to first order in the fluctuations is rhos u' + Us rho' = rhos (1 - rc4 Us) u' with the epilogue's rho' = -rc4 rhos u' and
// rc4 = -0.2 Ms^2 / Us (stepplan.cpp): g_j = rhos_j (1 + 0.2 Ms_j^2), written without the division so that a row with Us = 0 stays finite.
FluxTables flux_tables(const Plan& P, int mode) {
    if (mode != DFB_FLUX_MASS && mode != DFB_FLUX_VOLUME)
        throw Error{DFB_ERR_ARG, "unknown flux correction mode " + std::to_string(mode) +
                                     " (DFB_FLUX_OFF = 0, DFB_FLUX_MASS = 1, DFB_FLUX_VOLUME = 2)"};
    if (P.k0 != 0 || P.k1 != P.NzG)
        throw Error{DFB_ERR_ARG, "the flux correction needs the whole plane: a slab handle (k_begin, k_end) cannot form the plane's sum"};
    const int Ny = P.Ny, NzG = P.NzG;
    const double* R11 = P.rows.data();
    const double* Us = R11 + (size_t)4 * Ny;
    const double* rhos = R11 + (size_t)6 * Ny;
    const double* Ms = R11 + (size_t)7 * Ny;
    FluxTables T;
    T.mode = mode;
    T.wy.resize(Ny);
    T.rc0.resize(Ny);
    T.hz.resize(NzG);
    double Z = 0.0;
    for (int k = 0; k < NzG; ++k) {
        T.hz[k] = P.vert_z[k + 1] - P.vert_z[k];
        Z += T.hz[k];
    }
    double d = 0.0, mean = 0.0;
    if (P.cells) {
        // per-cell profiles: wy_j = hy_j, and g_jk hz_k per cell in wz
        const double* C = P.cells->data();
        const size_t n = (size_t)Ny * NzG;
        T.wz.resize(n);
        for (int j = 0; j < Ny; ++j) {
            const double hy = P.vert_y[j + 1] - P.vert_y[j];
            double dj = 0.0, mj = 0.0;
            for (int k = 0; k < NzG; ++k) {
                const size_t i = (size_t)j * NzG + k;
                const double r11 = C[i], us = C[4 * n + i], rho = C[6 * n + i], ms = C[7 * n + i];
                const double g = mode == DFB_FLUX_MASS ? rho * (1.0 + 0.2 * ms * ms) : 1.0;
                T.wz[i] = g * T.hz[k];
                dj += T.wz[i] * std::sqrt(r11);             // sqrt(R11): the per-cell constant rc0 (profile_consts), bit for bit
                mj += T.hz[k] * (mode == DFB_FLUX_MASS ? rho * us : us);
            }
            T.wy[j] = hy;
            d += hy * dj;
            mean += hy * mj;
        }
        T.rc0.clear();
        T.D = d;
        T.mean = mean;
    } else {
        for (int j = 0; j < Ny; ++j) {
            const double hy = P.vert_y[j + 1] - P.vert_y[j];
            const double g = mode == DFB_FLUX_MASS ? rhos[j] * (1.0 + 0.2 * Ms[j] * Ms[j]) : 1.0;
            T.rc0[j] = std::sqrt(R11[j]);                       // the epilogue's rowc[0] (stepplan.cpp), bit for bit
            T.wy[j] = g * hy;
            d += T.wy[j] * T.rc0[j];
            mean += hy * (mode == DFB_FLUX_MASS ? rhos[j] * Us[j] : Us[j]);
        }
        T.D = d * Z;
        T.mean = mean * Z;
    }
    if (!(T.D > 0.0) || !std::isfinite(T.D))
        throw Error{DFB_ERR_ARG, std::string("the flux correction needs sum A g sqrt(R11) > 0: R11 is zero on every ") + (P.cells ? "cell" : "row") + " of this plane"};
    return T;
}

}  // namespace dfb
