// csrc/profiles.cpp -- per-cell profiles (dfb_set_profiles): the checks of a whole-plane table and the epilogue constants of its cells.
// No CUDA call, no environment.
#include <cstdio>
#include <string>
#include "plan.hpp"

namespace dfb {

namespace {

const char* const QUANTITY[8] = {"R11", "R21", "R22", "R33", "Us", "Ts", "rhos", "Ms"};
// the constants of epilogue_consts; constant c is refused under quantity c
const char* const CONSTANT[PROFILE_CONSTS] = {"sqrt(R11)", "b = R21 / sqrt(R11)", "sqrt(R22 - b^2)", "sqrt(R33)", "-0.2 Ms^2 / Us", "Ts", "rhos"};

std::string at(int j, int k) { return " at row " + std::to_string(j) + ", column " + std::to_string(k); }

std::string num(double v) {
    char buf[32];
    std::snprintf(buf, sizeof(buf), "%.17g", v);
    return buf;
}

}  // namespace

std::vector<double> profile_consts(const Plan& P, const double* cells) {
    const int Ny = P.Ny, NzG = P.NzG, W = P.Nz();
    const size_t plane = (size_t)Ny * NzG, n = (size_t)Ny * W;
    std::vector<double> out((size_t)PROFILE_CONSTS * n);
    for (int j = 0; j < Ny; ++j)
        for (int k = 0; k < NzG; ++k) {
            double q[8], rc[PROFILE_CONSTS];
            for (int i = 0; i < 8; ++i) {
                q[i] = cells[(size_t)i * plane + (size_t)j * NzG + k];
                if (!std::isfinite(q[i]))
                    throw Error{DFB_ERR_ARG, std::string("dfb_set_profiles: ") + QUANTITY[i] + at(j, k) + " is not finite (" + num(q[i]) + ")"};
            }
            epilogue_consts(q, rc);
            for (int c = 0; c < PROFILE_CONSTS; ++c)
                if (!std::isfinite(rc[c]))
                    throw Error{DFB_ERR_ARG, std::string("dfb_set_profiles: ") + QUANTITY[c] + at(j, k) + " gives " + CONSTANT[c] +
                                                 " = " + num(rc[c]) + " (R11 = " + num(q[0]) + ", R21 = " + num(q[1]) + ", R22 = " +
                                                 num(q[2]) + ", R33 = " + num(q[3]) + ", Us = " + num(q[4]) + ", Ms = " + num(q[7]) + ")"};
            if (k >= P.k0 && k < P.k1)
                for (int c = 0; c < PROFILE_CONSTS; ++c) out[(size_t)c * n + (size_t)j * W + (k - P.k0)] = rc[c];
        }
    return out;
}

std::vector<double> profile_columns(const Plan& P, const double* cells) {
    const int Ny = P.Ny, NzG = P.NzG, W = P.Nz();
    std::vector<double> out((size_t)8 * Ny * W);
    for (int i = 0; i < 8; ++i)
        for (int j = 0; j < Ny; ++j)
            for (int k = 0; k < W; ++k)
                out[((size_t)i * Ny + j) * W + k] = cells[((size_t)i * Ny + j) * NzG + P.k0 + k];
    return out;
}

}  // namespace dfb
