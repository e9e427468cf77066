// tests/restart_cpp_test.cpp -- the C++ facade's restart calls: run A takes 2n steps; run B takes n, saves (with its N2 sums) and is
// destroyed; a fresh C loads and takes n more.  Every output of C's steps must equal A's bit for bit, and so must the N2 sums.
// Runs on the reference's default plane from a directory with ../files/RST.dat and ../line.dat (like examples/cpp-main.cpp).
//   usage: restart_cpp_test <restart file>      prints "RESTART_OK n" or exits non-zero
#include <cstdio>
#include <cstring>
#include <vector>
#include "digital_filter.hpp"

static std::vector<double> outputs(const DIGITAL_FILTER& df) {
    std::vector<double> o;
    for (const Vector* v : {&df.u.fluc, &df.v.fluc, &df.w.fluc, &df.T_fluc(), &df.rho_fluc()}) o.insert(o.end(), v->begin(), v->end());
    return o;
}

static std::vector<double> sums(const DIGITAL_FILTER& df, int64_t* count) {
    const size_t n = (size_t)df.get_Ny() * (size_t)df.get_Nz();
    std::vector<double> s(6 * n);
    for (int w = 0; w < 6; ++w)
        if (dfb_stats_get(df.handle(), w, 0, s.data() + w * n, count) != DFB_OK) return {};
    return s;
}

int main(int argc, char** argv) {
    if (argc < 2) return 2;
    const int n = 3;
    const double dts[2 * n] = {1e-6, 2e-7, 0.0, 3e-6, 5e-7, 1e-6};
    std::vector<std::vector<double>> ref;
    std::vector<double> ref_sums;
    int64_t ref_count = 0, count = 0;
    try {
        {
            DIGITAL_FILTER A{DFConfig{}};
            dfb_stats_enable(A.handle(), 1);
            for (int s = 0; s < 2 * n; ++s) { A.filter(dts[s]); if (s >= n) ref.push_back(outputs(A)); }
            ref_sums = sums(A, &ref_count);
        }
        {
            DIGITAL_FILTER B{DFConfig{}};
            dfb_stats_enable(B.handle(), 1);
            for (int s = 0; s < n; ++s) B.filter(dts[s]);
            B.save_restart(argv[1], DFB_RESTART_STATE | DFB_RESTART_STATS);
        }
        DIGITAL_FILTER C{DFConfig{}};
        C.load_restart(argv[1], DFB_RESTART_STATE | DFB_RESTART_STATS);
        for (int s = n; s < 2 * n; ++s) {
            C.filter(dts[s]);
            if (outputs(C) != ref[s - n]) { std::fprintf(stderr, "step %d differs from the uninterrupted run\n", s); return 3; }
        }
        if (sums(C, &count) != ref_sums || count != ref_count || count != 2 * n) { std::fprintf(stderr, "N2 sums differ\n"); return 4; }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 5;
    }
    std::printf("RESTART_OK %d\n", n);
    return 0;
}
