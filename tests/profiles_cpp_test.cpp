// tests/profiles_cpp_test.cpp -- the C++ facade's per-cell profiles (include/digital_filter.hpp: set_profiles, clear_profiles,
// profiles()) on the reference's default plane, run from a directory whose ../files/RST.dat and ../line.dat are the reference's inputs.
// The facade's handle equals one given the same profiles through the C ABI bit for bit; its filt_old equals a handle without profiles;
// a value that is not finite and a table of the wrong size are refused.
//   usage: profiles_cpp_test      prints "PROFILES_OK <Ny>" or exits non-zero
#include <cmath>
#include <cstdio>
#include <cstring>
#include <stdexcept>
#include <vector>
#include "digital_filter.hpp"

int main() {
    DFConfigEx c;
    c.seed = 37;
    DIGITAL_FILTER a(c);
    const int Ny = a.get_Ny(), Nz = a.get_Nz();
    // the row tables, thickened by up to 1.5x towards the last column
    std::vector<double> rows(Ny), cells((size_t)8 * Ny * Nz);
    for (int q = 0; q < 8; ++q) {
        if (dfb_get_table(a.handle(), q, 0, rows.data(), Ny) != DFB_OK) return 2;
        for (int j = 0; j < Ny; ++j)
            for (int k = 0; k < Nz; ++k) cells[((size_t)q * Ny + j) * Nz + k] = rows[j] * (q < 4 ? 1.0 + 0.5 * k / Nz : 1.0);
    }
    if (a.profiles()) return 3;
    a.set_profiles(cells);
    if (!a.profiles()) return 4;
    dfb_config k;
    dfb_config_init(&k);
    k.seed = 37;
    dfb_handle b = nullptr, off = nullptr;
    if (dfb_create(&k, &b) != DFB_OK || dfb_create(&k, &off) != DFB_OK || dfb_set_profiles(b, cells.data()) != DFB_OK) {
        std::fprintf(stderr, "C ABI: %s\n", dfb_last_error());
        return 5;
    }
    for (int s = 0; s < 4; ++s) {
        a.filter(1e-6 * (1 + s));
        if (dfb_filter(b, 1e-6 * (1 + s)) != DFB_OK || dfb_filter(off, 1e-6 * (1 + s)) != DFB_OK) return 6;
    }
    std::vector<double> x((size_t)Ny * Nz), y((size_t)Ny * Nz);
    for (int w = 0; w < 8; ++w) {
        if (dfb_get_field(a.handle(), w, x.data(), 0) != DFB_OK || dfb_get_field(b, w, y.data(), 0) != DFB_OK) return 7;
        if (std::memcmp(x.data(), y.data(), x.size() * sizeof(double)) != 0) { std::fprintf(stderr, "field %d differs\n", w); return 8; }
        if (dfb_get_field(off, w, y.data(), 0) != DFB_OK) return 9;
        const bool same = std::memcmp(x.data(), y.data(), x.size() * sizeof(double)) == 0;
        if (same != (w >= DFB_U_FILT)) { std::fprintf(stderr, "field %d against the handle without profiles\n", w); return 10; }
    }
    bool refused = false;
    std::vector<double> bad = cells;
    bad[5] = std::nan("");
    try { a.set_profiles(bad); } catch (const std::runtime_error&) { refused = true; }
    if (!refused || !a.profiles()) return 11;
    refused = false;
    try { a.set_profiles(std::vector<double>(8)); } catch (const std::invalid_argument&) { refused = true; }
    if (!refused) return 12;
    a.clear_profiles();
    if (a.profiles()) return 13;
    dfb_destroy(b);
    dfb_destroy(off);
    std::printf("PROFILES_OK %d\n", Ny);
    return 0;
}
