// tests/time_scales_cpp_test.cpp -- the C++ facade's per-row time scales (include/digital_filter.hpp: set_time_scales,
// clear_time_scales, time_scales_from_lengths) on the reference's default plane, run from a directory whose ../files/RST.dat and
// ../line.dat are the reference's inputs.  Rows from lengths set through the facade equal the same rows set through the C ABI, bit for
// bit; clearing them is the scalar path again; rows of the wrong size are refused.
//   usage: time_scales_cpp_test      prints "TIME_SCALES_OK <Ny>" or exits non-zero
#include <cstdio>
#include <cstring>
#include <stdexcept>
#include <vector>
#include "digital_filter.hpp"

int main() {
    DFConfigEx c;
    c.seed = 77;
    DIGITAL_FILTER a(c), b(c);
    const int Ny = a.get_Ny(), Nz = a.get_Nz();
    const double Ix[6] = {2e-4, 1.6e-3, 1e-4, 8e-4, 1.5e-4, 1.2e-3};
    const std::vector<double> rows = a.time_scales_from_lengths(Ix, 10.0);
    if ((int)rows.size() != 3 * Ny) return 3;
    a.set_time_scales(rows);
    if (dfb_set_time_scales(b.handle(), rows.data()) != DFB_OK) return 4;
    int64_t on = 0;
    if (dfb_info(a.handle(), 15, 0, &on) != DFB_OK || on != 1) return 5;
    for (int s = 0; s < 4; ++s) { a.filter(1e-6 * (1 + s)); b.filter(1e-6 * (1 + s)); }
    std::vector<double> x((size_t)Ny * Nz), y((size_t)Ny * Nz);
    for (int w = 0; w < 8; ++w) {
        if (dfb_get_field(a.handle(), w, x.data(), 0) != DFB_OK || dfb_get_field(b.handle(), w, y.data(), 0) != DFB_OK) return 6;
        if (std::memcmp(x.data(), y.data(), x.size() * sizeof(double)) != 0) { std::fprintf(stderr, "field %d differs\n", w); return 7; }
    }
    a.clear_time_scales();
    if (dfb_info(a.handle(), 15, 0, &on) != DFB_OK || on != 0) return 8;
    try {
        a.set_time_scales(std::vector<double>(5, 1.0));
        return 9;
    } catch (const std::invalid_argument&) {
    }
    std::printf("TIME_SCALES_OK %d\n", Ny);
    return 0;
}
