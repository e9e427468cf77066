// tests/flux_cpp_test.cpp -- the C++ facade's flux correction (include/digital_filter.hpp: set_flux_correction, flux_correction(),
// flux_info) on the reference's default plane, run from a directory whose ../files/RST.dat and ../line.dat are the reference's inputs.
// The facade's handle equals one corrected through the C ABI bit for bit and reports the same {c, m', mean}; its filt_old equals an
// uncorrected handle's; an unknown mode is refused.
//   usage: flux_cpp_test      prints "FLUX_OK <Ny>" or exits non-zero
#include <cstdio>
#include <cstring>
#include <stdexcept>
#include <vector>
#include "digital_filter.hpp"

int main() {
    DFConfigEx c;
    c.seed = 31;
    DIGITAL_FILTER a(c);
    a.set_flux_correction(DFB_FLUX_MASS);
    if (a.flux_correction() != DFB_FLUX_MASS) return 3;
    dfb_config k;
    dfb_config_init(&k);
    k.seed = 31;
    dfb_handle b = nullptr, off = nullptr;
    if (dfb_create(&k, &b) != DFB_OK || dfb_create(&k, &off) != DFB_OK || dfb_set_flux_correction(b, DFB_FLUX_MASS) != DFB_OK) {
        std::fprintf(stderr, "C ABI: %s\n", dfb_last_error());
        return 4;
    }
    for (int s = 0; s < 4; ++s) {
        a.filter(1e-6 * (1 + s));
        if (dfb_filter(b, 1e-6 * (1 + s)) != DFB_OK || dfb_filter(off, 1e-6 * (1 + s)) != DFB_OK) return 5;
    }
    const int Ny = a.get_Ny(), Nz = a.get_Nz();
    std::vector<double> x((size_t)Ny * Nz), y((size_t)Ny * Nz);
    for (int w = 0; w < 8; ++w) {
        if (dfb_get_field(a.handle(), w, x.data(), 0) != DFB_OK || dfb_get_field(b, w, y.data(), 0) != DFB_OK) return 6;
        if (std::memcmp(x.data(), y.data(), x.size() * sizeof(double)) != 0) { std::fprintf(stderr, "field %d differs\n", w); return 7; }
        if (w >= DFB_U_FILT || w == DFB_V_FLUC || w == DFB_W_FLUC) {
            if (dfb_get_field(off, w, y.data(), 0) != DFB_OK) return 8;
            if (std::memcmp(x.data(), y.data(), x.size() * sizeof(double)) != 0) { std::fprintf(stderr, "field %d differs from off\n", w); return 9; }
        }
    }
    const std::array<double, 3> fa = a.flux_info();
    double fb[3];
    if (dfb_flux_info(b, 0, fb) != DFB_OK || std::memcmp(fa.data(), fb, sizeof(fb)) != 0 || fa[0] == 0.0 || !(fa[2] > 0.0)) return 10;
    bool refused = false;
    try { a.set_flux_correction(7); } catch (const std::runtime_error&) { refused = true; }
    if (!refused || a.flux_correction() != DFB_FLUX_MASS) return 11;
    dfb_destroy(b);
    dfb_destroy(off);
    std::printf("FLUX_OK %d\n", Ny);
    return 0;
}
