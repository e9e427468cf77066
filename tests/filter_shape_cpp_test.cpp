// tests/filter_shape_cpp_test.cpp -- the C++ facade's filter shape (include/digital_filter.hpp: DFConfigEx::filter_shape,
// filter_shape()) on the reference's default plane, run from a directory whose ../files/RST.dat and ../line.dat are the reference's
// inputs.  The facade's Gaussian handle equals one made through the C ABI (skip_first_step, dfb_set_filter_shape, dfb_first_step) bit
// for bit; it runs the direct forms; a handle that has stepped refuses the call.
//   usage: filter_shape_cpp_test      prints "FILTER_SHAPE_OK <Ny>" or exits non-zero
#include <cstdio>
#include <cstring>
#include <vector>
#include "digital_filter.hpp"

int main() {
    DFConfigEx c;
    c.seed = 77;
    c.filter_shape = DFB_FILTER_GAUSSIAN;
    DIGITAL_FILTER a(c);
    if (a.filter_shape() != DFB_FILTER_GAUSSIAN) return 3;
    dfb_config k;
    dfb_config_init(&k);
    k.seed = 77;
    k.skip_first_step = 1;
    dfb_handle b = nullptr;
    if (dfb_create(&k, &b) != DFB_OK || dfb_set_filter_shape(b, DFB_FILTER_GAUSSIAN) != DFB_OK || dfb_first_step(b) != DFB_OK) {
        std::fprintf(stderr, "C ABI: %s\n", dfb_last_error());
        return 4;
    }
    int64_t tuned = 0, zmode = 1, yform = 1;
    if (dfb_info(a.handle(), 3, 0, &tuned) != DFB_OK || dfb_info(a.handle(), 7, 0, &zmode) != DFB_OK ||
        dfb_info(a.handle(), 10, 0, &yform) != DFB_OK || tuned != 1 || zmode != 0 || yform != 0) return 5;
    const int Ny = a.get_Ny(), Nz = a.get_Nz();
    for (int s = 0; s < 4; ++s) {
        a.filter(1e-6 * (1 + s));
        if (dfb_filter(b, 1e-6 * (1 + s)) != DFB_OK) return 6;
    }
    std::vector<double> x((size_t)Ny * Nz), y((size_t)Ny * Nz);
    for (int w = 0; w < 8; ++w) {
        if (dfb_get_field(a.handle(), w, x.data(), 0) != DFB_OK || dfb_get_field(b, w, y.data(), 0) != DFB_OK) return 7;
        if (std::memcmp(x.data(), y.data(), x.size() * sizeof(double)) != 0) { std::fprintf(stderr, "field %d differs\n", w); return 8; }
    }
    if (dfb_set_filter_shape(a.handle(), DFB_FILTER_EXPONENTIAL) != DFB_ERR_STATE) return 9;
    dfb_destroy(b);
    std::printf("FILTER_SHAPE_OK %d\n", Ny);
    return 0;
}
