/* tests/fortran_filter_shape_mimic.c -- the filter shape of fortran/digital_filtering.f90 (config%filter_shape in create_digital_filter,
 * set_filter_shape) made the way a Fortran compiler makes the calls, as tests/fortran_abi_mimic.c does for the rest of the module: the
 * config as fill_config leaves it (skip_first_step = 1 for another shape), every scalar by reference through dfb_set_filter_shape_f,
 * then dfb_first_step (the handle by value, as the module binds it).  Handle A is made that way, handle B through the C ABI; both take
 * the same steps through dfb_filter_to_host_f and must agree bit for bit.
 *   usage: fortran_filter_shape_mimic <RST.dat> <line.dat>      prints "FILTER_SHAPE_OK Ny" or exits non-zero */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "dfb200.h"

static void blank_pad(char* dst, const char* src, int n) {
    int l = (int)strlen(src);
    memset(dst, ' ', (size_t)n);
    memcpy(dst, src, (size_t)(l < n ? l : n));
}
static int len_trim(const char* s, int n) {
    while (n > 0 && s[n - 1] == ' ') --n;
    return n;
}

int main(int argc, char** argv) {
    if (argc < 3) { fprintf(stderr, "usage: %s RST.dat line.dat\n", argv[0]); return 2; }
    char vel_fluc_file[256], line_file[256];
    blank_pad(vel_fluc_file, argv[1], 256);
    blank_pad(line_file, argv[2], 256);
    dfb_config c;
    if (dfb_config_init(&c) != DFB_OK) return 3;
    c.d_i = 0.0013; c.rho_e = 0.044; c.U_e = 869.1; c.mu_e = 7.1212e-6;
    c.vel_file_offset = 0; c.vel_file_N_values = 330;
    c.honor_flow_config = 1;
    c.vel_fluc_file = vel_fluc_file; c.vel_fluc_file_len = len_trim(vel_fluc_file, 256);
    c.line_file = line_file;         c.line_file_len = len_trim(line_file, 256);
    c.seed = 4242; c.device = -1;
    c.skip_first_step = 1;                                        /* fill_config: filter_shape /= FILTER_EXPONENTIAL */

    dfb_handle a = NULL, b = NULL;
    const int shape = DFB_FILTER_GAUSSIAN;
    if (dfb_create_f(&c, &a) != DFB_OK || dfb_set_filter_shape_f(&a, &shape) != DFB_OK || dfb_first_step(a) != DFB_OK) {
        fprintf(stderr, "module path: %s\n", dfb_last_error()); return 4;
    }
    if (dfb_create(&c, &b) != DFB_OK || dfb_set_filter_shape(b, DFB_FILTER_GAUSSIAN) != DFB_OK || dfb_first_step(b) != DFB_OK) {
        fprintf(stderr, "C ABI: %s\n", dfb_last_error()); return 5;
    }
    int64_t v = -1;
    if (dfb_info(a, 17, 0, &v) != DFB_OK || v != DFB_FILTER_GAUSSIAN) return 6;
    int Ny = 0, Nz = 0;
    if (dfb_dims_f(&a, &Ny, &Nz) != DFB_OK) return 7;
    const size_t cells = (size_t)Ny * (size_t)Nz;
    double* x = malloc(8 * 5 * cells);
    double* y = malloc(8 * 5 * cells);
    const double dts[4] = {1e-6, 3e-6, 2e-6, 5e-6};
    for (int s = 0; s < 4; ++s) {
        if (dfb_filter_to_host_f(&a, &dts[s], x, x + cells, x + 2 * cells, x + 3 * cells, x + 4 * cells) != DFB_OK) return 8;
        if (dfb_filter_to_host_f(&b, &dts[s], y, y + cells, y + 2 * cells, y + 3 * cells, y + 4 * cells) != DFB_OK) return 9;
        if (memcmp(x, y, 8 * 5 * cells) != 0) { fprintf(stderr, "step %d differs\n", s); return 10; }
    }
    const int bad = 5;
    if (dfb_set_filter_shape_f(&a, &bad) != DFB_ERR_ARG) return 11;
    if (dfb_set_filter_shape_f(&a, &shape) != DFB_ERR_STATE) return 12;   /* it has stepped */
    printf("FILTER_SHAPE_OK %d\n", Ny);
    dfb_destroy_f(&a); dfb_destroy_f(&b);
    free(x); free(y);
    return 0;
}
