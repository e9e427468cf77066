/* tests/fortran_time_scales_mimic.c -- the per-row time scale calls of fortran/digital_filtering.f90 (set_time_scales,
 * clear_time_scales, time_scales_from_lengths) made the way a Fortran compiler makes them, as tests/fortran_abi_mimic.c does for the rest
 * of the module: every scalar by reference, the rows as a type(c_ptr) by reference (c_loc of the array; c_null_ptr clears) through
 * dfb_set_time_scales_f and dfb_time_scales_from_lengths_f.  Handle A takes its rows through these, handle B the same rows through the C
 * ABI; both take the same steps and must agree bit for bit.  Then A clears its rows and must equal C, a handle that never set rows,
 * restored to A's state.
 *   usage: fortran_time_scales_mimic <RST.dat> <line.dat>      prints "TIME_SCALES_OK Ny" or exits non-zero */
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

    dfb_handle a = NULL, b = NULL, h = NULL;
    if (dfb_create_f(&c, &a) != DFB_OK || dfb_create_f(&c, &b) != DFB_OK || dfb_create_f(&c, &h) != DFB_OK) {
        fprintf(stderr, "create: %s\n", dfb_last_error()); return 4;
    }
    int Ny = 0, Nz = 0;
    if (dfb_dims_f(&a, &Ny, &Nz) != DFB_OK) return 5;
    const size_t cells = (size_t)Ny * (size_t)Nz;
    const double Ix[6] = {2e-4, 1.6e-3, 1e-4, 8e-4, 1.5e-4, 1.2e-3}, u_min = 10.0;
    double* rows = malloc(8 * 3 * (size_t)Ny);                  /* Lt_rows(Ny, 3): column-major [3][Ny] */
    if (dfb_time_scales_from_lengths_f(&a, Ix, &u_min, rows) != DFB_OK) { fprintf(stderr, "from_lengths: %s\n", dfb_last_error()); return 6; }
    const double* p = rows;
    if (dfb_set_time_scales_f(&a, &p) != DFB_OK) { fprintf(stderr, "set: %s\n", dfb_last_error()); return 7; }
    if (dfb_set_time_scales(b, rows) != DFB_OK) return 8;
    double* x = malloc(8 * 5 * cells);
    double* y = malloc(8 * 5 * cells);
    const double dts[4] = {1e-6, 3e-6, 2e-6, 5e-6};
    for (int s = 0; s < 4; ++s) {
        if (dfb_filter_to_host_f(&a, &dts[s], x, x + cells, x + 2 * cells, x + 3 * cells, x + 4 * cells) != DFB_OK) return 9;
        if (dfb_filter_to_host_f(&b, &dts[s], y, y + cells, y + 2 * cells, y + 3 * cells, y + 4 * cells) != DFB_OK) return 10;
        if (memcmp(x, y, 8 * 5 * cells) != 0) { fprintf(stderr, "step %d differs\n", s); return 11; }
    }
    const double* null_rows = NULL;
    if (dfb_set_time_scales_f(&a, &null_rows) != DFB_OK) return 12;
    int64_t on = 1, step = 0;
    if (dfb_info(a, 15, 0, &on) != DFB_OK || on != 0) return 13;
    double* fo = malloc(8 * 3 * cells);
    if (dfb_get_state(a, fo, &step) != DFB_OK || dfb_set_state(h, fo, step) != DFB_OK) return 14;
    for (int s = 0; s < 4; ++s) {
        if (dfb_filter_to_host_f(&a, &dts[s], x, x + cells, x + 2 * cells, x + 3 * cells, x + 4 * cells) != DFB_OK) return 15;
        if (dfb_filter_to_host_f(&h, &dts[s], y, y + cells, y + 2 * cells, y + 3 * cells, y + 4 * cells) != DFB_OK) return 16;
        if (memcmp(x, y, 8 * 5 * cells) != 0) { fprintf(stderr, "after clearing, step %d differs\n", s); return 17; }
    }
    printf("TIME_SCALES_OK %d\n", Ny);
    dfb_destroy_f(&a); dfb_destroy_f(&b); dfb_destroy_f(&h);
    free(rows); free(x); free(y); free(fo);
    return 0;
}
