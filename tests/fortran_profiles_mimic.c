/* tests/fortran_profiles_mimic.c -- the per-cell profiles of fortran/digital_filtering.f90 (set_profiles, clear_profiles) made the way a
 * Fortran compiler makes the calls, as tests/fortran_abi_mimic.c does for the rest of the module: the table cells(k, j, q) passed by
 * the address of a c_loc through dfb_set_profiles_f, and c_null_ptr to clear.  Handle A is made that way, handle B through the C ABI;
 * both take the same steps through dfb_filter_to_host_f and must agree bit for bit.
 *   usage: fortran_profiles_mimic <RST.dat> <line.dat>      prints "PROFILES_OK Ny" or exits non-zero */
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
    c.seed = 4247; c.device = -1;

    dfb_handle a = NULL, b = NULL;
    if (dfb_create_f(&c, &a) != DFB_OK || dfb_create(&c, &b) != DFB_OK) { fprintf(stderr, "create: %s\n", dfb_last_error()); return 4; }
    int Ny = 0, Nz = 0;
    if (dfb_dims_f(&a, &Ny, &Nz) != DFB_OK) return 5;
    const size_t n = (size_t)Ny * Nz;
    double* cells = malloc(8 * n * sizeof(double));
    double* row = malloc((size_t)Ny * sizeof(double));
    for (int q = 0; q < 8; ++q) {
        if (dfb_get_table(a, q, 0, row, Ny) != DFB_OK) return 6;
        for (int j = 0; j < Ny; ++j)
            for (int k = 0; k < Nz; ++k) cells[(size_t)q * n + (size_t)j * Nz + k] = row[j] * (q == 4 ? 1.0 - 0.3 * k / Nz : 1.0);
    }
    const double* p = cells;
    const double* none = NULL;
    if (dfb_set_profiles_f(&a, &p) != DFB_OK || dfb_set_profiles(b, cells) != DFB_OK) { fprintf(stderr, "set: %s\n", dfb_last_error()); return 7; }
    if (dfb_set_profiles_f(&a, NULL) != DFB_ERR_ARG) return 8;
    double* x = malloc(5 * n * sizeof(double));
    double* y = malloc(5 * n * sizeof(double));
    for (int s = 0; s < 3; ++s) {
        const double dt = 2e-6 * (s + 1);
        if (dfb_filter_to_host_f(&a, &dt, x, x + n, x + 2 * n, x + 3 * n, x + 4 * n) != DFB_OK) return 9;
        if (dfb_filter_to_host(b, dt, y, y + n, y + 2 * n, y + 3 * n, y + 4 * n) != DFB_OK) return 10;
        if (memcmp(x, y, 5 * n * sizeof(double)) != 0) { fprintf(stderr, "step %d differs\n", s); return 11; }
    }
    int64_t m = -1;
    if (dfb_info(a, 19, 0, &m) != DFB_OK || m != 1) return 12;
    if (dfb_set_profiles_f(&a, &none) != DFB_OK || dfb_info(a, 19, 0, &m) != DFB_OK || m != 0) return 13;
    free(x); free(y); free(cells); free(row);
    dfb_destroy_f(&a);
    dfb_destroy(b);
    printf("PROFILES_OK %d\n", Ny);
    return 0;
}
