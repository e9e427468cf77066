/* tests/fortran_restart_mimic.c -- the restart calls of fortran/digital_filtering.f90 (save_restart / load_restart) made the way a
 * Fortran compiler makes them, as tests/fortran_abi_mimic.c does for the rest of the module: blank-padded character(len=256) paths
 * passed by c_loc + len_trim, every scalar by reference through dfb_save_restart_f / dfb_load_restart_f.  Run A takes 2n steps; run B
 * takes n, saves and is destroyed; a fresh C loads and takes n more, which must equal A's bit for bit.
 *   usage: fortran_restart_mimic <RST.dat> <line.dat> <restart file>      prints "RESTART_OK n" or exits non-zero */
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
    if (argc < 4) { fprintf(stderr, "usage: %s RST.dat line.dat restart\n", argv[0]); return 2; }
    char vel_fluc_file[256], line_file[256], path[256];
    blank_pad(vel_fluc_file, argv[1], 256);
    blank_pad(line_file, argv[2], 256);
    blank_pad(path, argv[3], 256);
    const int path_len = len_trim(path, 256), what = DFB_RESTART_STATE;

    dfb_config c;
    if (dfb_config_init(&c) != DFB_OK) return 3;
    c.d_i = 0.0013; c.rho_e = 0.044; c.U_e = 869.1; c.mu_e = 7.1212e-6;
    c.vel_file_offset = 0; c.vel_file_N_values = 330;
    c.honor_flow_config = 1;
    c.vel_fluc_file = vel_fluc_file; c.vel_fluc_file_len = len_trim(vel_fluc_file, 256);
    c.line_file = line_file;         c.line_file_len = len_trim(line_file, 256);
    c.seed = 12345; c.device = -1;

    enum { n = 3 };
    const double dts[2 * n] = {1e-8, 2e-8, 0.0, 5e-8, 1e-8, 3e-8};
    dfb_handle a = NULL, b = NULL, h = NULL;
    if (dfb_create_f(&c, &a) != DFB_OK || dfb_create_f(&c, &b) != DFB_OK) { fprintf(stderr, "create: %s\n", dfb_last_error()); return 4; }
    int Ny = 0, Nz = 0;
    if (dfb_dims_f(&a, &Ny, &Nz) != DFB_OK) return 5;
    const size_t cells = (size_t)Ny * (size_t)Nz;
    double* ref = malloc(8 * 5 * cells * n);
    double* got = malloc(8 * 5 * cells);
    for (int s = 0; s < 2 * n; ++s) {
        double* o = ref + (size_t)(s < n ? 0 : s - n) * 5 * cells;
        if (dfb_filter_to_host_f(&a, &dts[s], o, o + cells, o + 2 * cells, o + 3 * cells, o + 4 * cells) != DFB_OK) return 6;
    }
    for (int s = 0; s < n; ++s)
        if (dfb_filter_to_host_f(&b, &dts[s], got, got + cells, got + 2 * cells, got + 3 * cells, got + 4 * cells) != DFB_OK) return 7;
    if (dfb_save_restart_f(&b, path, &path_len, &what) != DFB_OK) { fprintf(stderr, "save_restart: %s\n", dfb_last_error()); return 8; }
    if (dfb_destroy_f(&b) != DFB_OK || b != NULL) return 9;
    if (dfb_create_f(&c, &h) != DFB_OK) return 10;
    if (dfb_load_restart_f(&h, path, &path_len, &what) != DFB_OK) { fprintf(stderr, "load_restart: %s\n", dfb_last_error()); return 11; }
    for (int s = n; s < 2 * n; ++s) {
        if (dfb_filter_to_host_f(&h, &dts[s], got, got + cells, got + 2 * cells, got + 3 * cells, got + 4 * cells) != DFB_OK) return 12;
        if (memcmp(got, ref + (size_t)(s - n) * 5 * cells, 8 * 5 * cells) != 0) { fprintf(stderr, "step %d differs\n", s); return 13; }
    }
    printf("RESTART_OK %d\n", n);
    dfb_destroy_f(&a); dfb_destroy_f(&h);
    free(ref); free(got);
    return 0;
}
