/* tests/fortran_facemap_mimic.c -- the face-map calls of fortran/digital_filtering.f90 (facemap_create, interp_to_host, interp_to_cells)
 * made the way a Fortran compiler makes them: every scalar by reference through the _f entry points, absent extents as NULL, and
 * interp_to_cells' type(c_ptr) mean(5), dst(5) as arrays of five addresses (c_null_ptr where unused).  On the reference's default plane:
 * an area map of faces equal to the cells returns the fields bit for bit, and to_cells equals to_host.
 *   usage: fortran_facemap_mimic <RST.dat> <line.dat>      prints "FACEMAP_OK <faces>" or exits non-zero */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <cuda_runtime.h>
#include "dfb200.h"

int main(int argc, char** argv) {
    if (argc < 3) { fprintf(stderr, "usage: %s RST.dat line.dat\n", argv[0]); return 2; }
    dfb_config c;
    if (dfb_config_init(&c) != DFB_OK) return 3;
    c.d_i = 0.0013; c.rho_e = 0.044; c.U_e = 869.1; c.mu_e = 7.1212e-6;
    c.vel_file_N_values = 330; c.honor_flow_config = 1;
    c.vel_fluc_file = argv[1]; c.vel_fluc_file_len = (int)strlen(argv[1]);
    c.line_file = argv[2];     c.line_file_len = (int)strlen(argv[2]);
    c.seed = 99; c.device = -1;
    dfb_handle h = NULL;
    if (dfb_create_f(&c, &h) != DFB_OK) { fprintf(stderr, "create: %s\n", dfb_last_error()); return 4; }
    int Ny = 0, Nz = 0;
    if (dfb_dims_f(&h, &Ny, &Nz) != DFB_OK) return 5;
    const int n = Ny * Nz;
    double* fld = malloc(8 * 5 * (size_t)n);
    const double dt = 1e-8;
    if (dfb_filter_to_host_f(&h, &dt, fld, fld + n, fld + 2 * n, fld + 3 * n, fld + 4 * n) != DFB_OK) return 6;
    double* vy = malloc(8 * (size_t)(Ny + 1));
    double* vz = malloc(8 * (size_t)(Nz + 1));
    if (dfb_get_table(h, 12, 0, vy, Ny + 1) != DFB_OK || dfb_get_table(h, 13, 0, vz, Nz + 1) != DFB_OK) return 7;
    double *yf = malloc(8 * (size_t)n), *zf = malloc(8 * (size_t)n), *hy = malloc(8 * (size_t)n), *hz = malloc(8 * (size_t)n);
    for (int j = 0; j < Ny; ++j)
        for (int k = 0; k < Nz; ++k) {
            const int i = j * Nz + k;
            yf[i] = 0.5 * (vy[j] + vy[j + 1]); zf[i] = 0.5 * (vz[k] + vz[k + 1]);
            hy[i] = vy[j + 1] - vy[j];         hz[i] = vz[k + 1] - vz[k];
        }
    const int kind_area = DFB_MAP_AREA, kind_point = DFB_MAP_POINT, zero = 0, wall = DFB_MAP_WALL_ZERO, all = 31, plane = 0, one = 1;
    int area = -1, point = -1;
    if (dfb_facemap_create_f(&h, &kind_area, &n, yf, zf, hy, hz, &zero, &zero, &zero, &area) != DFB_OK) { fprintf(stderr, "%s\n", dfb_last_error()); return 8; }
    int* served = malloc(sizeof(int) * (size_t)n);
    if (dfb_facemap_served_f(&h, &area, served) != DFB_OK) return 9;
    for (int i = 0; i < n; ++i) if (!served[i]) return 10;
    double* out = malloc(8 * 5 * (size_t)n);
    if (dfb_interp_to_host_f(&h, &area, &plane, &all, out) != DFB_OK) return 11;
    if (memcmp(out, fld, 8 * 5 * (size_t)n) != 0) { fprintf(stderr, "area map at the cells differs from the fields\n"); return 12; }
    for (int i = 0; i < n; ++i) { yf[i] += 0.25 * hy[i]; zf[i] += 0.4 * hz[i]; }
    if (dfb_facemap_create_f(&h, &kind_point, &n, yf, zf, NULL, NULL, &zero, &zero, &wall, &point) != DFB_OK) { fprintf(stderr, "%s\n", dfb_last_error()); return 13; }
    if (dfb_interp_to_host_f(&h, &point, &plane, &all, out) != DFB_OK) return 14;
    double* d = NULL;
    if (cudaMalloc((void**)&d, 8 * 5 * (size_t)n) != cudaSuccess || cudaMemset(d, 0, 8 * 5 * (size_t)n) != cudaSuccess) return 15;
    const double* mean[5] = {NULL, NULL, NULL, NULL, NULL};
    double* dst[5];
    for (int f = 0; f < 5; ++f) dst[f] = d + (size_t)f * n;
    const double scale[5] = {1, 1, 1, 1, 1};
    if (dfb_interp_to_cells_f(&h, &point, &plane, &all, NULL, mean, scale, dst, &one) != DFB_OK) return 16;
    double* back = malloc(8 * 5 * (size_t)n);
    if (dfb_sync(h) != DFB_OK || cudaMemcpy(back, d, 8 * 5 * (size_t)n, cudaMemcpyDeviceToHost) != cudaSuccess) return 17;
    if (memcmp(back, out, 8 * 5 * (size_t)n) != 0) { fprintf(stderr, "to_cells differs from to_host\n"); return 18; }
    if (dfb_facemap_destroy_f(&h, &point) != DFB_OK || dfb_facemap_destroy_f(&h, &area) != DFB_OK) return 19;
    if (dfb_interp_to_host_f(&h, &area, &plane, &all, out) != DFB_ERR_ARG) return 20;
    printf("FACEMAP_OK %d\n", n);
    cudaFree(d);
    dfb_destroy_f(&h);
    free(fld); free(vy); free(vz); free(yf); free(zf); free(hy); free(hz); free(served); free(out); free(back);
    return 0;
}
