/* tests/attached_capture_test.c -- a GPU-resident caller driving the generator from its own CUDA graph with the runtime API: handle A is
 * attached to the caller's stream, one dfb_filter_dev + one dfb_interp_to_cells are captured (cudaStreamCaptureModeGlobal) and the graph
 * is replayed K times with dt rewritten in device memory between replays; handle B runs the same sequence eagerly.  The five fields,
 * filt_old, the interpolated faces and the step counters must agree bit for bit.  Mode "fortran" makes the attach and the steps
 * through the by-reference entry points, as fortran/digital_filtering.f90 makes them (type(c_ptr) arguments by reference).
 *   usage: attached_capture_test <RST.dat> <line.dat> c|fortran     prints "CAPTURE_OK K" or exits non-zero */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <cuda_runtime.h>
#include "dfb200.h"

#define CK(x)                                                                              \
    do {                                                                                   \
        int rc_ = (x);                                                                     \
        if (rc_ != 0) { fprintf(stderr, "%s:%d %s -> %d %s\n", __FILE__, __LINE__, #x, rc_, dfb_last_error()); exit(10); } \
    } while (0)
#define CU(x)                                                                              \
    do {                                                                                   \
        cudaError_t e_ = (x);                                                              \
        if (e_ != cudaSuccess) { fprintf(stderr, "%s:%d %s -> %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); exit(11); } \
    } while (0)

enum { K = 50, NF = 64 };
static int fortran = 0;

static void attach(dfb_handle h, cudaStream_t s) {
    void* sp = s;
    if (fortran) CK(dfb_attach_stream_f(&h, &sp));
    else CK(dfb_attach_stream(h, sp));
}
static void step_dev(dfb_handle h, const double* dt_dev) {
    if (fortran) CK(dfb_filter_dev_f(&h, &dt_dev));
    else CK(dfb_filter_dev(h, dt_dev));
}
static void faces(dfb_handle h, int map, double** dst) { CK(dfb_interp_to_cells(h, map, 0, 31, NULL, NULL, NULL, dst, 1)); }

int main(int argc, char** argv) {
    if (argc < 4) { fprintf(stderr, "usage: %s RST.dat line.dat c|fortran\n", argv[0]); return 2; }
    fortran = strcmp(argv[3], "fortran") == 0;
    dfb_config c;
    CK(dfb_config_init(&c));
    c.d_i = 0.0013; c.rho_e = 0.044; c.U_e = 869.1; c.mu_e = 7.1212e-6;
    c.vel_file_N_values = 330; c.honor_flow_config = 1;
    c.vel_fluc_file = argv[1]; c.line_file = argv[2];
    c.seed = 4242; c.device = 0;
    dfb_handle a = NULL, b = NULL;
    CK(dfb_create(&c, &a));
    CK(dfb_create(&c, &b));
    int Ny = 0, Nz = 0;
    CK(dfb_dims(a, &Ny, &Nz));
    double vy[4096], vz[4096];
    CK(dfb_get_table(a, 12, 0, vy, 4096));
    CK(dfb_get_table(a, 13, 0, vz, 4096));
    double yf[NF], zf[NF];
    for (int i = 0; i < NF; ++i) {                       /* faces spread over the plane, off the cell centres */
        yf[i] = vy[0] + (vy[Ny] - vy[0]) * (i + 0.37) / NF;
        zf[i] = vz[0] + (vz[Nz] - vz[0]) * ((i * 7) % NF + 0.61) / NF;
    }
    int ma = -1, mb = -1;
    CK(dfb_facemap_create(a, DFB_MAP_POINT, NF, yf, zf, NULL, NULL, 0, 0, 0, &ma));
    CK(dfb_facemap_create(b, DFB_MAP_POINT, NF, yf, zf, NULL, NULL, 0, 0, 0, &mb));

    cudaStream_t s;
    CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    double *dt_a, *dt_b, *fa, *fb;
    CU(cudaMalloc((void**)&dt_a, 8)); CU(cudaMalloc((void**)&dt_b, 8));
    CU(cudaMalloc((void**)&fa, 5 * NF * 8)); CU(cudaMalloc((void**)&fb, 5 * NF * 8));
    CU(cudaMemset(fa, 0, 5 * NF * 8)); CU(cudaMemset(fb, 0, 5 * NF * 8));
    double* da[5]; double* db[5];
    for (int f = 0; f < 5; ++f) { da[f] = fa + f * NF; db[f] = fb + f * NF; }
    attach(a, s);
    attach(b, s);

    cudaGraph_t g;
    cudaGraphExec_t ge;
    CU(cudaStreamBeginCapture(s, cudaStreamCaptureModeGlobal));
    step_dev(a, dt_a);
    faces(a, ma, da);
    CU(cudaStreamEndCapture(s, &g));
    CU(cudaGraphInstantiate(&ge, g, 0));

    double* dts = malloc(sizeof(double) * K);           /* pinned would be faster; pageable keeps the copies ordered on s as well */
    for (int k = 0; k < K; ++k) dts[k] = (k % 5 == 3) ? 0.0 : 1e-8 * (1 + k % 7);
    for (int k = 0; k < K; ++k) {
        CU(cudaMemcpyAsync(dt_a, &dts[k], 8, cudaMemcpyHostToDevice, s));
        CU(cudaGraphLaunch(ge, s));
        CU(cudaMemcpyAsync(dt_b, &dts[k], 8, cudaMemcpyHostToDevice, s));
        step_dev(b, dt_b);
        faces(b, mb, db);
    }
    CK(dfb_sync(a));
    int64_t sa = 0, sb = 0;
    CK(dfb_info(a, 2, 0, &sa));
    CK(dfb_info(b, 2, 0, &sb));
    if (sa != sb || sa != 1 + K) { fprintf(stderr, "step counters %lld %lld\n", (long long)sa, (long long)sb); return 20; }
    const size_t n = (size_t)Ny * Nz;
    double* x = malloc(8 * n);
    double* y = malloc(8 * n);
    for (int w = 0; w < 8; ++w) {
        CK(dfb_get_field(a, w, x, 0));
        CK(dfb_get_field(b, w, y, 0));
        if (memcmp(x, y, 8 * n) != 0) { fprintf(stderr, "field %d differs\n", w); return 21; }
    }
    double hfa[5 * NF], hfb[5 * NF];
    CU(cudaMemcpy(hfa, fa, sizeof(hfa), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(hfb, fb, sizeof(hfb), cudaMemcpyDeviceToHost));
    if (memcmp(hfa, hfb, sizeof(hfa)) != 0) { fprintf(stderr, "faces differ\n"); return 22; }
    int nonzero = 0;
    for (int i = 0; i < 5 * NF; ++i) nonzero += hfa[i] != 0.0;
    if (nonzero < 4 * NF) { fprintf(stderr, "faces look unwritten (%d nonzero)\n", nonzero); return 23; }
    void* null_stream = NULL;
    if (fortran) CK(dfb_attach_stream_f(&a, &null_stream));
    else CK(dfb_attach_stream(a, NULL));
    CK(dfb_attach_stream(b, NULL));
    CU(cudaGraphExecDestroy(ge));
    CU(cudaGraphDestroy(g));
    CK(dfb_destroy(a));
    CK(dfb_destroy(b));
    CU(cudaStreamDestroy(s));
    printf("CAPTURE_OK %d\n", K);
    return 0;
}
