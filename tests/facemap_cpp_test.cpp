// tests/facemap_cpp_test.cpp -- the C++ facade's face maps (include/digital_filter.hpp: DIGITAL_FILTER::face_map_interp, FaceMap) on the
// reference's default plane, run from a directory whose ../files/RST.dat and ../line.dat are the reference's inputs.  An area map of
// faces equal to the cells returns the fields bit for bit; a point map delivers the same values to the host and to device cells.
//   usage: facemap_cpp_test      prints "FACEMAP_OK <faces>" or exits non-zero
#include <cstdio>
#include <cstring>
#include <vector>
#include <cuda_runtime.h>
#include "digital_filter.hpp"

int main() {
    DFConfigEx c;
    c.seed = 2024;
    DIGITAL_FILTER df(c);
    df.filter(1e-8);
    const int Ny = df.get_Ny(), Nz = df.get_Nz();
    std::vector<double> vy(Ny + 1), vz(Nz + 1);
    if (dfb_get_table(df.handle(), 12, 0, vy.data(), Ny + 1) != DFB_OK || dfb_get_table(df.handle(), 13, 0, vz.data(), Nz + 1) != DFB_OK) return 3;
    std::vector<double> yf, zf, hy, hz;
    for (int j = 0; j < Ny; ++j)
        for (int k = 0; k < Nz; ++k) {
            yf.push_back(0.5 * (vy[j] + vy[j + 1])); zf.push_back(0.5 * (vz[k] + vz[k + 1]));
            hy.push_back(vy[j + 1] - vy[j]); hz.push_back(vz[k + 1] - vz[k]);
        }
    const size_t n = yf.size();
    {
        FaceMap cells = df.face_map_interp(yf, zf, hy, hz);
        const std::vector<double> got = cells.to_host();
        const Vector* want[5] = {&df.u.fluc, &df.v.fluc, &df.w.fluc, &df.T_fluc(), &df.rho_fluc()};
        for (int f = 0; f < 5; ++f)
            if (std::memcmp(got.data() + f * n, want[f]->data(), n * sizeof(double)) != 0) { std::fprintf(stderr, "field %d differs\n", f); return 4; }
    }
    std::vector<double> ys(n), zs(n);
    for (size_t i = 0; i < n; ++i) { ys[i] = yf[(i * 7919) % n] + 0.3 * hy[(i * 7919) % n]; zs[i] = zf[(i * 104729) % n] - 0.2 * hz[0]; }
    FaceMap pts = df.face_map_interp(ys, zs);
    const std::vector<double> host = pts.to_host(1 << DFB_V_FLUC | 1 << DFB_RHO_FLUC);
    double* d = nullptr;
    if (cudaMalloc(&d, 2 * n * sizeof(double)) != cudaSuccess || cudaMemset(d, 0, 2 * n * sizeof(double)) != cudaSuccess) return 5;
    double* dst[5] = {nullptr, d, nullptr, nullptr, d + n};
    pts.to_cells(1 << DFB_V_FLUC | 1 << DFB_RHO_FLUC, nullptr, nullptr, nullptr, dst);
    std::vector<double> back(2 * n);
    if (dfb_sync(df.handle()) != DFB_OK || cudaMemcpy(back.data(), d, 2 * n * sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess) return 6;
    cudaFree(d);
    if (std::memcmp(back.data(), host.data(), 2 * n * sizeof(double)) != 0) { std::fprintf(stderr, "to_cells != to_host\n"); return 7; }
    std::printf("FACEMAP_OK %zu\n", n);
    return 0;
}
