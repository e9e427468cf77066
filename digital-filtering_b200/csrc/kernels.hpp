// csrc/kernels.hpp -- host launchers of the kernels in kernels.cu
#pragma once
#include "device.cuh"

namespace dfb {

cudaError_t launch_noise(const NoiseParams& P, const NoiseWindows& Wn, const PlaneDev& D, cudaStream_t st);
cudaError_t launch_ysweep_simple(const PlaneDev& D, cudaStream_t st);
cudaError_t launch_zsweep_simple(const PlaneDev& D, const StepConsts& S, const StepRecord* rec, const double2* rows, cudaStream_t st);
// attached steps (dfb_attach_stream): the step's first launch (with the per-row blend constants when A.rows is set), and loading
// every kernel such a step may launch
cudaError_t launch_advance(const AdvanceParams& A, cudaStream_t st);
cudaError_t attach_prepare();
cudaError_t ysweep_prepare();
// dense band-matrix tiles [0, n_dense) with ysweep_tma_kernel, then recursive tiles [n_dense, n_dense + n_rec) with ysweep_rec_kernel
cudaError_t launch_ysweep_tma(const YMaps& maps, const YParams& P, int n_dense, int n_rec, cudaStream_t st);
// run-recursive y-sweep (every row group through the exponential structure; resident window tiles)
cudaError_t ysweep_run_prepare(size_t smem);
cudaError_t launch_ysweep_run(const YRMaps& maps, const YParams& P, cudaStream_t st);
cudaError_t zsweep_prepare(int zk, int mode, size_t smem, int* blocks_per_sm);
cudaError_t launch_zsweep_tuned(const ZMaps& maps, const ZParams& P, cudaStream_t st);
cudaError_t launch_stats(const PlaneDev& D, double* sums, const StepRecord* rec, cudaStream_t st);
cudaError_t launch_scatter(const double* field, int n, const int* plane_index, const int* dst_index, const double* mean, double scale,
                           double* dst, cudaStream_t st);
// face maps (facemap.hpp): dst[f][dst_index[i] * stride] = base + scale[f] * sum_t w_t * field[f][idx_t] for the served faces i < n and
// the fields f in `fields`; base = mean[f][i], else dst's own value where bit f of `add` is set, else 0.  ptr == nullptr: 4 taps per face.
struct InterpArgs {
    const double* field[5];
    const double* mean[5];
    double scale[5];
    double* dst[5];
    const int* dst_index;             // nullptr: face i -> i
    long long stride;
    int n, fields, add;
    const int* idx;
    const double* w;
    const int* ptr;
};
cudaError_t launch_interp(const InterpArgs& a, cudaStream_t st);
cudaError_t launch_rebuild(double* plane, const double* rowc, int Ny, int NzG, int k0, int W, int first_only, cudaStream_t st);
cudaError_t launch_assemble(const double* slab, double* plane, const double* rowc, int Ny, int NzG, int k0, int W, int first_only, cudaStream_t st);
cudaError_t launch_dfma_peak(double* out, int blocks, int iters, cudaStream_t st);

// inflow mass-flux correction (flux.cu, dfb_set_flux_correction): u', T', rho' dense [P][Ny][W] (whole planes, W = Nz)
struct FluxParams {
    double* u;
    double* T;
    double* rho;
    const double* rowc;               // [Ny][ROWC]: rc0 = sqrt(R11), rc4, Ts, rhos of the epilogue
    const double* wy;                 // [Ny] g_j hy_j
    const double* hz;                 // [W]
    double* part;                     // [P][Ny] row partials
    unsigned* counter;                // [P] tickets of the row CTAs; 0 between launches
    double2* out;                     // [P] {c, m'} of the last corrected step
    double D;
    int Ny, W, P;
    size_t ps_cells;
};
// per-cell profiles (dfb_set_profiles): then wy_j = hy_j, the weights are wz and the constants pc
struct FluxCells {
    const double* wz;                 // [Ny][W] g_jk hz_k
    const double* pc;                 // [7][Ny][W] the epilogue's constants per cell (profile_consts): rc0, rc4, Ts, rhos at 0, 4, 5, 6
};
cudaError_t flux_prepare();
// cells: nullptr for the row tables; a void attached step (rec) changes nothing
cudaError_t launch_flux(const FluxParams& F, const FluxCells* cells, const StepRecord* rec, cudaStream_t st);

// per-cell profiles (profiles.cu, dfb_set_profiles): u', v', w' and, unless first, T', rho' of D[0]'s planes rescaled from filt_old with
// the constants pc [7][Ny][W] of every cell; a void attached step (rec) changes nothing
cudaError_t profiles_prepare();
cudaError_t launch_profiles(const PlaneDev& D, const double* pc, int first, const StepRecord* rec, cudaStream_t st);

// correlation statistics (corr.cu, dfb_corr_enable): sums [P][3][Ny][L_d + 1] per direction d = 0 z, 1 y, 2 t
struct CorrParams {
    const double* fluc[3];            // u', v', w': dense [P][Ny][W] (W = Nz: whole planes only)
    int P, Ny, W, periodic;
    int L[3];                         // lags per direction (0 = off)
    double* sum[3];
    double* part;                     // partial sums of the z segments / y column splits (corr_part_doubles)
    int y_nsplit, y_split_cols;       // corr_y_split
    double* ring;                     // [L_t][P][3][Ny][W]: the last L_t accumulated fields (allocated while accumulating)
    long long ring_count;             // fields written into the ring since it was emptied
};
void corr_y_split(int Ny, int W, int* nsplit, int* split_cols);
size_t corr_part_doubles(int P, int Ny, int W, int Lz, int Ly, int nsplit_y);
cudaError_t launch_corr_z(const CorrParams& p, cudaStream_t st);
cudaError_t launch_corr_y(const CorrParams& p, cudaStream_t st);
cudaError_t launch_corr_t(const CorrParams& p, int M, cudaStream_t st);   // lags 0..M (M = min(L_t, ring_count))

}  // namespace dfb
