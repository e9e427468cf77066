// csrc/profiles.cu -- per-cell profiles (dfb_set_profiles): after the z-sweep, the delivered fields are rescaled from filt_old with the
// epilogue's constants of every cell (profiles.cpp) instead of its row's.  filt_old, the noise and the sweeps do not depend on the profiles.
#include "kernels.hpp"

namespace dfb {

// One thread per cell, the operations and roundings of every form's epilogue: u' = rc0 zu, v' = fma(rc1, zu, rc2 zv), w' = rc3 zw,
// t2 = rc4 u', T' = t2 Ts, rho' = -t2 rhos.  The tuned z-sweeps write them so (epi_scale, epi_cross, the t2 products), and
// epilogue_cell compiles to the same contraction of v' in both one-thread-per-cell kernels.  So a cell whose constants equal its row's
// gets the bits the z-sweep wrote.  first: the constructor's step, whose T' and rho' stay untouched (df.cpp:65, quirk 3).
__global__ void __launch_bounds__(256) profiles_kernel(const PlaneDev D, const double* __restrict__ pc, size_t n, int first,
                                                       const StepRecord* rec) {
    const size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;       // cell within the plane
    if (c >= n || (rec && rec->void_step)) return;
    const size_t i = (size_t)blockIdx.y * n + c;                          // cell within the batch's dense arrays
    const double zu = D.f[0].filt_old[i], zv = D.f[1].filt_old[i], zw = D.f[2].filt_old[i];
    const double u = __dmul_rn(__ldg(pc + c), zu);
    D.f[0].fluc[i] = u;
    D.f[1].fluc[i] = __fma_rn(__ldg(pc + n + c), zu, __dmul_rn(__ldg(pc + 2 * n + c), zv));
    D.f[2].fluc[i] = __dmul_rn(__ldg(pc + 3 * n + c), zw);
    if (first) return;
    const double t2 = __dmul_rn(__ldg(pc + 4 * n + c), u);
    D.T_fluc[i] = __dmul_rn(t2, __ldg(pc + 5 * n + c));
    D.rho_fluc[i] = __dmul_rn(-t2, __ldg(pc + 6 * n + c));
}

cudaError_t profiles_prepare() {
    // load the kernel now, not while an attached handle's stream is being captured
    cudaFuncAttributes a;
    return cudaFuncGetAttributes(&a, (const void*)profiles_kernel);
}

cudaError_t launch_profiles(const PlaneDev& D, const double* pc, int first, const StepRecord* rec, cudaStream_t st) {
    const size_t n = (size_t)D.Ny * D.W;
    profiles_kernel<<<dim3((unsigned)((n + 255) / 256), (unsigned)D.P), 256, 0, st>>>(D, pc, n, first, rec);
    return cudaGetLastError();
}

}  // namespace dfb
