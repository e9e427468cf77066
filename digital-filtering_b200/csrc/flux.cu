// csrc/flux.cu -- inflow mass-flux correction (dfb_set_flux_correction): per plane and step, the plane sum m' = sum_j wy_j sum_k hz_k u'_jk
// in a fixed order, c = m' / D, then u' <- fma(-c, rc0_j, u') and T', rho' rebuilt from it.  The tables come from fluxtables.cpp.
// With per-cell profiles (dfb_set_profiles) the weights hz_k and the constants rc0_j, rc4_j, Ts_j, rhos_j are per cell.
#include "kernels.hpp"

namespace dfb {

namespace {

constexpr int FLUX_THREADS = 256;

// Sum over the block in a fixed order: each warp's butterfly (addition commutes exactly, so every lane holds the same bits), then
// the warps' sums in warp order.  The result is in every thread.
__device__ __forceinline__ double block_sum(double s) {
    __shared__ double warp_sum[FLUX_THREADS / 32];
    __shared__ double total;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = warp_sum[0];
        for (int w = 1; w < FLUX_THREADS / 32; ++w) t = __dadd_rn(t, warp_sum[w]);
        total = t;
    }
    __syncthreads();
    return total;
}

}  // namespace

// One CTA per (row, plane): the row's partial wy_j * sum_k hz_k u'_jk (each thread a strided sum in k, then block_sum).  The last CTA
// of a plane to finish (ticket counter) sums the plane's Ny partials in row order the same way, writes {c, m'} and puts the counter
// back to 0, so that the next step (or graph replay) needs no memset.  Neither order depends on the batch size or the launch.
// CELL: per-cell profiles, the weight of cell (j, k) is wz_jk instead of hz_k.
template <bool CELL>
__device__ __forceinline__ void flux_rows(const FluxParams& F, const double* wz, const StepRecord* rec) {
    if (rec && rec->void_step) return;
    const int j = blockIdx.x, p = blockIdx.y;
    const double* u = F.u + (size_t)p * F.ps_cells + (size_t)j * F.W;
    const double* w = CELL ? wz + (size_t)j * F.W : F.hz;
    double s = 0.0;
    for (int k = threadIdx.x; k < F.W; k += FLUX_THREADS) s = __fma_rn(__ldg(w + k), u[k], s);
    const double row = __dmul_rn(block_sum(s), __ldg(F.wy + j));
    __shared__ bool last;
    if (threadIdx.x == 0) {
        __stcg(F.part + (size_t)p * F.Ny + j, row);
        __threadfence();
        last = atomicAdd(F.counter + p, 1u) == (unsigned)F.Ny - 1u;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    double t = 0.0;
    for (int i = threadIdx.x; i < F.Ny; i += FLUX_THREADS) t = __dadd_rn(t, __ldcg(F.part + (size_t)p * F.Ny + i));
    const double m = block_sum(t);
    if (threadIdx.x == 0) {
        F.out[p] = make_double2(__ddiv_rn(m, F.D), m);
        F.counter[p] = 0u;
    }
}

__global__ void __launch_bounds__(FLUX_THREADS) flux_rows_kernel(const FluxParams F, const StepRecord* rec) { flux_rows<false>(F, nullptr, rec); }
__global__ void __launch_bounds__(FLUX_THREADS) flux_rows_cell_kernel(const FluxParams F, const FluxCells C, const StepRecord* rec) {
    flux_rows<true>(F, C.wz, rec);
}

// One thread per cell: u' <- fma(-c_p, rc0_j, u'), then T', rho' from it with the epilogue's roundings (as rebuild_kernel).
__global__ void __launch_bounds__(FLUX_THREADS) flux_apply_kernel(const FluxParams F, const StepRecord* rec) {
    if (rec && rec->void_step) return;
    const int k = blockIdx.x * FLUX_THREADS + threadIdx.x;
    const int j = blockIdx.y, p = blockIdx.z;
    if (k >= F.W) return;
    const size_t idx = (size_t)p * F.ps_cells + (size_t)j * F.W + k;
    const double* rc = F.rowc + (size_t)j * ROWC;
    const double c = F.out[p].x;
    const double u = __fma_rn(-c, __ldg(rc), F.u[idx]);
    const double t2 = __dmul_rn(__ldg(rc + 4), u);
    F.u[idx] = u;
    F.T[idx] = __dmul_rn(t2, __ldg(rc + 5));
    F.rho[idx] = __dmul_rn(-t2, __ldg(rc + 6));
}

// flux_apply_kernel with the constants of every cell (per-cell profiles): pc [7][Ny][W]
__global__ void __launch_bounds__(FLUX_THREADS) flux_apply_cell_kernel(const FluxParams F, const FluxCells C, const StepRecord* rec) {
    if (rec && rec->void_step) return;
    const int k = blockIdx.x * FLUX_THREADS + threadIdx.x;
    const int j = blockIdx.y, p = blockIdx.z;
    if (k >= F.W) return;
    const size_t n = (size_t)F.Ny * F.W, c = (size_t)j * F.W + k, idx = (size_t)p * F.ps_cells + c;
    const double cp = F.out[p].x;
    const double u = __fma_rn(-cp, __ldg(C.pc + c), F.u[idx]);
    const double t2 = __dmul_rn(__ldg(C.pc + 4 * n + c), u);
    F.u[idx] = u;
    F.T[idx] = __dmul_rn(t2, __ldg(C.pc + 5 * n + c));
    F.rho[idx] = __dmul_rn(-t2, __ldg(C.pc + 6 * n + c));
}

cudaError_t flux_prepare() {
    // load both kernels now, not while an attached handle's stream is being captured
    const void* fns[] = {(const void*)flux_rows_kernel, (const void*)flux_apply_kernel, (const void*)flux_rows_cell_kernel,
                         (const void*)flux_apply_cell_kernel};
    for (const void* fn : fns) {
        cudaFuncAttributes a;
        const cudaError_t e = cudaFuncGetAttributes(&a, fn);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t launch_flux(const FluxParams& F, const FluxCells* cells, const StepRecord* rec, cudaStream_t st) {
    const dim3 rows((unsigned)F.Ny, (unsigned)F.P), grid((unsigned)((F.W + FLUX_THREADS - 1) / FLUX_THREADS), (unsigned)F.Ny, (unsigned)F.P);
    if (cells) {
        flux_rows_cell_kernel<<<rows, FLUX_THREADS, 0, st>>>(F, *cells, rec);
        flux_apply_cell_kernel<<<grid, FLUX_THREADS, 0, st>>>(F, *cells, rec);
    } else {
        flux_rows_kernel<<<rows, FLUX_THREADS, 0, st>>>(F, rec);
        flux_apply_kernel<<<grid, FLUX_THREADS, 0, st>>>(F, rec);
    }
    return cudaGetLastError();
}

}  // namespace dfb
