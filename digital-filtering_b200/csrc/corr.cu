// csrc/corr.cu -- opt-in correlation statistics of u', v', w' (dfb_corr_enable, include/dfb200.h): per-row sums of lagged products
// along z, along y and in time, accumulated on the handle's stream after the z-sweep of every accumulated step.
//
// Every partial sum is reduced in a fixed order (no floating-point atomics): two identical runs give the same sums bit for bit, and
// the decomposition depends on the plane's shape and the lags only, so plane p of a batch sums exactly like a single plane.
#include <algorithm>
#include <cmath>
#include "kernels.hpp"

namespace dfb {

namespace {

constexpr int CZ_THREADS = 256;     // spanwise kernel: 8 warps per (row, segment)
constexpr int CZ_SEG = 4096;        // columns of x per spanwise CTA (plus the lag halo): the staged row fits shared memory at any Nz
constexpr int CZ_RMAX = 16;         // lags per lane
constexpr int CY_THREADS = 256;     // wall-normal kernel: 8 warps, each 64 rows x 32 lags
constexpr int CY_ROWS = 64;         // rows per CTA
constexpr int CY_LAGS = 256;        // lags per CTA
constexpr int CY_TK = 16;           // columns per staged chunk
constexpr int CT_THREADS = 256;

// field f's u' / v' / w' without indexing the parameter array at run time (which would copy it to the stack)
__device__ inline const double* fluc_of(const CorrParams& p, int f) { return f == 0 ? p.fluc[0] : (f == 1 ? p.fluc[1] : p.fluc[2]); }

__host__ __device__ inline int cy_pad(int r) { return r + 2 * (r >> 3); }     // 8 rows + 2 doubles: 16-byte loads without bank conflicts
__host__ __device__ inline int cy_pitch(int rows) { int p = cy_pad(rows); p = (p + 1) & ~1; return (p % 4 == 0) ? p + 2 : p; }

// ---- spanwise: S_z[row][d] over the columns of one segment ----------------------------------------------------------------------
// The segment's columns x are staged once; the columns x + d of one block of lags (the halo: the next columns, zero beyond the
// plane, or the wrapped columns with periodic_z) are staged per block, so shared memory stays bounded at any lag and width.  Lane l of every warp owns the lags d = lb*32R + l + 32r, r < R; warp w takes the residue classes
// c = w, w + 8, ... of x mod 32.  Along a class (x = c + 32m) the lane's operands f(x + d) = Y[m + r] slide by one per step, so a
// register ring of R samples turns one broadcast load of f(x) and one conflict-free load of the next Y into R FMAs.
template <int R>
__global__ void __launch_bounds__(CZ_THREADS) corr_z_kernel(const CorrParams p, int nseg) {
    extern __shared__ double csm[];
    const int seg = blockIdx.x, j = blockIdx.y, pf = blockIdx.z;
    const int f = pf % 3, pl = pf / 3;
    const int W = p.W, L = p.L[0], nlag = L + 1;
    const int LB = 32 * R, nlb = (nlag + LB - 1) / LB;
    const int ka = seg * CZ_SEG, nx = min(W, ka + CZ_SEG) - ka;
    const int ny = nx + LB + 32;                              // columns ka + lb*LB + [0, ny) of lag block lb
    const double* row = fluc_of(p, f) + ((size_t)pl * p.Ny + j) * W;
    double* xsm = csm;                                        // [nx]
    double* s = csm + nx;                                     // [ny]
    double* red = s + ny;                                     // [8 warps][LB]
    for (int i = threadIdx.x; i < nx; i += CZ_THREADS) xsm[i] = row[ka + i];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const size_t rowid = (size_t)pf * p.Ny + j;
    for (int lb = 0; lb < nlb; ++lb) {
        for (int i = threadIdx.x; i < ny; i += CZ_THREADS) {
            const int g = ka + lb * LB + i;
            s[i] = g < W ? row[g] : (p.periodic ? row[g % W] : 0.0);
        }
        __syncthreads();
        double acc[R];
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = 0.0;
        for (int c = warp; c < 32 && c < nx; c += CZ_THREADS / 32) {
            const int M = (nx - c + 31) >> 5;
            const double* xs = xsm + c;
            const double* ys = s + c + lane;
            double yr[R];
#pragma unroll
            for (int r = 0; r < R; ++r) yr[r] = ys[32 * r];
            int m = 0;
            for (; m + R <= M; m += R) {
#pragma unroll
                for (int i = 0; i < R; ++i) {
                    const double x = xs[32 * (m + i)];
#pragma unroll
                    for (int r = 0; r < R; ++r) acc[r] = fma(x, yr[(i + r) % R], acc[r]);
                    yr[i] = ys[32 * (m + i + R)];
                }
            }
            for (; m < M; ++m) {
                const double x = xs[32 * m];
#pragma unroll
                for (int r = 0; r < R; ++r) acc[r] = fma(x, ys[32 * (m + r)], acc[r]);
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) red[warp * LB + lane + 32 * r] = acc[r];
        __syncthreads();
        for (int t = threadIdx.x; t < LB; t += CZ_THREADS) {
            const int d = lb * LB + t;
            if (d > L) continue;
            double v = red[t];
            for (int w = 1; w < CZ_THREADS / 32; ++w) v += red[w * LB + t];
            if (nseg == 1) p.sum[0][rowid * nlag + d] += v;
            else p.part[((size_t)seg * p.P * 3 * p.Ny + rowid) * nlag + d] = v;
        }
        __syncthreads();
    }
}

// ---- wall-normal: S_y[row][d] over the columns of one column split -------------------------------------------------------------
// CTA = 64 rows j0.. x up to 256 lags d0.. x one split of the columns; thread = 8 rows x 8 lags (64 accumulators), warp = 64 rows x
// 32 lags; warps whose lags all lie beyond L only help staging.  Per column the thread loads its 8 rows (x) and the 16 rows j + d it pairs them with (y) -- 24 loads for 64 FMAs.  Columns are staged transposed
// in chunks of 16 (cp.async, two buffers; zero-filled beyond the plane), rows padded by 2 doubles per 8 so that the 16-byte loads
// of a warp hit distinct banks.  Rows beyond the plane are zero: their products vanish.
__device__ inline void cp_async8(double* dst, const double* src, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(d), "l"(src), "r"(valid ? 8 : 0));
}

__global__ void __launch_bounds__(CY_THREADS, 1) corr_y_kernel(const CorrParams p, int nsplit, int split_cols) {
    extern __shared__ __align__(16) double csm[];
    const int jb = blockIdx.x, pf = blockIdx.z;
    const int db = blockIdx.y / nsplit, split = blockIdx.y % nsplit;
    const int f = pf % 3, pl = pf / 3;
    const int Ny = p.Ny, W = p.W, L = p.L[1], nlag = L + 1;
    const int j0 = jb * CY_ROWS, d0 = db * CY_LAGS;
    const int nwd = min(CY_THREADS / 32, (nlag - d0 + 31) / 32);                  // warps with lags in this block
    const int yrows = 32 * nwd + CY_ROWS;                                         // rows j0 + d0 + [0, yrows)
    const int nrows = CY_ROWS + yrows;                                            // x rows, then y rows
    const int pitch = cy_pitch(nrows);
    const int kbeg = split * split_cols, kend = min(W, kbeg + split_cols);
    const double* base = fluc_of(p, f) + (size_t)pl * Ny * W;
    double* buf[2] = {csm, csm + (size_t)CY_TK * pitch};
    auto stage = [&](double* T, int k0) {
        for (int e = threadIdx.x; e < nrows * CY_TK; e += CY_THREADS) {
            const int r = e / CY_TK, kk = e % CY_TK;
            const int gr = r < CY_ROWS ? j0 + r : j0 + d0 + (r - CY_ROWS);
            const int gk = k0 + kk;
            const bool ok = gr < Ny && gk < kend;
            cp_async8(T + (size_t)kk * pitch + cy_pad(r), ok ? base + (size_t)gr * W + gk : base, ok);
        }
        asm volatile("cp.async.commit_group;\n" ::);
    };
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int jg = lane & 7, dg = warp * 4 + (lane >> 3);
    const bool active = warp < nwd;
    double acc[8][8];
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = 0.0;
    const int xo = cy_pad(8 * jg), yo0 = cy_pad(CY_ROWS + 8 * (jg + dg)), yo1 = cy_pad(CY_ROWS + 8 * (jg + dg) + 8);
    int nb = 0;
    if (kbeg < kend) stage(buf[0], kbeg);
    for (int k0 = kbeg; k0 < kend; k0 += CY_TK, nb ^= 1) {
        if (k0 + CY_TK < kend) { stage(buf[nb ^ 1], k0 + CY_TK); asm volatile("cp.async.wait_group 1;\n" ::); }
        else asm volatile("cp.async.wait_group 0;\n" ::);
        __syncthreads();
        if (active) {
            const double* T = buf[nb];
#pragma unroll 2
            for (int kk = 0; kk < CY_TK; ++kk) {
                const double* Tk = T + (size_t)kk * pitch;
                double x[8], y[16];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const double2 v = *reinterpret_cast<const double2*>(Tk + xo + 2 * q);
                    x[2 * q] = v.x; x[2 * q + 1] = v.y;
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const double2 v = *reinterpret_cast<const double2*>(Tk + yo0 + 2 * q);
                    y[2 * q] = v.x; y[2 * q + 1] = v.y;
                    const double2 u = *reinterpret_cast<const double2*>(Tk + yo1 + 2 * q);
                    y[8 + 2 * q] = u.x; y[8 + 2 * q + 1] = u.y;
                }
#pragma unroll
                for (int a = 0; a < 8; ++a)
#pragma unroll
                    for (int b = 0; b < 8; ++b) acc[a][b] = fma(x[a], y[a + b], acc[a][b]);
            }
        }
        __syncthreads();
    }
    if (!active) return;
    const size_t rows_all = (size_t)p.P * 3 * Ny;
#pragma unroll
    for (int a = 0; a < 8; ++a) {
        const int j = j0 + 8 * jg + a;
        if (j >= Ny) continue;
        const size_t rowid = (size_t)pf * Ny + j;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const int d = d0 + 8 * dg + b;
            if (d > L) continue;
            if (nsplit == 1) p.sum[1][rowid * nlag + d] += acc[a][b];
            else p.part[((size_t)split * rows_all + rowid) * nlag + d] = acc[a][b];
        }
    }
}

// sum[row][d] += the partials of the segments / splits, in their order
__global__ void corr_reduce_kernel(double* __restrict__ sum, const double* __restrict__ part, size_t n, int nparts) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double v = part[i];
    for (int s = 1; s < nparts; ++s) v += part[(size_t)s * n + i];
    sum[i] += v;
}

// ---- temporal: S_t[row][m] += sum_k f_s(k) f_{s-m}(k), m <= M; then f_s goes into the ring -----------------------------------
// CTA per (plane, field, row).  Each thread walks the same columns for every lag (the current row stays in L1), reduces its
// partial across the warp with a fixed xor tree, and the warps' sums are added in warp order.  The ring slot of this step is the
// one lag L_t read (the oldest): every thread reads its columns of it before it overwrites them.
__global__ void __launch_bounds__(CT_THREADS) corr_t_kernel(const CorrParams p, int M) {
    __shared__ double wsum[65][CT_THREADS / 32];
    const int j = blockIdx.x, pf = blockIdx.y;
    const int f = pf % 3, pl = pf / 3;
    const int W = p.W, Lt = p.L[2];
    const size_t rows_all = (size_t)p.P * 3 * p.Ny, rowid = (size_t)pf * p.Ny + j;
    const double* fr = fluc_of(p, f) + ((size_t)pl * p.Ny + j) * W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int m = 0; m <= M; ++m) {
        const double* rr = m == 0 ? fr : p.ring + ((size_t)((p.ring_count - m) % Lt) * rows_all + rowid) * W;
        double s = 0.0;
        for (int k = threadIdx.x; k < W; k += CT_THREADS) s = fma(fr[k], rr[k], s);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) wsum[m][warp] = s;
    }
    double* wr = p.ring + ((size_t)(p.ring_count % Lt) * rows_all + rowid) * W;
    for (int k = threadIdx.x; k < W; k += CT_THREADS) wr[k] = fr[k];
    __syncthreads();
    if (threadIdx.x <= M) {
        double v = wsum[threadIdx.x][0];
        for (int w = 1; w < CT_THREADS / 32; ++w) v += wsum[threadIdx.x][w];
        p.sum[2][rowid * (Lt + 1) + threadIdx.x] += v;
    }
}

int cz_r(int L) { return std::min(CZ_RMAX, (L + 1 + 31) / 32); }
size_t cz_smem(int W, int L) {
    const int LB = 32 * cz_r(L);
    const size_t nx = (size_t)std::min(W, CZ_SEG);
    return sizeof(double) * (nx + nx + LB + 32 + (size_t)(CZ_THREADS / 32) * LB);
}
size_t cy_smem(int L) {
    const int nwd = std::min(CY_THREADS / 32, (L + 1 + 31) / 32);
    return sizeof(double) * 2 * CY_TK * (size_t)cy_pitch(CY_ROWS + 32 * nwd + CY_ROWS);
}

template <int R>
cudaError_t launch_z(const CorrParams& p, cudaStream_t st) {
    const int nseg = (p.W + CZ_SEG - 1) / CZ_SEG;
    const size_t smem = cz_smem(p.W, p.L[0]);
    cudaError_t e = cudaFuncSetAttribute(corr_z_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    corr_z_kernel<R><<<dim3(nseg, p.Ny, 3 * p.P), CZ_THREADS, smem, st>>>(p, nseg);
    if ((e = cudaGetLastError()) != cudaSuccess || nseg == 1) return e;
    const size_t n = (size_t)p.P * 3 * p.Ny * (p.L[0] + 1);
    corr_reduce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p.sum[0], p.part, n, nseg);
    return cudaGetLastError();
}

}  // namespace

void corr_y_split(int Ny, int W, int* nsplit, int* split_cols) {
    // Column splits of one plane's rows: about 444 CTAs per block of lags for the three fields (three waves of one CTA per SM on a
    // 148-SM B200), at least 64 columns per split.  From the plane's shape alone -- never the batch size or the device -- so that
    // every plane of a batch adds its columns in the order a single plane does.
    const int per_split = 3 * ((Ny + CY_ROWS - 1) / CY_ROWS);
    const int best = std::max(1, std::min((444 + per_split - 1) / per_split, W / 64));
    *split_cols = ((W + best - 1) / best + CY_TK - 1) / CY_TK * CY_TK;
    *nsplit = (W + *split_cols - 1) / *split_cols;
}

size_t corr_part_doubles(int P, int Ny, int W, int Lz, int Ly, int nsplit_y) {
    const size_t rows = (size_t)P * 3 * Ny;
    const int nseg = (W + CZ_SEG - 1) / CZ_SEG;
    size_t n = 0;
    if (Lz > 0 && nseg > 1) n = std::max(n, (size_t)nseg * rows * (Lz + 1));
    if (Ly > 0 && nsplit_y > 1) n = std::max(n, (size_t)nsplit_y * rows * (Ly + 1));
    return n;
}

cudaError_t launch_corr_z(const CorrParams& p, cudaStream_t st) {
    switch (cz_r(p.L[0])) {
#define CZ_CASE(R) case R: return launch_z<R>(p, st);
        CZ_CASE(1) CZ_CASE(2) CZ_CASE(3) CZ_CASE(4) CZ_CASE(5) CZ_CASE(6) CZ_CASE(7) CZ_CASE(8)
        CZ_CASE(9) CZ_CASE(10) CZ_CASE(11) CZ_CASE(12) CZ_CASE(13) CZ_CASE(14) CZ_CASE(15) CZ_CASE(16)
#undef CZ_CASE
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_corr_y(const CorrParams& p, cudaStream_t st) {
    const size_t smem = cy_smem(p.L[1]);
    cudaError_t e = cudaFuncSetAttribute(corr_y_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int ndb = (p.L[1] + 1 + CY_LAGS - 1) / CY_LAGS;
    corr_y_kernel<<<dim3((p.Ny + CY_ROWS - 1) / CY_ROWS, ndb * p.y_nsplit, 3 * p.P), CY_THREADS, smem, st>>>(p, p.y_nsplit, p.y_split_cols);
    if ((e = cudaGetLastError()) != cudaSuccess || p.y_nsplit == 1) return e;
    const size_t n = (size_t)p.P * 3 * p.Ny * (p.L[1] + 1);
    corr_reduce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p.sum[1], p.part, n, p.y_nsplit);
    return cudaGetLastError();
}

cudaError_t launch_corr_t(const CorrParams& p, int M, cudaStream_t st) {
    corr_t_kernel<<<dim3(p.Ny, 3 * p.P), CT_THREADS, 0, st>>>(p, M);
    return cudaGetLastError();
}

}  // namespace dfb
