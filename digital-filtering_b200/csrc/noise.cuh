// csrc/noise.cuh -- device side of the white-noise contract in include/dfb_rng_spec.h (spec v2).
// Replaces DIGITAL_FILTER::generate_white_noise (df.cpp:332-349): per-element pcg32 streams
// (pcg_random.hpp:1866) addressed by jump-ahead (pcg_random.hpp:640-669) instead of one serial
// process-wide stream, and a Box-Muller pair transform made only of correctly rounded IEEE
// operations so that the host restatement (oracle/normal_oracle.c) matches bit for bit.
#pragma once
#include <cstdint>
#include "dfb_rng_spec.h"
#include "device.cuh"

namespace dfb {


__host__ __device__ inline uint64_t pcg_lcg(uint64_t s, uint64_t inc) { return s * DFB_PCG32_MULT + inc; }

// XSH-RR 64 -> 32 (pcg_random.hpp:845-872)
__host__ __device__ inline uint32_t pcg_xsh_rr(uint64_t s) {
    uint32_t x = (uint32_t)(((s >> 18) ^ s) >> 27);
    uint32_t r = (uint32_t)(s >> 59);
#ifdef __CUDA_ARCH__
    return __funnelshift_r(x, x, r);
#else
    return (x >> r) | (x << ((32u - r) & 31u));
#endif
}

// Brown's arbitrary-stride jump (pcg_random.hpp:640-669) as a composable affine map
__host__ __device__ inline Jump pcg_jump(uint64_t delta, uint64_t inc) {
    uint64_t acc_mult = 1u, acc_plus = 0u, cur_mult = DFB_PCG32_MULT, cur_plus = inc;
    while (delta > 0) {
        if (delta & 1u) { acc_mult *= cur_mult; acc_plus = acc_plus * cur_mult + cur_plus; }
        cur_plus = (cur_mult + 1u) * cur_plus;
        cur_mult *= cur_mult;
        delta >>= 1;
    }
    return Jump{acc_mult, acc_plus};
}

// increment of stream ((plane*3 + field)*2 + kind) of include/dfb_rng_spec.h, kind 0 = r_ys, 1 = r_zs halo
__host__ __device__ inline uint64_t noise_inc(int64_t plane, int field, int kind) {
    const uint64_t stream = (uint64_t)((plane * 3 + field) * 2 + kind);
    return (stream << 1) | 1u;
}

// pcg32 state at the first draw of step `step` of an array that draws `npairs` pairs per step: the host (fill_noise_states) and the
// step's advance kernel (dfb_attach_stream) both position the noise through this one function
__host__ __device__ inline uint64_t noise_step_state(uint64_t seed, uint64_t inc, int64_t step, uint64_t npairs) {
    const uint64_t state0 = pcg_lcg(seed + inc, inc);
    const Jump j = pcg_jump(4u * ((uint64_t)step * npairs), inc);
    return j.A * state0 + j.C;
}

#ifdef __CUDACC__
__constant__ double c_log1p[DFB_LOG1P_NC] = {DFB_LOG1P_C_LIST};
// per-lane index: global memory through the read-only path (a __constant__ table would serialise the divergent lookups)
__device__ const double2 g_logtab[64] = {DFB_LOGTAB_LIST};
__constant__ double c_sin[DFB_SIN_NC] = {DFB_SIN_C_LIST};
__constant__ double c_cos[DFB_COS_NC] = {DFB_COS_C_LIST};

// Four draws starting at `state` -> (z0, z1).  Every floating-point operation is an explicit
// round-to-nearest intrinsic: nvcc may not contract, reorder or substitute anything.
__device__ __forceinline__ void normal_pair(uint64_t state, uint64_t inc, double& z0, double& z1) {
    uint32_t o0 = pcg_xsh_rr(state); state = pcg_lcg(state, inc);
    uint32_t o1 = pcg_xsh_rr(state); state = pcg_lcg(state, inc);
    uint32_t o2 = pcg_xsh_rr(state); state = pcg_lcg(state, inc);
    uint32_t o3 = pcg_xsh_rr(state);
    uint64_t U1 = ((((uint64_t)o1 << 32) | o0) >> 11) | 1u;
    uint64_t U2 = (((uint64_t)o3 << 32) | o2) >> 11;

    double d = __ull2double_rn(U1);                         // exact: U1 < 2^53
    uint64_t bits = (uint64_t)__double_as_longlong(d);
    const unsigned i6 = (unsigned)(bits >> 46) & 63u, hi = i6 >> 5;
    const int e = (int)(bits >> 52) - 1023 + (int)hi - 53;
    const double m = __longlong_as_double((long long)((bits & 0x000FFFFFFFFFFFFFULL) | ((uint64_t)(0x3FFu - hi) << 52)));
    const double2 tab = __ldg(&g_logtab[i6]);               // (INV, L)
    const double rr = __fma_rn(m, tab.x, -1.0);
    double P = c_log1p[DFB_LOG1P_NC - 1];
#pragma unroll
    for (int k = DFB_LOG1P_NC - 2; k >= 0; --k) P = __fma_rn(P, rr, c_log1p[k]);
    const double lp = __fma_rn(__dmul_rn(rr, rr), P, rr);
    const double lnu = __fma_rn((double)e, DFB_LN2, __dadd_rn(tab.y, lp));
    double r = __dsqrt_rn(__dmul_rn(-2.0, lnu));

    unsigned oct = (unsigned)(U2 >> 50);
    uint64_t T = U2 & ((1ULL << 50) - 1u);
    if (oct & 1u) T = (1ULL << 50) - T;
    double t = __dmul_rn(__ull2double_rn(T), 0x1p-50);
    double x = __dmul_rn(t, DFB_PIO4);
    double x2 = __dmul_rn(x, x);
    double S = c_sin[DFB_SIN_NC - 1];
#pragma unroll
    for (int k = DFB_SIN_NC - 2; k >= 0; --k) S = __fma_rn(S, x2, c_sin[k]);
    double sx = __fma_rn(__dmul_rn(x, x2), S, x);
    double Cc = c_cos[DFB_COS_NC - 1];
#pragma unroll
    for (int k = DFB_COS_NC - 2; k >= 0; --k) Cc = __fma_rn(Cc, x2, c_cos[k]);
    double cx = __fma_rn(x2, Cc, 1.0);
    // octant -> (sin, cos) of the full angle without data-dependent branches (lanes of a warp sit in all eight octants):
    //   odd octant: swap;  quadrant q = oct >> 1:  q odd: (sn, cs) = (c, -s) else (s, c);  q >= 2: negate both.
    // Negation = sign-bit flip, the same value the host's unary minus produces.
    const bool swap_sc = ((oct ^ (oct >> 1)) & 1u) != 0;      // (oct & 1) swaps once, (q & 1) swaps again
    double sn = swap_sc ? cx : sx, cs = swap_sc ? sx : cx;
    const unsigned q = oct >> 1;
    const long long neg_sn = (long long)(q >> 1) << 63;                       // q = 2, 3
    const long long neg_cs = (long long)(((q + 1u) >> 1) & 1u) << 63;         // q = 1, 2
    sn = __longlong_as_double(__double_as_longlong(sn) ^ neg_sn);
    cs = __longlong_as_double(__double_as_longlong(cs) ^ neg_cs);
    z0 = __dmul_rn(r, cs);
    z1 = __dmul_rn(r, sn);
}
#endif  // __CUDACC__

}  // namespace dfb
