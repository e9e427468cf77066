// csrc/device.cuh -- device-side data layout of one inflow plane (or one spanwise slab of it) in HBM.
//
//   r_ys[f]   (Ny + 2*Ny_max[f]) x pitch_y   white noise of the y-sweep (df.cpp:197), columns = the slab's
//                                            EXTENDED range [xk0, xk1) = [k0-Nz_max, k1+Nz_max) clipped to the plane;
//                                            periodic_z: NOT clipped (xk0 may be negative), extended column x holds
//                                            global column (xk0 + x) mod NzG -- the plane part starts at column -xk0
//   r_zs[f]   Ny x pitch_z                   logical column c in [0, W+2*Nz_max) lives at zoff + c; c = Nz_max is
//                                            the slab's first column (df.cpp:157,363).  Columns whose GLOBAL
//                                            index falls outside [0,NzG) hold raw noise (SURVEY quirk 1),
//                                            the others are written by the y-sweep (incl. neighbours' columns,
//                                            recomputed locally instead of exchanged).  periodic_z: the y-sweep
//                                            writes every column (yshift = 0), those beyond an edge wrapped.
//   filt_old[f], fluc[f], T, rho   dense Ny x W, row-major j*W + k  (df.cpp:106) -> one memcpy to the caller
//   coefficients: one row per distinct half-width N (CSR keyed by N), plus per-row-group dense band
//   matrices for the tuned y-sweep; per-row epilogue constants.
#pragma once
#include <cmath>
#include <cstdint>
#include <cuda_runtime.h>
#include <cuda.h>

namespace dfb {

constexpr int YJ = 8;          // output rows per thread / per row group of the tuned y-sweep
constexpr int Y_G = 4;         // row groups (consumer warps) per y-sweep tile: 32 output rows share one sample stream
constexpr int Y_TK = 128;      // columns per y-sweep tile (each lane owns 4 of them)
constexpr int DFB_MAXP = 16;   // planes one handle can advance in one launch set (dfb_create_batch)
constexpr int Y_RC = 8;        // padded rows per chunk of the band-matrix y-sweep (ysweep_tma_kernel, ysweep_rec_kernel)
constexpr int Y_NS = 6;        // chunks it keeps in flight
// pairs per thread of the noise kernel, NOISE_THREADS pairs apart (one position jump per thread, stride jumps between its pairs).  Measured
// ms/step on 1024x2048 / 4096x8192 profile, pairs and NOISE_UNROLL: 4, 1: 0.1170 / 1.537; 4, 2: 0.1151 / 1.526; 4, 4: 0.1144 / 1.499; 8, 2: 0.1146 / 1.472
#ifndef NOISE_PAIRS
#define NOISE_PAIRS 8
#endif
#ifndef NOISE_THREADS
#define NOISE_THREADS 128
#endif

struct FieldDev {
    int Ny_max, Nz_max;
    int rows_y;            // Ny + 2*Ny_max
    int We, xk0;           // extended column count, global index of extended column 0
    int pitch_y;           // doubles
    int pitch_z, zoff;     // doubles
    int yshift;            // extended column x -> r_zs logical column x + yshift
    double* r_ys;          // plane p of a batch: + p * ps_ys
    double* r_zs;          //                     + p * ps_zs
    double* filt_old;      //                     + p * PlaneDev::ps_cells (also fluc, T_fluc, rho_fluc)
    double* fluc;
    size_t ps_ys, ps_zs;   // doubles per plane of r_ys / r_zs (planes of a batch are stacked along the rows)
    const int* Ny_row;     // [Ny]
    const int* Nz_row;     // [Ny]
    const int* Ny_cell;    // [Ny*NzG] or nullptr (row-uniform)
    const int* Nz_cell;
};

// per-row constants of the fused epilogue, computed on the host with the reference's expressions
// (df.cpp:425-438, 474): {sqrt(R11), b, sqrt(R22-b*b), sqrt(R33), temp1, Ts, rhos, pad}
constexpr int ROWC = 8;

struct PlaneDev {
    int Ny, W, NzG, k0;
    int P;                     // planes in this handle (1 unless dfb_create_batch): same geometry and tables, own noise streams and state
    size_t ps_cells;           // Ny * W
    FieldDev f[3];
    double* T_fluc;
    double* rho_fluc;
    const double* rowc;        // [Ny][ROWC]
    const int64_t* coef_ptr;   // [Nmax+1]
    const double* coef_vals;
};

// ---- tuned y-sweep work description ----
struct YGroup {                // YJ consecutive output rows of one field
    int field, j0, nrows, Nmax;
    int cstart;                // first chunk of the window on the field's absolute chunk grid (chunk c = padded rows [c*RC, (c+1)*RC))
    int nchunks;               // chunks the window touches
    long long cmat_off;        // doubles, into the band-matrix pool: Cmat[(row - cstart*RC)][YJ]
    int rec;                   // 1: every row has the same half-width N = Nmax >= 16: recursive evaluation (ysweep_rec_kernel)
    int w0;                    // padded row of the group's first window sample (= j0 + Ny_max - Nmax)
    int gc_off;                // recursive: index (x16 doubles) of the group's bulk factors in YParams::ygc
};
struct YTile {                 // up to Y_G consecutive groups x Y_TK columns
    int field, col0, g0, ngroups;
    int cbegin, cend;          // union of the groups' chunk ranges
};

struct YMaps { CUtensorMap m[3]; };

// ---- y-sweep, run-recursive form (ysweep_run_kernel): row groups of consecutive rows with ONE half-width ----
constexpr int YR_JL = 32;      // most rows of a long (lock-step) group; short groups hold <= YJ rows
constexpr int YR_LOCK_MIN_N = 25;
// Most rows a group of half-width N may hold.  Long groups walk the B sum against its stable direction (an error grows by
// 1/a = exp(2 pi / N) per row): bounded so that exp(2 pi R / N) <= 8, i.e. R <= N ln 8 / (2 pi) = 0.331 N.
inline int yr_group_cap(int N) { return N >= YR_LOCK_MIN_N ? (N * 331 / 1000 < YR_JL ? N * 331 / 1000 : YR_JL) : YJ; }
constexpr int YR_C = 32;       // columns per tile = lanes of a warp (one column each)
constexpr int YR_BOX = 32;     // padded rows per TMA box of the resident window
#ifndef YR_CONSUMERS_N
#define YR_CONSUMERS_N 8
#endif
constexpr int YR_CONSUMERS = YR_CONSUMERS_N;   // consumer warps of the persistent CTA (+ one producer warp).  Measured ms/step on 1024x2048 profile:
                                               // 4: 0.141, 6: 0.123, 8: 0.115, 12: 0.121, 16: 0.123 -- the kernel is bound by shared-memory bandwidth, and the registers
                                               // fewer warps leave free go to the next step's noise CTAs, which run beside it
constexpr int YR_MAXG = 128;   // most groups a tile can hold (a block of 128 rows, every row its own group)
struct YRGroup {               // 48 bytes
    int j0, nrows, N, pad;     // pad: 1 = long group (nrows > YJ), evaluated in lock step
    double a;                  // exp(-2 pi / N): ratio of neighbouring coefficients, b_i = a^|i| / s (df.cpp:168-177); 0 for N = 0
    double a4;                 // a^4 (the Horner starts run as four interleaved chains)
    double naN1;               // -a^(N+1): weight of the sample a sliding window drops
    double inv_s;              // centre coefficient b_0 = 1 / s
};
struct YRTile {                // row block x 32 columns of one field; its whole input window is staged in shared memory
    int field, col0, g0, ngroups;
    int wlo, wrows;            // first padded row and row count of the window (union of the groups' windows)
};
struct YRMaps { CUtensorMap m[3]; };   // r_ys[f] with box {YR_C columns, YR_BOX rows}
struct YRSmemCtl {                       // control block in front of the two window buffers
    uint64_t full[2], empty[2];
    int next_group[2];
    YRTile tile[2];
    int plane[2];
    int pad[2];
    alignas(16) YRGroup groups[2][YR_MAXG];      // cp.async.bulk destination
};
// dynamic shared memory of ysweep_run_kernel for `nbuf` window buffers of `wrows` rows
inline size_t ysweep_run_smem(int wrows, int nbuf) { return (sizeof(YRSmemCtl) + 127) / 128 * 128 + (size_t)nbuf * wrows * YR_C * sizeof(double); }

// Blend constants of one field (df.cpp:411-415): sa = sqrt(alpha), sb = sqrt(1 - alpha), alpha = exp(-pi dt / Lt).  The host evaluates
// them with its libm's exp (dfb_filter), step_advance_kernel with CUDA's (dfb_filter_dev); both are within one ulp of the exact value,
// so the two agree to rounding.  Multiply, divide and sqrt are correctly rounded on both sides.
__host__ __device__ inline void blend_consts(double dt, double Lt, double& sa, double& sb) {
    const double pi = 3.141592654;                             // df.cpp:411 (SURVEY quirk 2)
    const double alpha = exp(-pi * dt / Lt);                   // df.cpp:412
    sa = sqrt(alpha);                                          // df.cpp:415
    sb = sqrt(1.0 - alpha);
}

struct StepConsts {
    double sa[3], sb[3];       // sqrt(alpha), sqrt(1-alpha) per field (df.cpp:412-415), from the host's exp/sqrt
    int first_step;            // constructor semantics (df.cpp:57-62): no blend, T'/rho' untouched
};

// Step record of a handle attached to a caller's stream (dfb_attach_stream): what the host holds for a host-driven step, in device
// memory, so that a step needs no host decision and replays of a captured graph advance the generator.  Written by step_advance_kernel,
// the first launch of every attached step; read by the step's noise and z-sweep launches through their `rec` pointer.
struct StepRecord {
    long long step;            // steps completed (the host's dfb_filter_s::step)
    long long stats_count;     // N2: accumulated steps
    double dt;                 // dt of the current step
    double sa[3], sb[3];       // blend constants of the current step
    uint64_t pstate[DFB_MAXP][6];   // per plane and noise array: pcg32 state at the first draw of the current step (NoiseParams::pstate)
    int void_step;             // the current step is void (dt not finite or < 0): the z-sweep writes nothing
    int void_seen;             // sticky: a step was void since the host last read the record
};

struct AdvanceParams {
    StepRecord* rec;
    const double* dt_dev;      // dfb_filter_dev: dt in device memory; nullptr: dt, sa, sb below come from the host
    double dt, sa[3], sb[3];
    double Lt[3];              // time scales of u, v, w (df.cpp:412)
    uint64_t seed;
    uint64_t pinc[DFB_MAXP][6];     // stream increments, as NoiseParams::pinc
    uint64_t npairs[6];        // pairs one step draws from each array's stream
    int n_arrays, P;
    int stats;                 // this step accumulates N2: count it
    // per-row time scales (dfb_set_time_scales): step_advance_rows_kernel writes rows[i] = {sa, sb} of Lt_rows[i], i < n_rows = 3 Ny
    const double* Lt_rows;
    double2* rows;
    int n_rows;
};

// ---- noise generation work description (one segment = one row of one logical array, or one contiguous piece of a row) ----
struct NoiseArray {
    const void* seg_jump;      // Jump[n_seg]: jump from `state` to the segment's first pair
    const int* seg_off;        // r_ys: extended column of a segment's first pair, 2*q0 - (row * NzG + xk0) (a piece: + its first column,
                               // - its first stream element); halo: 0
    const int* seg_np;         // pairs in each segment
    int n_seg;
    int kind;                  // 0 = r_ys rows, 1 = r_zs halo rows
    int field;
};

struct Jump { uint64_t A, C; };   // affine map of the LCG state over a number of draws: state' = A*state + inc*C (noise.cuh)

struct NoiseParams {
    NoiseArray a[6];            // geometry of the (up to) six logical arrays, shared by the planes of a batch
    uint64_t pstate[DFB_MAXP][6];   // per plane and array: pcg32 state at the first draw of this step's array
    uint64_t pinc[DFB_MAXP][6];     //                      stream increment
    const Jump* slot_jump;      // (A, G) for delta = 4*t: state' = A*state + inc*G
    Jump stride;                // (A, G) for the 4*NOISE_THREADS draws between two consecutive pairs of one thread
    int n_arrays;
    int max_np;                 // largest segment (pairs)
    int chunks;                 // ceil(max_np / 128)
    unsigned long long* tl;     // development aid (DFB_TIMELINE): [start, end] globaltimer stamps of this launch, or nullptr
    const StepRecord* rec;      // attached step: the states come from rec->pstate instead of pstate; nullptr host-driven
};

// per array of NoiseParams: r_ys of a periodic plane whose extended rows wrap (periodic_z) -- {padded row, first, end extended column}
// of each segment, a row being up to three pieces of the stream (wrapped left piece, plane part, wrapped right piece); nullptr:
// segment = row, columns [0, We).  Only noise_pieces_kernel takes it: the parameters of noise_kernel stay those of a plane that
// does not wrap.
struct NoiseWindows { const int4* seg_win[6]; };

struct YParams {
    const YGroup* groups;
    const YTile* tiles;
    const double* cmat;
    int* zcounter;             // work counter of the z-sweep that follows (reset here ...
    int zcounter_init;         // ... to twice the z-sweep's warp count: its warps start on items they do not have to claim)
    const double* yrec;        // recursive groups, 16 doubles per half-width N: a at [0], a^2, a^4, a^8 at [10..12]
    const double* ygc;         // recursive groups, 16 doubles each: factors of the low-bulk sum [0..7] and of the high-bulk sum [8..15] per output row
    const YRGroup* rgroups;    // run-recursive form: groups and tiles (most expensive tile first), see ysweep_run_kernel
    const YRTile* rtiles;
    int n_rtiles;              // > 0: the run-recursive kernel is the y-sweep of this handle
    int r_smem;                // its dynamic shared memory: control block + two window buffers
    int r_wrows;               // rows of one window buffer (largest window, whole boxes)
    int r_nbuf;                // window buffers: 2, or 1 when two of the plane's tallest windows do not fit
    int r_grid;                // CTAs of the persistent grid (one per SM)
    int* rcounter;             // [2] tile queue of the run-recursive kernel: next tile (rests at r_grid between launches), CTAs done
    int tile0;                 // first tile of this launch in `tiles` (dense tiles first, then recursive tiles)
    int n_tiles;               // tiles of this launch (dense kernel: walked with stride gridDim.x)
    int tk;                    // columns per dense tile: 128, or 64 for planes that do not fill the GPU (never with recursive tiles)
    int resident_grid;         // > 0: launch the dense kernel with at most this many CTAs (one wave), each walking several tiles
    unsigned long long* prof;  // [8] cycle counters (development probe, filled when debug != 0)
    unsigned long long* tl;    // development aid (DFB_TIMELINE), see NoiseParams
    int debug;
    PlaneDev D;
};

struct ZUnit {                     // one row x one strip of 32*zk columns x one field: 8 ints
    int j, c0, f;
    int nchunk;                    // tap-loop chunks
    int line0;                     // first line (zk doubles) of the staged window
    int cbytes;                    // bytes staged after the window: the padded coefficient vector (direct form) or its 128-byte header (recursive form)
    int coff16;                    // offset of those bytes in coef_pad, in units of 16 doubles
    int pad;
};
static_assert(sizeof(ZUnit) == 32, "ZUnit is loaded as 8 ints, one per lane");
struct ZMaps { CUtensorMap m[3]; };   // r_zs[f] as {16 doubles, pitch/16 lines, Ny rows}, 128-byte swizzle

struct ZParams {
    PlaneDev D;
    StepConsts S;
    const ZUnit* units;          // n_uv items of two units (u, v of one (row, strip)), then n_items - n_uv items of one unit (w), each kind most expensive first
    int n_items, n_uv;           // items per plane; the work counter runs over n_items * D.P (item = c / P, plane = c % P)
    int* counter;                // work counter, zeroed by the y-sweep that precedes this launch
    const double* coef_pad;      // padded coefficient vectors B_N[m] = b_N[m - 16 - d(N)], zero elsewhere, + one 128-byte header line each
    const long long* coef_pad_ptr;   // [Nmax+1] offsets (doubles, 16-byte aligned) into coef_pad
    const double* unit_par;      // recursive form: per (row, field) the parameter line (16 doubles) followed by the row's ROWC epilogue
                                 // constants: what a unit stages after its window, as ONE record; nullptr in the direct form
    double* stats;               // N2 running sums [P][6][Ny*W] (u'^2, v'^2, w'^2, T'^2, rho'^2, u'v') accumulated by this launch, or nullptr
    int zk;                      // outputs per lane: 16 (128-byte lines) or 8 (64-byte lines); an item is 32*zk columns
    int box_lines;               // lines per staged window (box height of the tensor maps)
    int box_bytes;               // box_lines * zk * 8
    int unit_bytes;              // bytes per staging buffer: window | parameter line / coefficient vector | row constants | filt_old strip; 1024-aligned
    int rc_off, fo_off;          // offsets of the row constants (64 B) and of the staged filt_old strip (32 lines) in a staging buffer
    int nblocks;
    int smem_bytes;
    unsigned long long* tl;      // development aid (DFB_TIMELINE), see NoiseParams
    int zmode;                   // 0: direct Toeplitz tap loop; 1: recursive evaluation of the exponential window
    int debug;                   // development probes only (0 in production)
    unsigned long long* prof;    // [8] cycle counters filled when debug & 16
    const StepRecord* rec;       // attached step: sa, sb come from the record, and a void step writes nothing; nullptr host-driven
    const double2* rows;         // per-row time scales (dfb_set_time_scales): {sa, sb} of field f, row j at [f * Ny + j]; read by
                                 // zsweep_epilogue_rows_kernel only (sa, sb of S and rec are then unused)
};

}  // namespace dfb
