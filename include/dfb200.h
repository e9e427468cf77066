/* include/dfb200.h -- the C ABI of the B200 digital-filter inflow generator (libdfb200.so).
 *
 * The reference (connorswitala/digital-filtering) has no FFI: its surface is a C++ class
 * (digital-filtering-c++/df/df.hpp:38-125) and a Fortran module (digital-filtering-fortran/df/df.f90:3-6,
 * 59-63, 74, 621).  This header is the thin C boundary both facades bind to:
 *     include/digital_filter.hpp      class DIGITAL_FILTER / struct DFConfig  (C++ callers, cpp-main.cpp:6-17)
 *     fortran/digital_filtering.f90   module DIGITAL_FILTERING via iso_c_binding (fortran-main.f90:8-26)
 * Plain pointers and sizes only; every scalar a Fortran caller passes is also available by
 * reference through the *_f entry points at the bottom.  All functions return an int status
 * (DFB_OK = 0); none throws or exits across the boundary (the reference prints to cerr and returns
 * half-initialised, df.cpp:225-228, or `stop`s, df.f90:327-330).  dfb_last_error() gives the text.
 *
 * Layout everywhere: row-major idx = j*Nz + k, j = wall-normal (slow), k = spanwise (fast)
 * (df.cpp:106,364); Fortran sees the same memory as (j-1)*Nz + k, 1-based (df.f90:608-610).
 *
 * Threading: one handle = one CUDA stream on one device.  Calls on one handle must be serialised
 * by the caller; different handles are independent (the reference is not re-entrant at all:
 * function-static RNG, df.cpp:334-335).
 */
#ifndef DFB200_H
#define DFB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dfb_filter_s* dfb_handle;

enum {
    DFB_OK = 0,
    DFB_ERR_ARG = 1,        /* bad argument / inconsistent config */
    DFB_ERR_IO = 2,         /* a data file could not be opened or parsed (df.cpp:225-228,492-495) */
    DFB_ERR_CUDA = 3,       /* CUDA runtime error, or no sm_100 device: there is NO CPU fallback */
    DFB_ERR_STATE = 4,      /* call not valid in this state (e.g. inject mode without noise) */
    DFB_ERR_INTERP = 5      /* linear_interpolate's invalid_argument (df.cpp:810-815) */
};

/* which = field selector for dfb_get_field / dfb_device_ptr */
enum {
    DFB_U_FLUC = 0, DFB_V_FLUC = 1, DFB_W_FLUC = 2,   /* u.fluc, v.fluc, w.fluc   (df.hpp:28,87) */
    DFB_T_FLUC = 3, DFB_RHO_FLUC = 4,                 /* T_fluc, rho_fluc         (df.hpp:59)    */
    DFB_U_FILT = 5, DFB_V_FILT = 6, DFB_W_FILT = 7    /* filt == filt_old after a step (df.cpp:440-442) */
};

enum { DFB_NOISE_GENERATE = 0, DFB_NOISE_INJECT = 1 };

/* dfb_config: the reference's DFConfig (df.hpp:38-49 / df.f90:59-63), field for field, followed by
 * extensions.  dfb_config_init() zeroes everything; an all-zero extension block reproduces the
 * reference's hard-coded default plane (df.cpp:7-16, 73-74, 224). */
typedef struct dfb_config {
    /* ---- DFConfig ---- */
    double d_i;                 /* inlet boundary-layer height          df.hpp:39 */
    double rho_e;               /* freestream density                   df.hpp:40 */
    double U_e;                 /* freestream velocity                  df.hpp:41 */
    double mu_e;                /* freestream viscosity                 df.hpp:42 */
    int vel_file_offset;        /* header lines of the fluctuation file df.hpp:44; > 0 selects the DNS statistics layout
                                   (M6Tw025_Stat.dat: columns 1,8,10,9,15 as in RST.cpp:43-50), 0 the RST.dat layout */
    int vel_file_N_values;      /* data rows of the fluctuation file    df.hpp:45 */
    const char* grid_file;      /* df.hpp:47 (unused by the reference, kept for layout parity) */
    int grid_file_len;          /* <0: NUL-terminated; >=0: Fortran len_trim */
    const char* vel_fluc_file;  /* df.hpp:48; RST.dat-format file; NULL/empty -> "../files/RST.dat" (df.cpp:224) */
    int vel_fluc_file_len;
    /* ---- extensions ---- */
    int struct_bytes;           /* sizeof(dfb_config) as the caller compiled it (set by dfb_config_init) */
    int honor_flow_config;      /* 0: the C++ reference's hard-coded flow constants (df.cpp:7-16, DFConfig ignored);
                                   1: take d_i, rho_e, U_e, mu_e from above as the Fortran does (df.f90:80-87) */
    const char* line_file;      /* mean-profile file (x,y,z,n,rho,u,v,w,t,p); NULL/empty -> "../line.dat" (df.cpp:16) */
    int line_file_len;
    int Ny, Nz;                 /* plane size; 0,0 -> the reference's made-up grid (df.cpp:73-74, trimmed at 282-288) */
    int geom_per_row;           /* 1: yc,dy,dz hold Ny entries (grid uniform in z); 0: Ny*Nz entries */
    const double* yc;           /* cell-centre heights   (df.hpp:68) */
    const double* dy;           /* cell heights          (df.hpp:69) */
    const double* dz;           /* cell widths           (df.hpp:70) */
    const double* rows;         /* [8][Ny]: R11,R21,R22,R33 (df.hpp:60), Us,Ts,rhos,Ms (df.hpp:81);
                                   NULL -> read + interpolate the two files as get_RST_in/read_line_file do */
    const double* scales;       /* [3][3]: per field (u,v,w) Iz_inn, Iz_out, Lt (df.hpp:32); NULL -> df.cpp:35-45 */
    const int* N_y;             /* optional explicit half-widths [3][Ny*Nz] (or [3][Ny] if geom_per_row); */
    const int* N_z;             /*   NULL -> calculate_filter_properties (df.cpp:144-154,186-195)         */
    uint64_t seed;              /* pcg32 seed of the counter-based generator (include/dfb_rng_spec.h) */
    int noise_mode;             /* DFB_NOISE_GENERATE | DFB_NOISE_INJECT */
    int device;                 /* CUDA ordinal; -1 = current device */
    int plane_id;               /* RNG stream group of this plane (distinct planes -> independent noise) */
    int k_begin, k_end;         /* spanwise slab [k_begin,k_end) of the Nz-wide plane owned by this handle;
                                   0,0 -> the whole plane.  Noise is keyed by the GLOBAL index, so slabs
                                   reproduce the single-GPU plane bit for bit with no halo exchange
                                   (periodic_z included: a wrapped neighbour column is regenerated locally too). */
    int skip_first_step;        /* 1: do not run the constructor's first step (df.cpp:57-62) */
    int kernel_variant;         /* 0 = tuned kernels where they apply (row-uniform half-widths whose z window fits in shared memory,
                                 * dfb_info 3); 1 = simple cross-check kernels (same maths, one thread per cell) */
    int periodic_z;             /* 0 (default): the reference's plane, NOT periodic in z -- the z filter reads raw white noise for
                                   the Nz_max columns beyond each spanwise edge (SURVEY quirk 1);
                                   1: spanwise-periodic plane -- the z filter wraps, filt[j,k] = sum_i b_i * y_filtered[j, (k+i) mod Nz],
                                   for spanwise-periodic LES/DNS inflow.  Needs Nz_max <= Nz for every field.  r_ys is drawn exactly
                                   as with 0 (only columns whose window reaches an edge change); the r_zs halo is not drawn.
                                   (Occupies what was the struct's tail padding: sizeof(dfb_config) is unchanged.) */
} dfb_config;

int dfb_config_init(dfb_config* cfg);

/* DIGITAL_FILTER::DIGITAL_FILTER(DFConfig) df.cpp:4-66: setup + first step (no blend, T'/rho' = 0). */
int dfb_create(const dfb_config* cfg, dfb_handle* out);
int dfb_destroy(dfb_handle h);
/* BASELINE config 5 -- `nplanes` (1..16) independent planes of ONE geometry advanced by one handle: one launch set per step for all of
 * them (plane index = an extra tile / work-item coordinate; coefficient tables, band matrices and row constants shared), where one
 * handle per plane pays three launches per plane.  Plane p draws from RNG stream group cfg->plane_id + p, so it reproduces the
 * single-plane handle created with that plane_id bit for bit.  Every per-field array of a batch handle is [nplanes][Ny*Nz]:
 * dfb_filter_to_host fills nplanes*Ny*Nz doubles per pointer, dfb_get_state / dfb_set_state move [3][nplanes][Ny*Nz].
 * The us3d_user.f90-style caller (my_user_init once, my_user_main_pre every step: us3d_user.f90:21-48, 51-130) creates the batch once
 * and calls dfb_filter every step; fortran/digital_filtering.f90 exposes it as create_digital_filter_batch. */
int dfb_create_batch(const dfb_config* cfg, int nplanes, dfb_handle* out);
int dfb_num_planes(dfb_handle h, int* nplanes);

/* plane size as the reference ends up with it (Ny trimmed, df.cpp:282-288); Nz is this handle's slab width */
int dfb_dims(dfb_handle h, int* Ny, int* Nz);
/* what = 0 Ny_max, 1 Nz_max (per field f), 2 step counter, 3 row-uniform fast path in use (0/1): 0 for per-cell half-widths,
 *    kernel_variant = 1, or a z window too wide for shared memory -- on a B200 (232 448 bytes per block) the tuned z-sweep takes
 *    N_z <= 1120 in its recursive form and N_z <= 544 in its direct form (a row with N_z = 0, a slab cut off a 16-column boundary)
 *    with 16 outputs per lane (planes of >= 384 columns), N_z <= 888 / 720 with 8; a wider window runs the whole handle on the
 *    one-thread-per-cell kernels, which take any half-width (DFB_ZK / DFB_Z_MODE forcing a window that does not fit: DFB_ERR_ARG),
 *    while any N_y runs on the tuned y-sweep (rows too tall for the run-recursive form go to its band-matrix kernels),
 * 4 algorithmic tap-FMAs per step (as int64 via out64), 5 global Nz, 6 CUDA device ordinal,
 * 7 form of the z-sweep in use: 1 = recursive evaluation of the exponential window, 0 = direct Toeplitz sum,
 * 8 / 9 y-sweep tiles of the band-matrix kernels evaluated recursively / with dense band matrices,
 * 10 form of the y-sweep in use: 2 = run-recursive (every row group through the exponential window), 3 = run-recursive on the blocks of
 *    32 rows where it pays + dense band matrices on the rest (e.g. a batch of planes of the reference's default geometry), 1 = chunk-recursive band-matrix
 *    kernel, 0 = dense band matrices (DFB_Y_MODE=0|1|2 forces a form), 11 tiles of the run-recursive kernel, 12 transport of the config-4 hand-off: 2 = peer-to-peer copies (CUDA IPC + copy engines), 1 = NCCL
 *    send/recv, 0 = no communicator, 13 spanwise-periodic plane (dfb_config.periodic_z) in use (0/1),
 * 14 lags of correlation direction `field` (0 z, 1 y, 2 t; dfb_corr_enable), 0 when that direction is off or before any enable */
int dfb_info(dfb_handle h, int what, int field, int64_t* out64);
/* host copies of the setup tables (for parity tests): which = 0..7 rows R11,R21,R22,R33,Us,Ts,rhos,Ms [Ny];
 * 8 yc row [Ny]; 9 dy row [Ny]; 10 Lt[3]; 11 coefficients of half-width `arg` [2*arg+1];
 * 12 y of the vertex rows [Ny+1]; 13 z of the vertex columns [Nz_global+1] (df.cpp:99-100: the y / z the writers print) */
int dfb_get_table(dfb_handle h, int which, int arg, double* dst, int cap);
/* N_y / N_z of field f (dir 0 = y, 1 = z) for the local slab, [Ny*Nz] */
int dfb_get_half_widths(dfb_handle h, int field, int dir, int* dst);

/* DIGITAL_FILTER::filter(double dt_input) df.cpp:449-468 -- enqueues the whole step on the handle's
 * stream and returns; no print, no CSV (SURVEY quirk 8).  Results are read with dfb_get_field.
 * dt must be finite and >= 0 (here and in dfb_filter_to_host, _begin, dfb_get_rms, every entry of dfb_filter_batch's array, and the
 * _f entry points): otherwise DFB_ERR_ARG and nothing is enqueued -- the step counter, the fields, filt_old, the noise and the N2 and
 * correlation statistics stay as they were; dfb_filter_batch checks its whole array before the first step.  (A negative dt would give
 * the blend alpha = exp(-pi dt / Lt) > 1 and sqrt(1 - alpha) = NaN.)  dt = 0 gives alpha = 1: filt = filt_old; dt >> Lt gives
 * alpha = 0: no blend, the step of dfb_first_step. */
int dfb_filter(dfb_handle h, double dt);
/* The constructor's first step on demand (df.cpp:57-62: sweeps + RST scaling, no blend, T'/rho' untouched).
 * dfb_create runs it by itself in generate mode; in inject mode call it after the first dfb_set_noise x3. */
int dfb_first_step(dfb_handle h);
/* filter(dt) + copy the five outputs into caller (host) arrays of Ny*Nz doubles; any pointer may be
 * NULL.  This is the call the C++ / Fortran facades make every step (u.fluc ... live on the host). */
int dfb_filter_to_host(dfb_handle h, double dt, double* u, double* v, double* w, double* T, double* rho);
/* The same, pipelined: _begin enqueues the step and the copies and returns; _end blocks until the arrays of the OLDEST outstanding
 * _begin are filled.  At most two _begin may be outstanding, so a caller with two sets of (pinned) arrays overlaps the copy of step t
 * (84 MB at 1024x2048: 1.5 ms of PCIe) with the compute of step t+1:  begin(A); loop { begin(B); end(); use A; swap(A, B); } */
int dfb_filter_to_host_begin(dfb_handle h, double dt, double* u, double* v, double* w, double* T, double* rho);
int dfb_filter_to_host_end(dfb_handle h);
/* nsteps consecutive steps; out (optional, host) receives [nsteps][5][Ny*Nz] with D2H copies
 * overlapped with the following steps. */
int dfb_filter_batch(dfb_handle h, int nsteps, const double* dt, double* out);

/* copies one field (Ny*Nz doubles) to dst; dst_on_device != 0 -> dst is a device pointer */
int dfb_get_field(dfb_handle h, int which, double* dst, int dst_on_device);
/* the same for plane `plane` of a batch handle (dfb_get_field = plane 0) */
int dfb_get_field_plane(dfb_handle h, int plane, int which, double* dst, int dst_on_device);
/* device pointer to a field, valid until dfb_destroy (for GPU-resident CFD codes / NCCL gathers) */
int dfb_device_ptr(dfb_handle h, int which, void** ptr);
int dfb_device_ptr_plane(dfb_handle h, int plane, int which, void** ptr);
/* the handle's cudaStream_t */
int dfb_stream(dfb_handle h, void** stream);
/* CFD hand-off on the device (SURVEY 8f N3; the call a US3D-style plugin makes per inflow face, us3d_user.f90:88-113:
 * ghost-cell state = mean + fluctuation): dst[dst_index[i]] = mean[i] (or dst's own value when mean is NULL) +
 * scale * field[plane_index[i]], i < n, enqueued on the handle's stream after the step that produced `which`.
 * All four pointers are DEVICE pointers; plane_index is j*Nz + k within this handle's slab. */
int dfb_scatter_to_cells(dfb_handle h, int which, int n, const int* plane_index, const int* dst_index,
                         const double* mean, double scale, double* dst);
int dfb_sync(dfb_handle h);
/* page-lock (cudaHostRegister) / release a caller-owned host array: dfb_filter_to_host into registered arrays runs at the PCIe
 * rate; pageable arrays cost an extra staging pass inside the driver.  The C++ facade does this for its std::vectors. */
int dfb_host_register(void* ptr, size_t bytes);
int dfb_host_unregister(void* ptr);

/* BASELINE config 4 -- ONE plane in spanwise slabs over the ranks of a job (one process per GPU, each with a handle created with its
 * own k_begin/k_end; the filter itself needs no exchange, see k_begin).  NCCL over NVLink only hands the finished plane to the CFD rank
 * (README.md:55 "MPI support to distribute result"; the consumer is the per-rank face loop of us3d_user.f90:85-92):
 *   rank 0:     dfb_comm_unique_id(id)  -> ship the 128 bytes to every rank by the job's own means (MPI_Bcast, a file, ...)
 *   every rank: dfb_comm_init(h, id, rank, world)            collective; checks that the slabs tile [0, Nz) in rank order
 *   per step:   dfb_filter(h, dt); dfb_gather_begin(h, dst); [dfb_filter(h, dt) of the next step ...]; dfb_gather_end(h);
 * dfb_gather_begin stages u', v', w' of the step just enqueued (the next dfb_filter may follow at once) and ships them -- 24 bytes per
 * cell; T', rho' are row-wise multiples of u' (df.cpp:470-485) and are rebuilt on the destination, bit for bit -- on a communication
 * stream, into row-major [Ny][Nz] planes on the destination.  dfb_gather_end blocks until that is done; the gathered plane stays valid
 * until the next dfb_gather_begin.  Transport: NCCL sets the job up (communicator, exchange of the slab bounds and of CUDA IPC handles);
 * the data itself goes peer to peer -- each sender's copy engine writes its slab straight into the destination plane's final layout
 * over NVLink (strided 2-D copies), ordered by stream memory operations on flags: no SM is involved, so the hand-off of step t runs
 * under the persistent sweep kernels of step t+1.  Where CUDA IPC is not available between the ranks (or with
 * DFB_GATHER_TRANSPORT=nccl) the slabs go through ncclSend/ncclRecv and an assembly kernel instead.
 * A rank that only wants its own faces filled never gathers: it calls dfb_face_map + dfb_scatter_to_cells on its slab. */
#define DFB_COMM_ID_BYTES 128
int dfb_comm_unique_id(void* id128);
int dfb_comm_init(dfb_handle h, const void* id128, int rank, int world);
int dfb_comm_info(dfb_handle h, int* rank, int* world, int* bounds /* [2*world]: k_begin, k_end per rank; may be NULL */);
int dfb_gather_begin(dfb_handle h, int dst_rank);
int dfb_gather_end(dfb_handle h);
/* destination rank: device pointer to / host copy of gathered field `which` (DFB_U_FLUC .. DFB_RHO_FLUC), [Ny][Nz_global] */
int dfb_gathered_ptr(dfb_handle h, int which, void** ptr);
int dfb_gathered_to_host(dfb_handle h, int which, double* dst);
/* the cudaStream_t the hand-off runs on (for device-side timing of it) */
int dfb_comm_stream(dfb_handle h, void** stream);
/* bytes this rank put on / took off the wire in the last dfb_gather_begin */
int dfb_gather_wire_bytes(dfb_handle h, int64_t* bytes);
int dfb_comm_destroy(dfb_handle h);

/* noise injection ("ingest the reference's own draws", SURVEY quirk 4).  Host arrays in the
 * reference's layouts: r_ys (Ny+2*Ny_max) x Nz (df.cpp:197); halo Ny x (2*Nz_max) = the left and
 * right Nz_max raw-noise columns of r_zs, the only part of it that is read (df.cpp:157,398).
 * periodic_z = 1: r_ys alone is the noise (the z filter wraps onto y-filtered columns); r_zs_halo must be NULL. */
int dfb_set_noise(dfb_handle h, int field, const double* r_ys, const double* r_zs_halo);
/* same, but r_zs is the reference's full Ny x (Nz+2*Nz_max) array; its interior is ignored (all of it with periodic_z = 1; may be NULL) */
int dfb_set_noise_ref_layout(dfb_handle h, int field, const double* r_ys, const double* r_zs);
/* read back the noise of the last step in the same layouts (RNG gate); periodic_z = 1: r_zs_halo must be NULL */
int dfb_get_noise(dfb_handle h, int field, double* r_ys, double* r_zs_halo);
/* only generate the noise of step `step` (no filtering) -- used by the RNG gate and the benchmarks */
int dfb_generate_noise(dfb_handle h, int64_t step);

/* checkpoint (SURVEY section 5): filt_old[3][Ny*Nz] + step counter; the seed is in the config */
int dfb_get_state(dfb_handle h, double* filt_old3, int64_t* step);
int dfb_set_state(dfb_handle h, const double* filt_old3, int64_t step);

/* N2 -- running statistics, the reference's only validation tool (rms_add / plot_rms, df.cpp:571-621), on the device
 * and opt-in: after dfb_stats_enable(h, 1) every dfb_filter also accumulates per cell the sums of u'^2, v'^2, w'^2,
 * T'^2, rho'^2 and u'v' (which = 0..5).  dfb_stats_get copies one of them to the host (as_rms != 0: sqrt(sum/count)
 * like plot_rms, not for u'v') and returns the number of accumulated steps. */
int dfb_stats_enable(dfb_handle h, int on);
int dfb_stats_get(dfb_handle h, int which, int as_rms, double* dst, int64_t* count);
int dfb_stats_get_plane(dfb_handle h, int plane, int which, int as_rms, double* dst, int64_t* count);
/* get_rms (df.cpp:584-611), what the reference's own driver calls (test/cpp-main.cpp:17): reset the sums, run `nsteps` filter(dt)
 * steps (the reference: 500 steps of dt = 1e-5) accumulating on the device.  Results through dfb_stats_get(.., as_rms = 1, ..)
 * and dfb_write_rms_csv. */
int dfb_get_rms(dfb_handle h, int nsteps, double dt);
/* Correlation statistics -- does the generated field carry the integral scales it was configured with?  Opt-in: after
 * dfb_corr_enable(h, 1, lags) every dfb_filter (directly, or through _to_host, _begin, dfb_filter_batch, dfb_get_rms -- the steps N2
 * accumulates; not the constructor's step, not dfb_first_step) adds, on the handle's stream, per-row sums of lagged products of u', v'
 * and w' (field = 0, 1, 2; the fluc arrays, after blending and Lund scaling).  With f_s = field `field` of plane `plane` after
 * accumulated step s, L_d = lags[d], and per row j, summed over the columns k and over the accumulated steps:
 *   DFB_CORR_Z  S_z[j][d] = sum f(j,k) f(j,k+d),    d = 0..L_z; without periodic_z only k + d < Nz counts, with it the column
 *                                                    is (k+d) mod Nz and all Nz columns count
 *   DFB_CORR_Y  S_y[j][d] = sum f(j,k) f(j+d,k),    d = 0..L_y, j + d < Ny (one-sided: (j, j+d) gives the full two-point function)
 *   DFB_CORR_T  S_t[j][m] = sum f_s(j,k) f_{s-m}(j,k), m = 0..L_t; step s contributes to lag m only if step s-m was accumulated
 *                                                    too (a device ring holds the last L_t fields: L_t * nplanes * 3 * Ny * Nz doubles)
 * Lags: 0 turns a direction off; DFB_CORR_SUPPORT = the filter's whole support, where the expected correlation ends: z max over the
 * fields of 2 Nz_max, capped at Nz-1; y max of 2 Ny_max, capped at Ny-1 (DFB_ERR_ARG for t).  Otherwise 0 <= L_z <= Nz-1,
 * 0 <= L_y <= Ny-1, 0 <= L_t <= 64, else DFB_ERR_ARG.  Every field uses the same lags: dst is [Ny][L_d+1].
 * Whole planes only: a slab handle (k_begin/k_end narrower than the plane) gets DFB_ERR_ARG, "correlation statistics need the whole
 * plane" -- the spanwise sums need the neighbours' columns.  Single planes and batches, every kernel form, both periodic_z modes.
 * When they are off nothing is launched. */
enum { DFB_CORR_Z = 0, DFB_CORR_Y = 1, DFB_CORR_T = 2 };
#define DFB_CORR_SUPPORT (-1)
/* on = 1: allocates the sums (on the first call, or when the lags change), the ring and a scratch of partial sums (whenever they are
 * absent; a failed allocation is DFB_ERR_CUDA with a message), zeroes the sums, empties the ring and sets count = 0.  on = 0: stops
 * accumulating and frees the ring and the scratch; the sums stay readable (lags may be NULL).  Every valid lag fits the kernels'
 * shared memory: the z kernel stages its lag halo one block of lags at a time.
 * dfb_set_state empties the ring and keeps the sums: the next step follows the restored state, not the ring.
 * dfb_info selector 14 gives L_d of direction `field` (0 z, 1 y, 2 t) once enabled, 0 for an off direction and before any enable. */
int dfb_corr_enable(dfb_handle h, int on, const int lags[3]);
/* normalized = 0: the raw sums.  normalized = 1: correlation coefficients, z and t (S[j][d]/pairs[d]) / (S[j][0]/pairs[0]),
 * y S_y[j][d] / sqrt(S_y[j][0] S_y[j+d][0]); NaN where j + d >= Ny, where a variance is 0 (u' on rows with R11 = 0) or where a lag
 * has no pairs yet.  pairs (optional, [L_d+1]) = products per row behind each lag: z steps*(Nz-d) without periodic_z, steps*Nz with
 * it; y steps*Nz; t Nz times the number of steps that had a predecessor m steps back.  count (optional) = accumulated steps.
 * dst may be NULL.  Before any enable: DFB_ERR_STATE.  A field, direction (or one enabled with lag 0) or plane out of range: DFB_ERR_ARG. */
int dfb_corr_get(dfb_handle h, int field, int dir, int normalized, double* dst, int64_t* pairs, int64_t* count);
int dfb_corr_get_plane(dfb_handle h, int plane, int field, int dir, int normalized, double* dst, int64_t* pairs, int64_t* count);
/* Integral scale per row j from the normalised R: with d* the last lag such that R(e) > 0 for every e <= d*,
 * dst[j] = sum_{d=1..d*} (R(d-1) + R(d))/2 * (x(d) - x(d-1)), where x(d) = d * wbar for z, wbar = (z_v[NzG] - z_v[0]) / NzG of the
 * vertex table (dfb_get_table 13), metres; x(d) = yc[j+d] - yc[j] for y (dfb_get_table 8), metres, upward; x(m) = m for t, in steps
 * (multiply by dt).  NaN for a row with zero variance.  Host arithmetic on the copied-back sums, the same for every facade. */
int dfb_corr_integral_scales(dfb_handle h, int plane, int field, int dir, double* dst /* [Ny] */);
/* plot_rms (df.cpp:613-675): "z, y, u'_rms, v'_rms, w'_rms, T'_rms, rho'_rms " then one row per cell with the cell's lower-left VERTEX
 * coordinates (z[iidx], y[iidx]), default stream formatting (6 significant digits), ", " separators */
int dfb_write_rms_csv(dfb_handle h, const char* path);
/* N4 -- write_csv (df.cpp:764-803), opt-in and never called by dfb_filter: "z,y,u_fluc,v_fluc,w_fluc,T_fluc,rho_fluc",
 * fixed notation, 15 decimals, one row per cell in j-major order. */
int dfb_write_csv(dfb_handle h, const char* path);
/* write_tecplot (df.cpp:712-762): VARIABLES / ZONE (I = Nz+1, J = Ny+1, F=BLOCK) / VARLOCATION header, then the vertex z and y
 * blocks ((Ny+1)*(Nz+1) values, one per line) and the cell-centred u', v', w' blocks (Ny*Nz values each), default stream formatting.
 * (The reference's writer does not compile at HEAD -- member z is undeclared, SURVEY section 0 -- this follows its text.) */
int dfb_write_tecplot(dfb_handle h, const char* path);
/* N3 -- face -> (j,k) map for the CFD hand-off (us3d_user.f90:85-114: a plugin loops over its inflow faces j1..j2 and writes ghost cell
 * ii = ife(j,2)): for n face centres (yf[i], zf[i]) in the plane's coordinates, plane_index[i] = j*Nz + k of the cell of THIS handle's
 * slab that contains the point (clamped to the nearest cell in y and z), or -1 when the face lies in another rank's slab.  Host arrays;
 * the result is what dfb_scatter_to_cells takes as plane_index (after a copy to the device). */
int dfb_face_map(dfb_handle h, int n, const double* yf, const double* zf, int* plane_index);

/* CUDA-event time of the last dfb_filter, ms: stage 0 noise, 1 y-sweep, 2 z-sweep+epilogue, 3 whole step.
 * Only recorded when enabled with dfb_set_timing(h, 1). */
int dfb_set_timing(dfb_handle h, int on);
int dfb_last_ms(dfb_handle h, int stage, float* ms);

/* DFMA throughput microbenchmark on the handle's device -> TFLOP/s (the fp64 roofline denominator,
 * absent from MEASURED_PEAKS.json) */
int dfb_measure_fp64_peak(int device, double* tflops, double* sm_mhz_est);

const char* dfb_last_error(void);
const char* dfb_version(void);

/* ---- Fortran-friendly by-reference wrappers (iso_c_binding, all arguments by reference) ---- */
int dfb_create_f(const dfb_config* cfg, dfb_handle* out);
int dfb_filter_f(const dfb_handle* h, const double* dt);
int dfb_filter_to_host_f(const dfb_handle* h, const double* dt, double* u, double* v, double* w, double* T, double* rho);
int dfb_dims_f(const dfb_handle* h, int* Ny, int* Nz);
int dfb_create_batch_f(const dfb_config* cfg, const int* nplanes, dfb_handle* out);
int dfb_get_field_plane_f(const dfb_handle* h, const int* plane, const int* which, double* dst);
int dfb_comm_init_f(const dfb_handle* h, const void* id128, const int* rank, const int* world);
int dfb_gather_begin_f(const dfb_handle* h, const int* dst_rank);
int dfb_gather_end_f(const dfb_handle* h);
int dfb_gathered_to_host_f(const dfb_handle* h, const int* which, double* dst);
int dfb_face_map_f(const dfb_handle* h, const int* n, const double* yf, const double* zf, int* plane_index);
int dfb_destroy_f(dfb_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* DFB200_H */
