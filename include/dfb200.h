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
 *    N_z <= 1120 in its recursive form and N_z <= 544 in its direct form (a row with N_z = 0, a slab cut off a 16-column boundary,
 *    the Gaussian filter shape)
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
 * 14 lags of correlation direction `field` (0 z, 1 y, 2 t; dfb_corr_enable), 0 when that direction is off or before any enable,
 * 15 per-row time scales in use (dfb_set_time_scales, 0/1), 17 filter shape (dfb_set_filter_shape: DFB_FILTER_EXPONENTIAL /
 *    DFB_FILTER_GAUSSIAN), 18 flux correction mode (dfb_set_flux_correction: DFB_FLUX_OFF / _MASS / _VOLUME),
 * 19 per-cell profiles in use (dfb_set_profiles, 0/1) */
int dfb_info(dfb_handle h, int what, int field, int64_t* out64);
/* host copies of the setup tables (for parity tests): which = 0..7 rows R11,R21,R22,R33,Us,Ts,rhos,Ms [Ny];
 * 8 yc row [Ny]; 9 dy row [Ny]; 10 Lt[3]; 11 coefficients of half-width `arg` [2*arg+1], in the handle's filter shape;
 * 12 y of the vertex rows [Ny+1]; 13 z of the vertex columns [Nz_global+1] (df.cpp:99-100: the y / z the writers print);
 * 14 time scales Lt of field `arg` (0..2) per row in use [Ny]: the rows of dfb_set_time_scales, or the scalar Lt repeated;
 * 16 quantity `arg` (0..7, the order of 0..7) of the profiles in use for this handle's columns [Ny][Nz]: those of dfb_set_profiles, or
 *    the row table repeated along the span.  Tables 0..7 are the row tables whatever the profiles. */
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

/* GPU-resident CFD codes: run the steps on the caller's stream, with dt in device memory, capturable into a CUDA graph.
 * dfb_attach_stream(h, stream): from now on every call of this handle that enqueues device work goes on `stream` (a cudaStream_t of
 * the handle's device): steps, dfb_interp_to_cells, dfb_scatter_to_cells, and the copies of dfb_get_field / dfb_filter_to_host
 * (dfb_stream returns it).  The step's host state moves into device memory: step counter, pcg32 positions, blend constants, N2 count.
 * A step then needs no host decision: it is advance -> noise -> y-sweep -> z-sweep on `stream` alone, with no second stream, event,
 * synchronisation or allocation, so it can be captured with cudaStreamBeginCapture (cudaStreamCaptureModeGlobal included), and each
 * replay of the graph advances the generator by one step.  stream == NULL detaches: synchronises the attached stream, copies the device
 * step state back and continues host-driven.  An attached step does not overlap the next step's noise with this step's sweeps.
 * dfb_filter(h, dt) with a host dt still works while attached: the same device-driven step, with the blend constants computed on the
 * host as always, so a host-dt step is bit for bit the same attached or not.
 * dfb_filter_dev(h, dt_dev): one step whose dt is read from DEVICE memory (one double) when the step executes; the handle must be
 * attached (else DFB_ERR_STATE).  Nothing is read back and nothing synchronises.  The blend constants sqrt(exp(-3.141592654 dt / Lt))
 * are then computed on the device: CUDA's exp and the host's libm are each within one ulp, so they agree with dfb_filter's to rounding
 * (the fields to ~1e-15 of their rms), not bit for bit.  A dt that is not finite, or is < 0, voids the step: the fields, filt_old, the
 * N2 sums and the step counter stay as they were (the noise read back is the previous step's), and a sticky flag is set.  The next call
 * that synchronises (dfb_sync, dfb_info, dfb_get_state, dfb_set_state, dfb_get_field, dfb_filter_to_host, dfb_get_noise,
 * dfb_stats_get, dfb_save_restart, dfb_load_restart, dfb_interp_to_host, dfb_attach_stream(h, NULL)) returns DFB_ERR_ARG "dt must be
 * finite and >= 0 ..." once, does nothing else (a detach still detaches), and clears the flag.
 * While attached these return DFB_ERR_STATE, naming the call: dfb_comm_init and the gathers, dfb_corr_enable, dfb_stats_enable (set N2
 * on or off before attaching), dfb_set_timing(h, 1), dfb_filter_to_host_begin / _end, dfb_filter_batch, dfb_generate_noise,
 * dfb_get_rms.  Attaching an inject-mode handle, a handle with correlation statistics on or timing on, or while a _begin call is
 * outstanding is DFB_ERR_STATE; a stream of another device is DFB_ERR_ARG.  dfb_get_state / dfb_set_state, restart files, dfb_info,
 * dfb_stats_get, dfb_get_noise and face maps work: each synchronises the attached stream and reads or writes the device step record.
 * Load the kernels before capturing: dfb_attach_stream does it.  A captured graph references the handle's memory: it must not be
 * launched after a detach, a dfb_set_state / dfb_load_restart, or dfb_destroy; and the stream must outlive the attachment (dfb_destroy
 * of an attached handle synchronises it). */
int dfb_attach_stream(dfb_handle h, void* stream);
int dfb_filter_dev(dfb_handle h, const double* dt_dev);

/* Per-row temporal scales (opt-in).  The temporal blend of field f uses alpha = exp(-pi dt / Lt_f) with one Lt per field for the
 * whole plane (dfb_config.scales); under Taylor's hypothesis that fixes the streamwise length at row j to U(y_j) Lt_f, a small fraction
 * of its freestream value near the wall.  dfb_set_time_scales gives each field one Lt per row instead, e.g. Lt(y) = Ix(y) / U(y) for a
 * prescribed streamwise length Ix(y).
 * dfb_set_time_scales(h, Lt_rows): Lt_rows = [3][Ny] (u, v, w; Ny = dfb_dims, i.e. after the trim), every entry finite and > 0; NULL
 * returns to the config's scalar Lt.  Takes effect from the next step; the noise, filt_old and the step counter are untouched.  Rows
 * are global rows: every slab of a plane and every plane of a batch uses them, and slabs cut on multiples of 16 columns stay bit for
 * bit the whole plane.  Rows equal to the scalar Lt give the scalar path's results bit for bit.  Host-driven steps compute each row's
 * blend constants on the host with the scalar path's expressions and upload them when dt changes; attached steps (dfb_attach_stream)
 * compute them on the device, so with rows set an attached step agrees with a host-driven one to rounding (CUDA's exp against libm's),
 * also for a host dt.  Refused, leaving the handle as it was: an entry not finite or <= 0 (DFB_ERR_ARG, naming the field and row);
 * an attached handle (DFB_ERR_STATE: set the rows before attaching); an outstanding dfb_filter_to_host_begin or dfb_gather_begin
 * (DFB_ERR_STATE).  The rows are part of the restart fingerprint: a file saved with rows loads only into a handle with the same rows
 * (set them before dfb_load_restart); without rows the fingerprint is the one a handle without this feature has.
 * dfb_time_scales_from_lengths(h, Ix, u_min, Lt_rows): host only, fills Lt_rows[3][Ny] with Lt_f(j) = Ix_f(y_j) / max(Us_j, u_min),
 * Ix_f(y) = Ix_inn + (Ix_out - Ix_inn) * 0.5 * (1 + tanh((y / d_i - 0.2) / 0.03)) (the blend of Iz, df.cpp:146),
 * Ix = {inn_u, out_u, inn_v, out_v, inn_w, out_w} (metres, finite, > 0), y_j = dfb_get_table 8, Us = dfb_get_table 4, u_min > 0 (m/s). */
int dfb_set_time_scales(dfb_handle h, const double* Lt_rows);
int dfb_time_scales_from_lengths(dfb_handle h, const double Ix[6], double u_min, double* Lt_rows);
/* Filter shape (opt-in).  The spatial filters of every handle start as the reference's two-sided exponential (Xie & Castro),
 * b_i = exp(-2 pi |i| / N) / s: its correlation falls off as exp(-pi d / n) times a polynomial, and the integral scale it delivers is
 * about 0.64 of the configured Iz / Iy (N = 2 int(I / delta) = 2n).  DFB_FILTER_GAUSSIAN is the kernel of Klein, Sadiki & Janicka
 * (2003), b_i = exp(-2 pi i^2 / N^2) / s = exp(-pi i^2 / (2 n^2)) / s, whose correlation exp(-pi d^2 / (4 n^2)) has an integral scale of
 * n cells: the configured length to within one cell.  Both are normalised to sum b_i^2 = 1 over the same half-widths N (computed or
 * given in N_y / N_z); N = 0 is [1] in either shape.  The temporal blend is the exponential one in both: the temporal scale stays
 * 2 Lt / pi.
 * dfb_set_filter_shape(h, shape) sets the shape of a handle that has not stepped yet: in generate mode one created with
 * skip_first_step = 1 (call dfb_first_step afterwards for the constructor's step), in inject mode one whose step counter is still 0.  It
 * rebuilds the coefficient table and the step's whole plan (kernel forms, band matrices, z pads, tensor maps, grid sizes) and the
 * restart fingerprint; the noise, filt_old and the step counter are untouched.  A Gaussian has no exact sliding recursion, so a Gaussian
 * handle runs the direct forms: dense band matrices in y (dfb_info 10 = 0) and the direct z-sweep (dfb_info 7 = 0); a z window too
 * wide for the direct form runs the handle on the one-thread-per-cell kernels (dfb_info 3 = 0); DFB_Y_MODE=1|2 and DFB_Z_MODE=1 are
 * DFB_ERR_ARG.  Refused, leaving the handle as it was: an unknown shape (DFB_ERR_ARG); DFB_ERR_STATE, naming the reason, for a handle
 * that has stepped, is attached, has a communicator, has N2 or correlation statistics enabled, has per-row time scales or face maps,
 * or has a dfb_filter_to_host_begin outstanding.  The shape is part of the restart fingerprint when it is Gaussian (exponential
 * fingerprints are the ones handles without this call have) and is recorded in the file's header: a file written under the other
 * shape is DFB_ERR_ARG, naming both.  dfb_info 17 returns the shape. */
enum { DFB_FILTER_EXPONENTIAL = 0, DFB_FILTER_GAUSSIAN = 1 };
int dfb_set_filter_shape(dfb_handle h, int shape);
/* Inflow mass-flux correction (opt-in).  Every step's u' has a nonzero area-weighted plane mean, correlated over Lt: a low-frequency
 * pulsation of the inflow mass flow, which a compressible calculation receives as an acoustic disturbance.  With the correction on,
 * each plane p of each step (after the z-sweep) delivers
 *     u' <- fma(-c_p, sqrt(R11_j), u'),   c_p = m'_p / D,   m'_p = sum_jk A_jk g_j u'_jk,   D = sum_jk A_jk g_j sqrt(R11_j),
 * and T', rho' rebuilt from that u' with the epilogue's roundings (t2 = rc4 u'; T' = t2 Ts; rho' = -t2 rhos).  A_jk = hy_j hz_k are the
 * cells of the area face maps ([vert_y[j], vert_y[j+1]) x [vert_z[k], vert_z[k+1]), dfb_get_table 12, 13).  DFB_FLUX_MASS weighs with
 * g_j = rhos_j (1 + 0.2 Ms_j^2), the first-order mass flux rhos u' + Us rho' of the strong Reynolds analogy in use; DFB_FLUX_VOLUME with
 * g_j = 1.  The delivered first-order flux sum A g u' is then zero to rounding.  Rows with R11 = 0 are unchanged.
 * Only the delivered u', T', rho' change: filt_old (DFB_*_FILT), v' and w' are the same as with the correction off, so the generator
 * evolves the same way whatever the mode, and a restart file (its header and fingerprint) does not depend on it.  The second-order
 * flux rho' u' is not balanced (it has a nonzero mean of its own, fixed by the Reynolds stresses rather than by the filter's
 * sampling).  The constructor's step and dfb_first_step are never corrected.  N2 statistics, correlation statistics, face maps,
 * dfb_scatter_to_cells and every copy of the fields see the corrected fields.  Batches are corrected plane by plane, each plane bit for
 * bit as a single-plane handle of its plane_id.
 * dfb_set_flux_correction(h, mode): DFB_FLUX_OFF (default), DFB_FLUX_MASS or DFB_FLUX_VOLUME, from the next step on.  Refused,
 * leaving the handle as it was: an unknown mode or, for a mode other than DFB_FLUX_OFF, a slab handle (k_begin, k_end), or a plane with
 * R11 = 0 on every row (DFB_ERR_ARG); an attached handle or an outstanding dfb_filter_to_host_begin (DFB_ERR_STATE).  Attached steps and
 * graph replays take the correction; a void step changes nothing.  dfb_info 18 returns the mode.
 * dfb_flux_info(h, plane, out[3]): c_p and m'_p of the last corrected step of `plane`, and the mean flux sum A rhos Us (mass) or
 * sum A Us (volume) of the mode last enabled; before the first corrected step c_p = m'_p = 0.  DFB_ERR_STATE if the correction was
 * never enabled.  Synchronises the handle's stream (and an attached handle's step record). */
enum { DFB_FLUX_OFF = 0, DFB_FLUX_MASS = 1, DFB_FLUX_VOLUME = 2 };
int dfb_set_flux_correction(dfb_handle h, int mode);
int dfb_flux_info(dfb_handle h, int plane, double out[3]);
/* Per-cell profiles (opt-in), for planes whose boundary layer varies along the span (a cone at angle of attack, an elliptic cone, a
 * swept fin, a corner or duct inflow).  By default the eight quantities R11, R21, R22, R33, Us, Ts, rhos, Ms that scale the filtered
 * fields are one per row (dfb_config.rows, or interpolated from the data files at column 0's wall distance), so every column gets the
 * same boundary layer.  dfb_set_profiles(h, cells) gives every cell its own: cells is [8][Ny][Nz_global], the quantities in the order
 * of dfb_config.rows, Ny after the trim, for the whole plane (a slab handle uses its own columns; every plane of a batch the same table).
 * The epilogue's constants of each cell are derived on the host with the row path's expressions (b = R11 < 1e-10 ? 0 : R21 / sqrt(R11),
 * sqrt(R22 - b^2), -0.2 Ms^2 / Us, ...), so a cell whose eight values equal a row's gets that row's constants bit for bit.  After the
 * z-sweep each step rescales u', v', w' and T', rho' from filt_old with them (T', rho' stay untouched on the constructor's step and
 * dfb_first_step, quirk 3).  filt_old, the noise and the step counter do not depend on the profiles: a handle whose profiles equal its
 * rows delivers its own fields bit for bit.  N2 sums are then accumulated after the rescale; the flux correction uses g, sqrt(R11) and
 * the mean flux per cell.  The constructor's step is taken before any call, with the rows; on a handle created with skip_first_step,
 * dfb_first_step uses the profiles.
 * dfb_set_profiles(h, NULL) returns to the row tables.  Takes effect from the next step.  Refused, leaving the handle as it was: a value
 * that is not finite, or whose constant is not (R11 < 0, R22 < b^2, Us = 0, ...), naming the quantity, row and column (DFB_ERR_ARG);
 * with the flux correction on, profiles that make its D zero (DFB_ERR_ARG); an attached handle, a handle with a communicator
 * (dfb_comm_init, which refuses a handle with profiles in turn) or an outstanding dfb_filter_to_host_begin / dfb_gather_begin
 * (DFB_ERR_STATE).  dfb_info 19 tells whether profiles are in use, dfb_get_table 16 returns them.  The row tables (dfb_get_table 0..7),
 * the writers and dfb_time_scales_from_lengths keep using the rows.  A restart file saved with profiles loads only into a handle with
 * the same profiles; one saved without them only into a handle without. */
int dfb_set_profiles(dfb_handle h, const double* cells);
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

/* Restart files -- resume a generator across the jobs of a long run, bit for bit, whatever the decomposition on either side.
 * A file holds the plane's GLOBAL layout (filt_old [3][P][Ny][Nz_global] and, on request, the N2 sums [P][6][Ny][Nz_global] and the
 * correlation statistics), the step counter, and a fingerprint of the filter tables (half-widths, row tables, Lt, Ny, Nz, periodic_z).
 * Noise is keyed by (seed, step, global index), so the continued run equals the uninterrupted one bit for bit when it runs the same
 * kernel forms (dfb_info 3, 7, 10); a file written under other forms (DFB_Y_MODE, kernel_variant) is accepted and the continuation
 * then agrees to rounding.  Not saved: the outputs of the last step (u', v', w', T', rho', a gathered plane) -- the first dfb_filter
 * after a load produces step s+1 exactly as the uninterrupted run would.
 *
 * dfb_save_restart writes this handle's planes and columns (DFB_RESTART_STATE is always included).  Several writers may share one
 * file: the spanwise slabs of one plane or of one batch (one rank each, or several handles of one process).  Each opens the file without
 * truncating it and, under an open-file-description lock on the header, clears the writer records if they belong to another step (or
 * another plane range, geometry or set of sections), writes the header and sizes the file; then writes its rows; then adds its writer
 * record {plane range, k_begin, k_end, step, fingerprint} under the lock (at most 64 per file).  The file is complete when every
 * writer's call has returned: the caller's barrier (MPI_Barrier, a join) orders the saves before any load.  Saves are synchronous.
 *   DFB_RESTART_STATS without dfb_stats_enable ever called, DFB_RESTART_CORR without dfb_corr_enable: DFB_ERR_STATE.
 *   DFB_RESTART_CORR on a slab handle: DFB_ERR_ARG (correlation statistics are whole-plane only).
 *   A save while a dfb_filter_to_host_begin or dfb_gather_begin is outstanding: DFB_ERR_STATE.
 * dfb_load_restart restores any handle whose planes [plane_id, plane_id + nplanes) lie in the file's plane range and whose Ny, Nz,
 * periodic_z and filter tables match (and, in generate mode, its seed); it reads only its own columns, so a file written by 8 slabs
 * loads into 4, a batch file into single planes or smaller batches, slabs into a whole plane.  It checks everything before it touches
 * the device: a refused load leaves the handle as it was.  filt_old and the step go through dfb_set_state's path; with
 * DFB_RESTART_STATS the N2 sums, count and on/off state (the sums are allocated if needed); with DFB_RESTART_CORR (whole-plane handles)
 * the lags, sums, pair counts, the temporal ring and on/off state, so that the next steps add what the uninterrupted run would add.
 *   A mismatch (seed, geometry, filter tables, planes outside the file, a section the file lacks): DFB_ERR_ARG, naming it.
 *   A missing, short or foreign file, another format version, writer records that do not cover the handle's columns or carry another
 *   step or fingerprint: DFB_ERR_IO, naming the column range.
 * dfb_restart_info reads a file's header (no handle, no device) into out[0 .. min(cap, 30)):
 *   0 format version, 1 Ny, 2 Nz_global, 3 first plane id, 4 planes, 5 seed (bits), 6 periodic_z, 7 noise_mode, 8 step counter,
 *   9 sections (DFB_RESTART_* bits), 10 writer records, 11 fingerprint (bits), 12-14 Ny_max u v w, 15-17 Nz_max u v w,
 *   18-20 the last writer's dfb_info 3, 7, 10, 21 N2 count, 22 N2 on, 23-25 correlation lags z y t, 26 correlation count,
 *   27 correlation on, 28 ring fields saved, 29 file size in bytes. */
enum { DFB_RESTART_STATE = 1, DFB_RESTART_STATS = 2, DFB_RESTART_CORR = 4 };
int dfb_save_restart(dfb_handle h, const char* path, int what);
int dfb_load_restart(dfb_handle h, const char* path, int what);
int dfb_restart_info(const char* path, int64_t* out, int cap);

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

/* Face maps -- interpolate the outputs onto a CFD code's own inflow faces, on the device, all five fields in one pass.
 * A map is built once from the plane's global geometry: per face a fixed list of (plane cell, weight) taps.
 *   DFB_MAP_POINT  bilinear at the face centre (yf, zf) between the cell centres dfb_write_csv prints (at most 4 taps).  Beyond the
 *                  last centre z wraps with periodic_z (column Nz-1 with column 0) and clamps to the edge column without it; y clamps
 *                  to the top row above it and to the first row below csv_yc[0] -- with DFB_MAP_WALL_ZERO it goes linearly to 0 at the
 *                  wall vert_y[0] (dfb_get_table 12) instead and is 0 below it (no-slip fluctuations).  Needs increasing yc.
 *   DFB_MAP_AREA   the average over the face rectangle [yf -+ hy/2] x [zf -+ hz/2] of the cells [vert_y[j], vert_y[j+1]) x
 *                  [vert_z[k], vert_z[k+1]) (the cells dfb_face_map uses), weight = overlap area / face area, for finite-volume ghost
 *                  cells.  A part of a face outside the plane counts toward the nearest edge cell (wraps in z with periodic_z).  The
 *                  weights sum to 1; a face equal to a cell is that cell.
 * Serving: face i is served by the handle whose columns [own_begin, own_end) (0,0: its slab) contain the column of the cell holding the
 * face centre (dfb_face_map's clamped rule); every other face is not served (dfb_facemap_served).  A served face whose taps need a
 * column the handle does not compute (a bilinear tap across a slab cut, a wide area face) fails the creation with DFB_ERR_ARG naming
 * the face and the columns.  Remedy: create each slab 16 columns wider on each side (k_begin - 16, k_end + 16, within the plane) and
 * pass the unwidened columns as own_begin, own_end.  Slabs cut on multiples of 16 compute the whole plane's bits, so the overlap columns
 * hold the same values on both ranks and the faces of all ranks together are exactly the whole-plane result, with no communication.
 * (On a periodic plane, faces within half a cell of the seam -- bilinear between columns Nz-1 and 0 -- need a whole-plane handle.)
 * Errors: DFB_ERR_ARG for a bad kind, flag, mask, plane or map id, NULL arrays where n > 0, a non-finite coordinate, an extent <= 0
 * in an AREA map or extents given for a POINT map; DFB_ERR_STATE while a dfb_filter_to_host_begin or dfb_gather_begin is outstanding.
 * Maps are geometry only: they stay valid across dfb_set_state and dfb_load_restart, are not saved, and launch nothing per step.
 * dfb_destroy frees the maps still alive. */
enum { DFB_MAP_POINT = 0, DFB_MAP_AREA = 1 };
enum { DFB_MAP_WALL_ZERO = 1 };
int dfb_facemap_create(dfb_handle h, int kind, int n, const double* yf, const double* zf,
                       const double* hy, const double* hz,      /* face extents, AREA only (NULL for POINT) */
                       int own_begin, int own_end, int flags, int* map_id);
int dfb_facemap_served(dfb_handle h, int map_id, int* served /* [n] 0/1, host */);
int dfb_facemap_destroy(dfb_handle h, int map_id);
/* dst_f[dst_index[i] * stride] = mean_f[i] (dst's own value when mean or mean[f] is NULL) + scale_f * sum_t w_t * field_f[cell_t]
 * for every served face i and every field f in `fields` (bit 1 << DFB_U_FLUC .. 1 << DFB_RHO_FLUC) of plane `plane` of the handle.
 * Taps are summed in the map's fixed order (no atomics, no reduction across threads): a result depends on neither the launch, the
 * slab nor the batch.  dst_index, mean[f] ([n]) and dst[f] are DEVICE arrays; dst_index NULL means face i -> i; scale NULL means 1;
 * stride >= 1 lets dst be an array-of-structs state vector q(nvar, ncell) (dst[f] = &q(f, 0)).  Entries of unserved faces are not read
 * or written.  Enqueued on the handle's stream after the last enqueued step, like dfb_scatter_to_cells. */
int dfb_interp_to_cells(dfb_handle h, int map_id, int plane, int fields, const int* dst_index, const double* const mean[5],
                        const double scale[5], double* const dst[5], int stride);
/* The plain interpolated fluctuations of the served faces into host out[nfields][n] (the fields of the mask in increasing order):
 * sampled into a device staging buffer, then only those doubles cross PCIe.  Synchronous.  Entries of unserved faces are untouched. */
int dfb_interp_to_host(dfb_handle h, int map_id, int plane, int fields, double* out);

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
/* stream and dt_dev by reference: Fortran type(c_ptr) arguments (the stream as a cudaStream_t, dt_dev = the device address of dt) */
int dfb_attach_stream_f(const dfb_handle* h, void* const* stream);
int dfb_filter_dev_f(const dfb_handle* h, const double* const* dt_dev);
/* Lt_rows by reference as a Fortran type(c_ptr) (c_loc of a [Ny,3] array); c_null_ptr clears the rows */
int dfb_set_time_scales_f(const dfb_handle* h, const double* const* Lt_rows);
int dfb_time_scales_from_lengths_f(const dfb_handle* h, const double* Ix, const double* u_min, double* Lt_rows);
int dfb_set_filter_shape_f(const dfb_handle* h, const int* shape);
int dfb_set_flux_correction_f(const dfb_handle* h, const int* mode);
int dfb_set_profiles_f(const dfb_handle* h, const double* const* cells);
int dfb_flux_info_f(const dfb_handle* h, const int* plane, double* out);
/* path: Fortran character variable (c_loc) + its len_trim, as the file names of dfb_config (path_len < 0: NUL-terminated) */
int dfb_save_restart_f(const dfb_handle* h, const char* path, const int* path_len, const int* what);
int dfb_load_restart_f(const dfb_handle* h, const char* path, const int* path_len, const int* what);
/* face maps: hy, hz by address (NULL for a POINT map); mean, dst: five addresses (type(c_ptr) mean(5), dst(5)), mean may be NULL */
int dfb_facemap_create_f(const dfb_handle* h, const int* kind, const int* n, const double* yf, const double* zf, const double* hy,
                         const double* hz, const int* own_begin, const int* own_end, const int* flags, int* map_id);
int dfb_facemap_served_f(const dfb_handle* h, const int* map_id, int* served);
int dfb_facemap_destroy_f(const dfb_handle* h, const int* map_id);
int dfb_interp_to_host_f(const dfb_handle* h, const int* map_id, const int* plane, const int* fields, double* out);
int dfb_interp_to_cells_f(const dfb_handle* h, const int* map_id, const int* plane, const int* fields, const int* dst_index,
                          const double* const mean[5], const double scale[5], double* const dst[5], const int* stride);

#ifdef __cplusplus
}
#endif
#endif /* DFB200_H */
