! fortran/digital_filtering.f90 -- module DIGITAL_FILTERING over the B200 library (iso_c_binding).
!
! Drop-in for digital-filtering-fortran/df/df.f90: the same public names
!     public :: digital_filter_type, create_digital_filter, filter, DFConfig          (df.f90:6)
! so that a caller written like test/fortran-main.f90:8-26
!     type(digital_filter_type) :: df;  type(DFConfig) :: config
!     config%d_i = ...;  DF = create_digital_filter(config);  call filter(df, dt)
! compiles unchanged; results are read as DF%u%fluc(:), DF%v%fluc(:), DF%w%fluc(:), DF%T_fluc(:),
! DF%rho_fluc(:) in the reference's order idx = (j-1)*Nz + k (df.f90:608-610).
! Unlike the C++ reference, the Fortran one HONOURS DFConfig (df.f90:80-87): so does this module
! (honor_flow_config = 1).  The arithmetic follows the C++ code, which is normative for parity
! (SURVEY quirk 9).  Link with -ldfb200.
!
! Beyond the reference's surface (all optional):
!   create_digital_filter_batch / filter_batch   BASELINE config 5: P planes of one geometry behind one handle (one launch set per step)
!   config%k_begin / k_end, comm_unique_id, comm_init, gather_begin / gather_end / gathered_field
!                                                 BASELINE config 4: this rank's spanwise slab + the NCCL hand-off inside the library
!   config%periodic_z = 1                         spanwise-periodic plane: the z filter wraps around it
!   face_map, apply_inflow                        N3: inflow face -> plane cell, ghost cell = mean + fluctuation (us3d_user.f90:85-114)
!   corr_enable, corr_get, integral_scales        correlation statistics along z, y and in time (dfb_corr_*): the delivered scales
!   save_restart, load_restart                    restart files: resume a run across jobs, bit for bit, whatever the slab layout
!   facemap_create, interp_to_host,               the outputs interpolated onto the CFD code's own faces (bilinear or area-weighted),
!   interp_to_cells, filter_on_device               all five fields in one pass on the device; only the faces cross PCIe
!   attach_stream, filter_dev                     GPU-resident CFD codes: steps on the code's own CUDA stream with dt in device memory,
!                                                 capturable into its CUDA graph (include/dfb200.h, dfb_attach_stream)
!   set_time_scales, clear_time_scales,           per-row temporal scales Lt(y) for the temporal blend, e.g. from a prescribed
!   time_scales_from_lengths                        streamwise length: Lt = Ix(y) / U(y) (include/dfb200.h, dfb_set_time_scales)
!   config%filter_shape = FILTER_GAUSSIAN,        Klein et al.'s Gaussian filter kernel, which delivers the configured integral
!   set_filter_shape                                scales Iz / Iy (include/dfb200.h, dfb_set_filter_shape)
!   set_flux_correction, flux_info                each step's plane-integrated mass (or volume) flux of the inflow held at its mean
!                                                   (include/dfb200.h, dfb_set_flux_correction)
!   set_profiles, clear_profiles                  per-cell Reynolds stresses and mean state, for boundary layers that vary along the
!                                                   span (include/dfb200.h, dfb_set_profiles)
!
! NOTE: NEVER COMPILED -- no Fortran compiler exists in the build image or on the GPU boxes.  The binding is exercised through
! tests/fortran_abi_mimic.c, a C program that makes exactly these calls with exactly this struct layout and by-reference
! argument passing; tests/test_facades.py checks that the bind(C) type mirrors struct dfb_config field for field.
module DIGITAL_FILTERING
    use, intrinsic :: iso_c_binding
    implicit none
    private
    public :: digital_filter_type, create_digital_filter, filter, DFConfig, FilterField, destroy_digital_filter
    public :: digital_filter_batch_type, create_digital_filter_batch, filter_batch
    public :: comm_unique_id, comm_init, gather_begin, gather_end, gathered_field, face_map, apply_inflow
    public :: corr_enable, corr_get, integral_scales
    public :: save_restart, load_restart, RESTART_STATE, RESTART_STATS, RESTART_CORR
    public :: facemap_create, interp_to_host, interp_to_cells, facemap_destroy, MAP_POINT, MAP_AREA, MAP_WALL_ZERO, filter_on_device
    public :: attach_stream, filter_dev
    public :: set_time_scales, clear_time_scales, time_scales_from_lengths
    public :: set_filter_shape, FILTER_EXPONENTIAL, FILTER_GAUSSIAN
    public :: set_flux_correction, flux_info, FLUX_OFF, FLUX_MASS, FLUX_VOLUME
    public :: set_profiles, clear_profiles

    integer, parameter :: RESTART_STATE = 1, RESTART_STATS = 2, RESTART_CORR = 4   ! DFB_RESTART_* (what to save / load; added together)
    integer, parameter :: FILTER_EXPONENTIAL = 0, FILTER_GAUSSIAN = 1                ! DFB_FILTER_* (DFConfig%filter_shape)
    integer, parameter :: FLUX_OFF = 0, FLUX_MASS = 1, FLUX_VOLUME = 2               ! DFB_FLUX_* (set_flux_correction)

    integer, parameter :: dp = selected_real_kind(15)

    type :: FilterField                               ! df.f90:45-57 (the members a caller reads)
        real(kind=dp), allocatable :: fluc(:), filt(:)
        integer :: Ny_max = 0, Nz_max = 0
        real(kind=dp) :: Lt = 0.0_dp
    end type FilterField

    type :: DFConfig                                  ! df.f90:59-63
        real(kind=dp) :: d_i = 0.0_dp, rho_e = 0.0_dp, U_e = 0.0_dp, mu_e = 0.0_dp
        integer :: vel_file_offset = 0, vel_file_N_values = 0
        character(len=256) :: grid_file = ' ', vel_fluc_file = ' '
        ! extensions (not in the reference)
        character(len=256) :: line_file = ' '
        integer(c_int64_t) :: seed = 0_c_int64_t
        integer :: device = -1, plane_id = 0
        integer :: k_begin = 0, k_end = 0             ! this rank's spanwise slab [k_begin, k_end) (0-based, C convention); 0,0 = the whole plane
        integer :: periodic_z = 0                     ! 1: spanwise-periodic plane (the z filter wraps around it; needs Nz_max <= Nz)
        integer :: filter_shape = 0                   ! FILTER_EXPONENTIAL (the reference's) or FILTER_GAUSSIAN
    end type DFConfig

    type :: digital_filter_type
        type(c_ptr) :: handle = c_null_ptr
        integer :: Ny = 0, Nz = 0, n_cells = 0
        type(FilterField) :: u, v, w
        real(kind=dp), allocatable :: rho_fluc(:), T_fluc(:)
        real(kind=dp) :: dt = 0.0_dp
    end type digital_filter_type

    ! BASELINE config 5: nplanes independent planes of one geometry; arrays are (n_cells, nplanes), plane p uses stream group plane_id + p - 1
    type :: digital_filter_batch_type
        type(c_ptr) :: handle = c_null_ptr
        integer :: Ny = 0, Nz = 0, n_cells = 0, nplanes = 0
        real(kind=dp), allocatable :: u(:, :), v(:, :), w(:, :), T(:, :), rho(:, :)
    end type digital_filter_batch_type

    ! image of `struct dfb_config` (include/dfb200.h) -- keep the two in step
    ! face maps (include/dfb200.h, dfb_facemap_create); fields of interp_*: sum of 2**(0..4) for u', v', w', T', rho'
    integer, parameter :: MAP_POINT = 0, MAP_AREA = 1, MAP_WALL_ZERO = 1

    type, bind(C) :: dfb_config_c
        real(c_double) :: d_i, rho_e, U_e, mu_e
        integer(c_int) :: vel_file_offset, vel_file_N_values
        type(c_ptr) :: grid_file
        integer(c_int) :: grid_file_len
        type(c_ptr) :: vel_fluc_file
        integer(c_int) :: vel_fluc_file_len
        integer(c_int) :: struct_bytes, honor_flow_config
        type(c_ptr) :: line_file
        integer(c_int) :: line_file_len
        integer(c_int) :: Ny, Nz, geom_per_row
        type(c_ptr) :: yc, dy, dz, rows, scales, N_y, N_z
        integer(c_int64_t) :: seed
        integer(c_int) :: noise_mode, device, plane_id, k_begin, k_end, skip_first_step, kernel_variant
        integer(c_int) :: periodic_z
    end type dfb_config_c

    interface
        integer(c_int) function dfb_config_init(cfg) bind(C, name='dfb_config_init')
            import :: c_int, dfb_config_c
            type(dfb_config_c), intent(inout) :: cfg
        end function
        integer(c_int) function dfb_create_f(cfg, handle) bind(C, name='dfb_create_f')
            import :: c_int, c_ptr, dfb_config_c
            type(dfb_config_c), intent(in) :: cfg
            type(c_ptr), intent(out) :: handle
        end function
        integer(c_int) function dfb_dims_f(handle, Ny, Nz) bind(C, name='dfb_dims_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(out) :: Ny, Nz
        end function
        integer(c_int) function dfb_filter_to_host_f(handle, dt, u, v, w, T, rho) bind(C, name='dfb_filter_to_host_f')
            import :: c_int, c_ptr, c_double
            type(c_ptr), intent(in) :: handle
            real(c_double), intent(in) :: dt
            real(c_double), intent(inout) :: u(*), v(*), w(*), T(*), rho(*)
        end function
        integer(c_int) function dfb_get_field(handle, which, dst, on_device) bind(C, name='dfb_get_field')
            import :: c_int, c_ptr, c_double
            type(c_ptr), value :: handle
            integer(c_int), value :: which, on_device
            real(c_double), intent(inout) :: dst(*)
        end function
        integer(c_int) function dfb_create_batch_f(cfg, nplanes, handle) bind(C, name='dfb_create_batch_f')
            import :: c_int, c_ptr, dfb_config_c
            type(dfb_config_c), intent(in) :: cfg
            integer(c_int), intent(in) :: nplanes
            type(c_ptr), intent(out) :: handle
        end function
        integer(c_int) function dfb_host_register(ptr, bytes) bind(C, name='dfb_host_register')
            import :: c_int, c_ptr, c_size_t
            type(c_ptr), value :: ptr
            integer(c_size_t), value :: bytes
        end function
        integer(c_int) function dfb_comm_unique_id(id) bind(C, name='dfb_comm_unique_id')
            import :: c_int, c_char
            character(kind=c_char), intent(out) :: id(128)
        end function
        integer(c_int) function dfb_comm_init_f(handle, id, rank, world) bind(C, name='dfb_comm_init_f')
            import :: c_int, c_ptr, c_char
            type(c_ptr), intent(in) :: handle
            character(kind=c_char), intent(in) :: id(128)
            integer(c_int), intent(in) :: rank, world
        end function
        integer(c_int) function dfb_gather_begin_f(handle, dst_rank) bind(C, name='dfb_gather_begin_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(in) :: dst_rank
        end function
        integer(c_int) function dfb_gather_end_f(handle) bind(C, name='dfb_gather_end_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle
        end function
        integer(c_int) function dfb_gathered_to_host_f(handle, which, dst) bind(C, name='dfb_gathered_to_host_f')
            import :: c_int, c_ptr, c_double
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(in) :: which
            real(c_double), intent(inout) :: dst(*)
        end function
        integer(c_int) function dfb_face_map_f(handle, n, yf, zf, plane_index) bind(C, name='dfb_face_map_f')
            import :: c_int, c_ptr, c_double
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(in) :: n
            real(c_double), intent(in) :: yf(*), zf(*)
            integer(c_int), intent(inout) :: plane_index(*)
        end function
        integer(c_int) function dfb_destroy_f(handle) bind(C, name='dfb_destroy_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(inout) :: handle
        end function
        integer(c_int) function dfb_info(handle, what, field, out64) bind(C, name='dfb_info')
            import :: c_int, c_ptr, c_int64_t
            type(c_ptr), value :: handle
            integer(c_int), value :: what, field
            integer(c_int64_t), intent(out) :: out64
        end function
        integer(c_int) function dfb_corr_enable(handle, on, lags) bind(C, name='dfb_corr_enable')
            import :: c_int, c_ptr
            type(c_ptr), value :: handle
            integer(c_int), value :: on
            integer(c_int), intent(in) :: lags(3)
        end function
        integer(c_int) function dfb_corr_get(handle, field, dir, normalized, dst, pairs, count) bind(C, name='dfb_corr_get')
            import :: c_int, c_ptr, c_double
            type(c_ptr), value :: handle
            integer(c_int), value :: field, dir, normalized
            real(c_double), intent(inout) :: dst(*)
            type(c_ptr), value :: pairs, count
        end function
        integer(c_int) function dfb_corr_integral_scales(handle, plane, field, dir, dst) bind(C, name='dfb_corr_integral_scales')
            import :: c_int, c_ptr, c_double
            type(c_ptr), value :: handle
            integer(c_int), value :: plane, field, dir
            real(c_double), intent(inout) :: dst(*)
        end function
        integer(c_int) function dfb_save_restart_f(handle, path, path_len, what) bind(C, name='dfb_save_restart_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle
            type(c_ptr), value :: path
            integer(c_int), intent(in) :: path_len, what
        end function
        integer(c_int) function dfb_load_restart_f(handle, path, path_len, what) bind(C, name='dfb_load_restart_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle
            type(c_ptr), value :: path
            integer(c_int), intent(in) :: path_len, what
        end function
        integer(c_int) function dfb_filter_f(handle, dt) bind(C, name='dfb_filter_f')
            import :: c_int, c_ptr, c_double
            type(c_ptr), intent(in) :: handle
            real(c_double), intent(in) :: dt
        end function
        integer(c_int) function dfb_facemap_create_f(handle, kind, n, yf, zf, hy, hz, own_begin, own_end, flags, map_id) &
                bind(C, name='dfb_facemap_create_f')
            import :: c_int, c_ptr, c_double
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(in) :: kind, n, own_begin, own_end, flags
            real(c_double), intent(in) :: yf(*), zf(*)
            type(c_ptr), value :: hy, hz
            integer(c_int), intent(out) :: map_id
        end function
        integer(c_int) function dfb_facemap_destroy_f(handle, map_id) bind(C, name='dfb_facemap_destroy_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(in) :: map_id
        end function
        integer(c_int) function dfb_facemap_served_f(handle, map_id, served) bind(C, name='dfb_facemap_served_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(in) :: map_id
            integer(c_int), intent(inout) :: served(*)
        end function
        integer(c_int) function dfb_interp_to_host_f(handle, map_id, plane, fields, out) bind(C, name='dfb_interp_to_host_f')
            import :: c_int, c_ptr, c_double
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(in) :: map_id, plane, fields
            real(c_double), intent(inout) :: out(*)
        end function
        integer(c_int) function dfb_interp_to_cells_f(handle, map_id, plane, fields, dst_index, mean, scale, dst, stride) &
                bind(C, name='dfb_interp_to_cells_f')
            import :: c_int, c_ptr, c_double
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(in) :: map_id, plane, fields, stride
            type(c_ptr), value :: dst_index
            type(c_ptr), intent(in) :: mean(5), dst(5)
            real(c_double), intent(in) :: scale(5)
        end function
        integer(c_int) function dfb_attach_stream_f(handle, stream) bind(C, name='dfb_attach_stream_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle, stream
        end function
        integer(c_int) function dfb_filter_dev_f(handle, dt_dev) bind(C, name='dfb_filter_dev_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle, dt_dev
        end function
        integer(c_int) function dfb_set_time_scales_f(handle, Lt_rows) bind(C, name='dfb_set_time_scales_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle, Lt_rows
        end function
        integer(c_int) function dfb_set_filter_shape_f(handle, shape) bind(C, name='dfb_set_filter_shape_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(in) :: shape
        end function
        integer(c_int) function dfb_set_flux_correction_f(handle, mode) bind(C, name='dfb_set_flux_correction_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(in) :: mode
        end function
        integer(c_int) function dfb_set_profiles_f(handle, cells) bind(C, name='dfb_set_profiles_f')
            import :: c_int, c_ptr
            type(c_ptr), intent(in) :: handle, cells
        end function
        integer(c_int) function dfb_flux_info_f(handle, plane, out) bind(C, name='dfb_flux_info_f')
            import :: c_int, c_ptr, c_double
            type(c_ptr), intent(in) :: handle
            integer(c_int), intent(in) :: plane
            real(c_double), intent(out) :: out(3)
        end function
        integer(c_int) function dfb_first_step(handle) bind(C, name='dfb_first_step')
            import :: c_int, c_ptr
            type(c_ptr), value :: handle
        end function
        integer(c_int) function dfb_time_scales_from_lengths_f(handle, Ix, u_min, Lt_rows) bind(C, name='dfb_time_scales_from_lengths_f')
            import :: c_int, c_ptr, c_double
            type(c_ptr), intent(in) :: handle
            real(c_double), intent(in) :: Ix(6), u_min
            real(c_double), intent(out) :: Lt_rows(*)
        end function
        function dfb_last_error() bind(C, name='dfb_last_error') result(msg)
            import :: c_ptr
            type(c_ptr) :: msg
        end function
    end interface

contains

    subroutine check(rc, where)
        integer(c_int), intent(in) :: rc
        character(len=*), intent(in) :: where
        character(kind=c_char), pointer :: s(:)
        integer :: n
        if (rc == 0) return
        call c_f_pointer(dfb_last_error(), s, [512])
        n = 1
        do while (n < 512 .and. s(n) /= c_null_char)
            n = n + 1
        end do
        write(*, '(a,a,a,i0,a)', advance='no') 'DIGITAL_FILTERING: ', where, ' failed (', rc, '): '
        write(*, *) s(1:n-1)
        stop 1                                         ! the reference stops on I/O errors too (df.f90:327-330)
    end subroutine check

    subroutine fill_config(config, c)
        type(DFConfig), intent(in), target :: config
        type(dfb_config_c), intent(inout) :: c
        call check(dfb_config_init(c), 'dfb_config_init')
        c%d_i = config%d_i; c%rho_e = config%rho_e; c%U_e = config%U_e; c%mu_e = config%mu_e
        c%vel_file_offset = config%vel_file_offset; c%vel_file_N_values = config%vel_file_N_values
        c%honor_flow_config = 1
        c%grid_file = c_loc(config%grid_file);          c%grid_file_len = len_trim(config%grid_file)
        c%vel_fluc_file = c_loc(config%vel_fluc_file);  c%vel_fluc_file_len = len_trim(config%vel_fluc_file)
        c%line_file = c_loc(config%line_file);          c%line_file_len = len_trim(config%line_file)
        c%seed = config%seed; c%device = config%device; c%plane_id = config%plane_id
        c%k_begin = config%k_begin; c%k_end = config%k_end
        c%periodic_z = config%periodic_z
        if (config%filter_shape /= FILTER_EXPONENTIAL) c%skip_first_step = 1   ! shaped_start sets the shape, then takes the first step
    end subroutine fill_config

    ! a handle of another filter shape is created without its first step: set the shape, then take the constructor's step
    subroutine shaped_start(config, handle)
        type(DFConfig), intent(in) :: config
        type(c_ptr), intent(in) :: handle
        integer(c_int) :: shape
        if (config%filter_shape == FILTER_EXPONENTIAL) return
        shape = config%filter_shape
        call check(dfb_set_filter_shape_f(handle, shape), 'dfb_set_filter_shape')
        call check(dfb_first_step(handle), 'dfb_first_step')
    end subroutine shaped_start

    ! page-lock an array the library copies into every step (failure only costs speed)
    ! page-lock an array the library copies into every step (a failure only costs speed)
    subroutine pin(a, n)
        integer, intent(in) :: n
        real(kind=dp), intent(in), target :: a(n)
        integer(c_int) :: rc
        rc = dfb_host_register(c_loc(a), int(8, c_size_t) * int(n, c_size_t))
    end subroutine pin

    ! df.f90:74-138
    function create_digital_filter(config) result(DF)
        type(DFConfig), intent(in), target :: config
        type(digital_filter_type) :: DF
        type(dfb_config_c) :: c
        integer(c_int) :: Ny, Nz

        call fill_config(config, c)
        call check(dfb_create_f(c, DF%handle), 'create_digital_filter')
        call shaped_start(config, DF%handle)
        call check(dfb_dims_f(DF%handle, Ny, Nz), 'dfb_dims')
        DF%Ny = Ny; DF%Nz = Nz; DF%n_cells = Ny * Nz
        allocate(DF%u%fluc(DF%n_cells), DF%v%fluc(DF%n_cells), DF%w%fluc(DF%n_cells))
        allocate(DF%u%filt(DF%n_cells), DF%v%filt(DF%n_cells), DF%w%filt(DF%n_cells))
        allocate(DF%rho_fluc(DF%n_cells), DF%T_fluc(DF%n_cells))
        DF%rho_fluc = 0.0_dp; DF%T_fluc = 0.0_dp
        call pin(DF%u%fluc, DF%n_cells); call pin(DF%v%fluc, DF%n_cells); call pin(DF%w%fluc, DF%n_cells)     ! page-locked: filter()'s
        call pin(DF%T_fluc, DF%n_cells); call pin(DF%rho_fluc, DF%n_cells)                                     ! copies run at the PCIe rate
        ! fluctuations of the first step (df.f90:124-131)
        call check(dfb_get_field(DF%handle, 0_c_int, DF%u%fluc, 0_c_int), 'dfb_get_field')
        call check(dfb_get_field(DF%handle, 1_c_int, DF%v%fluc, 0_c_int), 'dfb_get_field')
        call check(dfb_get_field(DF%handle, 2_c_int, DF%w%fluc, 0_c_int), 'dfb_get_field')
    end function create_digital_filter

    ! df.f90:621-651.  dt_input must be finite and >= 0: otherwise the library returns DFB_ERR_ARG (check stops) and changes nothing.
    subroutine filter(DF, dt_input)
        type(digital_filter_type), intent(inout) :: DF
        real(kind=dp), intent(in) :: dt_input
        DF%dt = dt_input
        call check(dfb_filter_to_host_f(DF%handle, dt_input, DF%u%fluc, DF%v%fluc, DF%w%fluc, DF%T_fluc, DF%rho_fluc), 'filter')
    end subroutine filter

    ! ---- BASELINE config 5: nplanes planes of one geometry, one launch set per step for all of them ----
    function create_digital_filter_batch(config, nplanes) result(B)
        type(DFConfig), intent(in), target :: config
        integer, intent(in) :: nplanes
        type(digital_filter_batch_type) :: B
        type(dfb_config_c) :: c
        integer(c_int) :: Ny, Nz, np
        call fill_config(config, c)
        np = nplanes
        call check(dfb_create_batch_f(c, np, B%handle), 'create_digital_filter_batch')
        call shaped_start(config, B%handle)
        call check(dfb_dims_f(B%handle, Ny, Nz), 'dfb_dims')
        B%Ny = Ny; B%Nz = Nz; B%n_cells = Ny * Nz; B%nplanes = nplanes
        allocate(B%u(B%n_cells, nplanes), B%v(B%n_cells, nplanes), B%w(B%n_cells, nplanes), B%T(B%n_cells, nplanes), B%rho(B%n_cells, nplanes))
    end function create_digital_filter_batch

    subroutine filter_batch(B, dt_input)          ! every plane advances by dt_input; the fields of all planes land in B%u(:, p) ...
        type(digital_filter_batch_type), intent(inout) :: B
        real(kind=dp), intent(in) :: dt_input
        call check(dfb_filter_to_host_f(B%handle, dt_input, B%u, B%v, B%w, B%T, B%rho), 'filter_batch')
    end subroutine filter_batch

    ! ---- BASELINE config 4: the hand-off of the finished plane to the CFD rank (NCCL inside the library) ----
    subroutine comm_unique_id(id)                  ! rank 0; broadcast the 128 characters with MPI_Bcast
        character(kind=c_char), intent(out) :: id(128)
        call check(dfb_comm_unique_id(id), 'comm_unique_id')
    end subroutine comm_unique_id

    subroutine comm_init(DF, id, rank, world)      ! every rank (0-based rank, as MPI gives it)
        type(digital_filter_type), intent(inout) :: DF
        character(kind=c_char), intent(in) :: id(128)
        integer, intent(in) :: rank, world
        integer(c_int) :: r, w
        r = rank; w = world
        call check(dfb_comm_init_f(DF%handle, id, r, w), 'comm_init')
    end subroutine comm_init

    subroutine gather_begin(DF, dst_rank)          ! after filter(DF, dt); the next filter(DF, dt) may follow at once
        type(digital_filter_type), intent(inout) :: DF
        integer, intent(in) :: dst_rank
        integer(c_int) :: d
        d = dst_rank
        call check(dfb_gather_begin_f(DF%handle, d), 'gather_begin')
    end subroutine gather_begin

    subroutine gather_end(DF)
        type(digital_filter_type), intent(inout) :: DF
        call check(dfb_gather_end_f(DF%handle), 'gather_end')
    end subroutine gather_end

    subroutine gathered_field(DF, which, plane)    ! destination rank: which = 0..4 (u', v', w', T', rho'), plane(Ny * Nz_global)
        type(digital_filter_type), intent(inout) :: DF
        integer, intent(in) :: which
        real(kind=dp), intent(inout) :: plane(*)
        integer(c_int) :: wsel
        wsel = which
        call check(dfb_gathered_to_host_f(DF%handle, wsel, plane), 'gathered_field')
    end subroutine gathered_field

    ! ---- N3: inflow face -> plane cell, and the ghost-cell update of us3d_user.f90:85-114 ----
    subroutine face_map(DF, n, yf, zf, cell)       ! cell(i) = 1-based index into DF%u%fluc(:) of the cell holding face i, 0 = not in this rank's slab
        type(digital_filter_type), intent(in) :: DF
        integer, intent(in) :: n
        real(kind=dp), intent(in) :: yf(n), zf(n)
        integer, intent(out) :: cell(n)
        integer(c_int) :: nn
        nn = n
        call check(dfb_face_map_f(DF%handle, nn, yf, zf, cell), 'face_map')
        cell = cell + 1
    end subroutine face_map

    subroutine apply_inflow(n, cell, ghost, mean, fluc, q)    ! q(ghost(i)) = mean(i) + fluc(cell(i)): r(ii), u(ii), ... of us3d_user.f90:106-114
        integer, intent(in) :: n, cell(n), ghost(n)
        real(kind=dp), intent(in) :: mean(n), fluc(:)
        real(kind=dp), intent(inout) :: q(:)
        integer :: i
        do i = 1, n
            if (cell(i) > 0) q(ghost(i)) = mean(i) + fluc(cell(i))
        end do
    end subroutine apply_inflow

    ! ---- face maps: the outputs interpolated onto this rank's own faces (include/dfb200.h, dfb_facemap_create) ----
    subroutine filter_on_device(DF, dt_input)     ! filter(DF, dt) without the copy of the five fields to DF%u%fluc ... (face maps read them)
        type(digital_filter_type), intent(inout) :: DF
        real(kind=dp), intent(in) :: dt_input
        real(c_double) :: dt
        dt = dt_input
        call check(dfb_filter_f(DF%handle, dt), 'filter_on_device')
    end subroutine filter_on_device

    ! every later step, interp_to_cells and copy of DF goes on `stream` (a cudaStream_t, e.g. from CUDA Fortran or the CFD code's own
    ! C layer; c_null_ptr detaches), with the step's state in device memory, so that filter_dev can be captured into a CUDA graph
    subroutine attach_stream(DF, stream)
        type(digital_filter_type), intent(in) :: DF
        type(c_ptr), intent(in) :: stream
        call check(dfb_attach_stream_f(DF%handle, stream), 'attach_stream')
    end subroutine attach_stream

    ! one step with dt read from device memory (dt_dev: the device address of one real(c_double)) when it runs; DF must be attached
    subroutine filter_dev(DF, dt_dev)
        type(digital_filter_type), intent(in) :: DF
        type(c_ptr), intent(in) :: dt_dev
        call check(dfb_filter_dev_f(DF%handle, dt_dev), 'filter_dev')
    end subroutine filter_dev

    ! per-row time scales of the temporal blend from the next step on: Lt_rows(j, f), j = 1..Ny (after the trim), f = 1..3 (u, v, w),
    ! finite and > 0; set them before attach_stream and before load_restart of a file saved with them
    subroutine set_time_scales(DF, Lt_rows)
        type(digital_filter_type), intent(in) :: DF
        real(c_double), intent(in), target, contiguous :: Lt_rows(:, :)
        call check(dfb_set_time_scales_f(DF%handle, c_loc(Lt_rows)), 'set_time_scales')
    end subroutine set_time_scales

    ! FILTER_EXPONENTIAL or FILTER_GAUSSIAN on a handle that has not stepped (config%filter_shape does this in create_digital_filter)
    subroutine set_filter_shape(DF, shape)
        type(digital_filter_type), intent(in) :: DF
        integer, intent(in) :: shape
        integer(c_int) :: s
        s = shape
        call check(dfb_set_filter_shape_f(DF%handle, s), 'set_filter_shape')
    end subroutine set_filter_shape

    ! FLUX_OFF, FLUX_MASS or FLUX_VOLUME from the next step on (whole planes only; not while attached)
    subroutine set_flux_correction(DF, mode)
        type(digital_filter_type), intent(in) :: DF
        integer, intent(in) :: mode
        integer(c_int) :: m
        m = mode
        call check(dfb_set_flux_correction_f(DF%handle, m), 'set_flux_correction')
    end subroutine set_flux_correction

    ! out = (c, m', mean flux) of the last corrected step of the (0-based) plane
    subroutine flux_info(DF, plane, out)
        type(digital_filter_type), intent(in) :: DF
        integer, intent(in) :: plane
        real(c_double), intent(out) :: out(3)
        integer(c_int) :: p
        p = plane
        call check(dfb_flux_info_f(DF%handle, p, out), 'flux_info')
    end subroutine flux_info

    ! per-cell profiles from the next step on: cells(k, j, q), k = 1..Nz (the whole plane), j = 1..Ny (after the trim), q = 1..8 in the
    ! order R11, R21, R22, R33, Us, Ts, rhos, Ms of config%rows; set them before attach_stream and before load_restart of a file saved
    ! with them
    subroutine set_profiles(DF, cells)
        type(digital_filter_type), intent(in) :: DF
        real(c_double), intent(in), target, contiguous :: cells(:, :, :)
        call check(dfb_set_profiles_f(DF%handle, c_loc(cells)), 'set_profiles')
    end subroutine set_profiles

    ! back to the row tables
    subroutine clear_profiles(DF)
        type(digital_filter_type), intent(in) :: DF
        call check(dfb_set_profiles_f(DF%handle, c_null_ptr), 'clear_profiles')
    end subroutine clear_profiles

    ! back to the scalar Lt of the configuration
    subroutine clear_time_scales(DF)
        type(digital_filter_type), intent(in) :: DF
        call check(dfb_set_time_scales_f(DF%handle, c_null_ptr), 'clear_time_scales')
    end subroutine clear_time_scales

    ! Lt_rows(j, f) = Ix_f(y_j) / max(U(y_j), u_min): Ix = (inn_u, out_u, inn_v, out_v, inn_w, out_w) blended across the boundary layer
    ! like Iz; host only, sets nothing (pass the result to set_time_scales)
    subroutine time_scales_from_lengths(DF, Ix, u_min, Lt_rows)
        type(digital_filter_type), intent(in) :: DF
        real(c_double), intent(in) :: Ix(6), u_min
        real(c_double), intent(out) :: Lt_rows(:, :)
        call check(dfb_time_scales_from_lengths_f(DF%handle, Ix, u_min, Lt_rows), 'time_scales_from_lengths')
    end subroutine time_scales_from_lengths

    subroutine facemap_create(DF, n, yf, zf, map_id, hy, hz, own_begin, own_end, wall_zero, served)
        ! bilinear at the face centres, or with hy, hz the average over each face; own_begin/own_end: 0-based columns [own_begin,
        ! own_end) whose faces this rank serves (default: its slab); served(i) = 1 where it serves face i
        type(digital_filter_type), intent(in) :: DF
        integer, intent(in) :: n
        real(kind=dp), intent(in) :: yf(n), zf(n)
        integer, intent(out) :: map_id
        real(kind=dp), intent(in), target, optional :: hy(n), hz(n)
        integer, intent(in), optional :: own_begin, own_end
        logical, intent(in), optional :: wall_zero
        integer, intent(out), optional :: served(n)
        integer(c_int) :: nn, kind, o0, o1, flags, id
        type(c_ptr) :: phy, phz
        nn = n; kind = MAP_POINT; o0 = 0; o1 = 0; flags = 0
        phy = c_null_ptr; phz = c_null_ptr
        if (present(hy) .and. present(hz)) then
            kind = MAP_AREA; phy = c_loc(hy); phz = c_loc(hz)
        end if
        if (present(own_begin)) o0 = own_begin
        if (present(own_end)) o1 = own_end
        if (present(wall_zero)) then
            if (wall_zero) flags = MAP_WALL_ZERO
        end if
        call check(dfb_facemap_create_f(DF%handle, kind, nn, yf, zf, phy, phz, o0, o1, flags, id), 'facemap_create')
        map_id = id
        if (present(served)) call check(dfb_facemap_served_f(DF%handle, id, served), 'facemap_create')
    end subroutine facemap_create

    subroutine interp_to_host(DF, map_id, fields, out, plane)   ! out(n, nfields): the served faces' entries, fields in increasing order
        type(digital_filter_type), intent(in) :: DF
        integer, intent(in) :: map_id, fields
        real(kind=dp), intent(inout) :: out(:, :)
        integer, intent(in), optional :: plane
        integer(c_int) :: id, f, p
        id = map_id; f = fields; p = 0
        if (present(plane)) p = plane
        call check(dfb_interp_to_host_f(DF%handle, id, p, f, out), 'interp_to_host')
    end subroutine interp_to_host

    subroutine interp_to_cells(DF, map_id, fields, dst_index, mean, scale, dst, stride, plane)
        ! device arrays (CUDA Fortran / OpenACC host_data): dst(f)[dst_index(i) * stride] = mean(f)[i] (or dst's own value where
        ! mean(f) is c_null_ptr) + scale(f) * interpolated field f; 0-based dst_index, c_null_ptr for face i -> i
        type(digital_filter_type), intent(in) :: DF
        integer, intent(in) :: map_id, fields, stride
        type(c_ptr), intent(in) :: dst_index, mean(5), dst(5)
        real(kind=dp), intent(in) :: scale(5)
        integer, intent(in), optional :: plane
        integer(c_int) :: id, f, s, p
        id = map_id; f = fields; s = stride; p = 0
        if (present(plane)) p = plane
        call check(dfb_interp_to_cells_f(DF%handle, id, p, f, dst_index, mean, scale, dst, s), 'interp_to_cells')
    end subroutine interp_to_cells

    subroutine facemap_destroy(DF, map_id)
        type(digital_filter_type), intent(in) :: DF
        integer, intent(in) :: map_id
        integer(c_int) :: id
        id = map_id
        call check(dfb_facemap_destroy_f(DF%handle, id), 'facemap_destroy')
    end subroutine facemap_destroy

    ! ---- correlation statistics (like the rest of this module, never compiled: see the note at the top) ----
    subroutine corr_enable(DF, lz, ly, lt)         ! lags along z, y (0 = off, -1 = the filter's whole support) and t (0..64 steps)
        type(digital_filter_type), intent(inout) :: DF
        integer, intent(in) :: lz, ly, lt
        integer(c_int) :: lags(3)
        lags = [int(lz, c_int), int(ly, c_int), int(lt, c_int)]
        call check(dfb_corr_enable(DF%handle, 1_c_int, lags), 'corr_enable')
    end subroutine corr_enable

    subroutine corr_get(DF, field, dir, R)         ! R(0:L, Ny): correlation coefficients of field 0..2 (u', v', w'), dir 0 z, 1 y, 2 t
        type(digital_filter_type), intent(in) :: DF
        integer, intent(in) :: field, dir
        real(kind=dp), allocatable, intent(out) :: R(:, :)
        integer(c_int64_t) :: L
        call check(dfb_info(DF%handle, 14_c_int, int(dir, c_int), L), 'corr_get')
        allocate(R(0:L, DF%Ny))
        call check(dfb_corr_get(DF%handle, int(field, c_int), int(dir, c_int), 1_c_int, R, c_null_ptr, c_null_ptr), 'corr_get')
    end subroutine corr_get

    subroutine integral_scales(DF, field, dir, L)  ! L(Ny): per-row integral scale, metres for z and y, steps for t
        type(digital_filter_type), intent(in) :: DF
        integer, intent(in) :: field, dir
        real(kind=dp), intent(inout) :: L(:)
        call check(dfb_corr_integral_scales(DF%handle, 0_c_int, int(field, c_int), int(dir, c_int), L), 'integral_scales')
    end subroutine integral_scales

    ! ---- restart files (include/dfb200.h, dfb_save_restart): what = RESTART_STATE (default) [+ RESTART_STATS] [+ RESTART_CORR] ----
    subroutine save_restart(DF, path, what)         ! every rank of a slab job may save its slab into the same file; MPI_Barrier after
        type(digital_filter_type), intent(in) :: DF
        character(len=*), intent(in), target :: path
        integer, intent(in), optional :: what
        integer(c_int) :: w, n
        w = RESTART_STATE
        if (present(what)) w = what
        n = len_trim(path)
        call check(dfb_save_restart_f(DF%handle, c_loc(path), n, w), 'save_restart')
    end subroutine save_restart

    subroutine load_restart(DF, path, what)         ! after the writers' barrier; the next filter(DF, dt) continues the saved run
        type(digital_filter_type), intent(in) :: DF
        character(len=*), intent(in), target :: path
        integer, intent(in), optional :: what
        integer(c_int) :: w, n
        w = RESTART_STATE
        if (present(what)) w = what
        n = len_trim(path)
        call check(dfb_load_restart_f(DF%handle, c_loc(path), n, w), 'load_restart')
    end subroutine load_restart

    subroutine destroy_digital_filter(DF)
        type(digital_filter_type), intent(inout) :: DF
        integer(c_int) :: rc
        rc = dfb_destroy_f(DF%handle)
    end subroutine destroy_digital_filter

end module DIGITAL_FILTERING
