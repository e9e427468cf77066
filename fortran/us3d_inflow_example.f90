! fortran/us3d_inflow_example.f90 -- where a US3D-style plugin calls the generator (model: the
! reference's us3d_user.f90:21-48 my_user_init, 51-130 my_user_main_pre, 184-201 user_initialize).
! NEVER COMPILED (needs the proprietary US3D modules, and there is no Fortran compiler in the image); it documents the call shape.
module inflow_df_plugin
    use DIGITAL_FILTERING
    implicit none
    type(digital_filter_type), save :: df
    integer, allocatable, save :: cell(:), ghost(:)        ! inflow face -> cell of the filter plane / ghost cell of the CFD grid
    character(len=*), parameter :: restart_file = 'inflow_df.restart'   ! one file for all ranks: each saves / loads its own slab
contains
    subroutine my_user_init(rank, world, id, nface, yface, zface, ife)   ! once, like us3d_user.f90:21-48
        integer, intent(in) :: rank, world, nface, ife(:, :)
        character(kind=c_char), intent(inout) :: id(128)   ! NCCL id: rank 0 fills it (comm_unique_id), MPI_Bcast before this call
        real(8), intent(in) :: yface(nface), zface(nface)  ! centres of this rank's inflow faces in the plane's coordinates
        type(DFConfig) :: config
        integer :: f
        logical :: have_restart
        config%d_i = 0.0013d0; config%rho_e = 0.044d0; config%U_e = 869.1d0; config%mu_e = 7.1212d-6
        config%vel_fluc_file = '../files/RST.dat'
        config%line_file = '../line.dat'
        ! one plane shared by the ranks: each rank filters the spanwise slab that holds its faces (no halo exchange:
        ! the noise is keyed by the global cell index), e.g. equal slabs of the 400 columns
        config%k_begin = (400 * rank) / world
        config%k_end = (400 * (rank + 1)) / world
        df = create_digital_filter(config)
        ! a job of a restarted run resumes the inflow where the last checkpoint left it (the file holds the whole plane, so the
        ! previous job may have run on another number of ranks); the first job starts from the constructor's step
        inquire(file=restart_file, exist=have_restart)
        if (have_restart) call load_restart(df, restart_file)
        call comm_init(df, id, rank, world)                ! only needed if some rank wants the WHOLE plane (gather_begin / gather_end)
        allocate(cell(nface), ghost(nface))
        call face_map(df, nface, yface, zface, cell)       ! "provide the current rank", us3d_user.f90:87-89
        do f = 1, nface
            ghost(f) = ife(f, 2)                           ! us3d_user.f90:92
        end do
    end subroutine my_user_init

    subroutine my_user_main_pre(dt, nface, u, v, w, t, r, umean, vmean, wmean, tmean, rmean)
        ! per timestep, like us3d_user.f90:51-130: ghost cell ii = ife(j,2) gets mean + fluctuation (us3d_user.f90:106-114)
        real(8), intent(in) :: dt
        integer, intent(in) :: nface
        real(8), intent(inout) :: u(:), v(:), w(:), t(:), r(:)
        real(8), intent(in) :: umean(:), vmean(:), wmean(:), tmean(:), rmean(:)
        call filter(df, dt)
        call apply_inflow(nface, cell, ghost, umean, df%u%fluc, u)
        call apply_inflow(nface, cell, ghost, vmean, df%v%fluc, v)
        call apply_inflow(nface, cell, ghost, wmean, df%w%fluc, w)
        call apply_inflow(nface, cell, ghost, tmean, df%T_fluc, t)
        call apply_inflow(nface, cell, ghost, rmean, df%rho_fluc, r)
    end subroutine my_user_main_pre

    subroutine my_user_checkpoint()
        ! wherever the CFD code writes its own restart: every rank saves its slab into the one file; the code's barrier
        ! (MPI_Barrier) after the checkpoint is what makes the file complete before any later job reads it
        call save_restart(df, restart_file)
    end subroutine my_user_checkpoint
end module inflow_df_plugin
