! fortran/us3d_inflow_interp_example.f90 -- us3d_inflow_example.f90 with face maps: each rank receives only its own faces' values,
! interpolated onto the face centres (or averaged over the faces) on the GPU, instead of copying the five whole fields to the host
! every step.  NEVER COMPILED (needs the proprietary US3D modules, and there is no Fortran compiler in the image); it documents the
! call shape.
module inflow_df_interp_plugin
    use DIGITAL_FILTERING
    implicit none
    type(digital_filter_type), save :: df
    integer, save :: map_id
    integer, allocatable, save :: ghost(:), served(:)
    real(8), allocatable, save :: fluc(:, :)               ! (nface, 5): u', v', w', T', rho' at this rank's faces
contains
    subroutine my_user_init(rank, world, nface, yface, zface, hface, wface, ife)
        integer, intent(in) :: rank, world, nface, ife(:, :)
        real(8), intent(in) :: yface(nface), zface(nface)  ! centres of this rank's inflow faces in the plane's coordinates
        real(8), intent(in) :: hface(nface), wface(nface)  ! their heights and widths (finite-volume ghost cells: area-weighted)
        type(DFConfig) :: config
        integer :: f, k0, k1
        config%d_i = 0.0013d0; config%rho_e = 0.044d0; config%U_e = 869.1d0; config%mu_e = 7.1212d-6
        config%vel_fluc_file = '../files/RST.dat'
        config%line_file = '../line.dat'
        ! this rank serves the faces of the columns [k0, k1) (cut on multiples of 16) and filters 16 more columns on each side, so
        ! that a face near a cut finds every cell it overlaps; the overlap columns are bit for bit the neighbours' columns
        k0 = 16 * ((25 * rank) / world)
        k1 = 16 * ((25 * (rank + 1)) / world)
        config%k_begin = max(0, k0 - 16)
        config%k_end = min(400, k1 + 16)
        df = create_digital_filter(config)
        allocate(ghost(nface), served(nface), fluc(nface, 5))
        call facemap_create(df, nface, yface, zface, map_id, hy=hface, hz=wface, own_begin=k0, own_end=k1, served=served)
        do f = 1, nface
            ghost(f) = ife(f, 2)                           ! us3d_user.f90:92
        end do
    end subroutine my_user_init

    subroutine my_user_main_pre(dt, nface, u, v, w, t, r, umean, vmean, wmean, tmean, rmean)
        real(8), intent(in) :: dt
        integer, intent(in) :: nface
        real(8), intent(inout) :: u(:), v(:), w(:), t(:), r(:)
        real(8), intent(in) :: umean(:), vmean(:), wmean(:), tmean(:), rmean(:)
        integer :: i
        call filter_on_device(df, dt)                      ! no whole-plane copy
        call interp_to_host(df, map_id, 31, fluc)          ! 5 x nface doubles cross PCIe
        do i = 1, nface
            if (served(i) == 0) cycle
            u(ghost(i)) = umean(i) + fluc(i, 1)
            v(ghost(i)) = vmean(i) + fluc(i, 2)
            w(ghost(i)) = wmean(i) + fluc(i, 3)
            t(ghost(i)) = tmean(i) + fluc(i, 4)
            r(ghost(i)) = rmean(i) + fluc(i, 5)
        end do
    end subroutine my_user_main_pre
end module inflow_df_interp_plugin
