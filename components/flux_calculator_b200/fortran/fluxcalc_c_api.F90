!> ISO_C_BINDING interfaces of libfluxcalc_b200.so (include/fluxcalc.h).
!! Source only: this image has no Fortran compiler, so the module is compile-untested here; it follows the
!! reference's own C-interop precedent (src/pyfort/call_python.f90:19-26, :32-35: bind(c, name=...) interfaces,
!! NUL-terminated character(c_char) strings, integer(c_int) status, "stop" on a non-zero status).
module fluxcalc_c_api
  use, intrinsic :: iso_c_binding
  implicit none
  public

  interface
    integer(c_int) function fc_create(ctx, grid_size, num_surface_types, device) bind(c, name='fc_create')
      import :: c_ptr, c_int, c_int64_t
      type(c_ptr), intent(out) :: ctx
      integer(c_int64_t), intent(in) :: grid_size(3)
      integer(c_int), value :: num_surface_types, device
    end function
    integer(c_int) function fc_destroy(ctx) bind(c, name='fc_destroy')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
    end function
    function fc_last_error(ctx) bind(c, name='fc_last_error') result(msg)
      import :: c_ptr
      type(c_ptr), value :: ctx
      type(c_ptr) :: msg
    end function
    integer(c_int) function fc_bind_field(ctx, surface_type, grid, var_idx, p, n) bind(c, name='fc_bind_field')
      import :: c_ptr, c_int, c_int64_t
      type(c_ptr), value :: ctx
      integer(c_int), value :: surface_type, grid, var_idx
      type(c_ptr), value :: p                       ! c_loc(local_field(i,g)%var(idx)%field)
      integer(c_int64_t), value :: n
    end function
    integer(c_int) function fc_set_method(ctx, which, surface_type, method) bind(c, name='fc_set_method')
      import :: c_ptr, c_int, c_char
      type(c_ptr), value :: ctx
      character(kind=c_char), intent(in) :: which(*), method(*)
      integer(c_int), value :: surface_type
    end function
    integer(c_int) function fc_set_distribute_shortwave(ctx, on) bind(c, name='fc_set_distribute_shortwave')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
      integer(c_int), value :: on
    end function
    integer(c_int) function fc_set_corrections(ctx, which, corr, n, enabled, init_date) bind(c, name='fc_set_corrections')
      import :: c_ptr, c_int, c_int64_t
      type(c_ptr), value :: ctx
      integer(c_int), value :: which, enabled, init_date
      type(c_ptr), value :: corr                    ! c_loc(corrections) : corrections(1,12,n), Fortran order
      integer(c_int64_t), value :: n
    end function
    integer(c_int) function fc_add_output_field(ctx, surface_type, grid, var_idx) bind(c, name='fc_add_output_field')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
      integer(c_int), value :: surface_type, grid, var_idx
    end function
    integer(c_int) function fc_set_area(ctx, grid, area, n) bind(c, name='fc_set_area')
      import :: c_ptr, c_int, c_int64_t
      type(c_ptr), value :: ctx
      integer(c_int), value :: grid
      type(c_ptr), value :: area
      integer(c_int64_t), value :: n
    end function
    integer(c_int) function fc_set_time(ctx, current_step_time) bind(c, name='fc_set_time')
      import :: c_ptr, c_int, c_int64_t
      type(c_ptr), value :: ctx
      integer(c_int64_t), value :: current_step_time
    end function
    integer(c_int) function fc_prepare(ctx, strict) bind(c, name='fc_prepare')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
      integer(c_int), value :: strict
    end function
    integer(c_int) function fc_set_option(ctx, name, value) bind(c, name='fc_set_option')
      import :: c_ptr, c_int, c_char, c_int64_t
      type(c_ptr), value :: ctx
      character(kind=c_char), intent(in) :: name(*)
      integer(c_int64_t), value :: value
    end function
    ! ---- the nine calculators (flux_calculator_calculate.F90:25-385) ----
    integer(c_int) function fc_calc_spec_vapor_surface(ctx, which_grid) bind(c, name='fc_calc_spec_vapor_surface')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
      integer(c_int), value :: which_grid
    end function
    integer(c_int) function fc_calc_flux_mass_evap(ctx) bind(c, name='fc_calc_flux_mass_evap')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
    end function
    integer(c_int) function fc_calc_flux_heat_latent(ctx) bind(c, name='fc_calc_flux_heat_latent')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
    end function
    integer(c_int) function fc_calc_flux_heat_sensible(ctx) bind(c, name='fc_calc_flux_heat_sensible')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
    end function
    integer(c_int) function fc_calc_flux_momentum_east(ctx, which_grid) bind(c, name='fc_calc_flux_momentum_east')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
      integer(c_int), value :: which_grid
    end function
    integer(c_int) function fc_calc_flux_momentum_north(ctx, which_grid) bind(c, name='fc_calc_flux_momentum_north')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
      integer(c_int), value :: which_grid
    end function
    integer(c_int) function fc_calc_flux_radiation_blackbody(ctx) bind(c, name='fc_calc_flux_radiation_blackbody')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
    end function
    integer(c_int) function fc_distribute_shortwave_radiation_flux(ctx) bind(c, name='fc_distribute_shortwave_radiation_flux')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
    end function
    integer(c_int) function fc_average_across_surface_types(ctx, which_grid, var_idx) &
        bind(c, name='fc_average_across_surface_types')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
      integer(c_int), value :: which_grid, var_idx
    end function
    ! ---- fused phases of the time loop (flux_calculator.F90:902 / :972-991) ----
    integer(c_int) function fc_step_early(ctx, current_step_time) bind(c, name='fc_step_early')
      import :: c_ptr, c_int, c_int64_t
      type(c_ptr), value :: ctx
      integer(c_int64_t), value :: current_step_time
    end function
    integer(c_int) function fc_step_normal(ctx, current_step_time) bind(c, name='fc_step_normal')
      import :: c_ptr, c_int, c_int64_t
      type(c_ptr), value :: ctx
      integer(c_int64_t), value :: current_step_time
    end function
    integer(c_int) function fc_step_all(ctx, current_step_time) bind(c, name='fc_step_all')
      import :: c_ptr, c_int, c_int64_t
      type(c_ptr), value :: ctx
      integer(c_int64_t), value :: current_step_time
    end function
    integer(c_int) function fc_synchronize(ctx) bind(c, name='fc_synchronize')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
    end function
    integer(c_int) function fc_get_diagnostics(ctx, surface_type, grid, var_idx, out) bind(c, name='fc_get_diagnostics')
      import :: c_ptr, c_int, c_double
      type(c_ptr), value :: ctx
      integer(c_int), value :: surface_type, grid, var_idx
      real(c_double), intent(out) :: out(3)
    end function
    integer(c_int) function fc_get_diagnostics_history(ctx, surface_type, grid, var_idx, first_step, count, out) &
        bind(c, name='fc_get_diagnostics_history')
      import :: c_ptr, c_int, c_int64_t, c_double
      type(c_ptr), value :: ctx
      integer(c_int), value :: surface_type, grid, var_idx
      integer(c_int64_t), value :: first_step, count
      real(c_double), intent(out) :: out(3, *)      ! out(:, j + 1) = sum, min, max after step first_step + j
    end function
    integer(c_int) function fc_comm_get_unique_id(id) bind(c, name='fc_comm_get_unique_id')
      import :: c_int, c_char
      character(kind=c_char), intent(out) :: id(128)
    end function
    integer(c_int) function fc_comm_init(ctx, id, rank, nranks) bind(c, name='fc_comm_init')
      import :: c_ptr, c_int, c_char
      type(c_ptr), value :: ctx
      character(kind=c_char), intent(in) :: id(128)
      integer(c_int), value :: rank, nranks
    end function
    ! the reference's own configuration files ("next" rows 3-4): flux_calculator.nml and corrections/mass_evap-MM.nc
    integer(c_int) function fc_configure_from_namelist(ctx, nml_path, bottom_model) bind(c, name='fc_configure_from_namelist')
      import :: c_ptr, c_int, c_char
      type(c_ptr), value :: ctx
      character(kind=c_char), intent(in) :: nml_path(*)      ! NUL-terminated
      integer(c_int), value :: bottom_model
    end function
    integer(c_int) function fc_load_corrections(ctx, root_dir, grid_offset, reference_start_quirk) &
        bind(c, name='fc_load_corrections')
      import :: c_ptr, c_int, c_int64_t, c_char
      type(c_ptr), value :: ctx
      character(kind=c_char), intent(in) :: root_dir(*)      ! NUL-terminated; contains corrections/
      integer(c_int64_t), value :: grid_offset
      integer(c_int), value :: reference_start_quirk
    end function
    ! peer-memory exchange fused into the step (one process per GPU on one NVLink node): export the mailbox handle,
    ! MPI_Allgather the 64-byte handles, connect; afterwards every step posts its diagnostics to all ranks
    integer(c_int) function fc_comm_p2p_handle(ctx, handle) bind(c, name='fc_comm_p2p_handle')
      import :: c_ptr, c_int, c_char
      type(c_ptr), value :: ctx
      character(kind=c_char), intent(out) :: handle(64)
    end function
    integer(c_int) function fc_comm_p2p_connect(ctx, handles, rank, nranks) bind(c, name='fc_comm_p2p_connect')
      import :: c_ptr, c_int, c_char
      type(c_ptr), value :: ctx
      character(kind=c_char), intent(in) :: handles(*)     ! nranks x 64 bytes, rank order
      integer(c_int), value :: rank, nranks
    end function
    integer(c_int) function fc_allreduce_diagnostics(ctx) bind(c, name='fc_allreduce_diagnostics')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
    end function
    integer(c_int) function fc_current_month(init_date, seconds) bind(c, name='fc_current_month')
      import :: c_int, c_int64_t
      integer(c_int), value :: init_date
      integer(c_int64_t), value :: seconds
    end function
    integer(c_int) function fc_shard_range(n, rank, nranks, align, offset, size) bind(c, name='fc_shard_range')
      import :: c_int, c_int64_t
      integer(c_int64_t), value :: n, align
      integer(c_int), value :: rank, nranks
      integer(c_int64_t), intent(out) :: offset, size
    end function
    ! %allocated of a registry slot as the host has it (flux_calculator_basic.F90:88); -1 = infer from the aliasing
    integer(c_int) function fc_set_allocated(ctx, surface_type, grid, var_idx, allocated) bind(c, name='fc_set_allocated')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
      integer(c_int), value :: surface_type, grid, var_idx, allocated
    end function
    ! host-pointer mode: what does not have to cross PCIe every step (namelist constants val_*, flux_calculator.F90:444-449)
    integer(c_int) function fc_mark_static(ctx, surface_type, grid, var_idx, is_static) bind(c, name='fc_mark_static')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
      integer(c_int), value :: surface_type, grid, var_idx, is_static
    end function
    integer(c_int) function fc_mark_dirty(ctx, surface_type, grid, var_idx) bind(c, name='fc_mark_dirty')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
      integer(c_int), value :: surface_type, grid, var_idx
    end function
    integer(c_int) function fc_bind_thread_to_device_numa(device) bind(c, name='fc_bind_thread_to_device_numa')
      import :: c_int
      integer(c_int), value :: device
    end function
    ! nsteps consecutive coupling steps without host synchronisation (device-resident fields; CUDA graph per month)
    integer(c_int) function fc_run_steps(ctx, t0, timestep, nsteps) bind(c, name='fc_run_steps')
      import :: c_ptr, c_int, c_int64_t
      type(c_ptr), value :: ctx
      integer(c_int64_t), value :: t0, timestep
      integer(c_int), value :: nsteps
    end function
    ! do_regridding (flux_calculator_basic.F90:463-522): direction 0 = u->t, 1 = v->t, 2 = t->u, 3 = t->v; 1-based indices
    integer(c_int) function fc_set_regrid_matrix(ctx, direction, num_elements, src_index, dst_index, weight) &
        bind(c, name='fc_set_regrid_matrix')
      import :: c_ptr, c_int, c_int64_t
      type(c_ptr), value :: ctx
      integer(c_int), value :: direction
      integer(c_int64_t), value :: num_elements
      type(c_ptr), value :: src_index, dst_index, weight     ! c_loc(matrix%src_index%field) ... (integer(4), real(8))
    end function
    integer(c_int) function fc_regrid(ctx, direction, dst, src) bind(c, name='fc_regrid')
      import :: c_ptr, c_int
      type(c_ptr), value :: ctx
      integer(c_int), value :: direction
      type(c_ptr), value :: dst, src
    end function
    ! ---- Level 1: the 14 array routines are declared in the GENERATED module fluxcalc_level1_api
    !      (fluxcalc_level1_api.F90, written by gen_fortran_api.py from include/fluxcalc.h); MODULE flux_library with the
    !      reference's public names on top of them is flux_library_gpu.F90 ----
  end interface

contains

  !> same policy as call_python.f90:13-16 / prepare.F90:31-33: log and stop on a non-zero status
  subroutine fc_check(ctx, status, where)
    type(c_ptr), intent(in) :: ctx
    integer(c_int), intent(in) :: status
    character(len=*), intent(in) :: where
    character(kind=c_char), pointer :: msg(:)
    type(c_ptr) :: cmsg
    integer :: k
    if (status /= 0) then
      cmsg = fc_last_error(ctx)
      call c_f_pointer(cmsg, msg, [1024])
      k = 1
      do while (k < 1024 .and. msg(k) /= c_null_char)
        k = k + 1
      end do
      write (*,*) 'fluxcalc error ', status, ' in ', where, ': ', msg(1:k-1)
      stop -1
    end if
  end subroutine fc_check

end module fluxcalc_c_api
