module dang_gpu_mod
  ! ======================================================================================
  ! iso_c_binding shim between dang's Fortran host code and libdang_gpu.so
  ! (include/dang_gpu.h).  It replaces the BODIES of three call sites of the Gibbs loop and
  ! nothing else; dang_params / dang_data / dang_comps, the parameter file and all FITS /
  ! HEALPix I/O stay as they are:
  !
  !   call sample_cg_groups(dpar,ddata)            dang.f90:101  ->  sample_cg_groups_gpu
  !   call sample_spectral_parameters(dpar,ddata)  dang.f90:106  ->  sample_spectral_parameters_gpu
  !   call compute_chisq(self)  (write_stats_to_term, dang_data_mod.f90:537)
  !                                                              ->  compute_chisq_gpu
  !
  ! plus dang_gpu_init after initialize_cg_groups (dang.f90:73) and dang_gpu_finalize before
  ! mpi_finalize (dang.f90:127).  See INTEGRATION.md for the exact edits and link line.
  !
  ! NOTE: this image has no Fortran compiler, so this file is checked by review only; the
  ! same entry points are exercised through ctypes by dang_b200/engine.py and tests/.
  ! ======================================================================================
  use iso_c_binding
  use healpix_types
  use dang_util_mod
  use dang_param_mod
  use dang_bp_mod
  use dang_data_mod
  use dang_component_mod
  use dang_cg_mod
  implicit none

  private
  public :: dang_gpu_init, dang_gpu_finalize, dang_gpu_upload_ddata
  public :: sample_cg_groups_gpu, sample_spectral_parameters_gpu, compute_chisq_gpu, sample_calibrators_gpu
  public :: dang_gpu_download_components, dang_gpu_download_sky_model
  public :: posterior_begin_gpu, posterior_accumulate_gpu, posterior_get_gpu
  public :: posterior_begin_batched_gpu, posterior_ess_gpu
  public :: POST_AMPLITUDE, POST_INDICES, POST_CHI_MAP, POST_RESIDUAL, POST_TEMPLATE_AMPLITUDES

  type(c_ptr), save :: handle = c_null_ptr
  integer(i8b), save :: gpu_seed = 20260101_i8b   ! device Philox seed, advanced every draw

  ! enums of include/dang_gpu.h
  integer(c_int), parameter :: COMP_POWERLAW = 1, COMP_MBB = 2, COMP_FREEFREE = 3, COMP_LOGNORMAL = 4, COMP_CMB = 5, &
       COMP_TEMPLATE = 6, COMP_T_CMB = 7, COMP_MONOPOLE = 8, COMP_HI_FIT = 9
  integer(c_int), parameter :: LNL_CHISQ = 0, LNL_MARGINAL = 1, LNL_PRIOR = 2
  integer(c_int), parameter :: PRIOR_UNIFORM = 0, PRIOR_GAUSSIAN = 1, PRIOR_JEFFREYS = 2
  integer(c_int), parameter :: ML_OPTIMIZE = 0, ML_SAMPLE = 1
  integer(c_int), parameter :: POST_AMPLITUDE = 1, POST_INDICES = 2, POST_CHI_MAP = 4, POST_RESIDUAL = 8, &
       POST_TEMPLATE_AMPLITUDES = 16

  interface
     integer(c_int) function dang_gpu_create(device, nside, npix, nmaps, nbands, ncomp, pix_lo, pix_hi, h) &
          bind(C, name='dang_gpu_create')
       import :: c_int, c_int64_t, c_ptr
       integer(c_int), value :: device, nside, nmaps, nbands, ncomp
       integer(c_int64_t), value :: npix, pix_lo, pix_hi
       type(c_ptr) :: h
     end function dang_gpu_create
     integer(c_int) function dang_gpu_destroy(h) bind(C, name='dang_gpu_destroy')
       import :: c_int, c_ptr
       type(c_ptr), value :: h
     end function dang_gpu_destroy
     type(c_ptr) function dang_gpu_last_error(h) bind(C, name='dang_gpu_last_error')
       import :: c_ptr
       type(c_ptr), value :: h
     end function dang_gpu_last_error
     integer(c_int) function dang_gpu_set_band(h, band, nu_c, n_bp, nu0, tau0) bind(C, name='dang_gpu_set_band')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: band, n_bp
       real(c_double), value :: nu_c
       real(c_double), intent(in) :: nu0(*), tau0(*)
     end function dang_gpu_set_band
     integer(c_int) function dang_gpu_upload_maps(h, sig, rms, mask, gain, offset) bind(C, name='dang_gpu_upload_maps')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       real(c_double), intent(in) :: sig(*), rms(*), mask(*), gain(*), offset(*)
     end function dang_gpu_upload_maps
     integer(c_int) function dang_gpu_set_component(h, ic, ctype, label, nu_ref, cg_group, sample_amp, amp, idx) &
          bind(C, name='dang_gpu_set_component')
       import :: c_int, c_double, c_ptr, c_char
       type(c_ptr), value :: h
       integer(c_int), value :: ic, ctype, cg_group, sample_amp
       character(kind=c_char), intent(in) :: label(*)
       real(c_double), value :: nu_ref
       real(c_double), intent(in) :: amp(*), idx(*)
     end function dang_gpu_set_component
     integer(c_int) function dang_gpu_set_index(h, ic, nind, sample_index, index_mode, lnl_type, prior_type, &
          gauss, uni, step, sample_nside, pol_flags, nflag) bind(C, name='dang_gpu_set_index')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic, nind, sample_index, index_mode, lnl_type, prior_type, sample_nside, nflag
       real(c_double), intent(in) :: gauss(2), uni(2)
       real(c_double), value :: step
       integer(c_int), intent(in) :: pol_flags(*)
     end function dang_gpu_set_index
     integer(c_int) function dang_gpu_set_cg_group(h, cg_group, i_max, converge, pol_flags, nflag) &
          bind(C, name='dang_gpu_set_cg_group')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: cg_group, i_max, nflag
       real(c_double), value :: converge
       integer(c_int), intent(in) :: pol_flags(*)
     end function dang_gpu_set_cg_group
     integer(c_int) function dang_gpu_cg_solve(h, cg_group, flag_n, ml_mode, eta, seed, n_iter, delta) &
          bind(C, name='dang_gpu_cg_solve')
       import :: c_int, c_double, c_ptr, c_int64_t
       type(c_ptr), value :: h, eta           ! eta = c_null_ptr: device RNG
       integer(c_int), value :: cg_group, flag_n, ml_mode
       integer(c_int64_t), value :: seed
       integer(c_int) :: n_iter
       real(c_double) :: delta
     end function dang_gpu_cg_solve
     integer(c_int) function dang_gpu_sample_index(h, ic, nind, map_n, nsample, ml_mode, z, u, seed, accept) &
          bind(C, name='dang_gpu_sample_index')
       import :: c_int, c_double, c_ptr, c_int64_t
       type(c_ptr), value :: h, z, u          ! c_null_ptr: device RNG
       integer(c_int), value :: ic, nind, map_n, nsample, ml_mode
       integer(c_int64_t), value :: seed
       real(c_double) :: accept
     end function dang_gpu_sample_index
     integer(c_int) function dang_gpu_chisq(h, pol_lo, pol_hi, planes, n_unmasked) bind(C, name='dang_gpu_chisq')
       import :: c_int, c_double, c_ptr, c_int64_t
       type(c_ptr), value :: h
       integer(c_int), value :: pol_lo, pol_hi
       real(c_double) :: planes(*)
       integer(c_int64_t) :: n_unmasked
     end function dang_gpu_chisq
     integer(c_int) function dang_gpu_get_amplitude(h, ic, amp) bind(C, name='dang_gpu_get_amplitude')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic
       real(c_double) :: amp(*)
     end function dang_gpu_get_amplitude
     integer(c_int) function dang_gpu_get_indices(h, ic, idx) bind(C, name='dang_gpu_get_indices')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic
       real(c_double) :: idx(*)
     end function dang_gpu_get_indices
     integer(c_int) function dang_gpu_get_sky_model(h, pol_lo, pol_hi, sky, res, chi) bind(C, name='dang_gpu_get_sky_model')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: pol_lo, pol_hi
       real(c_double) :: sky(*), res(*), chi(*)
     end function dang_gpu_get_sky_model
     integer(c_int) function dang_gpu_fit_band_gain(h, map_n, band, ml_mode, z, seed, gain) &
          bind(C, name='dang_gpu_fit_band_gain')
       import :: c_int, c_double, c_ptr, c_int64_t
       type(c_ptr), value :: h, z             ! z = c_null_ptr: device RNG
       integer(c_int), value :: map_n, band, ml_mode
       integer(c_int64_t), value :: seed
       real(c_double) :: gain
     end function dang_gpu_fit_band_gain
     integer(c_int) function dang_gpu_index_mean(h, ic, nind, map_n, mean) bind(C, name='dang_gpu_index_mean')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic, nind, map_n
       real(c_double) :: mean
     end function dang_gpu_index_mean
     integer(c_int) function dang_gpu_set_option(h, option, value) bind(C, name='dang_gpu_set_option')
       import :: c_int, c_double, c_ptr          ! option ids: the DANG_OPT_* enum of include/dang_gpu.h
       type(c_ptr), value :: h
       integer(c_int), value :: option
       real(c_double), value :: value
     end function dang_gpu_set_option
     integer(c_int) function dang_gpu_set_template(h, ic, template, template_amplitudes, corr, nfit) &
          bind(C, name='dang_gpu_set_template')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic, nfit
       real(c_double) :: template(*), template_amplitudes(*)   ! (0:npix-1,nmaps), (nbands,nmaps)
       integer(c_int) :: corr(*)
     end function dang_gpu_set_template
     integer(c_int) function dang_gpu_get_template_amplitudes(h, ic, template_amplitudes) &
          bind(C, name='dang_gpu_get_template_amplitudes')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic
       real(c_double) :: template_amplitudes(*)
     end function dang_gpu_get_template_amplitudes
     integer(c_int) function dang_gpu_get_index_fullsky(h, ic, nind, map_n, value) &
          bind(C, name='dang_gpu_get_index_fullsky')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic, nind, map_n
       real(c_double) :: value
     end function dang_gpu_get_index_fullsky
     ! ---- multi-GPU (INTEGRATION.md section 3): one MPI rank per GPU
     integer(c_int) function dang_gpu_comm_unique_id(id) bind(C, name='dang_gpu_comm_unique_id')
       import :: c_int, c_char
       character(kind=c_char) :: id(128)
     end function dang_gpu_comm_unique_id
     integer(c_int) function dang_gpu_comm_init(h, nranks, rank, id) bind(C, name='dang_gpu_comm_init')
       import :: c_int, c_char, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: nranks, rank
       character(kind=c_char), intent(in) :: id(128)
     end function dang_gpu_comm_init
     integer(c_int) function dang_gpu_comm_ipc_handle(h, handle) bind(C, name='dang_gpu_comm_ipc_handle')
       import :: c_int, c_char, c_ptr
       type(c_ptr), value :: h
       character(kind=c_char) :: handle(64)
     end function dang_gpu_comm_ipc_handle
     integer(c_int) function dang_gpu_comm_open_peers(h, handles) bind(C, name='dang_gpu_comm_open_peers')
       import :: c_int, c_char, c_ptr
       type(c_ptr), value :: h
       character(kind=c_char), intent(in) :: handles(*)       ! nranks * 64 bytes, rank-major
     end function dang_gpu_comm_open_peers
     integer(c_int) function dang_gpu_comm_check(h) bind(C, name='dang_gpu_comm_check')
       import :: c_int, c_ptr
       type(c_ptr), value :: h
     end function dang_gpu_comm_check
     ! ---- staging (INTEGRATION.md section 4): copies on dedicated streams, host arrays page-locked
     integer(c_int) function dang_gpu_stage_eta(h, eta, nplanes) bind(C, name='dang_gpu_stage_eta')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       real(c_double), intent(in) :: eta(*)
       integer(c_int), value :: nplanes
     end function dang_gpu_stage_eta
     integer(c_int) function dang_gpu_get_amplitude_async(h, ic, k_lo, k_hi, amplitude) &
          bind(C, name='dang_gpu_get_amplitude_async')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic, k_lo, k_hi
       real(c_double) :: amplitude(*)
     end function dang_gpu_get_amplitude_async
     integer(c_int) function dang_gpu_get_indices_async(h, ic, nind, k_lo, k_hi, indices) &
          bind(C, name='dang_gpu_get_indices_async')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic, nind, k_lo, k_hi
       real(c_double) :: indices(*)
     end function dang_gpu_get_indices_async
     integer(c_int) function dang_gpu_download_wait(h) bind(C, name='dang_gpu_download_wait')
       import :: c_int, c_ptr
       type(c_ptr), value :: h
     end function dang_gpu_download_wait
     integer(c_int) function dang_gpu_host_alloc(ptr, bytes) bind(C, name='dang_gpu_host_alloc')
       import :: c_int, c_int64_t, c_ptr
       type(c_ptr) :: ptr                                     ! c_f_pointer it onto the allocatable's shape
       integer(c_int64_t), value :: bytes
     end function dang_gpu_host_alloc
     integer(c_int) function dang_gpu_host_free(ptr) bind(C, name='dang_gpu_host_free')
       import :: c_int, c_ptr
       type(c_ptr), value :: ptr
     end function dang_gpu_host_free
     integer(c_int) function dang_gpu_sync(h) bind(C, name='dang_gpu_sync')
       import :: c_int, c_ptr
       type(c_ptr), value :: h
     end function dang_gpu_sync
     ! ---- state pushed again by the host (swap_cg_maps, offsets / gains read from file, warm starts)
     integer(c_int) function dang_gpu_set_gain_offset(h, gain, offset) bind(C, name='dang_gpu_set_gain_offset')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       real(c_double), intent(in) :: gain(*), offset(*)
     end function dang_gpu_set_gain_offset
     integer(c_int) function dang_gpu_set_amplitude(h, ic, amplitude) bind(C, name='dang_gpu_set_amplitude')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic
       real(c_double), intent(in) :: amplitude(*)
     end function dang_gpu_set_amplitude
     integer(c_int) function dang_gpu_set_indices(h, ic, indices) bind(C, name='dang_gpu_set_indices')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic
       real(c_double), intent(in) :: indices(*)
     end function dang_gpu_set_indices
     ! ---- tune_spectral_parameter_length (dang_sample_mod.f90:623-717)
     integer(c_int) function dang_gpu_tune_index(h, ic, nind, map_n, nsample, ml_mode, z, u, seed, max_blocks, &
          blocks_run, step_size) bind(C, name='dang_gpu_tune_index')
       import :: c_int, c_double, c_ptr, c_int64_t
       type(c_ptr), value :: h, z, u                          ! z = u = c_null_ptr: device RNG
       integer(c_int), value :: ic, nind, map_n, nsample, ml_mode, max_blocks
       integer(c_int64_t), value :: seed
       integer(c_int) :: blocks_run
       real(c_double) :: step_size
     end function dang_gpu_tune_index
     ! ---- udgrade_ring / udgrade_rms / udgrade_mask (dang_util_mod.f90:341-376, dang_sample_mod.f90:204-217, 480)
     integer(c_int) function dang_gpu_udgrade(h, kind, data_in, nside_in, data_out, nside_out, nmaps, threshold) &
          bind(C, name='dang_gpu_udgrade')
       import :: c_ptr, c_int, c_double
       type(c_ptr),    value :: h
       integer(c_int), value :: kind, nside_in, nside_out, nmaps
       real(c_double), value :: threshold
       real(c_double), intent(in)  :: data_in(*)
       real(c_double), intent(out) :: data_out(*)
     end function dang_gpu_udgrade
     ! ---- global T_CMB after a 'T_cmb' draw (dang_sample_mod.f90:76-78)
     integer(c_int) function dang_gpu_set_t_cmb(h, t_cmb) bind(C, name='dang_gpu_set_t_cmb')
       import :: c_ptr, c_int, c_double
       type(c_ptr),    value :: h
       real(c_double), value :: t_cmb
     end function dang_gpu_set_t_cmb
     integer(c_int) function dang_gpu_get_step_size(h, ic, nind, step_size) bind(C, name='dang_gpu_get_step_size')
       import :: c_int, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: ic, nind
       real(c_double) :: step_size
     end function dang_gpu_get_step_size
     ! ---- samples of bp(band) the device sums over: 0 delta, n_bp table, else the verified Gauss rule's nodes
     integer(c_int) function dang_gpu_band_samples(h, band, n_samples) bind(C, name='dang_gpu_band_samples')
       import :: c_int, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: band
       integer(c_int) :: n_samples
     end function dang_gpu_band_samples
     ! ---- deferred scalars (DANG_OPT_DEFER_SCALARS = 18): the numbers of write_stats_to_term (dang.f90:100-104)
     !      one iteration late; a host that prints every iteration calls _mark at the end of iteration k and
     !      _scalars(ticket of k-1) right after it
     integer(c_int) function dang_gpu_iteration_mark(h, ticket) bind(C, name='dang_gpu_iteration_mark')
       import :: c_int, c_int64_t, c_ptr
       type(c_ptr), value :: h
       integer(c_int64_t) :: ticket
     end function dang_gpu_iteration_mark
     integer(c_int) function dang_gpu_iteration_scalars(h, ticket, n_iter, delta_final, chisq_after_amplitudes, accept, &
          index_value, chisq_after_index) bind(C, name='dang_gpu_iteration_scalars')
       import :: c_int, c_int64_t, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int64_t), value :: ticket
       integer(c_int) :: n_iter
       real(c_double) :: delta_final, accept, index_value
       real(c_double), intent(out) :: chisq_after_amplitudes(*), chisq_after_index(*)
     end function dang_gpu_iteration_scalars
     ! ---- posterior summaries on the device (not in the reference): running mean / M2 of the chain state, added by
     !      _accumulate after each iteration past burn-in; _get downloads mean and std where write_maps is due
     integer(c_int) function dang_gpu_posterior_begin(h, what, pol_lo, pol_hi) bind(C, name='dang_gpu_posterior_begin')
       import :: c_int, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: what, pol_lo, pol_hi
     end function dang_gpu_posterior_begin
     integer(c_int) function dang_gpu_posterior_accumulate(h) bind(C, name='dang_gpu_posterior_accumulate')
       import :: c_int, c_ptr
       type(c_ptr), value :: h
     end function dang_gpu_posterior_accumulate
     integer(c_int) function dang_gpu_posterior_get(h, kind, ic, nind, mean, stddev, n) bind(C, name='dang_gpu_posterior_get')
       import :: c_int, c_int64_t, c_double, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: kind, ic, nind
       real(c_double), intent(out) :: mean(*), stddev(*)
       integer(c_int64_t) :: n
     end function dang_gpu_posterior_get
     integer(c_int) function dang_gpu_posterior_end(h) bind(C, name='dang_gpu_posterior_end')
       import :: c_int, c_ptr
       type(c_ptr), value :: h
     end function dang_gpu_posterior_end
     integer(c_int) function dang_gpu_posterior_rhat(hs, m, kind, ic, nind, rhat) bind(C, name='dang_gpu_posterior_rhat')
       import :: c_int, c_double, c_ptr
       type(c_ptr), intent(in) :: hs(*)
       integer(c_int), value :: m, kind, ic, nind
       real(c_double), intent(out) :: rhat(*)
     end function dang_gpu_posterior_rhat
     ! batch means next to the moments (b = batch_len consecutive samples), for the effective sample size and the
     ! Monte Carlo standard error of the posterior mean
     integer(c_int) function dang_gpu_posterior_begin_batched(h, what, pol_lo, pol_hi, batch_len) &
          bind(C, name='dang_gpu_posterior_begin_batched')
       import :: c_int, c_ptr
       type(c_ptr), value :: h
       integer(c_int), value :: what, pol_lo, pol_hi, batch_len
     end function dang_gpu_posterior_begin_batched
     integer(c_int) function dang_gpu_posterior_ess(hs, m, kind, ic, nind, ess, mcse) bind(C, name='dang_gpu_posterior_ess')
       import :: c_int, c_double, c_ptr
       type(c_ptr), intent(in) :: hs(*)
       integer(c_int), value :: m, kind, ic, nind
       real(c_double), intent(out) :: ess(*), mcse(*)
     end function dang_gpu_posterior_ess
  end interface

contains

  subroutine gpu_check(rc, where)
    ! Fatal, like the reference's `write(*,*) ...; stop` (e.g. dang_cg_mod.f90:97-101)
    integer(c_int),   intent(in) :: rc
    character(len=*), intent(in) :: where
    character(kind=c_char), pointer :: msg(:)
    integer(i4b) :: n
    if (rc == 0) return
    call c_f_pointer(dang_gpu_last_error(handle), msg, [1024])
    n = 1
    do while (n < 1024 .and. msg(n) /= c_null_char)
       n = n + 1
    end do
    write(*,*) 'dang_gpu error in '//trim(where)//': ', msg(1:n-1)
    stop
  end subroutine gpu_check

  integer(c_int) function comp_type_enum(ctype)
    character(len=*), intent(in) :: ctype
    if (trim(ctype) == 'power-law') then
       comp_type_enum = COMP_POWERLAW
    else if (trim(ctype) == 'mbb') then
       comp_type_enum = COMP_MBB
    else if (trim(ctype) == 'freefree') then
       comp_type_enum = COMP_FREEFREE
    else if (trim(ctype) == 'lognormal') then
       comp_type_enum = COMP_LOGNORMAL
    else if (trim(ctype) == 'cmb') then
       comp_type_enum = COMP_CMB
    else if (trim(ctype) == 'template') then
       comp_type_enum = COMP_TEMPLATE
    else if (trim(ctype) == 'T_cmb') then
       comp_type_enum = COMP_T_CMB
    else if (trim(ctype) == 'monopole') then
       comp_type_enum = COMP_MONOPOLE
    else if (trim(ctype) == 'hi_fit') then
       comp_type_enum = COMP_HI_FIT
    else
       write(*,*) 'dang_gpu: component type '//trim(ctype)//' is not on the GPU path yet'
       stop
    end if
  end function comp_type_enum

  subroutine dang_gpu_init(dpar, ddata, device)
    ! After initialize_components / initialize_data_module / initialize_cg_groups (dang.f90:71-73)
    type(dang_params), intent(in) :: dpar
    type(dang_data),   intent(in) :: ddata
    integer(i4b), intent(in), optional :: device
    type(dang_comps), pointer :: c
    integer(i4b)   :: i, j, dev
    integer(c_int) :: lnl, prior
    real(dp)       :: dummy(1)

    dev = 0; if (present(device)) dev = device
    call gpu_check(dang_gpu_create(int(dev,c_int), int(nside,c_int), int(npix,c_int64_t), int(nmaps,c_int), &
         int(nbands,c_int), int(ncomp,c_int), 0_c_int64_t, int(npix,c_int64_t), handle), 'dang_gpu_create')

    do j = 1, nbands                         ! bp(:) as left by init_bp_mod (dang_bp_mod.f90:19-60)
       if (trim(bp(j)%id) == 'delta') then
          call gpu_check(dang_gpu_set_band(handle, int(j-1,c_int), bp(j)%nu_c, 0_c_int, dummy, dummy), 'set_band')
       else
          call gpu_check(dang_gpu_set_band(handle, int(j-1,c_int), bp(j)%nu_c, int(bp(j)%n,c_int), &
               bp(j)%nu0, bp(j)%tau0), 'set_band')
       end if
    end do

    call dang_gpu_upload_ddata(ddata)

    do i = 1, ncomp                          ! component_list (dang_component_mod.f90:12-65)
       c => component_list(i)%p
       if (trim(c%type) == 'template') then   ! dang_component_mod.f90:536-577: c%template is already / temp_norm
          call gpu_check(dang_gpu_set_component(handle, int(i-1,c_int), COMP_TEMPLATE, &
               trim(c%label)//c_null_char, c%nu_ref, int(c%cg_group,c_int), merge(1_c_int,0_c_int,c%sample_amplitude), &
               dummy, dummy), 'set_component')   ! (amplitude / indices are ignored for this type)
          call gpu_check(dang_gpu_set_template(handle, int(i-1,c_int), c%template, c%template_amplitudes, &
               merge(1_c_int,0_c_int,c%corr), int(c%nfit,c_int)), 'set_template')
          cycle
       end if
       if (trim(c%type) == 'monopole') then   ! dang_component_mod.f90:579-597: the library builds the (1,0,0) map itself
          call gpu_check(dang_gpu_set_component(handle, int(i-1,c_int), COMP_MONOPOLE, &
               trim(c%label)//c_null_char, c%nu_ref, int(c%cg_group,c_int), merge(1_c_int,0_c_int,c%sample_amplitude), &
               dummy, dummy), 'set_component')
          call gpu_check(dang_gpu_set_template(handle, int(i-1,c_int), c%template, c%template_amplitudes, &
               merge(1_c_int,0_c_int,c%corr), int(c%nfit,c_int)), 'set_template')
          cycle
       end if
       call gpu_check(dang_gpu_set_component(handle, int(i-1,c_int), comp_type_enum(c%type), &
            trim(c%label)//c_null_char, c%nu_ref, int(c%cg_group,c_int), merge(1_c_int,0_c_int,c%sample_amplitude), &
            c%amplitude, c%indices), 'set_component')
       if (trim(c%type) == 'hi_fit') then      ! dang_component_mod.f90:599-700: template + per-band amplitudes + T_d map
          call gpu_check(dang_gpu_set_template(handle, int(i-1,c_int), c%template, c%template_amplitudes, &
               merge(1_c_int,0_c_int,c%corr), int(c%nfit,c_int)), 'set_template')
       end if
       do j = 1, c%nindices
          lnl = LNL_CHISQ
          if (trim(c%lnl_type(j)) == 'marginal') lnl = LNL_MARGINAL
          if (trim(c%lnl_type(j)) == 'prior')    lnl = LNL_PRIOR
          prior = PRIOR_UNIFORM
          if (trim(c%prior_type(j)) == 'gaussian') prior = PRIOR_GAUSSIAN
          if (trim(c%prior_type(j)) == 'jeffreys') prior = PRIOR_JEFFREYS
          call gpu_check(dang_gpu_set_index(handle, int(i-1,c_int), int(j-1,c_int), &
               merge(1_c_int,0_c_int,c%sample_index(j)), int(c%index_mode(j),c_int), lnl, prior, &
               c%gauss_prior(j,:), c%uni_prior(j,:), c%step_size(j), int(c%sample_nside(j),c_int), &
               int(c%pol_flag(j,1:c%nflag(j)),c_int), int(c%nflag(j),c_int)), 'set_index')
       end do
    end do

    do i = 1, ncg_groups                     ! cg_groups (dang_cg_mod.f90:57-120)
       call gpu_check(dang_gpu_set_cg_group(handle, int(cg_groups(i)%p%cg_group,c_int), &
            int(cg_groups(i)%p%i_max,c_int), cg_groups(i)%p%converge, &
            int(cg_groups(i)%p%pol_flag,c_int), int(cg_groups(i)%p%nflag,c_int)), 'set_cg_group')
    end do
  end subroutine dang_gpu_init

  subroutine dang_gpu_upload_ddata(ddata)
    ! sig_map / rms_map / masks(:,1) / gain / offset; call again after swap_cg_maps (dang.f90:92-97)
    type(dang_data), intent(in) :: ddata
    call gpu_check(dang_gpu_upload_maps(handle, ddata%sig_map, ddata%rms_map, ddata%masks(:,1), &
         ddata%gain, ddata%offset), 'upload_maps')
  end subroutine dang_gpu_upload_ddata

  subroutine dang_gpu_finalize()
    if (c_associated(handle)) call gpu_check(dang_gpu_destroy(handle), 'destroy')
    handle = c_null_ptr
  end subroutine dang_gpu_finalize

  subroutine sample_cg_groups_gpu(dpar, ddata)
    ! Drop-in for sample_cg_groups (dang_cg_mod.f90:142-177)
    type(dang_params) :: dpar
    type(dang_data)   :: ddata
    integer(i4b)      :: i, f
    integer(c_int)    :: n_iter, mode
    real(c_double)    :: delta

    mode = ML_OPTIMIZE; if (trim(dpar%ml_mode) == 'sample') mode = ML_SAMPLE
    do i = 1, ncg_groups
       if (cg_groups(i)%p%sample) then
          write(*,fmt='(a,i4)') "Computing a CG search of CG group ", i
          do f = 1, cg_groups(i)%p%nflag
             gpu_seed = gpu_seed + 1
             call gpu_check(dang_gpu_cg_solve(handle, int(cg_groups(i)%p%cg_group,c_int), int(f-1,c_int), mode, &
                  c_null_ptr, int(gpu_seed,c_int64_t), n_iter, delta), 'cg_solve')
             write(*,fmt='(a,i4,a,e12.5)') 'Final CG Iter: ', n_iter, ' | delta: ', delta
          end do
          call compute_chisq_gpu(ddata)
          call write_stats_gpu(ddata, iter)
       end if
    end do
  end subroutine sample_cg_groups_gpu

  subroutine sample_spectral_parameters_gpu(dpar, ddata)
    ! Drop-in for sample_spectral_parameters (dang_sample_mod.f90:21-86)
    type(dang_params) :: dpar
    type(dang_data)   :: ddata
    type(dang_comps), pointer :: c
    integer(i4b)   :: i, j, k, map_n
    integer(c_int) :: mode, blocks_run
    real(c_double) :: accept, step
    logical(lgt)   :: sampled

    mode = ML_OPTIMIZE; if (trim(ml_mode) == 'sample') mode = ML_SAMPLE
    sampled = .false.
    do i = 1, ncomp
       c => component_list(i)%p
       if (c%nindices == 0) cycle
       if (.not. any(c%sample_index)) cycle
       sampled = .true.
       do j = 1, c%nindices
          if (.not. c%sample_index(j)) cycle
          do k = 1, c%nflag(j)
             if (iand(c%pol_flag(j,k),1) .ne. 0) then
                map_n = 1
             else if (iand(c%pol_flag(j,k),2) .ne. 0) then
                map_n = 2
             else if (iand(c%pol_flag(j,k),4) .ne. 0) then
                map_n = 3
             else if (iand(c%pol_flag(j,k),8) .ne. 0) then
                map_n = -1
             else
                write(*,*) "There is something wrong with the poltype flag"
                cycle
             end if
             ! sample_index_mh tunes the step first whenever .not. c%tuned(j) (tuned = .not. fg_spec_tune,
             ! dang_sample_mod.f90:270-273 full-sky, :341-347 per-pixel with the mean index as the start) and the
             ! tuner sets ALL of c%tuned (:711); the tuned step comes back into c%step_size(j)
             if (.not. c%tuned(j) .and. trim(c%lnl_type(j)) /= 'prior') then
                write(*,*) 'Tuning!'
                gpu_seed = gpu_seed + 1
                call gpu_check(dang_gpu_tune_index(handle, int(i-1,c_int), int(j-1,c_int), int(map_n,c_int), &
                     int(nsample,c_int), mode, c_null_ptr, c_null_ptr, int(gpu_seed,c_int64_t), 1000_c_int, &
                     blocks_run, step), 'tune_index')
                c%step_size(j) = step
                c%tuned        = .true.
             end if
             gpu_seed = gpu_seed + 1
             call gpu_check(dang_gpu_sample_index(handle, int(i-1,c_int), int(j-1,c_int), int(map_n,c_int), &
                  int(nsample,c_int), mode, c_null_ptr, c_null_ptr, int(gpu_seed,c_int64_t), accept), 'sample_index')
          end do
       end do
       if (trim(c%type) == 'T_cmb') then       ! dang_sample_mod.f90:76-78: update the global variable T_CMB
          call dang_gpu_download_fullsky_index(c, i, 1, 1)
          T_CMB = c%indices(0,1,1)
          call gpu_check(dang_gpu_set_t_cmb(handle, T_CMB), 'set_t_cmb')
       end if
    end do
    if (sampled) then
       call compute_chisq_gpu(ddata)
       call write_stats_gpu(ddata, iter)
    end if
  end subroutine sample_spectral_parameters_gpu

  subroutine sample_calibrators_gpu(ddata)
    ! Drop-in for sample_calibrators / fit_band_gain (dang_sample_mod.f90:487-518, 570-621)
    type(dang_data), intent(inout) :: ddata
    integer(i4b)   :: j
    integer(c_int) :: mode
    real(c_double) :: gain
    logical(lgt)   :: sampled
    mode = ML_OPTIMIZE; if (trim(ml_mode) == 'sample') mode = ML_SAMPLE
    sampled = any(ddata%fit_gain(:))
    if (sampled) write(*,*) "Sampling band calibrators"
    do j = 1, nbands
       if (ddata%fit_gain(j)) then
          gpu_seed = gpu_seed + 1
          call gpu_check(dang_gpu_fit_band_gain(handle, 1_c_int, int(j-1,c_int), mode, c_null_ptr, &
               int(gpu_seed,c_int64_t), gain), 'fit_band_gain')
          ddata%gain(j) = gain
       end if
    end do
    if (sampled) then
       call compute_chisq_gpu(ddata)
       call write_stats_gpu(ddata, iter)
    end if
  end subroutine sample_calibrators_gpu

  subroutine compute_chisq_gpu(ddata)
    ! Drop-in for update_sky_model + compute_chisq (dang_data_mod.f90:339-396,494-526).
    ! The device returns the un-normalised per-plane sums; nump stays the host's (SURVEY Q9).
    type(dang_data), intent(inout) :: ddata
    real(c_double)     :: planes(3)
    integer(c_int64_t) :: n_unmasked
    integer(i4b)       :: k
    call gpu_check(dang_gpu_chisq(handle, int(ddata%pol_type(1),c_int), &
         int(ddata%pol_type(size(ddata%pol_type)),c_int), planes, n_unmasked), 'chisq')
    ddata%chisq = 0.d0
    do k = 1, nmaps
       ddata%chisq = ddata%chisq + planes(k)
    end do
    ddata%chisq = ddata%chisq/nump
  end subroutine compute_chisq_gpu

  subroutine write_stats_gpu(ddata, iter)
    ! The prints of write_stats_to_term (dang_data_mod.f90:528-570) from device-side reductions
    type(dang_data), intent(in) :: ddata
    integer(i4b),    intent(in) :: iter
    type(dang_comps), pointer   :: c
    integer(i4b)   :: i, j, k, map_n
    real(c_double) :: mean
    write(*,fmt='(a)') '---------------------------------------------'
    write(*,fmt='(i6,a,E16.5)') iter, " - Chisq: ", ddata%chisq
    do i = 1, ncomp
       c => component_list(i)%p
       do j = 1, c%nindices
          if (.not. c%sample_index(j)) cycle
          do k = 1, c%nflag(j)
             map_n = 1
             if (iand(c%pol_flag(j,k),2) .ne. 0 .or. iand(c%pol_flag(j,k),8) .ne. 0) map_n = 2
             if (iand(c%pol_flag(j,k),4) .ne. 0) map_n = 3
             call gpu_check(dang_gpu_index_mean(handle, int(i-1,c_int), int(j-1,c_int), int(map_n,c_int), mean), &
                  'index_mean')
             write(*,fmt='(a,a,a,a,a,f12.5)') '     ', trim(c%label), ' ', trim(c%ind_label(j)), ' mean:   ', mean
          end do
       end do
    end do
    write(*,fmt='(a)') '---------------------------------------------'
  end subroutine write_stats_gpu

  subroutine dang_gpu_download_components()
    ! c%amplitude / c%indices <- device; call before write_data / write_maps need them
    ! (dang.f90:116-121) and before anything else on the host reads the component maps.
    type(dang_comps), pointer :: c
    integer(i4b) :: i
    do i = 1, ncomp
       c => component_list(i)%p
       if (trim(c%type) == 'template') then   ! unpack_amplitudes :1374-1392 left them in the handle
          call gpu_check(dang_gpu_get_template_amplitudes(handle, int(i-1,c_int), c%template_amplitudes), &
               'get_template_amplitudes')
          cycle
       end if
       call gpu_check(dang_gpu_get_amplitude(handle, int(i-1,c_int), c%amplitude), 'get_amplitude')
       if (c%nindices > 0) call gpu_check(dang_gpu_get_indices(handle, int(i-1,c_int), c%indices), 'get_indices')
    end do
  end subroutine dang_gpu_download_components

  subroutine dang_gpu_download_fullsky_index(c, ic, nind, map_n)
    ! After a full-sky draw the whole plane holds one value (dang_sample_mod.f90:329,483): fetch the
    ! 8 bytes and do the reference's own assignment on the host instead of downloading the map.
    type(dang_comps), pointer, intent(inout) :: c
    integer(i4b),              intent(in)    :: ic, nind, map_n
    real(c_double) :: value
    integer(i4b)   :: k
    if (map_n == -1) then
       do k = 2, 3
          call gpu_check(dang_gpu_get_index_fullsky(handle, int(ic-1,c_int), int(nind-1,c_int), int(k,c_int), value), &
               'get_index_fullsky')
          c%indices(:,k,nind) = value
       end do
    else
       call gpu_check(dang_gpu_get_index_fullsky(handle, int(ic-1,c_int), int(nind-1,c_int), int(map_n,c_int), value), &
            'get_index_fullsky')
       c%indices(:,map_n,nind) = value
    end if
  end subroutine dang_gpu_download_fullsky_index

  subroutine dang_gpu_download_sky_model(ddata)
    ! sky_model / res_map / chi_map <- device, only when write_maps is due (dang.f90:119-121)
    type(dang_data), intent(inout) :: ddata
    call gpu_check(dang_gpu_get_sky_model(handle, int(ddata%pol_type(1),c_int), &
         int(ddata%pol_type(size(ddata%pol_type)),c_int), ddata%sky_model, ddata%res_map, ddata%chi_map), &
         'get_sky_model')
  end subroutine dang_gpu_download_sky_model

  subroutine posterior_begin_gpu(ddata, what)
    ! zero the running moments of the POST_* kinds in `what`; CHI_MAP / RESIDUAL over ddata%pol_type
    type(dang_data), intent(in) :: ddata
    integer(c_int),  intent(in) :: what
    call gpu_check(dang_gpu_posterior_begin(handle, what, int(ddata%pol_type(1),c_int), &
         int(ddata%pol_type(size(ddata%pol_type)),c_int)), 'posterior_begin')
  end subroutine posterior_begin_gpu

  subroutine posterior_accumulate_gpu()
    ! add the current state as one sample: stream ordered, no host wait
    call gpu_check(dang_gpu_posterior_accumulate(handle), 'posterior_accumulate')
  end subroutine posterior_accumulate_gpu

  subroutine posterior_get_gpu(kind, ic, nind, mean, stddev, n)
    ! mean / std of one kind, in the layout of the matching array (ic, nind: 1-based, as c%indices(:,:,nind))
    integer(c_int),     intent(in)  :: kind, ic, nind
    real(dp),           intent(out) :: mean(*), stddev(*)
    integer(c_int64_t), intent(out) :: n
    call gpu_check(dang_gpu_posterior_get(handle, kind, int(ic-1,c_int), int(nind-1,c_int), mean, stddev, n), &
         'posterior_get')
  end subroutine posterior_get_gpu

  subroutine posterior_begin_batched_gpu(ddata, what, batch_len)
    ! posterior_begin_gpu plus batch means of batch_len consecutive samples (about sqrt of the planned samples,
    ! at least 20 batches), which posterior_ess_gpu reads
    type(dang_data), intent(in) :: ddata
    integer(c_int),  intent(in) :: what, batch_len
    call gpu_check(dang_gpu_posterior_begin_batched(handle, what, int(ddata%pol_type(1),c_int), &
         int(ddata%pol_type(size(ddata%pol_type)),c_int), batch_len), 'posterior_begin_batched')
  end subroutine posterior_begin_batched_gpu

  subroutine posterior_ess_gpu(kind, ic, nind, ess, mcse)
    ! effective sample size and Monte Carlo standard error of the posterior mean of this chain, in the layout of
    ! posterior_get_gpu (ic, nind: 1-based)
    integer(c_int), intent(in)  :: kind, ic, nind
    real(dp),       intent(out) :: ess(*), mcse(*)
    type(c_ptr) :: hs(1)
    hs(1) = handle
    call gpu_check(dang_gpu_posterior_ess(hs, 1_c_int, kind, int(ic-1,c_int), int(nind-1,c_int), ess, mcse), &
         'posterior_ess')
  end subroutine posterior_ess_gpu

end module dang_gpu_mod
