!=======================================================================
!  rfinv_b200_capi.f90 -- Fortran 2003 interface to librfinv_b200.so
!
!  UNTESTED SOURCE: no Fortran compiler exists in the build image (SURVEY.md F2).  It declares, with
!  iso_c_binding, the entry points of include/rfinv_b200.h that rf_inv.f90 / pt_mcmc.f90 / likelihood.f90
!  would call instead of calc_likelihood / mcmc / pt_control.  See INTEGRATION.md for the call sites.
!=======================================================================
module rfinv_b200_capi
  use iso_c_binding
  implicit none

  ! struct rfinv_config (field order and types must match include/rfinv_b200.h)
  type, bind(C) :: rfinv_config
     integer(c_int32_t) :: ntrc, nfft, nsmp, deconv_mode
     real(c_double)     :: delta, t_start, sdep
     type(c_ptr)        :: rayps, a_gus, ipha, obs, r_inv
     integer(c_int32_t) :: nref, pad0
     real(c_double)     :: z_ref_min, dz_ref
     type(c_ptr)        :: vp_ref, vs_ref
     integer(c_int32_t) :: vp_mode, k_min, k_max, prior_mode
     real(c_double)     :: z_min, z_max, h_min, dvs_prior, dvp_prior
     type(c_ptr)        :: sig_min, sig_max
     real(c_double)     :: vp_min, vp_max, vs_min, vs_max, vpvs_min, vpvs_max
     real(c_double)     :: dev_z, dev_dvs, dev_dvp, dev_sig
     integer(c_int32_t) :: nburn, niter, ncorr, nchains, ncool, iseed
     real(c_double)     :: t_high
     integer(c_int32_t) :: nbin_z, nbin_vs, nbin_vp, nbin_vpvs, nbin_sig, nbin_amp
     real(c_double)     :: amp_min, amp_max
     real(c_double)     :: bdep
  end type rfinv_config

  interface
     integer(c_int32_t) function rfinv_create(cfg, device, handle) bind(C, name="rfinv_create")
       import :: c_int32_t, c_ptr, rfinv_config
       type(rfinv_config), intent(in) :: cfg
       integer(c_int32_t), value :: device
       type(c_ptr), intent(out) :: handle
     end function rfinv_create

     subroutine rfinv_destroy(handle) bind(C, name="rfinv_destroy")
       import :: c_ptr
       type(c_ptr), value :: handle
     end subroutine rfinv_destroy

     ! calc_likelihood(fwd_flag=.true.) for C models; arrays exactly as the reference holds them:
     ! z(k_max-1, C), dvp(k_max, C), dvs(k_max, C), sig(ntrc, C), logl(C), rft(nfft, ntrc, C)
     integer(c_int32_t) function rfinv_eval_batch(handle, c, k, z, dvp, dvs, sig, logl, rft, is_valid) &
          & bind(C, name="rfinv_eval_batch")
       import :: c_int32_t, c_ptr, c_double
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: c
       integer(c_int32_t), intent(in) :: k(*)
       real(c_double), intent(in) :: z(*), dvp(*), dvs(*), sig(*)
       real(c_double), intent(out) :: logl(*)
       type(c_ptr), value :: rft        ! c_loc(rft) or c_null_ptr
       type(c_ptr), value :: is_valid   ! c_loc(int8 array) or c_null_ptr
     end function rfinv_eval_batch

     ! calc_likelihood with its per-call fwd_flag, batched (src/likelihood.f90:74-82): phi(ntrc, C) is written for the models
     ! with fwd_flag /= 0 and read (the cached values of the chain's current RF) for sigma-only proposals
     integer(c_int32_t) function rfinv_eval_batch_flags(handle, c, fwd_flag, k, z, dvp, dvs, sig, phi, logl, is_valid) &
          & bind(C, name="rfinv_eval_batch_flags")
       import :: c_int32_t, c_int8_t, c_ptr, c_double
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: c
       integer(c_int8_t), intent(in) :: fwd_flag(*)
       integer(c_int32_t), intent(in) :: k(*)
       real(c_double), intent(in) :: z(*), dvp(*), dvs(*), sig(*)
       real(c_double), intent(inout) :: phi(*)
       real(c_double), intent(out) :: logl(*)
       type(c_ptr), value :: is_valid
     end function rfinv_eval_batch_flags

     ! asynchronous pair: two groups of chains in flight, slot = 0 or 1 (arrays must stay untouched until _end returns)
     integer(c_int32_t) function rfinv_eval_batch_begin(handle, slot, c, k, z, dvp, dvs, sig, logl, is_valid) &
          & bind(C, name="rfinv_eval_batch_begin")
       import :: c_int32_t, c_ptr, c_double
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: slot, c
       integer(c_int32_t), intent(in) :: k(*)
       real(c_double), intent(in) :: z(*), dvp(*), dvs(*), sig(*)
       real(c_double), intent(out) :: logl(*)
       type(c_ptr), value :: is_valid
     end function rfinv_eval_batch_begin

     integer(c_int32_t) function rfinv_eval_batch_end(handle, slot) bind(C, name="rfinv_eval_batch_end")
       import :: c_int32_t, c_ptr
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: slot
     end function rfinv_eval_batch_end

     ! communicator of the distributed run: the id is created on one MPI rank and broadcast by the host, e.g.
     !   if (rank == 0) ierr = rfinv_comm_create_id(id);  call mpi_bcast(id, 128, MPI_BYTE, 0, MPI_COMM_WORLD, ierr)
     !   ierr = rfinv_comm_init(handle, id, nproc_gpu, rank)
     integer(c_int32_t) function rfinv_comm_id_bytes() bind(C, name="rfinv_comm_id_bytes")
       import :: c_int32_t
     end function rfinv_comm_id_bytes

     integer(c_int32_t) function rfinv_comm_create_id(id) bind(C, name="rfinv_comm_create_id")
       import :: c_int32_t, c_int8_t
       integer(c_int8_t), intent(out) :: id(*)
     end function rfinv_comm_create_id

     integer(c_int32_t) function rfinv_comm_init(handle, id, world, rank) bind(C, name="rfinv_comm_init")
       import :: c_int32_t, c_int8_t, c_ptr
       type(c_ptr), value :: handle
       integer(c_int8_t), intent(in) :: id(*)
       integer(c_int32_t), value :: world, rank
     end function rfinv_comm_init

     ! pt_control over all processes (in-library ncclAllGather per iteration), then output_results' reduces and gathers
     integer(c_int32_t) function rfinv_pt_run_distributed(handle, n_iter) bind(C, name="rfinv_pt_run_distributed")
       import :: c_int32_t, c_ptr
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: n_iter
     end function rfinv_pt_run_distributed

     integer(c_int32_t) function rfinv_pt_reduce_outputs(handle) bind(C, name="rfinv_pt_reduce_outputs")
       import :: c_int32_t, c_ptr
       type(c_ptr), value :: handle
     end function rfinv_pt_reduce_outputs

     ! 1: pair and swap tables stored straight into peer memory (NVLink) from a side branch of the iteration; 2: one ncclAllGather per iteration
     integer(c_int32_t) function rfinv_pt_exchange_mode(handle) bind(C, name="rfinv_pt_exchange_mode")
       import :: c_int32_t, c_ptr
       type(c_ptr), value :: handle
     end function rfinv_pt_exchange_mode

     integer(c_int32_t) function rfinv_pt_init(handle, nproc_total, rank_begin, rank_count) bind(C, name="rfinv_pt_init")
       import :: c_int32_t, c_ptr
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: nproc_total, rank_begin, rank_count
     end function rfinv_pt_init

     integer(c_int32_t) function rfinv_pt_run(handle, n_iter) bind(C, name="rfinv_pt_run")
       import :: c_int32_t, c_ptr
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: n_iter
     end function rfinv_pt_run

     integer(c_int32_t) function rfinv_pt_local_step(handle) bind(C, name="rfinv_pt_local_step")
       import :: c_int32_t, c_ptr
       type(c_ptr), value :: handle
     end function rfinv_pt_local_step

     integer(c_int32_t) function rfinv_pt_swap_table(handle, dev_ptr, n_doubles) bind(C, name="rfinv_pt_swap_table")
       import :: c_int32_t, c_int64_t, c_ptr
       type(c_ptr), value :: handle
       integer(c_int64_t), intent(out) :: dev_ptr
       integer(c_int32_t), intent(out) :: n_doubles
     end function rfinv_pt_swap_table

     integer(c_int32_t) function rfinv_pt_apply_swap(handle, gathered_dev_ptr, world) bind(C, name="rfinv_pt_apply_swap")
       import :: c_int32_t, c_int64_t, c_ptr
       type(c_ptr), value :: handle
       integer(c_int64_t), value :: gathered_dev_ptr
       integer(c_int32_t), value :: world
     end function rfinv_pt_apply_swap

     integer(c_int32_t) function rfinv_pt_get_state(handle, k, z, dvp, dvs, sig, logl, temps) bind(C, name="rfinv_pt_get_state")
       import :: c_int32_t, c_ptr, c_double
       type(c_ptr), value :: handle
       integer(c_int32_t), intent(out) :: k(*)
       real(c_double), intent(out) :: z(*), dvp(*), dvs(*), sig(*), logl(*), temps(*)
     end function rfinv_pt_get_state

     integer(c_int32_t) function rfinv_pt_get_counters(handle, nprop, naccept, likelihood_hist, n_hist, n_eval) &
          & bind(C, name="rfinv_pt_get_counters")
       import :: c_int32_t, c_int64_t, c_ptr, c_double
       type(c_ptr), value :: handle
       integer(c_int64_t), intent(out) :: nprop(*), naccept(*)
       real(c_double), intent(out) :: likelihood_hist(*)
       integer(c_int32_t), value :: n_hist
       integer(c_int64_t), intent(out) :: n_eval
     end function rfinv_pt_get_counters

     integer(c_int32_t) function rfinv_pt_draw(handle, local_rank, kind, n, out) bind(C, name="rfinv_pt_draw")
       import :: c_int32_t, c_ptr, c_double
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: local_rank, kind, n
       real(c_double), intent(out) :: out(*)
     end function rfinv_pt_draw

     integer(c_int32_t) function rfinv_filter_traces(handle, n_series, trace_of, in, out) bind(C, name="rfinv_filter_traces")
       import :: c_int32_t, c_ptr, c_double
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: n_series
       integer(c_int32_t), intent(in) :: trace_of(*)
       real(c_double), intent(in) :: in(*)
       real(c_double), intent(out) :: out(*)
     end function rfinv_filter_traces

     ! checkpoint / resume (ABI version 4): path is a NUL-terminated string, e.g. trim(fname)//c_null_char
     integer(c_int32_t) function rfinv_pt_save(handle, path) bind(C, name="rfinv_pt_save")
       import :: c_int32_t, c_ptr, c_char
       type(c_ptr), value :: handle
       character(kind=c_char), intent(in) :: path(*)
     end function rfinv_pt_save

     integer(c_int32_t) function rfinv_pt_restore(handle, path) bind(C, name="rfinv_pt_restore")
       import :: c_int32_t, c_ptr, c_char
       type(c_ptr), value :: handle
       character(kind=c_char), intent(in) :: path(*)
     end function rfinv_pt_restore

     ! even/odd temperature swaps inside every virtual rank (ABI version 6): mode 0 the reference, 1 the sweep
     integer(c_int32_t) function rfinv_pt_set_rank_swaps(handle, mode) bind(C, name="rfinv_pt_set_rank_swaps")
       import :: c_int32_t, c_ptr
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: mode
     end function rfinv_pt_set_rank_swaps

     ! mode, then swaps proposed / accepted per neighbour pair: n_prop(nchains-1), n_acc(nchains-1)
     integer(c_int32_t) function rfinv_pt_get_rank_swaps(handle, mode, n_prop, n_acc) bind(C, name="rfinv_pt_get_rank_swaps")
       import :: c_int32_t, c_int64_t, c_ptr
       type(c_ptr), value :: handle
       integer(c_int32_t), intent(out) :: mode
       integer(c_int64_t), intent(out) :: n_prop(*), n_acc(*)
     end function rfinv_pt_get_rank_swaps

     ! ladder tuning during the burn-in on top of the rank swaps (ABI version 7): on 0 or 1, before the first iteration
     integer(c_int32_t) function rfinv_pt_set_ladder_tuning(handle, on) bind(C, name="rfinv_pt_set_ladder_tuning")
       import :: c_int32_t, c_ptr
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: on
     end function rfinv_pt_set_ladder_tuning

     ! the setting, and the tuning points passed with it on
     integer(c_int32_t) function rfinv_pt_get_ladder_tuning(handle, on, n_points) bind(C, name="rfinv_pt_get_ladder_tuning")
       import :: c_int32_t, c_ptr
       type(c_ptr), value :: handle
       integer(c_int32_t), intent(out) :: on, n_points
     end function rfinv_pt_get_ladder_tuning

     ! random-walk width tuning during the burn-in on top of the rank swaps (ABI version 8): on 0 or 1, target in (0, 1)
     integer(c_int32_t) function rfinv_pt_set_step_tuning(handle, on, target) bind(C, name="rfinv_pt_set_step_tuning")
       import :: c_int32_t, c_double, c_ptr
       type(c_ptr), value :: handle
       integer(c_int32_t), value :: on
       real(c_double), value :: target
     end function rfinv_pt_set_step_tuning

     ! the setting, target, tuning points passed; widths / n_prop / n_acc (4, nchains, rank_count) in the order z, dvs, dvp, sig
     integer(c_int32_t) function rfinv_pt_get_step_tuning(handle, on, target, n_points, widths, n_prop, n_acc) &
         bind(C, name="rfinv_pt_get_step_tuning")
       import :: c_int32_t, c_int64_t, c_double, c_ptr
       type(c_ptr), value :: handle
       integer(c_int32_t), intent(out) :: on, n_points
       real(c_double), intent(out) :: target, widths(*)
       integer(c_int64_t), intent(out) :: n_prop(*), n_acc(*)
     end function rfinv_pt_get_step_tuning

     ! several stations advanced together (ABI version 5): handles(n) are the c_ptr of n handles after rfinv_pt_init
     integer(c_int32_t) function rfinv_pt_group_create(handles, n, group) bind(C, name="rfinv_pt_group_create")
       import :: c_int32_t, c_ptr
       type(c_ptr), intent(in) :: handles(*)
       integer(c_int32_t), value :: n
       type(c_ptr), intent(out) :: group
     end function rfinv_pt_group_create

     integer(c_int32_t) function rfinv_pt_group_run(group, n_iter) bind(C, name="rfinv_pt_group_run")
       import :: c_int32_t, c_ptr
       type(c_ptr), value :: group
       integer(c_int32_t), value :: n_iter
     end function rfinv_pt_group_run

     subroutine rfinv_pt_group_destroy(group) bind(C, name="rfinv_pt_group_destroy")
       import :: c_ptr
       type(c_ptr), value :: group
     end subroutine rfinv_pt_group_destroy

     function rfinv_last_error() bind(C, name="rfinv_last_error") result(msg)
       import :: c_ptr
       type(c_ptr) :: msg
     end function rfinv_last_error
  end interface
end module rfinv_b200_capi
