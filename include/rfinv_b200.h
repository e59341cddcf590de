/*
 * rfinv_b200.h -- C-ABI of the B200-native forward-model + likelihood path of RF_INV.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  Every entry point is `extern "C"`, takes
 * plain pointers, int32_t and double, and returns an int status (0 = ok, non-zero = error, text via
 * rfinv_last_error()).  The library never calls exit(); NaN log-likelihoods are values, not errors.
 * A Fortran host binds these with `interface ... bind(C)` blocks (see include/rfinv_b200_capi.f90
 * and INTEGRATION.md).
 *
 * Reference interfaces replaced (paths relative to the reference checkout):
 *   rfinv_create            <- module globals set up by get_params/read_obs (src/params.f90:101-476),
 *                              read_ref_model (src/model.f90:109-171), init_filter (src/forward.f90:95-119),
 *                              init_fftw (src/fftw.f90:41-48), init_r_inv (src/likelihood.f90:168-241)
 *   rfinv_eval_batch        <- calc_likelihood (src/likelihood.f90:56-101), batched over chains; the
 *                              call sites are src/pt_mcmc.f90:178-180 and src/likelihood.f90:156-160
 *   rfinv_format_model_batch<- format_model (src/model.f90:175-290)
 *   rfinv_pt_*              <- init_model (src/model.f90:43-107), init_sig/init_rft
 *                              (src/likelihood.f90:107-163), init_pt_mcmc (src/pt_mcmc.f90:296-464),
 *                              mcmc (src/pt_mcmc.f90:54-290), pt_control (src/pt_mcmc.f90:468-576)
 *   rfinv_write_outputs     <- output_results (src/mcmc_out.f90:35-322)
 *   rfinv_params_*          <- get_params / read_obs / read_ref_model (file formats are a contract)
 *
 * Array layouts follow the reference's Fortran arrays with the chain as the slowest index, i.e. what a
 * Fortran caller already holds: z(k_max-1, C), dvp(k_max, C), dvs(k_max, C), sig(ntrc, C),
 * rft(nfft, ntrc, C).  On device the library re-lays them out chain-fastest (structure of arrays).
 */
#ifndef RFINV_B200_H
#define RFINV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RFINV_ABI_VERSION 9

/* status codes */
#define RFINV_OK 0
#define RFINV_ERR_ARG 1      /* bad argument / unsupported configuration */
#define RFINV_ERR_CUDA 2     /* CUDA runtime failure (no device, launch failure, out of memory) */
#define RFINV_ERR_IO 3       /* file could not be read / written / parsed */
#define RFINV_ERR_STATE 4    /* call out of order (e.g. pt_step before pt_init) */

/* Immutable configuration: the reference's module globals (src/params.f90:50-96, src/model.f90:35-36). */
typedef struct rfinv_config {
  /* observation and RF synthesis */
  int32_t ntrc;         /* N_TRC */
  int32_t nfft;         /* N_FFT; must be a power of two, 64 <= nfft <= 4096 */
  int32_t nsmp;         /* samples in [T_START, T_END] (src/params.f90:446-448); nsmp <= nfft */
  int32_t deconv_mode;  /* 0: normalise by vertical, 1: water-level deconvolution */
  double delta;         /* sampling interval as read from the SAC header (float32 promoted) */
  double t_start;       /* T_START */
  double sdep;          /* SEA_DEP (km); > 0 prepends a water layer */
  const double* rayps;  /* [ntrc] ray parameters (s/km) */
  const double* a_gus;  /* [ntrc] Gaussian filter parameters */
  const int32_t* ipha;  /* [ntrc] 1 = P receiver function, -1 = S receiver function */
  const double* obs;    /* [ntrc][nsmp] observed traces = Fortran obs(1:nsmp, itrc) */
  const double* r_inv;  /* [ntrc][nsmp][nsmp] inverse data covariance (src/likelihood.f90:222), or NULL:
                           the library then builds it itself from a_gus/delta (symmetric eigen-solver) */
  /* reference velocity model */
  int32_t nref;
  int32_t pad0_;
  double z_ref_min;
  double dz_ref;
  const double* vp_ref; /* [nref] */
  const double* vs_ref; /* [nref] */
  /* prior and model validity */
  int32_t vp_mode;      /* 0: dVp fixed at 0, 1: solved */
  int32_t k_min;
  int32_t k_max;        /* 2 <= k_max <= 64 (fixed device layout) */
  int32_t prior_mode;   /* 1: Laplace, 2: Gaussian */
  double z_min, z_max, h_min;
  double dvs_prior, dvp_prior;
  const double* sig_min; /* [ntrc] */
  const double* sig_max; /* [ntrc] */
  double vp_min, vp_max, vs_min, vs_max, vpvs_min, vpvs_max;
  /* proposal widths */
  double dev_z, dev_dvs, dev_dvp, dev_sig;
  /* parallel tempering */
  int32_t nburn, niter, ncorr;
  int32_t nchains;      /* chains per (virtual) rank = per mt19937 stream */
  int32_t ncool;        /* non-tempered chains per rank */
  int32_t iseed;        /* I_SEED; rank r is seeded iseed + r*r*10000 + 23*r (src/rf_inv.f90:75) */
  double t_high;
  /* posterior histograms (src/pt_mcmc.f90:396-433) */
  int32_t nbin_z, nbin_vs, nbin_vp, nbin_vpvs, nbin_sig, nbin_amp;
  double amp_min, amp_max;
  /* Buried station ("BOREHOLE_DEP", the optional second number of the SEA_DEP line; disabled by comment markers in the
   * reference: src/params.f90:67,203-224, src/forward.f90:289-338,493-516): depth of the receiver below the free surface /
   * the sea floor in km.  0 = receiver at the surface, which is all the reference can run today.  (ABI version 2.) */
  double bdep;
} rfinv_config;

typedef struct rfinv_handle rfinv_handle;

/* ---- library -------------------------------------------------------------------------------- */
int32_t rfinv_abi_version(void);
/* Thread-local text of the last error returned to this thread. */
const char* rfinv_last_error(void);
/* Number of CUDA devices visible; negative status on CUDA failure. */
int32_t rfinv_device_count(void);

/* ---- evaluator ------------------------------------------------------------------------------ */
/* Uploads the configuration (filters, twiddles, observed data, R^-1, reference model) to `device`
 * and creates one stream.  The handle is single-owner: one call at a time per handle.           */
int32_t rfinv_create(const rfinv_config* cfg, int32_t device, rfinv_handle** out);
void rfinv_destroy(rfinv_handle* h);
/* Use an externally owned cudaStream_t (passed as an integer) for all work of this handle. */
int32_t rfinv_set_stream(rfinv_handle* h, uint64_t cuda_stream);

/* calc_likelihood(fwd_flag=.true.) for C models at once.  HOST pointers in and out.
 *   k[C], z[C][k_max-1], dvp[C][k_max], dvs[C][k_max], sig[C][ntrc]
 *   logl[C]               out
 *   rft[C][ntrc][nfft]    out, may be NULL
 *   is_valid[C]           out, may be NULL (format_model's flag; logl is computed regardless, like the reference) */
int32_t rfinv_eval_batch(rfinv_handle* h, int32_t C, const int32_t* k, const double* z, const double* dvp,
                         const double* dvs, const double* sig, double* logl, double* rft, uint8_t* is_valid);

/* calc_likelihood with its per-call fwd_flag (src/likelihood.f90:56-82), batched: fwd_flag[c] != 0 evaluates model c like
 * rfinv_eval_batch and RETURNS its per-trace quadratic forms phi[c][t] = m^T R^-1 m; fwd_flag[c] == 0 -- a sigma-only
 * proposal -- skips the forward model: phi[c][:] is READ (the values the host kept from the evaluation that produced the
 * chain's current RF) and logL follows from them with the proposed sig, which is what the reference computes by taking the
 * chain's cached rft through the same misfit and quadratic form again.  phi[C][ntrc] in / out; k, z, dvp, dvs of the models
 * with fwd_flag == 0 are not looked at; their is_valid comes back 1 (format_model is not run for them). */
int32_t rfinv_eval_batch_flags(rfinv_handle* h, int32_t C, const uint8_t* fwd_flag, const int32_t* k, const double* z,
                               const double* dvp, const double* dvs, const double* sig, double* phi, double* logl,
                               uint8_t* is_valid);

/* Asynchronous form of rfinv_eval_batch for hosts that keep two (or more) groups of chains in flight, e.g. the two halves of
 * the chains of one MPI rank of the reference (src/pt_mcmc.f90:77-201 proposes and judges every chain independently):
 * _begin queues upload, evaluation and the read-back of logl (and is_valid, may be NULL) of one batch on the stream and
 * workspace of `slot` (0 or 1) and returns at once; _end waits until logl[] is filled.  With two slots in flight the
 * transfers of one batch hide behind the kernels of the other.  The host arrays must stay untouched until _end returns
 * (page-locked memory for real overlap; pageable memory works, synchronously).  The complete RF (rft) is not returned. */
int32_t rfinv_eval_batch_begin(rfinv_handle* h, int32_t slot, int32_t C, const int32_t* k, const double* z, const double* dvp,
                               const double* dvs, const double* sig, double* logl, uint8_t* is_valid);
int32_t rfinv_eval_batch_end(rfinv_handle* h, int32_t slot);

/* Same evaluation with DEVICE pointers in the library's chain-fastest layout:
 *   k[C], z[k_max-1][C], dvp[k_max][C], dvs[k_max][C], sig[ntrc][C], logl[C],
 *   rft_smp[ntrc][C][nsmp] (first nsmp samples only; may be 0), is_valid[C] (may be 0).
 * Asynchronous on the handle's stream.                                                          */
int32_t rfinv_eval_batch_device(rfinv_handle* h, int32_t C, uint64_t d_k, uint64_t d_z, uint64_t d_dvp,
                                uint64_t d_dvs, uint64_t d_sig, uint64_t d_logl, uint64_t d_rft_smp,
                                uint64_t d_is_valid);

/* format_model for C models (HOST pointers): nlay[C], alpha/beta/rho/h [C][k_max+1] (k_max+1 is the
 * largest nlay: k_max-1 interfaces + half space + optional sea layer), is_valid[C].             */
int32_t rfinv_format_model_batch(rfinv_handle* h, int32_t C, const int32_t* k, const double* z,
                                 const double* dvp, const double* dvs, int32_t* nlay, double* alpha,
                                 double* beta, double* rho, double* hthick, uint8_t* is_valid);

/* out = c2r( r2c(in) * flt(:, trace_of[i]) ) for n_series real series of nfft samples, both transforms unnormalised like
 * FFTW's: the noise shaping of make_syn (src/make_syn.f90:96-100, plans src/fftw.f90:44-45).  HOST pointers:
 * trace_of[n_series] (0-based trace whose Gaussian filter is applied), in/out [n_series][nfft].                      */
int32_t rfinv_filter_traces(rfinv_handle* h, int32_t n_series, const int32_t* trace_of, const double* in, double* out);

/* Copies the R^-1 actually in use back to the host ([ntrc][nsmp][nsmp]). */
int32_t rfinv_get_r_inv(rfinv_handle* h, double* r_inv);
/* Waits for all work queued on the handle's stream. */
int32_t rfinv_synchronize(rfinv_handle* h);

/* Timing / accounting of the last rfinv_eval_batch* call: number of kernels launched by it. */
int32_t rfinv_last_launch_count(rfinv_handle* h);
/* enable != 0: bracket every kernel of the evaluation with CUDA events on the handle's stream. */
int32_t rfinv_set_timing(rfinv_handle* h, int32_t enable);
/* Device time (ms) of the kernels of the last evaluation: ms[0] forward, ms[1] quadratic form, ms[2] logL.
 * Synchronises the stream.  Requires rfinv_set_timing(h, 1).                                      */
int32_t rfinv_get_timing(rfinv_handle* h, double* ms);
/* Form of the quadratic form chosen at rfinv_create, per trace (arrays of ntrc): rank[t] = 0: dense m^T R^-1 m; > 0: factor
 * form |W^T m|^2 with that many columns; split[t] = 1: the factor acts on sums / differences of mirrored samples (R^-1
 * commutes with the exchange matrix), rank_s[t] columns on the sums and rank[t] - rank_s[t] on the differences.     */
int32_t rfinv_get_quadform_form(rfinv_handle* h, int32_t* rank, int32_t* rank_s, int32_t* split);
/* FP64 roofline denominators measured on `device` right now: dense DFMA and DMMA (mma.sync m8n8k4)
 * loops on all SMs, best of a few repetitions; TFLOP/s.                                           */
int32_t rfinv_measure_fp64_peak(int32_t device, double* dfma_tflops, double* dmma_tflops);

/* ---- parallel tempering (device-resident chains) ---------------------------------------------------
 * The job consists of `nproc_total` virtual ranks (= MPI ranks of the reference: cfg.nchains chains and ONE
 * mt19937 stream each, seeded iseed + r*r*10000 + 23*r, src/rf_inv.f90:75).  This handle owns the ranks
 * [rank_begin, rank_begin + rank_count); with several processes every process must own the same number of
 * ranks and process q owns [q*rank_count, (q+1)*rank_count).                                               */
/* init_model + init_sig + init_rft + temperatures (src/rf_inv.f90:86-91), on device. */
int32_t rfinv_pt_init(rfinv_handle* h, int32_t nproc_total, int32_t rank_begin, int32_t rank_count);
/* Draws n deviates from the mt19937 stream of local virtual rank `local_rank`, advancing it: kind 0 = grnd()
 * (src/mt19937.f90:92-130), kind 1 = gauss() (src/math.f90:34-50).  out[n] is a HOST pointer.  With cfg.ncool = cfg.nchains
 * (no temperature draws) the stream after rfinv_pt_init(h, 1, 0, 1) is where make_syn starts its noise draws
 * (src/make_syn.f90:52-65, 80-110). */
int32_t rfinv_pt_draw(rfinv_handle* h, int32_t local_rank, int32_t kind, int32_t n, double* out);
/* Number of proposal types (src/pt_mcmc.f90:311-365): 4 (+1 if vp_mode) (+1 if a sigma is solved). */
int32_t rfinv_pt_ntype(rfinv_handle* h);
/* Keep per-iteration logs for the next `cap_iters` iterations (0 disables): accept flags, proposal types, swaps. */
int32_t rfinv_pt_set_logging(rfinv_handle* h, int32_t cap_iters);
/* pt_control (src/pt_mcmc.f90:468-576) for n_iter iterations when this handle owns ALL ranks. */
int32_t rfinv_pt_run(rfinv_handle* h, int32_t n_iter);
/* ---- one process per GPU: the collectives of the path, inside the library (NCCL over NVLink) ---------------------
 * Replaces the reference's MPI traffic on this path: pt_control's swap exchange (src/pt_mcmc.f90:518-571: mpi_bcast of the
 * pair, mpi_send / mpi_recv of temperature and likelihood) becomes ONE ncclAllGather of the swap tables per iteration on the
 * handle's stream -- or, when every GPU can map its peers' memory (one NVLink / NVSwitch box), no collective call at all: the
 * pair and the tables are stored into peer memory by two small kernels on a side branch of the iteration's graph and the swap
 * is applied one iteration later (rfinv_pt_exchange_mode); output_results' 14 mpi_reduce and 2 mpi_gather (src/mcmc_out.f90:52-93) become rfinv_pt_reduce_outputs.
 * NCCL is bound at run time (libnccl.so.2, or the file named by RFINV_NCCL_LIB).  The host only carries the communicator id
 * from one process to the others (MPI_Bcast of rfinv_comm_id_bytes() bytes in the Fortran host).                          */
int32_t rfinv_comm_id_bytes(void);
/* On ONE process: a fresh communicator id (ncclUniqueId), id_out[rfinv_comm_id_bytes()]. */
int32_t rfinv_comm_create_id(void* id_out);
/* On EVERY process (collective): joins the communicator of `world` processes as process `rank`. */
int32_t rfinv_comm_init(rfinv_handle* h, const void* id, int32_t world, int32_t rank);
int32_t rfinv_comm_destroy(rfinv_handle* h);
/* world / rank of the handle's communicator (1 / 0 without one) and the version of the NCCL library bound (0: none). */
int32_t rfinv_comm_info(rfinv_handle* h, int32_t* world, int32_t* rank, int32_t* nccl_version);
/* How rfinv_pt_run_distributed exchanges the swap tables: 0 = not decided yet (no distributed run since rfinv_pt_init) or a
 * single process; 1 = peer memory -- every process stores the pair and its table straight into the buffers of all processes
 * (CUDA IPC mappings over NVLink) from a side branch of the iteration's graph and raises a flag; no collective call, and no
 * process waits for another at the end of an iteration (the swap is applied one iteration later, where its parts are needed);
 * 2 = one ncclAllGather per iteration (some process could not map its peers, or RFINV_PT_EXCHANGE=nccl). */
int32_t rfinv_pt_exchange_mode(rfinv_handle* h);
/* pt_control (src/pt_mcmc.f90:468-576) for n_iter iterations over the processes of the communicator; process q must have
 * called rfinv_pt_init(h, nproc_total, q * G, G).  Bit-identical to the single-process run of the same nproc_total.
 * Like rfinv_pt_run, the launch sequence of an iteration is captured once in a CUDA graph and replayed. */
int32_t rfinv_pt_run_distributed(rfinv_handle* h, int32_t n_iter);
/* Collective, once, after the last iteration: process 0 then holds the job-wide sums of the bookkeeping arrays, counters and
 * likelihood history and the recorded models of every process in process order -- what mpi_reduce / mpi_gather deliver on
 * rank 0 -- and returns them through rfinv_pt_get_hist / _get_counters / _get_models. */
int32_t rfinv_pt_reduce_outputs(rfinv_handle* h);

/* Multi-process iteration, step 1: every chain proposes, is evaluated and accepted/rejected; fills this
 * process's swap table [temps(Cl) | logL(Cl) | next uniform of each local stream (G) | itarget1, itarget2]. */
int32_t rfinv_pt_local_step(rfinv_handle* h);
/* Device pointer and length (doubles) of the swap table: the payload of the per-iteration all-gather. */
int32_t rfinv_pt_swap_table(rfinv_handle* h, uint64_t* dev_ptr, int32_t* n_doubles);
/* Step 2: `gathered_dev_ptr` holds the `world` tables in process order (device memory); every process evaluates
 * the one global swap proposal of the iteration identically (src/pt_mcmc.f90:501-571) and updates its chains. */
int32_t rfinv_pt_apply_swap(rfinv_handle* h, uint64_t gathered_dev_ptr, int32_t world);
/* Host copies of the local chain state, chain-major like the Fortran arrays (any pointer may be NULL):
 * k[Cl], z[Cl][k_max-1], dvp[Cl][k_max], dvs[Cl][k_max], sig[Cl][ntrc], logl[Cl], temps[Cl]. */
int32_t rfinv_pt_get_state(rfinv_handle* h, int32_t* k, double* z, double* dvp, double* dvs, double* sig, double* logl,
                           double* temps);
/* nprop[ntype], naccept[ntype] of the non-tempered chains (src/pt_mcmc.f90:196-198), likelihood_hist[0..n_hist)
 * (sum of logL over the local non-tempered chains per iteration, :199-200), forward evaluations executed. */
int32_t rfinv_pt_get_counters(rfinv_handle* h, int64_t* nprop, int64_t* naccept, double* likelihood_hist, int32_t n_hist,
                              int64_t* n_eval);
int32_t rfinv_pt_iterations_done(rfinv_handle* h);
/* Logs kept by rfinv_pt_set_logging: flags[n][Cl] (-1 null proposal, 0 rejected, 1 accepted), itypes[n][Cl]
 * (1-based), swaps[n][3] (itarget1, itarget2, accepted). */
int32_t rfinv_pt_get_log(rfinv_handle* h, int8_t* flags, int8_t* itypes, int32_t* swaps, int32_t* n_logged);

/* Posterior bookkeeping of the non-tempered chains, recorded every ncorr iterations after nburn
 * (src/pt_mcmc.f90:204-286); local sums of this handle.  Layouts: nk[k_max], nz[nbin_z], nsig[ntrc][nbin_sig],
 * namp[ntrc][nsmp][nbin_amp], nvpz[nbin_vp][nbin_z], nvsz[nbin_vs][nbin_z], nvpvsz[nbin_vpvs][nbin_z], *_mean[nbin_z].
 * Requires cfg.niter > 0 and all nbin_* > 0 at rfinv_pt_init.  Any pointer may be NULL. */
int32_t rfinv_pt_get_hist(rfinv_handle* h, int64_t* nmod, int64_t* nk, int64_t* nz, int64_t* nsig, int64_t* namp,
                          int64_t* nvpz, int64_t* nvsz, int64_t* nvpvsz, double* vp_mean, double* vs_mean,
                          double* vpvs_mean);
/* Recorded models (all_models): vp_model/vs_model [n_models][nbin_z]. */
int32_t rfinv_pt_get_models(rfinv_handle* h, int64_t max_models, double* vp_model, double* vs_model, int64_t* n_models);

/* ---- checkpoint / resume (ABI version 4) ---------------------------------------------------------------------------
 * Writes this handle's complete PT state to `path` (atomically: path + ".tmp", fsync, rename): mt19937 streams, chain state
 * and RF buffers, swap table, counters, likelihood history and, with the bookkeeping on, histograms, means and recorded
 * models.  Per-iteration logs are not saved.  A distributed run writes one file per process (its own virtual ranks).
 * RFINV_ERR_STATE between rfinv_pt_local_step and rfinv_pt_apply_swap, and after rfinv_pt_reduce_outputs. */
int32_t rfinv_pt_save(rfinv_handle* h, const char* path);
/* Loads a state written by rfinv_pt_save into a handle on which rfinv_pt_init(h, nproc_total, rank_begin, rank_count)
 * was called with the same arguments and no iteration has run since.  Continues at iterations_done = the saved count;
 * the continued run is bit-identical to an uninterrupted one.  The configuration must be the one the file was written
 * with, except that cfg.niter may be larger.  Logging is switched off (call rfinv_pt_set_logging again).
 * RFINV_ERR_IO: unreadable, short, bad magic / version / checksum.  RFINV_ERR_ARG: other rank layout, nchains, a smaller
 * niter, or a configuration group that differs (named in rfinv_last_error()).  RFINV_ERR_STATE: not fresh from pt_init. */
int32_t rfinv_pt_restore(rfinv_handle* h, const char* path);

/* ---- several runs advanced together on one GPU (ABI version 5) -------------------------------------------------------
 * A study inverts many stations, each an independent PT run of its own handle.  A group advances n such handles by one
 * iteration in ONE graph launch with n parallel branches, so the small kernels of many runs share the GPU instead of taking
 * turns.  Members stay ordinary handles: rfinv_pt_get_*, rfinv_pt_set_logging, rfinv_pt_save / _restore and a solo rfinv_pt_run
 * keep working between group runs.  A group iteration lasts as long as its slowest member's. */
typedef struct rfinv_pt_group rfinv_pt_group;
/* n >= 1 distinct handles on the same device, each after rfinv_pt_init as a single process (rank_count == nproc_total).  The
 * handles must outlive the group.  RFINV_ERR_ARG: NULL or duplicate handles, members on different devices; RFINV_ERR_STATE:
 * a member without rfinv_pt_init or with a distributed layout.  The message names the member index. */
int32_t rfinv_pt_group_create(rfinv_handle* const* handles, int32_t n, rfinv_pt_group** out);
/* n_iter iterations of every member, as if each had called rfinv_pt_run(member, n_iter): every member ends with the same bits
 * (state, RF buffers, counters, likelihood history, histograms, recorded models, logs; the profile means are summed with fp64
 * atomics and agree to rounding).  Synchronous.  RFINV_ERR_STATE, naming the member, when the members differ in nburn, ncorr
 * or iterations done, or a member is between rfinv_pt_local_step and rfinv_pt_apply_swap or after rfinv_pt_reduce_outputs. */
int32_t rfinv_pt_group_run(rfinv_pt_group* g, int32_t n_iter);
/* Frees the group; the member handles are untouched. */
void rfinv_pt_group_destroy(rfinv_pt_group* g);

/* ---- even/odd temperature swaps inside every virtual rank (ABI version 6, DESIGN.md 7c) ----------------------------------
 * The reference proposes one swap per iteration for the whole job, between two chains drawn from all of them.  Mode 1 adds,
 * every iteration i, a sweep inside each virtual rank: its chains sorted by (temperature, chain index) form levels 0..nchains-1,
 * and each level l = i (mod 2) proposes to swap temperatures with level l + 1 (judge_pt's test, a Philox4x64-10 uniform of
 * counter (i, rank, l, 0) and key (iseed, 0)).  The sweep runs after the posterior bookkeeping and before the global swap,
 * and leaves the mt19937 streams untouched.  Mode 0 (the default after rfinv_pt_init) is the reference, bit for bit.  May be
 * called after rfinv_pt_init and between runs; a distributed run needs the same mode on every process (the caller's
 * contract, like the rank layout), and a checkpoint restores only into a handle set to the mode it was saved in.
 * RFINV_ERR_ARG: a mode other than 0 or 1.  RFINV_ERR_STATE: between rfinv_pt_local_step and rfinv_pt_apply_swap, or after
 * rfinv_pt_reduce_outputs. */
int32_t rfinv_pt_set_rank_swaps(rfinv_handle* h, int32_t mode);
/* The mode and, per level pair l = 0..nchains-2, the swaps proposed and accepted by the sweep, summed over this handle's ranks
 * (after rfinv_pt_reduce_outputs in mode 1: over the job, on process 0).  n_prop / n_acc have nchains - 1 entries; any
 * pointer may be NULL. */
int32_t rfinv_pt_get_rank_swaps(rfinv_handle* h, int32_t* mode, int64_t* n_prop, int64_t* n_acc);

/* ---- ladder tuning during the burn-in (ABI version 7, DESIGN.md 7d) --------------------------------------------------------
 * On top of the rank sweep (mode 1): at the tuning points e = 64, 128, 256, ... <= nburn (inside iteration e - 1, after its
 * sweep, before its global swap) every virtual rank moves the temperatures of its levels above the cold ones so that the
 * rejection rates its neighbour pairs showed in the round [e/2, e) (from 0 for e = 64) would be equal: the ladder of equal
 * rejection rates of Syed, Bouchard-Cote, Deligiannidis & Doucet (JRSS-B 2021).  The coldest level, the hottest and every cold
 * chain keep their temperatures; models, logL and every random stream are untouched.  After the burn-in the ladders stay
 * fixed.  Off (the default) leaves the mode-1 run bit for bit as it is.  A checkpoint restores only into a handle with the same
 * setting; a distributed run needs it on every process.
 * RFINV_ERR_ARG: a value other than 0 or 1.  RFINV_ERR_STATE: switching it on without rfinv_pt_init, after an iteration has
 * run, or while the rank swaps are not mode 1; either way between rfinv_pt_local_step and rfinv_pt_apply_swap or after
 * rfinv_pt_reduce_outputs.  rfinv_pt_set_rank_swaps(h, 0) switches the tuning off as well. */
int32_t rfinv_pt_set_ladder_tuning(rfinv_handle* h, int32_t on);
/* The setting and the number of tuning points passed with it on; either pointer may be NULL. */
int32_t rfinv_pt_get_ladder_tuning(rfinv_handle* h, int32_t* on, int32_t* n_points);

/* ---- random-walk width tuning during the burn-in (ABI version 8, DESIGN.md 7e) ----------------------------------------------
 * On top of the rank sweep (mode 1), independent of the ladder tuning: the chains at level l of virtual rank r propose the
 * moves z, dVs, dVp and sigma with width dev_tau * scale[r][l][tau] (scale 1 when switched on); the two chains of the
 * previous iteration's global swap propose with the params.in widths.  At the tuning points e = 64, 128, 256, ... <= nburn
 * (inside iteration e - 1, after the sweep and the ladder tuning) every (rank, level, type) with at least 16 proposals since
 * the previous point multiplies its scale by (acceptance / target) clamped to [1/2, 2], the scale staying in [2^-8, 2^8].
 * After the burn-in the widths stay fixed.  Off (the default) leaves the mode-1 run bit for bit as it is.  A checkpoint
 * restores only into a handle with the same setting and target; a distributed run needs it on every process.
 * on: 0/1; target in (0, 1), e.g. 0.44.
 * RFINV_ERR_ARG: on other than 0 or 1, a target outside (0, 1), or switching it on with nchains < 2.  RFINV_ERR_STATE:
 * switching it on without rfinv_pt_init, after an iteration has run, or while the rank swaps are not mode 1; either way
 * between rfinv_pt_local_step and rfinv_pt_apply_swap or after rfinv_pt_reduce_outputs.  Off returns the widths to the
 * params.in values; rfinv_pt_set_rank_swaps(h, 0) switches the tuning off as well. */
int32_t rfinv_pt_set_step_tuning(rfinv_handle* h, int32_t on, double target);
/* widths[G][nchains][4]: absolute dev_tau * scale in the order z, dvs, dvp, sig (params.in value for a type the run does not
 * propose); n_prop / n_acc [G][nchains][4] since the last tuning point; any pointer may be NULL */
int32_t rfinv_pt_get_step_tuning(rfinv_handle* h, int32_t* on, double* target, int32_t* n_points, double* widths,
                                 int64_t* n_prop, int64_t* n_acc);

/* ---- convergence diagnostics (ABI version 9, DESIGN.md 7f) ---------------------------------------------------------------
 * Level 0 of virtual rank r is its chain of lowest (temperature, local chain index), the order of the rank sweep.  With the
 * diagnostics on, every iteration that records the posterior bookkeeping (it > nburn, it % ncorr == 0) also records, right
 * after the bookkeeping (the temperatures at acceptance, before the sweep and the global swap), one row per local rank from
 * its level-0 chain: k, logL, sig[t] of every trace t with sig_mode[t] on (trace order), and the Vs the bookkeeping assigns
 * to each chosen depth bin b (1-based; vs_min inside the sea layer); and beside it the temperature T0 of that chain.  Layout
 * trace[sample][local rank][quantity] (fp64), t0[sample][local rank]; the capacity is the number of recording iterations in
 * [1, nburn + niter]; later samples are not recorded.  In iterations that run the rank sweep (mode 1), each chain also keeps a
 * round-trip state on the levels the sweep finds before deciding any pair: reaching level 0 sets "came from level 0";
 * reaching level nchains - 1 from it moves on to "reached the top"; reaching level 0 from there completes one round trip of
 * the chain's rank, counted during the burn-in (it <= nburn) or after it.  The diagnostics only read: state, counters, logs,
 * histograms and recorded models stay bit for bit those of the same run without them.
 * on: 0/1; vs_bins[n_bins], 0 <= n_bins <= 16, each in [1, nbin_z].  Only after rfinv_pt_init and before the first
 * iteration, or before rfinv_pt_restore (a checkpoint restores only into a handle with the same setting and bins).
 * RFINV_ERR_ARG: on other than 0 or 1, bad bins or more than 16.  RFINV_ERR_STATE: after an iteration has run, between
 * rfinv_pt_local_step and rfinv_pt_apply_swap, after rfinv_pt_reduce_outputs, or switching on without the bookkeeping
 * (niter > 0 and all nbin_* > 0). */
int32_t rfinv_pt_set_diagnostics(rfinv_handle* h, int32_t on, int32_t n_bins, const int32_t* vs_bins);
/* The setting, quantities per row (2 + solved sigmas + n_bins), the bins, and the first min(recorded, max_samples) samples of
 * this process's trace: trace[n][G][n_quantities], t0[n][G]; vs_bins has up to 16 entries.  Any pointer may be NULL. */
int32_t rfinv_pt_get_cold_trace(rfinv_handle* h, int32_t* on, int32_t* n_quantities, int32_t* n_bins, int32_t* vs_bins,
                                int64_t max_samples, int64_t* n_samples, double* trace, double* t0);
/* Statistics of the n recorded samples, computed on the device.  rows[n_ranks][n_quantities][9], one per rank and quantity
 * from its series alone: mean, variance (n - 1), tau (integrated autocorrelation time: autocovariance with divisor n over
 * lag 0, tau = 1 + 2 sum rho(t) up to the first m >= 5 tau; NaN for n < 4 or a constant series), ESS = n / tau, the mean and
 * variance (h - 1) of the halves [0, h) and [n - h, n) with h = n / 2, and the rank's samples with T0 > 1 + 1e-6f.
 * summary[n_quantities][4] over the ranks in global rank order: split-R-hat (BDA3) over the 2 n_ranks half-chains (NaN for
 * h < 2 or a zero within-variance), the sum of the ESS and the median tau over the ranks with finite tau, and the share of
 * (rank, sample) entries whose T0 is tempered.  trips[n_ranks][2]: round trips during the burn-in and after it (zero in
 * mode 0 and with one chain per rank).  n_ranks is this process's G -- after rfinv_pt_reduce_outputs, on process 0, every
 * virtual rank of the job, with the same result as one process holding them all.  Any pointer may be NULL.
 * RFINV_ERR_STATE: the diagnostics are off. */
int32_t rfinv_pt_get_diagnostics(rfinv_handle* h, int64_t* n_samples, int32_t* n_ranks, int32_t* n_quantities, double* rows,
                                 double* summary, int64_t* trips);

/* ---- file formats either side of the path (host only, no CUDA) ---------------------------------------
 * params.in (positional, '#' comment lines; src/params.f90:101-405), SAC traces cut to [T_START, T_END]
 * (src/params.f90:422-476), reference velocity model (src/model.f90:109-171).                        */
typedef struct rfinv_problem rfinv_problem;
int32_t rfinv_problem_load(const char* params_path, const char* base_dir, rfinv_problem** out);
void rfinv_problem_free(rfinv_problem* p);
/* The configuration read (pointers owned by the problem; r_inv is NULL). */
const rfinv_config* rfinv_problem_config(const rfinv_problem* p);
const char* rfinv_problem_out_dir(const rfinv_problem* p);
double rfinv_problem_t_end(const rfinv_problem* p);
/* <out_dir>/params.in.copy and <input_dir>/inputNN, the side outputs of get_params / read_obs. */
int32_t rfinv_problem_write_copies(const rfinv_problem* p, const char* out_dir, const char* input_dir);
/* output_results (src/mcmc_out.f90:97-318): writes all_models, likelihood, num_interface.ppd, syn_trace.ppd,
 * interface_depth.ppd, sigma.ppd, vs_z.ppd, vp_z.ppd, vpvs_z.ppd, vs_z.mean, vp_z.mean, vpvs_z.mean into out_dir
 * from job-wide sums (the caller reduces over processes, like the reference's mpi_reduce at :52-93). */
int32_t rfinv_write_outputs(const rfinv_config* c, const char* out_dir, int32_t nproc_total, int64_t nmod, const int64_t* nk,
                            const int64_t* nz, const int64_t* nsig, const int64_t* namp, const int64_t* nvpz,
                            const int64_t* nvsz, const int64_t* nvpvsz, const double* vp_mean, const double* vs_mean,
                            const double* vpvs_mean, const double* likelihood_hist, int32_t n_hist, const double* vp_model,
                            const double* vs_model, int64_t n_models);

#ifdef __cplusplus
}
#endif
#endif /* RFINV_B200_H */
