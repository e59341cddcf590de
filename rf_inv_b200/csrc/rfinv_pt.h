// Device-resident parallel-tempering state (pt.cu).
#pragma once
#include <atomic>
#include "rfinv_common.cuh"

// Passed to the PT kernels by value.  Arrays are chain-fastest: x[i*Cl + c].
struct PtDev {
  int nproc_total, rank_begin, G, nchains, Cl, ncool, iseed;
  int ntype, it_birth, it_death, it_z, it_dvs, it_dvp, it_sig, nsig_trc;
  int isig_trc[RFINV_MAX_TRC], sig_mode[RFINV_MAX_TRC];
  double sig_min[RFINV_MAX_TRC], sig_max[RFINV_MAX_TRC];
  double t_high, dev_z, dev_dvs, dev_dvp, dev_sig, dvs_prior, dvp_prior;
  // mt19937 streams, one per virtual rank: word i of stream r at mt[r*624 + i]
  uint32_t* mt;
  int* mti;
  // current state
  int* k;
  double *z, *dvp, *dvs, *sig, *logl, *temps, *phi;   // [k_max-1|k_max|k_max|ntrc][Cl], [Cl], [Cl], [ntrc][Cl]
  uint8_t* slot;                                      // which rft_smp buffer holds the current RF of chain c
  double* rft_smp[2];                                 // [ntrc][Cl][nsmp] x 2 (current / proposal, selected by slot)
  // proposal
  int* pk;
  double *pz, *pdvp, *pdvs, *psig, *pphi, *log_r, *log_prior12;
  int8_t *itype, *pflag;                              // pflag: -1 null proposal, 1 forward needed, 2 cached RF
  int* active;                                        // compacted list of chains with pflag == 1
  int* n_active;
  unsigned long long *nprop, *naccept, *n_eval;       // counters of the non-tempered chains; evaluations executed
  // posterior bookkeeping of the non-tempered chains (src/pt_mcmc.f90:204-286); layouts as in rfinv_pt_get_hist
  int nburn, ncorr, nbin_z, nbin_vs, nbin_vp, nbin_vpvs, nbin_sig, nbin_amp;
  double amp_min, amp_max;
  unsigned long long *nk, *nz, *nsig, *namp, *nvpz, *nvsz, *nvpvsz, *nmod;
  double *vp_mean, *vs_mean, *vpvs_mean;
  uint8_t* ocean_bin;                                 // [nbin_z] depth bins inside the sea layer: their vs / vpvs means are ASSIGNED (src/pt_mcmc.f90:260-263)
  double *vp_model, *vs_model;                        // [cap_models][nbin_z] (all_models), may be null
  long long cap_models;
  int *cold_ordinal, *cold_count;                     // ordered numbering of the chains recorded this iteration
  // optional per-iteration logs (tests): iteration `it` (0-based, read from *it_dev) goes to slot it - log_base if that is
  // inside [0, log_cap)
  int8_t *log_flags, *log_itypes;
  int32_t* log_swaps;
  int log_base, log_cap;
  // iterations completed, on the device: advanced by pt_swap_kernel, read by the kernels that index by iteration
  // (likelihood history, logs) -- nothing of an iteration's launch sequence depends on the host's counter, so the sequence
  // can be captured once in a CUDA graph and replayed
  int* it_dev;
  // even/odd swaps inside every virtual rank (rfinv_pt_set_rank_swaps, DESIGN.md 7c); allocated by the first switch to mode 1
  unsigned long long* rs_nprop;   // [nchains - 1] proposals per level, summed over the local ranks
  unsigned long long* rs_nacc;    // [G][nchains - 1] accepted swaps per rank and level (rows: no same-address atomics)
  int* rs_arrived;                // arrival counter of pt_rank_swap_kernel
  // ladder tuning during the burn-in (rfinv_pt_set_ladder_tuning, DESIGN.md 7d); allocated by the first switch on
  unsigned long long* rs_base;    // [G][nchains - 1] rs_nacc at the last tuning point: the acceptances of a round are the difference
  int rs_tune;                    // 1: pt_rank_swap_kernel retunes the ladders at the tuning points
  // random-walk width tuning during the burn-in (rfinv_pt_set_step_tuning, DESIGN.md 7e); allocated by the first switch on.
  // Rows [G][nchains][4]: virtual rank, level, type (0 move z, 1 dVs, 2 dVp, 3 sigma)
  double* st_scale;               // factor on the params.in width, 1 when switched on
  unsigned long long *st_nprop, *st_nacc;   // proposals / accepted ones since the last tuning point (one writer per row)
  int* st_lvl;                    // [Cl] each chain's level after the previous iteration's rank sweep
  int* st_pair;                   // [2] global chains of the previous iteration's global swap (-1: none yet)
  double st_target;               // acceptance rate the widths are tuned towards
  int st_on;                      // 1: proposals use the tuned widths, pt_rank_swap_kernel tunes them at the tuning points
};

struct ncclComm;   // NCCL communicator (comm.cu)

// Swap exchange over peer memory (one process per GPU on one NVLink / NVSwitch box).  Every process owns ONE buffer, opened
// by every other process through CUDA IPC:
//   gather [2][world][table_len] doubles | table flags [world] | error word | pair flag | pair [4][2] doubles
// Stores into peer memory, system-scope fences and release stores cost microseconds each, so none of them sits on the
// iteration's critical path: two small kernels on a SIDE BRANCH of the iteration's graph do them while the main branch computes.
// * pt_pairpush_kernel (behind pt_propose_kernel, beside prep / forward / quadform): the process that owns virtual rank 0
//   stores the pair of iteration i into pair slot i & 3 of EVERY process and raises pair flag = i + 1 everywhere (four slots:
//   the pair of iteration i may be drawn while the slowest process still reads that of iteration i - 2);
// * pt_push_kernel (at the top of iteration i + 1, beside pt_propose_kernel): stores the swap table of iteration i -- which
//   pt_finish_kernel left in the local table, parity i & 1 -- into slot `me` of EVERY process's gather buffer and raises table
//   flag[me] = i + 1 everywhere.
// And nobody waits for the exchange at the end of the iteration: swap i is APPLIED one iteration later, where its parts are
// needed -- the stream shift of rank1 (judge_pt's draw, src/pt_mcmc.f90:590) at the top of pt_propose_kernel of iteration i + 1,
// which only needs the pair; the exchange of the two temperatures at the top of pt_finish_kernel of iteration i + 1 (the
// acceptance test is the first reader of a temperature), which needs the tables.  By then both arrived most of an iteration
// ago, so the processes drift by up to an iteration instead of meeting at every swap.  pt_drain_kernel applies the last swap of
// a run.  (Double buffering suffices: a process needs every table flag of iteration i - 1 to finish iteration i, so it is
// never two iterations ahead of anyone.)
#define RFINV_MAX_PEERS 16
struct PtPeers {
  int world, me, table_len;
  double* gather[RFINV_MAX_PEERS];               // buffer of process q (own: local memory, others: IPC mappings)
  unsigned long long* flag[RFINV_MAX_PEERS];     // its flag words: [world] table epochs, [world] error, [world + 1] pair epoch;
                                                 // the pair slots follow as doubles (pt_pair_slot)
  double* own_gather;                            // = gather[me], flag[me]: kept apart so that no kernel indexes the arrays above with
  unsigned long long* own_flag;                  // a run-time value (the parameter block would be copied to local memory per thread)
  int* done;                                     // local: [0] swaps whose stream shift is applied, [1] swaps whose temperatures are,
                                                 // [2] tables pushed, [3] arrival counter of pt_push_kernel
};
// words of 8 bytes behind the gather buffer
inline size_t pt_peer_tail_words(int world) { return (size_t)world + 2 + 8; }

// unique over the process: a PtState that rfinv_pt_init creates again at the same address still gets a new generation
inline uint64_t rfinv_pt_next_generation() {
  static std::atomic<uint64_t> n{0};
  return ++n;
}

struct PtState {
  PtDev dev;
  int it_done = 0;
  // one iteration as a CUDA graph: [0] plain, [1] with the posterior bookkeeping kernels (every ncorr-th iteration after
  // the burn-in); invalidated when something that is baked into the launches changes (logging, capacity)
  cudaGraphExec_t graph[2] = {nullptr, nullptr};
  uint64_t generation = rfinv_pt_next_generation();   // renewed whenever the graphs are dropped (groups capture again)
  int graph_world = 0;
  cudaStream_t capture_stream = nullptr;
  cudaStream_t side_stream = nullptr;      // side branch of the iteration (peer-memory exchange)
  cudaEvent_t ev_side[3] = {nullptr, nullptr, nullptr};
  double* d_gather = nullptr;  // swap tables of all processes (distributed run, NCCL all-gather)
  int cap_gather = 0;
  // peer-memory exchange (comm.cu: rfinv_comm_peer_setup); peer_state 0 = not tried, 1 = on, -1 = unavailable (NCCL all-gather)
  PtPeers peers = {};
  int peer_state = 0;
  double* d_peer_gather = nullptr;
  unsigned long long* d_peer_flags = nullptr;
  int cap_lhist = 0;
  double* d_lhist = nullptr;   // likelihood_hist(it), src/pt_mcmc.f90:199-200
  double* d_lh_part = nullptr; // per-CTA sums of the likelihood history (pt_finish_kernel)
  int* d_lh_cnt = nullptr;     // its arrival counter
  double* d_table = nullptr;   // swap table of this process, [2][table_len] (the peer-memory exchange alternates, the others use [0])
  int table_len = 0;
  int log_cap = 0, log_base = 0;
  long long n_eval = 0;
  bool record = false;
  bool step_pending = false;   // rfinv_pt_local_step has run, rfinv_pt_apply_swap not yet: no checkpoint in between
  bool reduced = false;        // rfinv_pt_reduce_outputs has run: the bookkeeping may hold job-wide sums
  int rank_swaps = 0;          // rfinv_pt_set_rank_swaps: 0 the reference's global swap only, 1 the rank sweep before it
  int tune_points_off = 0;     // tuning points passed while the ladder tuning was on, frozen when it is switched off
  int step_points_off = 0;     // likewise for the step tuning
};

// does an iteration of this state run the rank sweep?  (nothing to pair with fewer than two chains per rank)
inline bool pt_sweeps(const PtState* s) { return s->rank_swaps == 1 && s->dev.nchains >= 2; }

// the tuning points e = 2^j, j >= 6, e <= nburn among the first it_done iterations (DESIGN.md 7d, 7e)
inline int pt_tuning_points(int it_done, int nburn) {
  int n = 0;
  for (long long e = 64; e <= it_done && e <= nburn; e *= 2) ++n;
  return n;
}
