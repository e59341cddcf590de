// Internal definition of the opaque rfinv_handle.
#pragma once
#include <vector>
#include "rfinv_common.cuh"

struct PtState;  // pt.cu

// Device buffers of one evaluation in flight (grown on demand).  The handle itself is workspace 0 (synchronous calls and the
// parallel-tempering driver); rfinv_eval_batch_begin / _end use one more workspace and stream per slot.
struct EvalWorkspace {
  int cap = 0;
  int* d_k = nullptr;
  double *d_z = nullptr, *d_dvp = nullptr, *d_dvs = nullptr, *d_sig = nullptr, *d_stage = nullptr;
  double *d_misfit = nullptr, *d_phi = nullptr, *d_logl = nullptr, *d_rft_full = nullptr, *d_scratch = nullptr;
  uint8_t* d_valid = nullptr;
  double* d_qpart = nullptr;    // quadform_kernel partial sums
  int* d_qcnt = nullptr;        // quadform_kernel work / arrival counters
  size_t cap_rft_full = 0;
  int grow(const DevConfig& dc, const rfinv_config& cfg, int device, int C);
  void release();
};

constexpr int RFINV_ASYNC_SLOTS = 2;
constexpr int RFINV_UPLOAD_PIECES = 4;

struct rfinv_handle : EvalWorkspace {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  rfinv_config cfg;  // deep copy; pointers refer to the vectors below
  std::vector<double> h_rayps, h_a_gus, h_obs, h_vp_ref, h_vs_ref, h_sig_min, h_sig_max, h_r_inv;
  std::vector<int32_t> h_ipha;
  DevConfig dc;
  // constants in HBM
  double* d_flt = nullptr;
  double2* d_tw = nullptr;
  double2 *d_chirp = nullptr, *d_chirp_b = nullptr, *d_twq = nullptr;   // Bluestein tables (nfft not a power of two)
  double* d_obs = nullptr;
  double* d_vp_ref = nullptr;
  double* d_vs_ref = nullptr;
  double* d_r_inv = nullptr;
  double* d_w_fac = nullptr;
  // rfinv_eval_batch: the models go up as the caller holds them (chain slowest, no layout kernels); large batches in
  // pieces on a second stream, prep_kernel launched per piece behind the piece's event
  cudaStream_t stream_copy = nullptr;
  cudaEvent_t ev_copy[RFINV_UPLOAD_PIECES + 2] = {};
  // rfinv_eval_batch_begin / _end: one workspace and stream per slot
  EvalWorkspace* async_ws[RFINV_ASYNC_SLOTS] = {};
  cudaStream_t async_stream[RFINV_ASYNC_SLOTS] = {};
  bool async_pending[RFINV_ASYNC_SLOTS] = {};
  int launches = 0;
  bool timing = false;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  // parallel-tempering state (pt.cu)
  PtState* pt = nullptr;
  // NCCL communicator of the distributed parallel-tempering run (comm.cu); one process per GPU
  void* comm = nullptr;
  int comm_world = 1, comm_rank = 0;

  // (growing the workspace moves the buffers the captured parallel-tempering launches point at)
  int ensure_capacity(int C) { if (C > cap) invalidate_pt_graphs(); return grow(dc, cfg, device, C); }
  void invalidate_pt_graphs();
  void free_workspace() { release(); }
  void free_pt();
  // forward + quadratic form (+ logL) for device-resident arrays on workspace `w` / stream `s` (defaults: the handle's own)
  int eval_device(int C, const int* k, const double* z, const double* dvp, const double* dvs, const double* sig,
                  double* logl, double* rft_smp, double* rft_full, uint8_t* is_valid, const int* active, int n_active,
                  const ModelBatch* layout = nullptr, EvalWorkspace* w = nullptr, cudaStream_t s = nullptr,
                  bool prep_done = false,    // layout: chain_major field to take over (host path); prep_done: prep_kernel already ran
                  cudaEvent_t before_quadform = nullptr);   // the quadratic form (which reads sig) waits for this event
};

// comm.cu: all-gather of `count` doubles per process over the handle's communicator, on stream s (capturable)
int rfinv_comm_allgather(rfinv_handle* h, const double* send, double* recv, size_t count, cudaStream_t s);
extern "C" int32_t rfinv_comm_destroy(rfinv_handle* h);
// comm.cu: peer-memory swap exchange (CUDA IPC over NVLink); collective over the handle's communicator.  Leaves
// h->pt->peer_state = 1 (on) or -1 (some process cannot map its peers: the NCCL all-gather stays)
int rfinv_comm_peer_setup(rfinv_handle* h);
void rfinv_comm_peer_release(rfinv_handle* h);
// pt.cu: after the job-wide sum, the bins whose means the reference assigns go back to the assigned value
int rfinv_pt_fix_assigned_bins(rfinv_handle* h);
// pt.cu: room in the likelihood history for iterations [0, upto)
int rfinv_pt_reserve_lhist(rfinv_handle* h, int upto);
// capi.cu: the environment switches that change the arithmetic, as read once per process: bit 0 RFINV_FULL_BAND, bit 1
// RFINV_QF_DENSE, bit 2 RFINV_QF_NOSPLIT
int rfinv_arith_switches();
