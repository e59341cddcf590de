// Shared device-side definitions of the B200 forward+likelihood path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <map>
#include <mutex>
#include <utility>
#include "../../include/rfinv_b200.h"

#define RFINV_MAX_TRC 16     // traces per model (kernel parameter arrays)
#define RFINV_MAX_K 64       // k_max upper bound: fixed per-chain layer storage
#define RFINV_MAX_LAY (RFINV_MAX_K + 2)
#define RFINV_MAX_QF_TILES 64   // nsmp_pad / 64 with nsmp <= nfft <= 4096

#define RFINV_PI 3.1415926535897931  // src/forward.f90:33

// Immutable per-handle constants, passed to kernels by value (the reference's module globals).
struct DevConfig {
  int ntrc, nfft, nh, nsmp;
  int log2n;                    // log2 of fft_len
  // Transform lengths.  nfft a power of two: the shared-memory FFT runs on nfft points directly (fft_general = 0,
  // nfft_p2 = fft_len = nfft).  Any other length (FFTW accepts any, src/fftw.f90:43-45): threads and bin groups are laid
  // out for nfft_p2 = the next power of two (bins beyond nfft/2 are masked) and the transform is Bluestein's chirp-z
  // convolution on fft_len = 2 nfft_p2 points (forward.cu, bluestein_inverse).
  int fft_general, nfft_p2, fft_len;
  int deconv_mode, vp_mode, k_min, k_max, prior_mode, nref, ray_common;
  int nsmp_pad;                 // nsmp rounded up to the likelihood tile (64)
  double bdep;                  // receiver depth below the surface / sea floor (0 = at the surface)
  double delta, t_start, sdep, z_ref_min, dz_ref, z_min, z_max, h_min;
  double vp_min, vp_max, vs_min, vs_max, vpvs_min, vpvs_max;
  double domg;                  // 2 pi / (nfft * delta), src/forward.f90:241
  double rayp[RFINV_MAX_TRC];
  int ipha[RFINV_MAX_TRC];
  int jbins[RFINV_MAX_TRC];     // frequency-bin groups (of blockDim bins each) of forward_kernel that carry signal for the trace
  int jb_max;                   // largest jbins[]: picks the kernel variant
  const double* flt;            // [ntrc][nh]   Gaussian filter, src/forward.f90:95-119
  const double2* tw;            // [fft_len]    exp(+2 pi i m / fft_len)
  const double2* twq;           // fft_general: the per-stage twiddle tables of the radix-8 stages for fft_len points (layout of
                                // fill_fft_twiddles, forward.cu), read from global memory / L1 instead of a shared-memory copy
  const double2* chirp;         // [nfft]       fft_general: exp(+i pi m^2 / nfft)
  const double2* chirp_b;       // [fft_len]    fft_general: FFT_fft_len(conj(chirp) wrapped around fft_len) / fft_len
  const double* obs;            // [ntrc][nsmp]
  const double* vp_ref;         // [nref]
  const double* vs_ref;         // [nref]
  const double* r_inv;          // [ntrc][nsmp_pad][nsmp_pad] zero padded, symmetric
  // factor R^-1 = W W^T of the traces whose R^-1 is positive semi-definite of low rank (0 = use the dense form):
  const double* w_fac;          // [ntrc][qf_wrows][nsmp_pad]: row e = sqrt(lambda_e) * eigenvector e, zero padded
  int qf_rank[RFINV_MAX_TRC];   // kept eigenpairs per trace, 0 = dense
  int qf_split[RFINV_MAX_TRC];  // 1: split form -- the misfit row holds (s | a) = (m_i + m_{S-1-i} | m_i - m_{S-1-i}) in its two
                                // halves [0, nsmp_pad/2) and [nsmp_pad/2, nsmp_pad); factor rows 0.. act on s, rows 64*ceil(rank_s/64).. on a
  int qf_rank_s[RFINV_MAX_TRC]; // split form: eigenpairs of the symmetric block (the antisymmetric block has qf_rank - qf_rank_s)
  int qf_tiles[RFINV_MAX_TRC];  // 64-column work items per (64 chains, trace): nsmp_pad/64 when dense, ceil(rank/64), or
                                // ceil(rank_s/64) + ceil(rank_a/64) in the split form
  int qf_tiles_max, qf_wrows;
  int qf_order[RFINV_MAX_QF_TILES];   // hand-out order of the column tiles inside a scheduling chunk (most expensive first)
};

// Chain-fastest (structure-of-arrays) model batch in HBM.
struct ModelBatch {
  int C;                        // number of models
  const int* k;                 // [C]
  const double* z;              // [k_max-1][C]
  const double* dvp;            // [k_max][C]
  const double* dvs;            // [k_max][C]
  const double* sig;            // [ntrc][C]
  const int* active;            // optional list of model indices to evaluate (nullptr = all)
  int n_active;                 // length of `active` (upper bound when n_active_dev is set)
  const int* n_active_dev;      // optional: actual length of `active`, resident on device (grids are sized by n_active)
  // Host-layout batch (rfinv_eval_batch): z / dvp / dvs as the caller holds them, chain slowest -- z[c*(k_max-1) + i],
  // dvp / dvs[c*k_max + i] -- so the upload is a plain copy.  (sig stays chain-fastest: only loglik_kernel reads it.)
  int chain_major = 0;
};

// Fortran NINT (round half away from zero)
__host__ __device__ __forceinline__ int f_nint(double x) {
  return x >= 0.0 ? (int)floor(x + 0.5) : -(int)floor(-x + 0.5);
}

// src/model.f90:298-314 -- Brocher (2005) with the reference's float32 coefficients.  Written with
// explicit round-to-nearest mul/add so no FMA contraction changes the bits (the top-layer validity test
// and the densities in mcmc_out depend on it).
__device__ __forceinline__ double vp_to_rho(double a1) {
  double a2 = __dmul_rn(a1, a1), a3 = __dmul_rn(a2, a1), a4 = __dmul_rn(a3, a1), a5 = __dmul_rn(a4, a1);
  double p = __dmul_rn((double)1.6612f, a1);
  p = __dsub_rn(p, __dmul_rn((double)0.4721f, a2));
  p = __dadd_rn(p, __dmul_rn((double)0.0671f, a3));
  p = __dsub_rn(p, __dmul_rn((double)0.0043f, a4));
  p = __dadd_rn(p, __dmul_rn((double)0.000106f, a5));
  return p;
}

// One layer of format_model (src/model.f90:209-283): reference velocity lookup at the layer's mid depth.
// Returns false when the layer violates the velocity bounds (src/model.f90:219-224).
__device__ __forceinline__ bool layer_velocity(const DevConfig& cfg, double zc, double d_vs, double d_vp, double& alpha,
                                               double& beta) {
  int iz = f_nint(__ddiv_rn(__dsub_rn(zc, cfg.z_ref_min), cfg.dz_ref)) + 1;
  iz = iz < 1 ? 1 : (iz > cfg.nref ? cfg.nref : iz);  // the reference would index out of bounds
  beta = __dadd_rn(cfg.vs_ref[iz - 1], d_vs);
  alpha = cfg.vp_mode == 1 ? __dadd_rn(cfg.vp_ref[iz - 1], d_vp) : cfg.vp_ref[iz - 1];
  double ratio = __ddiv_rn(alpha, beta);
  return !(alpha < cfg.vp_min || alpha > cfg.vp_max || beta < cfg.vs_min || beta > cfg.vs_max ||
           ratio < cfg.vpvs_min || ratio > cfg.vpvs_max);
}

#define RFINV_CUDA_CHECK(expr)                                                        \
  do {                                                                                \
    cudaError_t e__ = (expr);                                                         \
    if (e__ != cudaSuccess) {                                                         \
      rfinv_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); \
      return RFINV_ERR_CUDA;                                                          \
    }                                                                                 \
  } while (0)

void rfinv_set_error(const char* fmt, ...);

// cudaFuncAttributeMaxDynamicSharedMemorySize of `kernel` on the current device raised to at least `bytes`, never lowered.  The
// attribute is process-wide per kernel while the size a launch needs depends on the handle's shape (nfft, k_max, ntrc, nchains):
// a handle of another shape that set a smaller value would invalidate the launches another handle has captured in a graph.
inline cudaError_t rfinv_raise_smem_limit(const void* kernel, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, size_t> limit;   // (device, kernel) -> largest value set
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  size_t& cur = limit[{dev, kernel}];
  if (bytes <= cur) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) cur = bytes;
  return e;
}

// Programmatic dependent launch (sm_90+): a kernel launched with rfinv_launch_pdl may start while the kernel before it on the
// stream is still draining -- its CTAs take the SM slots the predecessor's last CTAs free, run their prologue, and block in
// pdl_wait() until the predecessor has completed and its writes are visible.  The predecessor calls pdl_trigger() early
// (a kernel that never does releases its dependents when it exits).  Opt-in (RFINV_PDL=1): measured slower, see capi.cu.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
int rfinv_pdl_mode();   // bit 0: prep_kernel -> forward_kernel edge, bit 1: forward_kernel -> quadform_kernel edge
template <typename... KArgs, typename... Args>
cudaError_t rfinv_launch_pdl(int edge_bit, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = (rfinv_pdl_mode() & edge_bit) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// kernel launchers (forward.cu, likelihood.cu); all asynchronous on `stream`
struct EvalOutputs {
  double* misfit;     // [ntrc][C][nsmp_pad]  rft(1:nsmp) - obs, zero padded          (required)
  double* rft_smp;    // [ntrc][C][nsmp]      first nsmp samples of the RF (optional)
  double* rft_smp_alt;  // second buffer of the same shape: model c writes to (slot[c] ^ slot_invert) ? alt : rft_smp
  const uint8_t* slot;  // optional, with rft_smp_alt
  int slot_invert;
  double* rft_full;   // [C][ntrc][nfft]      complete RF, the reference's prop_rft (optional)
  uint8_t* is_valid;  // [C]                  format_model's flag (optional)
};
// prep_kernel + forward_kernel.  scratch: rfinv_forward_scratch_doubles(cfg, n_models) doubles in HBM
size_t rfinv_forward_scratch_doubles(const DevConfig& cfg, long long n_models);
int rfinv_launch_forward(const DevConfig& cfg, const ModelBatch& mb, const EvalOutputs& out, double* scratch,
                         cudaStream_t stream, int* n_kernels = nullptr,    // n_kernels: kernels launched (optional)
                         bool prep_done = false);                          // prep_done: rfinv_launch_prep already covered the batch
// prep_kernel alone for the models [m_begin, m_begin + m_count) of the batch (index into `active` when that is set): the
// host path launches it piece by piece behind the pieces of the upload
int rfinv_launch_prep(const DevConfig& cfg, const ModelBatch& mb, uint8_t* is_valid, double* scratch, cudaStream_t stream,
                      int m_begin, int m_count);
// bins per thread of forward_kernel for the full band (threads per CTA = nfft_p2/2 / this); nfft_p2 = DevConfig::nfft_p2
int rfinv_forward_bins_per_thread(int nfft_p2);
inline int rfinv_forward_threads(const DevConfig& cfg) { return (cfg.nfft_p2 / 2) / rfinv_forward_bins_per_thread(cfg.nfft_p2); }
// phi[ntrc][C] = m^T R^-1 m per trace and model.  partial / counters: scratch sized by the two functions below, the
// counters zeroed at allocation
size_t rfinv_quadform_partial_doubles(const DevConfig& cfg, int C);
size_t rfinv_quadform_counter_ints(const DevConfig& cfg, int C);
// sig / logl (optional, chain fastest): logl[c] = sum_t -0.5 phi/sig^2 - nsmp log(sig) is written by the same kernel
int rfinv_launch_quadform(const DevConfig& cfg, int C, const double* misfit, double* phi, double* partial, int* counters,
                          const int* active, int n_active, const int* n_active_dev, cudaStream_t stream,
                          const double* sig = nullptr, double* logl = nullptr);
// logl[c] = sum_t -0.5 phi/sig^2 - nsmp log(sig)   (src/likelihood.f90:94-96)
int rfinv_launch_loglik(const DevConfig& cfg, int C, const double* phi, const double* sig, double* logl,
                        cudaStream_t stream);
int rfinv_launch_format_model(const DevConfig& cfg, const ModelBatch& mb, int* nlay, double* alpha, double* beta,
                              double* rho, double* h, uint8_t* is_valid, cudaStream_t stream);
// y = c2r(r2c(x) * flt(:, trace_of[series])) for n_series real series of nfft samples (make_syn's noise shaping)
int rfinv_launch_filter_traces(const DevConfig& cfg, int n_series, const double* in, const int* trace_of, double* out,
                               cudaStream_t stream);
