// C-ABI of the evaluator (include/rfinv_b200.h): handle life cycle, configuration upload, batched
// calc_likelihood with host or device buffers.  No torch types, no CPU compute fallback: every entry
// point that evaluates models launches the CUDA kernels or fails with RFINV_ERR_CUDA.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <vector>
#include <algorithm>
#include "rfinv_handle.h"

static thread_local char g_err[1024] = "";

int rfinv_pdl_mode() {
  // Programmatic dependent launch per kernel boundary, measured on B200 (target shape, 16 384 chains, 30 interleaved rounds):
  //   none 1.2933 / 1.2953 ms per step;  prep -> forward only 1.3076 (forward_kernel's early CTAs cost prep_kernel's last wave
  //   more than the hidden launch gains);  forward -> quadform only 1.2913 / 1.2933 (quadform_kernel's CTAs take the slots
  //   forward_kernel's CTAs free one by one);  both 1.3056.  Default: the forward -> quadform edge.
  // RFINV_PDL: bit 0 = the prep_kernel -> forward_kernel edge, bit 1 = the forward_kernel -> quadform_kernel edge.
  static const int mode = getenv("RFINV_PDL") ? atoi(getenv("RFINV_PDL")) : 2;
  return mode;
}

int rfinv_arith_switches() {
  auto on = [](const char* name) { return getenv(name) && atoi(getenv(name)) != 0; };
  static const int bits = (on("RFINV_FULL_BAND") ? 1 : 0) | (on("RFINV_QF_DENSE") ? 2 : 0) | (on("RFINV_QF_NOSPLIT") ? 4 : 0);
  return bits;
}

void rfinv_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

namespace {

// ---- host-side init services ------------------------------------------------------------------
// init_filter, src/forward.f90:95-119 (same operation order)
void build_filter(const rfinv_config& c, std::vector<double>& flt) {
  const int nh = c.nfft / 2 + 1;
  flt.resize((size_t)c.ntrc * nh);
  const double df = 1.0 / (c.delta * c.nfft);
  for (int t = 0; t < c.ntrc; ++t) {
    const double fac_norm = c.nfft * c.a_gus[t] * c.delta / std::sqrt(RFINV_PI);
    for (int i = 0; i < nh; ++i) {
      const double omega = i * 2.0 * RFINV_PI * df;
      const double q = omega / (2.0 * c.a_gus[t]);
      flt[(size_t)t * nh + i] = std::exp(-(q * q)) / fac_norm;
    }
  }
}

// Band limit of the forward kernel.  The Gaussian filter (src/forward.f90:95-119) multiplies every spectrum before the
// inverse FFT; bins whose total weight is below 2^-52 of the filter's mass change no bit of the fp64 trace and are not
// propagated.  forward_kernel computes bins in groups of `nthr` (thread t owns bins t + m*nthr): jbins[t] = number of
// groups kept for trace t, rounded up to a value the kernel is instantiated for.  Full band when the water-level
// deconvolution is on (its water level is the maximum over all bins) or RFINV_FULL_BAND=1.
void band_limits(DevConfig& d, const std::vector<double>& flt) {
  const int nh = d.nh, jfull = rfinv_forward_bins_per_thread(d.nfft_p2), nthr = (d.nfft_p2 / 2) / jfull;
  const bool full_band = (rfinv_arith_switches() & 1) != 0;
  const int allowed[6] = {1, 2, 3, 4, 6, 8};
  d.jb_max = 1;
  for (int t = 0; t < d.ntrc; ++t) {
    int g = jfull;
    if (!full_band && d.deconv_mode == 0) {
      const double* f = flt.data() + (size_t)t * nh;
      double total = 0.0;
      for (int j = 0; j < nh; ++j) total += f[j];
      double tail = 0.0;
      g = jfull;
      // largest cut (in whole groups) whose tail -- bins g*nthr .. nh-1 -- stays below 2^-52 of the total
      for (int cand = jfull - 1; cand >= 1; --cand) {
        tail = 0.0;
        for (int j = cand * nthr; j < nh; ++j) tail += f[j];
        if (tail <= total * 2.220446049250313e-16) g = cand; else break;
      }
    }
    int r = jfull;
    for (int i = 5; i >= 0; --i) if (allowed[i] >= g && allowed[i] <= jfull) r = allowed[i];
    d.jbins[t] = r;
    if (r > d.jb_max) d.jb_max = r;
  }
  if (d.ray_common) for (int t = 0; t < d.ntrc; ++t) d.jbins[t] = d.jb_max;   // one propagation serves every trace
}

// exp(+2 pi i m / n), exact symmetries of the octants
void build_twiddles(int n, std::vector<double2>& tw) {
  tw.resize(n);
  for (int m = 0; m < n; ++m) {
    const double ang = 2.0 * RFINV_PI * (double)m / (double)n;
    tw[m] = make_double2(std::cos(ang), std::sin(ang));
  }
  tw[0] = make_double2(1.0, 0.0);
  if (n % 4 == 0) { tw[n / 4] = make_double2(0.0, 1.0); tw[n / 2] = make_double2(-1.0, 0.0); tw[3 * n / 4] = make_double2(0.0, -1.0); }
}

// Bluestein tables for a transform length n that is not a power of two (forward.cu, bluestein_inverse): the chirp
// w[m] = exp(+i pi m^2 / n) -- m^2 reduced mod 2n in integers, so the angle stays in [0, 2 pi) -- and
// B = FFT_M(b) / M with b[m mod M] = conj(w[m]) for |m| < n, zero elsewhere (M >= 2n - 1 a power of two).  B is computed
// in long double by a plain radix-2 transform: it multiplies every spectrum, so it should carry no error of its own.
void build_chirp(int n, int M, std::vector<double2>& chirp, std::vector<double2>& chirp_b) {
  const long double pi = 3.14159265358979323846264338327950288L;
  std::vector<long double> wr(n), wi(n);
  chirp.resize(n);
  for (long long m = 0; m < n; ++m) {
    const long long r = (m * m) % (2LL * n);
    const long double ang = pi * (long double)r / (long double)n;
    wr[m] = cosl(ang); wi[m] = sinl(ang);
    chirp[m] = make_double2((double)wr[m], (double)wi[m]);
  }
  std::vector<long double> br(M, 0.0L), bi(M, 0.0L);
  for (int m = 0; m < n; ++m) {
    br[m] = wr[m]; bi[m] = -wi[m];
    if (m) { br[M - m] = wr[m]; bi[M - m] = -wi[m]; }
  }
  // forward transform (sign -), decimation in time
  int bits = 0; while ((1 << bits) < M) ++bits;
  for (int i = 0; i < M; ++i) {
    int r = 0;
    for (int b = 0; b < bits; ++b) if (i & (1 << b)) r |= 1 << (bits - 1 - b);
    if (r > i) { std::swap(br[i], br[r]); std::swap(bi[i], bi[r]); }
  }
  for (int len = 2; len <= M; len <<= 1) {
    const int hl = len / 2;
    for (int j = 0; j < hl; ++j) {
      const long double ang = -2.0L * pi * (long double)j / (long double)len;
      const long double c = cosl(ang), s_ = sinl(ang);
      for (int s0 = 0; s0 < M; s0 += len) {
        const long double xr = br[s0 + j + hl] * c - bi[s0 + j + hl] * s_, xi = br[s0 + j + hl] * s_ + bi[s0 + j + hl] * c;
        br[s0 + j + hl] = br[s0 + j] - xr; bi[s0 + j + hl] = bi[s0 + j] - xi;
        br[s0 + j] += xr; bi[s0 + j] += xi;
      }
    }
  }
  chirp_b.resize(M);
  for (int m = 0; m < M; ++m) chirp_b[m] = make_double2((double)(br[m] / M), (double)(bi[m] / M));
}

// Eigen-decomposition of a symmetric matrix (row-major n x n): A = V diag(w) V^T, v[i*n + e] = component i of
// eigenvector e.  Householder tridiagonalisation followed by the implicit QL algorithm (the classical EISPACK
// tred2 / tql2 pair, O(n^3) with a small constant: ~1 s at n = 1000).  Used (i) for init_r_inv when the caller passes
// no R^-1 -- R = r^((i-j)^2) is symmetric positive semi-definite, so its SVD (what the reference asks LAPACK dgesvd for,
// src/likelihood.f90:197-205) is its eigen-decomposition -- and (ii) to factor R^-1 = W W^T for the quadratic form.
void sym_eigh(std::vector<double>& a, int n, std::vector<double>& w, std::vector<double>& v) {
  std::vector<double> d(n), e(n);
  auto V = [&](int i, int j) -> double& { return a[(size_t)i * n + j]; };
  for (int j = 0; j < n; ++j) d[j] = V(n - 1, j);
  for (int i = n - 1; i > 0; --i) {   // Householder reduction to tridiagonal form
    double scale = 0.0, h = 0.0;
    for (int k = 0; k < i; ++k) scale += std::fabs(d[k]);
    if (scale == 0.0) {
      e[i] = d[i - 1];
      for (int j = 0; j < i; ++j) { d[j] = V(i - 1, j); V(i, j) = 0.0; V(j, i) = 0.0; }
    } else {
      for (int k = 0; k < i; ++k) { d[k] /= scale; h += d[k] * d[k]; }
      double f = d[i - 1], g = std::sqrt(h);
      if (f > 0) g = -g;
      e[i] = scale * g; h -= f * g; d[i - 1] = f - g;
      for (int j = 0; j < i; ++j) e[j] = 0.0;
      for (int j = 0; j < i; ++j) {
        f = d[j]; V(j, i) = f; g = e[j] + V(j, j) * f;
        for (int k = j + 1; k <= i - 1; ++k) { g += V(k, j) * d[k]; e[k] += V(k, j) * f; }
        e[j] = g;
      }
      f = 0.0;
      for (int j = 0; j < i; ++j) { e[j] /= h; f += e[j] * d[j]; }
      const double hh = f / (h + h);
      for (int j = 0; j < i; ++j) e[j] -= hh * d[j];
      for (int j = 0; j < i; ++j) {
        f = d[j]; g = e[j];
        for (int k = j; k <= i - 1; ++k) V(k, j) -= (f * e[k] + g * d[k]);
        d[j] = V(i - 1, j); V(i, j) = 0.0;
      }
    }
    d[i] = h;
  }
  for (int i = 0; i < n - 1; ++i) {   // accumulate the transformations
    V(n - 1, i) = V(i, i); V(i, i) = 1.0;
    const double h = d[i + 1];
    if (h != 0.0) {
      for (int k = 0; k <= i; ++k) d[k] = V(k, i + 1) / h;
      for (int j = 0; j <= i; ++j) {
        double g = 0.0;
        for (int k = 0; k <= i; ++k) g += V(k, i + 1) * V(k, j);
        for (int k = 0; k <= i; ++k) V(k, j) -= g * d[k];
      }
    }
    for (int k = 0; k <= i; ++k) V(k, i + 1) = 0.0;
  }
  for (int j = 0; j < n; ++j) { d[j] = V(n - 1, j); V(n - 1, j) = 0.0; }
  V(n - 1, n - 1) = 1.0; e[0] = 0.0;
  // implicit QL on the tridiagonal matrix; eigenvectors kept transposed (z[e*n + i]) so the plane rotations stream
  std::vector<double> z((size_t)n * n);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) z[(size_t)j * n + i] = V(i, j);
  for (int i = 1; i < n; ++i) e[i - 1] = e[i];
  e[n - 1] = 0.0;
  double f = 0.0, tst1 = 0.0;
  const double eps = 2.220446049250313e-16;
  for (int l = 0; l < n; ++l) {
    tst1 = std::max(tst1, std::fabs(d[l]) + std::fabs(e[l]));
    int m = l;
    while (m < n) { if (std::fabs(e[m]) <= eps * tst1) break; ++m; }
    if (m > l) {
      int iter = 0;
      do {
        ++iter;
        double g = d[l], p = (d[l + 1] - g) / (2.0 * e[l]), r = std::hypot(p, 1.0);
        if (p < 0) r = -r;
        d[l] = e[l] / (p + r); d[l + 1] = e[l] * (p + r);
        const double dl1 = d[l + 1];
        double h = g - d[l];
        for (int i = l + 2; i < n; ++i) d[i] -= h;
        f += h;
        p = d[m];
        double c = 1.0, c2 = c, c3 = c, s = 0.0, s2 = 0.0;
        const double el1 = e[l + 1];
        for (int i = m - 1; i >= l; --i) {
          c3 = c2; c2 = c; s2 = s;
          g = c * e[i]; h = c * p; r = std::hypot(p, e[i]);
          e[i + 1] = s * r; s = e[i] / r; c = p / r; p = c * d[i] - s * g;
          d[i + 1] = h + s * (c * g + s * d[i]);
          double* zi = &z[(size_t)i * n];
          double* zi1 = &z[(size_t)(i + 1) * n];
          for (int k = 0; k < n; ++k) { const double hk = zi1[k]; zi1[k] = s * zi[k] + c * hk; zi[k] = c * zi[k] - s * hk; }
        }
        p = -s * s2 * c3 * el1 * e[l] / dl1; e[l] = s * p; d[l] = c * p;
      } while (std::fabs(e[l]) > eps * tst1 && iter < 200);
    }
    d[l] += f; e[l] = 0.0;
  }
  w.assign(d.begin(), d.end());
  v.resize((size_t)n * n);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) v[(size_t)i * n + j] = z[(size_t)j * n + i];
}

// init_r_inv, src/likelihood.f90:168-241: R^-1 = sum_{s_i > 1e-3} v_i v_i^T / s_i
void build_r_inv(const rfinv_config& c, std::vector<double>& rinv) {
  const int S = c.nsmp;
  rinv.assign((size_t)c.ntrc * S * S, 0.0);
  std::vector<double> a, w, v;
  for (int t = 0; t < c.ntrc; ++t) {
    bool same = false;  // traces with the same Gaussian width share R^-1
    for (int u = 0; u < t; ++u)
      if (c.a_gus[u] == c.a_gus[t]) {
        std::memcpy(&rinv[(size_t)t * S * S], &rinv[(size_t)u * S * S], sizeof(double) * (size_t)S * S);
        same = true;
        break;
      }
    if (same) continue;
    const double r = std::exp(-(c.a_gus[t] * c.a_gus[t]) * (c.delta * c.delta));
    a.resize((size_t)S * S);
    for (int i = 0; i < S; ++i)
      for (int j = 0; j < S; ++j) a[(size_t)i * S + j] = std::pow(r, (double)((i - j) * (i - j)));
    sym_eigh(a, S, w, v);
    double* out = &rinv[(size_t)t * S * S];
    for (int e = 0; e < S; ++e) {
      if (!(w[e] > 1.0e-3)) continue;
      const double inv = 1.0 / w[e];
      for (int i = 0; i < S; ++i) {
        const double vi = v[(size_t)i * S + e] * inv;
        for (int j = 0; j < S; ++j) out[(size_t)i * S + j] += vi * v[(size_t)j * S + e];
      }
    }
  }
}

template <typename T>
int upload(const std::vector<T>& h, T** d) {
  RFINV_CUDA_CHECK(cudaMalloc((void**)d, sizeof(T) * std::max<size_t>(h.size(), 1)));
  if (!h.empty()) RFINV_CUDA_CHECK(cudaMemcpy(*d, h.data(), sizeof(T) * h.size(), cudaMemcpyHostToDevice));
  return RFINV_OK;
}

int check_config(const rfinv_config* c) {
  if (!c) { rfinv_set_error("config is NULL"); return RFINV_ERR_ARG; }
  if (c->ntrc < 1 || c->ntrc > RFINV_MAX_TRC) { rfinv_set_error("ntrc must be in [1,%d]", RFINV_MAX_TRC); return RFINV_ERR_ARG; }
  // powers of two run the shared-memory FFT directly; any other length goes through Bluestein's convolution on twice the
  // next power of two, which must still fit the shared memory of an SM
  if (c->nfft < 64 || c->nfft > 4096 || ((c->nfft & (c->nfft - 1)) && c->nfft > 2048)) {
    rfinv_set_error("nfft=%d unsupported: the shared-memory FFT takes powers of two in [64,4096] and any other length in [64,2048]", c->nfft);
    return RFINV_ERR_ARG;
  }
  if (c->nsmp < 1 || c->nsmp > c->nfft) { rfinv_set_error("nsmp must be in [1,nfft]"); return RFINV_ERR_ARG; }
  if (c->deconv_mode != 0 && c->deconv_mode != 1) { rfinv_set_error("deconv_mode must be either 0 or 1"); return RFINV_ERR_ARG; }
  if (c->vp_mode != 0 && c->vp_mode != 1) { rfinv_set_error("vp_mode should be 0 or 1"); return RFINV_ERR_ARG; }
  if (c->k_max < 2 || c->k_max > RFINV_MAX_K || c->k_min < 1 || c->k_min >= c->k_max) {
    rfinv_set_error("need 1 <= k_min < k_max <= %d", RFINV_MAX_K);
    return RFINV_ERR_ARG;
  }
  if (!c->rayps || !c->a_gus || !c->ipha || !c->obs || !c->vp_ref || !c->vs_ref || !c->sig_min || !c->sig_max || c->nref < 1) {
    rfinv_set_error("rayps/a_gus/ipha/obs/vp_ref/vs_ref/sig_min/sig_max must be set");
    return RFINV_ERR_ARG;
  }
  for (int t = 0; t < c->ntrc; ++t)
    if (c->ipha[t] != 1 && c->ipha[t] != -1) { rfinv_set_error("ipha must be 1 or -1"); return RFINV_ERR_ARG; }
  if (c->bdep < 0.0) { rfinv_set_error("BOREHOLE_DEP must be positive"); return RFINV_ERR_ARG; }
  if (!(c->delta > 0.0) || !(c->dz_ref > 0.0)) { rfinv_set_error("delta and dz_ref must be positive"); return RFINV_ERR_ARG; }
  return RFINV_OK;
}

// chain-major host layout -> chain-fastest device layout for the n models from c0 on: out[i*C + c0 + c] = in[c*len + i]
__global__ void to_soa_kernel(const double* __restrict__ in, double* __restrict__ out, int C, int c0, int n, int len) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)n * len) return;
  const int c = (int)(idx % n), i = (int)(idx / n);
  out[(size_t)i * C + c0 + c] = in[(size_t)c * len + i];
}
// chain-fastest device layout -> chain-major host layout: out[c*len + i] = in[i*C + c]
__global__ void from_soa_kernel(const double* __restrict__ in, double* __restrict__ out, int C, int len) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)C * len) return;
  const int i = (int)(idx % len), c = (int)(idx / len);
  out[idx] = in[(size_t)i * C + c];
}
// Large uploads (rfinv_eval_batch) go up in RFINV_UPLOAD_PIECES pieces of at least UPLOAD_PIECE_MIN models: measured at
// 16 384 models, pieces of 1024 / 2048 / 4096 / 8192 give 9.3 / 9.9 / 10.2 / 9.8 M evals/s end to end (every copy costs a few
// microseconds of set-up; the first piece is exposed).
constexpr int UPLOAD_PIECE_MIN = 2048;
static int upload_pieces() {   // RFINV_UPLOAD_PIECES_N=1..4 (tuning)
  static const int n = getenv("RFINV_UPLOAD_PIECES_N") ? std::min(RFINV_UPLOAD_PIECES, std::max(1, atoi(getenv("RFINV_UPLOAD_PIECES_N")))) : RFINV_UPLOAD_PIECES;
  return n;
}
static int upload_piece(int C) { return std::max(UPLOAD_PIECE_MIN, ((C / upload_pieces() + 255) / 256) * 256); }

}  // namespace

int EvalWorkspace::grow(const DevConfig& dc, const rfinv_config& cfg, int device, int C) {
  if (C <= cap) return RFINV_OK;
  release();
  const int km = cfg.k_max, T = cfg.ntrc;
  const size_t Cz = (size_t)C;
  RFINV_CUDA_CHECK(cudaSetDevice(device));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_k, sizeof(int) * Cz));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_z, sizeof(double) * Cz * (km - 1)));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_dvp, sizeof(double) * Cz * km));
  RFINV_CUDA_CHECK(cudaMemset(d_dvp, 0, sizeof(double) * Cz * km));   // stays zero with vp_mode = 0 (never uploaded, never used)
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_dvs, sizeof(double) * Cz * km));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_sig, sizeof(double) * Cz * T));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_stage, sizeof(double) * Cz * (size_t)std::max(km, T)));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_misfit, sizeof(double) * Cz * T * dc.nsmp_pad));
  RFINV_CUDA_CHECK(cudaMemset(d_misfit, 0, sizeof(double) * Cz * T * dc.nsmp_pad));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_phi, sizeof(double) * Cz * T));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_logl, sizeof(double) * Cz));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_valid, Cz));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_scratch, sizeof(double) * rfinv_forward_scratch_doubles(dc, C)));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_qpart, sizeof(double) * rfinv_quadform_partial_doubles(dc, C)));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_qcnt, sizeof(int) * rfinv_quadform_counter_ints(dc, C)));
  RFINV_CUDA_CHECK(cudaMemset(d_qcnt, 0, sizeof(int) * rfinv_quadform_counter_ints(dc, C)));
  cap = C;
  return RFINV_OK;
}

void EvalWorkspace::release() {
  cudaFree(d_k); cudaFree(d_z); cudaFree(d_dvp); cudaFree(d_dvs); cudaFree(d_sig); cudaFree(d_stage);
  cudaFree(d_misfit); cudaFree(d_phi); cudaFree(d_logl); cudaFree(d_valid); cudaFree(d_rft_full); cudaFree(d_scratch); cudaFree(d_qpart); cudaFree(d_qcnt);
  d_qpart = nullptr; d_qcnt = nullptr;
  d_k = nullptr; d_z = d_dvp = d_dvs = d_sig = d_stage = d_misfit = d_phi = d_logl = d_rft_full = d_scratch = nullptr;
  d_valid = nullptr;
  cap = 0; cap_rft_full = 0;
}

int rfinv_handle::eval_device(int C, const int* k, const double* z, const double* dvp, const double* dvs,
                              const double* sig, double* logl, double* rft_smp, double* rft_full, uint8_t* is_valid,
                              const int* active, int n_active, const ModelBatch* layout, EvalWorkspace* w, cudaStream_t s,
                              bool prep_done, cudaEvent_t before_quadform) {
  if (!w) w = this;
  if (!s) s = stream;
  // misfit scratch is sized by capacity; its [t][c] stride uses the C of this call
  ModelBatch mb;
  if (layout) mb = *layout;
  mb.C = C; mb.k = k; mb.z = z; mb.dvp = dvp; mb.dvs = dvs; mb.sig = sig; mb.active = active; mb.n_active = n_active; mb.n_active_dev = nullptr;
  EvalOutputs out;
  out.misfit = w->d_misfit; out.rft_smp = rft_smp; out.rft_smp_alt = nullptr; out.slot = nullptr; out.slot_invert = 0;
  out.rft_full = rft_full; out.is_valid = is_valid;
  int st;
  launches = 0;
  const bool timed = timing && w == this;
  if (timed) cudaEventRecord(ev[0], s);
  int n_fwd = 0;
  if ((st = rfinv_launch_forward(dc, mb, out, w->d_scratch, s, &n_fwd, prep_done)) != RFINV_OK) return st;
  launches += n_fwd;
  if (timed) cudaEventRecord(ev[1], s);
  if (before_quadform) RFINV_CUDA_CHECK(cudaStreamWaitEvent(s, before_quadform, 0));
  // logL leaves the same kernel (its last CTA per block of 64 chains sums the traces): no separate loglik_kernel launch
  if ((st = rfinv_launch_quadform(dc, C, w->d_misfit, w->d_phi, w->d_qpart, w->d_qcnt, active, n_active, nullptr, s, logl ? sig : nullptr, logl)) != RFINV_OK) return st;
  ++launches;
  if (timed) { cudaEventRecord(ev[2], s); cudaEventRecord(ev[3], s); }
  return RFINV_OK;
}

extern "C" {

int32_t rfinv_abi_version(void) { return RFINV_ABI_VERSION; }
const char* rfinv_last_error(void) { return g_err; }

int32_t rfinv_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    rfinv_set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
    return -RFINV_ERR_CUDA;
  }
  return n;
}

int32_t rfinv_create(const rfinv_config* cfg, int32_t device, rfinv_handle** out) {
  if (!out) { rfinv_set_error("out is NULL"); return RFINV_ERR_ARG; }
  *out = nullptr;
  int st = check_config(cfg);
  if (st != RFINV_OK) return st;
  int ndev = 0;
  RFINV_CUDA_CHECK(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) {
    rfinv_set_error("device %d not available (%d CUDA devices visible); this library has no CPU path", device, ndev);
    return RFINV_ERR_CUDA;
  }
  RFINV_CUDA_CHECK(cudaSetDevice(device));
  rfinv_handle* h = new rfinv_handle();
  h->device = device;
  // deep copy of the configuration
  h->cfg = *cfg;
  const int T = cfg->ntrc, S = cfg->nsmp;
  h->h_rayps.assign(cfg->rayps, cfg->rayps + T);
  h->h_a_gus.assign(cfg->a_gus, cfg->a_gus + T);
  h->h_ipha.assign(cfg->ipha, cfg->ipha + T);
  h->h_obs.assign(cfg->obs, cfg->obs + (size_t)T * S);
  h->h_vp_ref.assign(cfg->vp_ref, cfg->vp_ref + cfg->nref);
  h->h_vs_ref.assign(cfg->vs_ref, cfg->vs_ref + cfg->nref);
  h->h_sig_min.assign(cfg->sig_min, cfg->sig_min + T);
  h->h_sig_max.assign(cfg->sig_max, cfg->sig_max + T);
  if (cfg->r_inv) h->h_r_inv.assign(cfg->r_inv, cfg->r_inv + (size_t)T * S * S);
  else build_r_inv(*cfg, h->h_r_inv);
  h->cfg.rayps = h->h_rayps.data(); h->cfg.a_gus = h->h_a_gus.data(); h->cfg.ipha = h->h_ipha.data();
  h->cfg.obs = h->h_obs.data(); h->cfg.vp_ref = h->h_vp_ref.data(); h->cfg.vs_ref = h->h_vs_ref.data();
  h->cfg.sig_min = h->h_sig_min.data(); h->cfg.sig_max = h->h_sig_max.data(); h->cfg.r_inv = h->h_r_inv.data();

  DevConfig& d = h->dc;
  std::memset(&d, 0, sizeof(d));
  d.ntrc = T; d.nfft = cfg->nfft; d.nh = cfg->nfft / 2 + 1; d.nsmp = S;
  d.nfft_p2 = 64; while (d.nfft_p2 < cfg->nfft) d.nfft_p2 <<= 1;
  d.fft_general = d.nfft_p2 != cfg->nfft;
  d.fft_len = d.fft_general ? 2 * d.nfft_p2 : cfg->nfft;
  d.log2n = 0; while ((1 << d.log2n) < d.fft_len) ++d.log2n;
  d.deconv_mode = cfg->deconv_mode; d.vp_mode = cfg->vp_mode; d.k_min = cfg->k_min; d.k_max = cfg->k_max;
  d.prior_mode = cfg->prior_mode; d.nref = cfg->nref;
  d.ray_common = 1;  // check_ray, src/forward.f90:59-76
  for (int t = 1; t < T; ++t)
    if (cfg->rayps[t] != cfg->rayps[0] || cfg->ipha[t] != cfg->ipha[0]) d.ray_common = 0;
  d.nsmp_pad = ((S + 63) / 64) * 64;
  d.delta = cfg->delta; d.t_start = cfg->t_start; d.sdep = cfg->sdep; d.bdep = cfg->bdep; d.z_ref_min = cfg->z_ref_min; d.dz_ref = cfg->dz_ref;
  d.z_min = cfg->z_min; d.z_max = cfg->z_max; d.h_min = cfg->h_min;
  d.vp_min = cfg->vp_min; d.vp_max = cfg->vp_max; d.vs_min = cfg->vs_min; d.vs_max = cfg->vs_max;
  d.vpvs_min = cfg->vpvs_min; d.vpvs_max = cfg->vpvs_max;
  d.domg = 2.0 * RFINV_PI / (cfg->nfft * cfg->delta);  // src/forward.f90:241
  for (int t = 0; t < T; ++t) { d.rayp[t] = cfg->rayps[t]; d.ipha[t] = cfg->ipha[t]; }

  std::vector<double> flt;
  build_filter(*cfg, flt);
  band_limits(d, flt);
  std::vector<double2> tw;
  build_twiddles(d.fft_len, tw);
  std::vector<double2> chirp, chirp_b;
  std::vector<double2> twq;
  if (d.fft_general) {
    build_chirp(cfg->nfft, d.fft_len, chirp, chirp_b);
    // per-stage twiddle tables of the radix-8 stages, [q - 1][offset] per stage (what fill_fft_twiddles builds in shared memory)
    for (int N = d.fft_len; N > 8; N >>= 3) {
      const int stride = N >> 3, tmul = d.fft_len / N;
      for (int i = 0; i < 7 * stride; ++i) { const int q = i / stride + 1, o = i - (q - 1) * stride; twq.push_back(tw[(size_t)q * o * tmul]); }
    }
  }
  // R^-1: symmetrised (the quadratic form only sees the symmetric part) and zero padded to the tile
  const int Sp = d.nsmp_pad;
  std::vector<double> rpad((size_t)T * Sp * Sp, 0.0);
  for (int t = 0; t < T; ++t)
    for (int i = 0; i < S; ++i)
      for (int j = 0; j < S; ++j)
        rpad[((size_t)t * Sp + i) * Sp + j] =
            0.5 * (h->h_r_inv[((size_t)t * S + i) * S + j] + h->h_r_inv[((size_t)t * S + j) * S + i]);
  // Factor form of the quadratic form: when the symmetrised R^-1 is positive semi-definite of rank r << S (it is, by
  // construction: a truncated pseudo-inverse, src/likelihood.f90:212-222), phi = m^T R^-1 m = |W^T m|^2 with
  // W = V_r diag(sqrt(lambda_r)) costs 2 S r flop instead of S^2 and sums non-negative terms only.  Eigenvalues below
  // 1e-12 of the largest are rounding residue of the construction (they change phi by < 1e-10 relative) and are
  // dropped; any eigenvalue below -1e-12 lambda_max, or a rank that does not pay, keeps the dense form for that trace.
  //
  // Split form.  R_ij = r^((i-j)^2) is a symmetric Toeplitz matrix, so R^-1 commutes with the exchange matrix J
  // (R^-1[i][j] = R^-1[S-1-i][S-1-j]) and its eigenvectors are symmetric or antisymmetric about the centre of the
  // window.  In the basis q_i^+- = (e_i +- e_{S-1-i})/sqrt2 (plus the centre sample when S is odd) R^-1 is block
  // diagonal: phi = s^T M+ s + a^T M- a with s_i = m_i + m_{S-1-i}, a_i = m_i - m_{S-1-i} (the 1/sqrt2 goes into the
  // factors), two quadratic forms of half the length -- half the flop of the factor form, and two half-size
  // eigenproblems at create.  Used when R^-1 passes the symmetry test (any R^-1 the reference can build does);
  // forward_kernel then writes (s | a) instead of m into the misfit rows (DevConfig::qf_split).
  std::vector<double> wfac;
  {
    const bool force_dense = (rfinv_arith_switches() & 2) != 0;
    const bool no_split = (rfinv_arith_switches() & 4) != 0;
    const int ntile_dense = Sp / 64;
    std::vector<std::vector<double>> Wt(T);      // per trace: [wrows_t][Sp], row = one column of W, K contiguous
    std::vector<int> wrows_t(T, 0);
    std::vector<double> a, w, v, a2, w2, v2;
    d.qf_tiles_max = 0;
    int wrows = 64;
    const double rs2 = 0.70710678118654752440;
    for (int t = 0; t < T; ++t) {
      d.qf_rank[t] = 0; d.qf_rank_s[t] = 0; d.qf_split[t] = 0;
      d.qf_tiles[t] = ntile_dense;
      const double* Rm = &rpad[(size_t)t * Sp * Sp];
      auto R = [&](int i, int j) { return Rm[(size_t)i * Sp + j]; };
      int same = -1;
      for (int u = 0; u < t && same < 0; ++u)
        if (std::memcmp(&rpad[(size_t)u * Sp * Sp], Rm, sizeof(double) * (size_t)Sp * Sp) == 0) same = u;
      if (force_dense) { /* keep dense */ }
      else if (same >= 0) {
        d.qf_rank[t] = d.qf_rank[same]; d.qf_rank_s[t] = d.qf_rank_s[same]; d.qf_split[t] = d.qf_split[same];
        d.qf_tiles[t] = d.qf_tiles[same]; Wt[t] = Wt[same]; wrows_t[t] = wrows_t[same];
      } else {
        double rmax = 0.0, asym = 0.0;
        for (int i = 0; i < S; ++i)
          for (int j = 0; j < S; ++j) {
            rmax = std::max(rmax, std::fabs(R(i, j)));
            asym = std::max(asym, std::fabs(R(i, j) - R(S - 1 - i, S - 1 - j)));
          }
        const int ha = S / 2, hs = S - ha;            // antisymmetric / symmetric subspace dimensions
        const bool split = !no_split && rmax > 0.0 && asym <= 1e-10 * rmax && hs <= Sp / 2;
        const double units_dense = 0.5 * ntile_dense * (ntile_dense + 1);
        auto tile_units = [&](int r) { return r / 64 + (r % 64 ? 0.4 : 0.0); };
        if (split) {
          // blocks of R^-1 in the orthonormal (+, -) basis; forward_kernel writes the unnormalised sums and differences, so
          // the 1/sqrt2 of the paired basis vectors goes into the rows of W below
          a.assign((size_t)hs * hs, 0.0); a2.assign((size_t)ha * ha, 0.0);
          for (int i = 0; i < ha; ++i)
            for (int j = 0; j < ha; ++j) {
              const int ir = S - 1 - i, jr = S - 1 - j;
              a[(size_t)i * hs + j] = 0.5 * ((R(i, j) + R(ir, jr)) + (R(i, jr) + R(ir, j)));
              a2[(size_t)i * ha + j] = 0.5 * ((R(i, j) + R(ir, jr)) - (R(i, jr) + R(ir, j)));
            }
          if (hs > ha) {                               // centre sample: a basis vector of its own in the + block
            const int c = ha;
            a[(size_t)c * hs + c] = R(c, c);
            for (int i = 0; i < ha; ++i) a[(size_t)i * hs + c] = a[(size_t)c * hs + i] = rs2 * (R(i, c) + R(S - 1 - i, c));
          }
          sym_eigh(a, hs, w, v);
          if (ha > 0) sym_eigh(a2, ha, w2, v2); else { w2.clear(); v2.clear(); }
          double lmax = 0.0, lmin = 0.0;
          for (double x : w) { lmax = std::max(lmax, x); lmin = std::min(lmin, x); }
          for (double x : w2) { lmax = std::max(lmax, x); lmin = std::min(lmin, x); }
          const double tol = 1e-12 * lmax;
          std::vector<int> os, oa;
          for (int e = 0; e < hs; ++e) if (w[e] > tol) os.push_back(e);
          for (int e = 0; e < ha; ++e) if (w2[e] > tol) oa.push_back(e);
          std::sort(os.begin(), os.end(), [&](int x, int y) { return w[x] > w[y] || (w[x] == w[y] && x < y); });
          std::sort(oa.begin(), oa.end(), [&](int x, int y) { return w2[x] > w2[y] || (w2[x] == w2[y] && x < y); });
          const int rs = (int)os.size(), ra = (int)oa.size(), ts = (rs + 63) / 64, ta = (ra + 63) / 64;
          const double units_split = 0.5 * (tile_units(rs) + tile_units(ra)) * ntile_dense;
          if (lmax > 0.0 && lmin >= -tol && rs + ra > 0 && units_split < 0.9 * units_dense) {
            d.qf_rank[t] = rs + ra; d.qf_rank_s[t] = rs; d.qf_split[t] = 1;
            d.qf_tiles[t] = ts + ta;
            wrows_t[t] = 64 * (ts + ta);
            Wt[t].assign((size_t)wrows_t[t] * Sp, 0.0);
            for (int row = 0; row < rs; ++row) {        // + block: K range [0, Sp/2)
              const int e = os[row];
              const double sc = std::sqrt(w[e]);
              double* dst = &Wt[t][(size_t)row * Sp];
              for (int i = 0; i < ha; ++i) dst[i] = sc * rs2 * v[(size_t)i * hs + e];
              if (hs > ha) dst[ha] = sc * v[(size_t)ha * hs + e];
            }
            for (int row = 0; row < ra; ++row) {        // - block: rows from 64 ts on, K range [Sp/2, Sp)
              const int e = oa[row];
              const double sc = std::sqrt(w2[e]);
              double* dst = &Wt[t][(size_t)(64 * ts + row) * Sp + Sp / 2];
              for (int i = 0; i < ha; ++i) dst[i] = sc * rs2 * v2[(size_t)i * ha + e];
            }
          }
        }
        if (d.qf_rank[t] == 0 && rmax > 0.0) {          // plain factor form over the whole window
          a.resize((size_t)S * S);
          for (int i = 0; i < S; ++i)
            for (int j = 0; j < S; ++j) a[(size_t)i * S + j] = R(i, j);
          sym_eigh(a, S, w, v);
          double lmax = 0.0, lmin = 0.0;
          for (int e = 0; e < S; ++e) { lmax = std::max(lmax, w[e]); lmin = std::min(lmin, w[e]); }
          const double tol = 1e-12 * lmax;
          int r = 0;
          for (int e = 0; e < S; ++e) r += w[e] > tol;
          if (lmax > 0.0 && lmin >= -tol && r > 0 && tile_units(r) * ntile_dense < 0.9 * units_dense) {
            d.qf_rank[t] = r;
            d.qf_tiles[t] = (r + 63) / 64;
            wrows_t[t] = 64 * d.qf_tiles[t];
            Wt[t].assign((size_t)wrows_t[t] * Sp, 0.0);
            std::vector<int> order;
            for (int e = 0; e < S; ++e) if (w[e] > tol) order.push_back(e);
            std::sort(order.begin(), order.end(), [&](int x, int y) { return w[x] > w[y] || (w[x] == w[y] && x < y); });
            for (int row = 0; row < r; ++row) {         // largest eigenvalue first
              const int e = order[row];
              const double sc = std::sqrt(w[e]);
              for (int i = 0; i < S; ++i) Wt[t][(size_t)row * Sp + i] = sc * v[(size_t)i * S + e];
            }
          }
        }
      }
      d.qf_tiles_max = std::max(d.qf_tiles_max, d.qf_tiles[t]);
      wrows = std::max(wrows, wrows_t[t]);
    }
    d.qf_wrows = wrows;
    wfac.assign((size_t)T * wrows * Sp, 0.0);
    for (int t = 0; t < T; ++t)
      if (!Wt[t].empty()) std::memcpy(&wfac[(size_t)t * wrows * Sp], Wt[t].data(), sizeof(double) * Wt[t].size());
    // hand-out order of the column tiles inside a scheduling chunk: most expensive first (dense form: the cost grows
    // with jt; factor forms: full tiles before partial ones), judged on the trace with the most tiles
    {
      int tr = 0;
      for (int t = 0; t < T; ++t) if (d.qf_tiles[t] > d.qf_tiles[tr]) tr = t;
      std::vector<std::pair<double, int>> cost;
      for (int jt = 0; jt < d.qf_tiles_max && jt < RFINV_MAX_QF_TILES; ++jt) {
        double cst;
        if (d.qf_rank[tr] == 0) cst = jt + 1;
        else if (d.qf_split[tr]) {
          const int rs = d.qf_rank_s[tr], ts = (rs + 63) / 64;
          cst = std::min(64, jt < ts ? rs - 64 * jt : (d.qf_rank[tr] - rs) - 64 * (jt - ts));
        } else cst = std::min(64, d.qf_rank[tr] - 64 * jt);
        cost.push_back({-cst, jt});
      }
      std::sort(cost.begin(), cost.end());
      for (size_t q = 0; q < cost.size(); ++q) d.qf_order[q] = cost[q].second;
    }
  }
#define RFINV_TRY(x) do { st = (x); if (st != RFINV_OK) { rfinv_destroy(h); return st; } } while (0)
  RFINV_TRY(upload(flt, &h->d_flt));
  RFINV_TRY(upload(tw, &h->d_tw));
  if (d.fft_general) { RFINV_TRY(upload(chirp, &h->d_chirp)); RFINV_TRY(upload(chirp_b, &h->d_chirp_b)); RFINV_TRY(upload(twq, &h->d_twq)); }
  RFINV_TRY(upload(h->h_obs, &h->d_obs));
  RFINV_TRY(upload(h->h_vp_ref, &h->d_vp_ref));
  RFINV_TRY(upload(h->h_vs_ref, &h->d_vs_ref));
  RFINV_TRY(upload(rpad, &h->d_r_inv));
  RFINV_TRY(upload(wfac, &h->d_w_fac));
#undef RFINV_TRY
  d.flt = h->d_flt; d.tw = h->d_tw; d.chirp = h->d_chirp; d.chirp_b = h->d_chirp_b; d.twq = h->d_twq; d.obs = h->d_obs; d.vp_ref = h->d_vp_ref; d.vs_ref = h->d_vs_ref; d.r_inv = h->d_r_inv; d.w_fac = h->d_w_fac;
  cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { rfinv_set_error("cudaStreamCreate: %s", cudaGetErrorString(e)); rfinv_destroy(h); return RFINV_ERR_CUDA; }
  h->own_stream = true;
  *out = h;
  return RFINV_OK;
}

void rfinv_destroy(rfinv_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  h->free_pt();              // first: the captured iteration graphs hold references on the communicator (ncclCommDestroy waits for them)
  rfinv_comm_destroy(h);
  h->free_workspace();
  cudaFree(h->d_flt); cudaFree(h->d_tw); cudaFree(h->d_chirp); cudaFree(h->d_chirp_b); cudaFree(h->d_twq); cudaFree(h->d_obs); cudaFree(h->d_vp_ref); cudaFree(h->d_vs_ref); cudaFree(h->d_r_inv); cudaFree(h->d_w_fac);
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  if (h->stream_copy) {
    cudaStreamSynchronize(h->stream_copy);
    cudaStreamDestroy(h->stream_copy);
    for (cudaEvent_t e : h->ev_copy) if (e) cudaEventDestroy(e);
  }
  for (int i = 0; i < RFINV_ASYNC_SLOTS; ++i) {
    if (h->async_stream[i]) { cudaStreamSynchronize(h->async_stream[i]); cudaStreamDestroy(h->async_stream[i]); }
    if (h->async_ws[i]) { h->async_ws[i]->release(); delete h->async_ws[i]; }
  }
  for (int i = 0; i < 4; ++i)
    if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  delete h;
}

int32_t rfinv_set_stream(rfinv_handle* h, uint64_t cuda_stream) {
  if (!h) { rfinv_set_error("handle is NULL"); return RFINV_ERR_ARG; }
  if (h->own_stream && h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
  h->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  h->own_stream = false;
  return RFINV_OK;
}

int32_t rfinv_synchronize(rfinv_handle* h) {
  if (!h) { rfinv_set_error("handle is NULL"); return RFINV_ERR_ARG; }
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  return RFINV_OK;
}

int32_t rfinv_last_launch_count(rfinv_handle* h) { return h ? h->launches : 0; }

int32_t rfinv_set_timing(rfinv_handle* h, int32_t enable) {
  if (!h) { rfinv_set_error("handle is NULL"); return RFINV_ERR_ARG; }
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  if (enable && !h->ev[0])
    for (int i = 0; i < 4; ++i) RFINV_CUDA_CHECK(cudaEventCreate(&h->ev[i]));
  h->timing = enable != 0;
  return RFINV_OK;
}

int32_t rfinv_get_quadform_form(rfinv_handle* h, int32_t* rank, int32_t* rank_s, int32_t* split) {
  if (!h || !rank || !rank_s || !split) { rfinv_set_error("rfinv_get_quadform_form: NULL argument"); return RFINV_ERR_ARG; }
  for (int t = 0; t < h->dc.ntrc; ++t) { rank[t] = h->dc.qf_rank[t]; rank_s[t] = h->dc.qf_rank_s[t]; split[t] = h->dc.qf_split[t]; }
  return RFINV_OK;
}

int32_t rfinv_get_timing(rfinv_handle* h, double* ms) {
  if (!h || !ms) { rfinv_set_error("NULL argument"); return RFINV_ERR_ARG; }
  if (!h->timing) { rfinv_set_error("rfinv_get_timing: call rfinv_set_timing(h, 1) first"); return RFINV_ERR_STATE; }
  RFINV_CUDA_CHECK(cudaEventSynchronize(h->ev[3]));
  for (int i = 0; i < 3; ++i) {
    float f = 0.f;
    RFINV_CUDA_CHECK(cudaEventElapsedTime(&f, h->ev[i], h->ev[i + 1]));
    ms[i] = f;
  }
  return RFINV_OK;
}

int32_t rfinv_get_r_inv(rfinv_handle* h, double* r_inv) {
  if (!h || !r_inv) { rfinv_set_error("NULL argument"); return RFINV_ERR_ARG; }
  std::memcpy(r_inv, h->h_r_inv.data(), sizeof(double) * h->h_r_inv.size());
  return RFINV_OK;
}

// models [c0, c0 + n) of a batch of C: host (chain-major) -> device (chain-fastest), asynchronous on stream s
static int upload_models(rfinv_handle* h, int C, const int32_t* k, const double* z, const double* dvp, const double* dvs,
                         const double* sig, cudaStream_t s, int c0 = 0, int n = -1) {
  const int km = h->cfg.k_max, T = h->cfg.ntrc;
  if (n < 0) n = C;
  RFINV_CUDA_CHECK(cudaMemcpyAsync(h->d_k + c0, k + c0, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, s));
  struct Item { const double* src; double* dst; int len; } items[4] = {
      {z, h->d_z, km - 1}, {dvp, h->d_dvp, km}, {dvs, h->d_dvs, km}, {sig, h->d_sig, T}};
  for (const Item& it : items) {
    // vp_mode = 0: format_model never looks at dVp (src/model.f90:214-218, 271-275) -- a third of the upload
    if (it.src == dvp && h->cfg.vp_mode == 0) continue;
    const size_t nel = (size_t)n * it.len;
    RFINV_CUDA_CHECK(cudaMemcpyAsync(h->d_stage, it.src + (size_t)c0 * it.len, sizeof(double) * nel, cudaMemcpyHostToDevice, s));
    to_soa_kernel<<<(unsigned)((nel + 255) / 256), 256, 0, s>>>(h->d_stage, it.dst, C, c0, n, it.len);
    RFINV_CUDA_CHECK(cudaGetLastError());
  }
  return RFINV_OK;
}

static int check_models(const rfinv_handle* h, const char* who, int32_t C, const int32_t* k, const double* z, const double* dvp,
                        const double* dvs, const double* sig, const double* logl) {
  if (!h || C < 0 || (C > 0 && (!k || !z || !dvp || !dvs || !sig || !logl))) {
    rfinv_set_error("%s: NULL argument", who);
    return RFINV_ERR_ARG;
  }
  for (int c = 0; c < C; ++c)
    if (k[c] < 1 || k[c] > h->cfg.k_max - 1) {
      rfinv_set_error("%s: k[%d]=%d outside [1,k_max-1]", who, c, k[c]);
      return RFINV_ERR_ARG;
    }
  return RFINV_OK;
}

int32_t rfinv_eval_batch(rfinv_handle* h, int32_t C, const int32_t* k, const double* z, const double* dvp,
                         const double* dvs, const double* sig, double* logl, double* rft, uint8_t* is_valid) {
  int st = check_models(h, "rfinv_eval_batch", C, k, z, dvp, dvs, sig, logl);
  if (st != RFINV_OK) return st;
  if (C == 0) return RFINV_OK;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  if ((st = h->ensure_capacity(C)) != RFINV_OK) return st;
  if (rft) {
    const size_t need = (size_t)C * h->cfg.ntrc * h->cfg.nfft;
    if (need > h->cap_rft_full) {
      cudaFree(h->d_rft_full);
      h->d_rft_full = nullptr; h->cap_rft_full = 0;
      RFINV_CUDA_CHECK(cudaMalloc((void**)&h->d_rft_full, sizeof(double) * need));
      h->cap_rft_full = need;
    }
  }
  // Upload.  z / dvp / dvs go up exactly as the caller holds them (chain slowest): prep_kernel reads that layout
  // directly, one warp per model reading consecutive words, so no layout kernels run (only sig, which the likelihood wants
  // chain fastest, is transposed).  dVp stays on the host at vp_mode 0: format_model never looks at it
  // (src/model.f90:214-218, 271-275).  Large batches go up in pieces (upload_piece()) on a second stream; prep_kernel is
  // launched per piece on the handle's stream behind the event that marks the piece's arrival, so only the first piece's
  // transfer is exposed and nothing ever polls (RFINV_UPLOAD_OVERLAP=0: plain copies on the handle's stream).
  static const bool overlap_ok = !(getenv("RFINV_UPLOAD_OVERLAP") && atoi(getenv("RFINV_UPLOAD_OVERLAP")) == 0);
  const int km = h->cfg.k_max, T = h->cfg.ntrc;
  const bool pieces = overlap_ok && upload_pieces() > 1 && C >= upload_pieces() * UPLOAD_PIECE_MIN;
  const int piece = pieces ? upload_piece(C) : C;
  ModelBatch mb;
  mb.chain_major = 1;
  mb.C = C; mb.k = h->d_k; mb.z = h->d_z; mb.dvp = h->d_dvp; mb.dvs = h->d_dvs; mb.sig = h->d_sig;
  mb.active = nullptr; mb.n_active = 0; mb.n_active_dev = nullptr;
  cudaStream_t up = h->stream;
  if (pieces) {
    if (!h->stream_copy) {
      RFINV_CUDA_CHECK(cudaStreamCreateWithFlags(&h->stream_copy, cudaStreamNonBlocking));
      for (cudaEvent_t& e : h->ev_copy) RFINV_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    up = h->stream_copy;
    RFINV_CUDA_CHECK(cudaEventRecord(h->ev_copy[RFINV_UPLOAD_PIECES], h->stream));   // earlier work on the handle's stream reads these buffers
    RFINV_CUDA_CHECK(cudaStreamWaitEvent(up, h->ev_copy[RFINV_UPLOAD_PIECES], 0));
  }
  if (h->timing) cudaEventRecord(h->ev[0], h->stream);
  int ip = 0;
  for (int c0 = 0; c0 < C; c0 += piece, ++ip) {
    const size_t n = (size_t)std::min(piece, C - c0);
    RFINV_CUDA_CHECK(cudaMemcpyAsync(h->d_k + c0, k + c0, sizeof(int) * n, cudaMemcpyHostToDevice, up));
    RFINV_CUDA_CHECK(cudaMemcpyAsync(h->d_z + (size_t)c0 * (km - 1), z + (size_t)c0 * (km - 1), sizeof(double) * n * (km - 1), cudaMemcpyHostToDevice, up));
    RFINV_CUDA_CHECK(cudaMemcpyAsync(h->d_dvs + (size_t)c0 * km, dvs + (size_t)c0 * km, sizeof(double) * n * km, cudaMemcpyHostToDevice, up));
    if (h->cfg.vp_mode == 1)
      RFINV_CUDA_CHECK(cudaMemcpyAsync(h->d_dvp + (size_t)c0 * km, dvp + (size_t)c0 * km, sizeof(double) * n * km, cudaMemcpyHostToDevice, up));
    if (pieces) {
      RFINV_CUDA_CHECK(cudaEventRecord(h->ev_copy[ip], up));
      RFINV_CUDA_CHECK(cudaStreamWaitEvent(h->stream, h->ev_copy[ip], 0));
    }
    if ((st = rfinv_launch_prep(h->dc, mb, is_valid ? h->d_valid : nullptr, h->d_scratch, h->stream, c0, (int)n)) != RFINV_OK) return st;
  }
  {  // sig: only the likelihood (the tail of quadform_kernel) reads it; it travels last and forward_kernel does not wait for it
    const size_t nel = (size_t)C * T;
    RFINV_CUDA_CHECK(cudaMemcpyAsync(h->d_stage, sig, sizeof(double) * nel, cudaMemcpyHostToDevice, up));
    to_soa_kernel<<<(unsigned)((nel + 255) / 256), 256, 0, up>>>(h->d_stage, h->d_sig, C, 0, C, T);
    RFINV_CUDA_CHECK(cudaGetLastError());
    if (pieces) RFINV_CUDA_CHECK(cudaEventRecord(h->ev_copy[RFINV_UPLOAD_PIECES + 1], up));
  }
  const bool timing_saved = h->timing;
  h->timing = false;   // ev[0] is already on the stream (before the first piece of prep_kernel)
  st = h->eval_device(C, h->d_k, h->d_z, h->d_dvp, h->d_dvs, h->d_sig, h->d_logl, nullptr, rft ? h->d_rft_full : nullptr,
                      is_valid ? h->d_valid : nullptr, nullptr, 0, &mb, nullptr, nullptr, /*prep_done=*/true,
                      pieces ? h->ev_copy[RFINV_UPLOAD_PIECES + 1] : nullptr);
  h->timing = timing_saved;
  if (st != RFINV_OK) return st;
  h->launches += ip + 1;   // prep_kernel per piece, sig layout kernel
  if (h->timing) { cudaEventRecord(h->ev[1], h->stream); cudaEventRecord(h->ev[2], h->stream); cudaEventRecord(h->ev[3], h->stream); }
  RFINV_CUDA_CHECK(cudaMemcpyAsync(logl, h->d_logl, sizeof(double) * (size_t)C, cudaMemcpyDeviceToHost, h->stream));
  if (rft)
    RFINV_CUDA_CHECK(cudaMemcpyAsync(rft, h->d_rft_full, sizeof(double) * (size_t)C * h->cfg.ntrc * h->cfg.nfft,
                                     cudaMemcpyDeviceToHost, h->stream));
  if (is_valid) RFINV_CUDA_CHECK(cudaMemcpyAsync(is_valid, h->d_valid, (size_t)C, cudaMemcpyDeviceToHost, h->stream));
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  return RFINV_OK;
}

// calc_likelihood with a per-model fwd_flag (src/likelihood.f90:74-82).  The reference's fwd_flag = .false. branch takes the
// chain's cached rft and evaluates the same misfit and quadratic form again: phi does not change, only sigma does.  The
// stateless batched form carries the cached quantity through the caller: phi[c][t] is written for the models that were
// propagated and read for the others.
int32_t rfinv_eval_batch_flags(rfinv_handle* h, int32_t C, const uint8_t* fwd_flag, const int32_t* k, const double* z,
                               const double* dvp, const double* dvs, const double* sig, double* phi, double* logl,
                               uint8_t* is_valid) {
  int st = RFINV_OK;
  if (!h || C < 0 || (C > 0 && (!fwd_flag || !k || !z || !dvp || !dvs || !sig || !phi || !logl))) {
    rfinv_set_error("rfinv_eval_batch_flags: NULL argument");
    return RFINV_ERR_ARG;
  }
  if (C == 0) return RFINV_OK;
  std::vector<int> active;
  active.reserve(C);
  for (int c = 0; c < C; ++c)
    if (fwd_flag[c]) {
      if (k[c] < 1 || k[c] > h->cfg.k_max - 1) { rfinv_set_error("rfinv_eval_batch_flags: k[%d]=%d outside [1,k_max-1]", c, k[c]); return RFINV_ERR_ARG; }
      active.push_back(c);
    }
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  if ((st = h->ensure_capacity(C)) != RFINV_OK) return st;
  const int km = h->cfg.k_max, T = h->cfg.ntrc;
  const size_t n = (size_t)C;
  cudaStream_t s = h->stream;
  int* d_active = nullptr;
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_active, sizeof(int) * std::max<size_t>(active.size(), 1)));
  auto fail = [&](int code) { cudaFree(d_active); return code; };
#define TRY_CUDA(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { rfinv_set_error("rfinv_eval_batch_flags: %s", cudaGetErrorString(e__)); return fail(RFINV_ERR_CUDA); } } while (0)
  TRY_CUDA(cudaMemcpyAsync(h->d_k, k, sizeof(int) * n, cudaMemcpyHostToDevice, s));
  TRY_CUDA(cudaMemcpyAsync(h->d_z, z, sizeof(double) * n * (km - 1), cudaMemcpyHostToDevice, s));
  TRY_CUDA(cudaMemcpyAsync(h->d_dvs, dvs, sizeof(double) * n * km, cudaMemcpyHostToDevice, s));
  if (h->cfg.vp_mode == 1) TRY_CUDA(cudaMemcpyAsync(h->d_dvp, dvp, sizeof(double) * n * km, cudaMemcpyHostToDevice, s));
  TRY_CUDA(cudaMemcpyAsync(h->d_stage, sig, sizeof(double) * n * T, cudaMemcpyHostToDevice, s));
  to_soa_kernel<<<(unsigned)((n * T + 255) / 256), 256, 0, s>>>(h->d_stage, h->d_sig, C, 0, C, T);
  // the cached quadratic forms of every model, chain fastest; the propagated models overwrite theirs
  TRY_CUDA(cudaMemcpyAsync(h->d_stage, phi, sizeof(double) * n * T, cudaMemcpyHostToDevice, s));
  to_soa_kernel<<<(unsigned)((n * T + 255) / 256), 256, 0, s>>>(h->d_stage, h->d_phi, C, 0, C, T);
  TRY_CUDA(cudaGetLastError());
  if (is_valid) TRY_CUDA(cudaMemsetAsync(h->d_valid, 1, n, s));   // models that are not propagated are not re-validated
  if (!active.empty()) {
    TRY_CUDA(cudaMemcpyAsync(d_active, active.data(), sizeof(int) * active.size(), cudaMemcpyHostToDevice, s));
    ModelBatch layout;
    layout.chain_major = 1;
    st = h->eval_device(C, h->d_k, h->d_z, h->d_dvp, h->d_dvs, h->d_sig, nullptr, nullptr, nullptr, is_valid ? h->d_valid : nullptr,
                        d_active, (int)active.size(), &layout);
    if (st != RFINV_OK) return fail(st);
  }
  if ((st = rfinv_launch_loglik(h->dc, C, h->d_phi, h->d_sig, h->d_logl, s)) != RFINV_OK) return fail(st);
  h->launches += 3;
  TRY_CUDA(cudaMemcpyAsync(logl, h->d_logl, sizeof(double) * n, cudaMemcpyDeviceToHost, s));
  // phi back, chain slowest like the caller's array (through the staging buffer)
  from_soa_kernel<<<(unsigned)((n * T + 255) / 256), 256, 0, s>>>(h->d_phi, h->d_stage, C, T);
  TRY_CUDA(cudaGetLastError());
  TRY_CUDA(cudaMemcpyAsync(phi, h->d_stage, sizeof(double) * n * T, cudaMemcpyDeviceToHost, s));
  if (is_valid) TRY_CUDA(cudaMemcpyAsync(is_valid, h->d_valid, n, cudaMemcpyDeviceToHost, s));
  TRY_CUDA(cudaStreamSynchronize(s));
#undef TRY_CUDA
  cudaFree(d_active);
  return RFINV_OK;
}

// Asynchronous form of rfinv_eval_batch: everything of one batch -- upload, kernels, read-back of logL -- is queued on the
// slot's own stream and workspace; with two slots in flight the transfers of one batch hide behind the kernels of the other.
int32_t rfinv_eval_batch_begin(rfinv_handle* h, int32_t slot, int32_t C, const int32_t* k, const double* z, const double* dvp,
                               const double* dvs, const double* sig, double* logl, uint8_t* is_valid) {
  int st = check_models(h, "rfinv_eval_batch_begin", C, k, z, dvp, dvs, sig, logl);
  if (st != RFINV_OK) return st;
  if (slot < 0 || slot >= RFINV_ASYNC_SLOTS) { rfinv_set_error("rfinv_eval_batch_begin: slot must be in [0,%d)", RFINV_ASYNC_SLOTS); return RFINV_ERR_ARG; }
  if (h->async_pending[slot]) { rfinv_set_error("rfinv_eval_batch_begin: slot %d is in flight; call rfinv_eval_batch_end first", slot); return RFINV_ERR_STATE; }
  if (C == 0) return RFINV_OK;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  if (!h->async_ws[slot]) {
    h->async_ws[slot] = new EvalWorkspace();
    RFINV_CUDA_CHECK(cudaStreamCreateWithFlags(&h->async_stream[slot], cudaStreamNonBlocking));
  }
  EvalWorkspace* w = h->async_ws[slot];
  cudaStream_t s = h->async_stream[slot];
  if ((st = w->grow(h->dc, h->cfg, h->device, C)) != RFINV_OK) return st;
  const int km = h->cfg.k_max, T = h->cfg.ntrc;
  const size_t n = (size_t)C;
  RFINV_CUDA_CHECK(cudaMemcpyAsync(w->d_k, k, sizeof(int) * n, cudaMemcpyHostToDevice, s));
  RFINV_CUDA_CHECK(cudaMemcpyAsync(w->d_z, z, sizeof(double) * n * (km - 1), cudaMemcpyHostToDevice, s));
  RFINV_CUDA_CHECK(cudaMemcpyAsync(w->d_dvs, dvs, sizeof(double) * n * km, cudaMemcpyHostToDevice, s));
  if (h->cfg.vp_mode == 1) RFINV_CUDA_CHECK(cudaMemcpyAsync(w->d_dvp, dvp, sizeof(double) * n * km, cudaMemcpyHostToDevice, s));
  RFINV_CUDA_CHECK(cudaMemcpyAsync(w->d_stage, sig, sizeof(double) * n * T, cudaMemcpyHostToDevice, s));
  to_soa_kernel<<<(unsigned)((n * T + 255) / 256), 256, 0, s>>>(w->d_stage, w->d_sig, C, 0, C, T);
  RFINV_CUDA_CHECK(cudaGetLastError());
  ModelBatch layout;
  layout.chain_major = 1;
  st = h->eval_device(C, w->d_k, w->d_z, w->d_dvp, w->d_dvs, w->d_sig, w->d_logl, nullptr, nullptr, is_valid ? w->d_valid : nullptr,
                      nullptr, 0, &layout, w, s);
  if (st != RFINV_OK) return st;
  RFINV_CUDA_CHECK(cudaMemcpyAsync(logl, w->d_logl, sizeof(double) * n, cudaMemcpyDeviceToHost, s));
  if (is_valid) RFINV_CUDA_CHECK(cudaMemcpyAsync(is_valid, w->d_valid, n, cudaMemcpyDeviceToHost, s));
  h->async_pending[slot] = true;
  return RFINV_OK;
}

int32_t rfinv_eval_batch_end(rfinv_handle* h, int32_t slot) {
  if (!h || slot < 0 || slot >= RFINV_ASYNC_SLOTS) { rfinv_set_error("rfinv_eval_batch_end: bad handle or slot"); return RFINV_ERR_ARG; }
  if (!h->async_pending[slot]) return RFINV_OK;
  h->async_pending[slot] = false;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->async_stream[slot]));
  return RFINV_OK;
}

int32_t rfinv_filter_traces(rfinv_handle* h, int32_t n_series, const int32_t* trace_of, const double* in, double* out) {
  if (!h || n_series < 0 || (n_series > 0 && (!trace_of || !in || !out))) {
    rfinv_set_error("rfinv_filter_traces: NULL argument");
    return RFINV_ERR_ARG;
  }
  for (int i = 0; i < n_series; ++i)
    if (trace_of[i] < 0 || trace_of[i] >= h->cfg.ntrc) {
      rfinv_set_error("rfinv_filter_traces: trace_of[%d]=%d outside [0,ntrc)", i, trace_of[i]);
      return RFINV_ERR_ARG;
    }
  if (n_series == 0) return RFINV_OK;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  const size_t n = (size_t)n_series * h->cfg.nfft;
  double *d_in = nullptr, *d_out = nullptr;
  int* d_tr = nullptr;
  cudaError_t e = cudaMalloc((void**)&d_in, sizeof(double) * n);
  if (e == cudaSuccess) e = cudaMalloc((void**)&d_out, sizeof(double) * n);
  if (e == cudaSuccess) e = cudaMalloc((void**)&d_tr, sizeof(int) * (size_t)n_series);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_in, in, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_tr, trace_of, sizeof(int) * (size_t)n_series, cudaMemcpyHostToDevice, h->stream);
  int st = RFINV_OK;
  if (e == cudaSuccess) st = rfinv_launch_filter_traces(h->dc, n_series, d_in, d_tr, d_out, h->stream);
  if (e == cudaSuccess && st == RFINV_OK) e = cudaMemcpyAsync(out, d_out, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess && st == RFINV_OK) e = cudaStreamSynchronize(h->stream);
  cudaFree(d_in); cudaFree(d_out); cudaFree(d_tr);
  if (e != cudaSuccess) { rfinv_set_error("rfinv_filter_traces: %s", cudaGetErrorString(e)); return RFINV_ERR_CUDA; }
  return st;
}

int32_t rfinv_eval_batch_device(rfinv_handle* h, int32_t C, uint64_t d_k, uint64_t d_z, uint64_t d_dvp, uint64_t d_dvs,
                                uint64_t d_sig, uint64_t d_logl, uint64_t d_rft_smp, uint64_t d_is_valid) {
  if (!h || C < 0 || (C > 0 && (!d_k || !d_z || !d_dvp || !d_dvs || !d_sig || !d_logl))) {
    rfinv_set_error("rfinv_eval_batch_device: NULL argument");
    return RFINV_ERR_ARG;
  }
  if (C == 0) return RFINV_OK;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  int st = h->ensure_capacity(C);
  if (st != RFINV_OK) return st;
  return h->eval_device(C, reinterpret_cast<const int*>(d_k), reinterpret_cast<const double*>(d_z),
                        reinterpret_cast<const double*>(d_dvp), reinterpret_cast<const double*>(d_dvs),
                        reinterpret_cast<const double*>(d_sig), reinterpret_cast<double*>(d_logl),
                        reinterpret_cast<double*>(d_rft_smp), nullptr, reinterpret_cast<uint8_t*>(d_is_valid), nullptr, 0);
}

int32_t rfinv_format_model_batch(rfinv_handle* h, int32_t C, const int32_t* k, const double* z, const double* dvp,
                                 const double* dvs, int32_t* nlay, double* alpha, double* beta, double* rho,
                                 double* hthick, uint8_t* is_valid) {
  if (!h || C < 0 || (C > 0 && (!k || !z || !dvp || !dvs || !nlay || !alpha || !beta || !rho || !hthick || !is_valid))) {
    rfinv_set_error("rfinv_format_model_batch: NULL argument");
    return RFINV_ERR_ARG;
  }
  if (C == 0) return RFINV_OK;
  for (int c = 0; c < C; ++c)
    if (k[c] < 1 || k[c] > h->cfg.k_max - 1) {
      rfinv_set_error("rfinv_format_model_batch: k[%d]=%d outside [1,k_max-1]", c, k[c]);
      return RFINV_ERR_ARG;
    }
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  int st = h->ensure_capacity(C);
  if (st != RFINV_OK) return st;
  std::vector<double> sig((size_t)C * h->cfg.ntrc, 1.0);
  if ((st = upload_models(h, C, k, z, dvp, dvs, sig.data(), h->stream)) != RFINV_OK) return st;
  const int stride = h->cfg.k_max + 1;
  int* d_nlay = nullptr;
  double* d_out = nullptr;
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_nlay, sizeof(int) * (size_t)C));
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_out, sizeof(double) * (size_t)C * stride * 4));
  RFINV_CUDA_CHECK(cudaMemsetAsync(d_out, 0, sizeof(double) * (size_t)C * stride * 4, h->stream));
  ModelBatch mb;
  mb.C = C; mb.k = h->d_k; mb.z = h->d_z; mb.dvp = h->d_dvp; mb.dvs = h->d_dvs; mb.sig = h->d_sig; mb.active = nullptr; mb.n_active = 0; mb.n_active_dev = nullptr;
  const size_t blk = (size_t)C * stride;
  st = rfinv_launch_format_model(h->dc, mb, d_nlay, d_out, d_out + blk, d_out + 2 * blk, d_out + 3 * blk, h->d_valid, h->stream);
  if (st == RFINV_OK) {
    cudaMemcpyAsync(nlay, d_nlay, sizeof(int) * (size_t)C, cudaMemcpyDeviceToHost, h->stream);
    cudaMemcpyAsync(alpha, d_out, sizeof(double) * blk, cudaMemcpyDeviceToHost, h->stream);
    cudaMemcpyAsync(beta, d_out + blk, sizeof(double) * blk, cudaMemcpyDeviceToHost, h->stream);
    cudaMemcpyAsync(rho, d_out + 2 * blk, sizeof(double) * blk, cudaMemcpyDeviceToHost, h->stream);
    cudaMemcpyAsync(hthick, d_out + 3 * blk, sizeof(double) * blk, cudaMemcpyDeviceToHost, h->stream);
    cudaMemcpyAsync(is_valid, h->d_valid, (size_t)C, cudaMemcpyDeviceToHost, h->stream);
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { rfinv_set_error("format_model: %s", cudaGetErrorString(e)); st = RFINV_ERR_CUDA; }
  }
  cudaFree(d_nlay); cudaFree(d_out);
  return st;
}

}  // extern "C"
