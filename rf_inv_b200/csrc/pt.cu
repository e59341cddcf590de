// Parallel-tempering reversible-jump MCMC on device: the caller of the forward+likelihood path.
//
// Replaces, with all chain state resident in HBM (structure of arrays, chain fastest):
//   init_model        src/model.f90:43-107        init_sig     src/likelihood.f90:107-139
//   init_rft          src/likelihood.f90:143-163  temperatures src/pt_mcmc.f90:444-452
//   mcmc              src/pt_mcmc.f90:54-201      judge_mcmc   src/pt_mcmc.f90:600-621
//   pt_control        src/pt_mcmc.f90:468-576     judge_pt     src/pt_mcmc.f90:580-595
//   mt19937 grnd      src/mt19937.f90:78-130      gauss        src/math.f90:34-50
//   laplace, log_prior_ratio                      src/prior.f90:36-123
//
// RNG semantics (SURVEY.md F6, section 3.3): the reference has ONE mt19937 stream per MPI rank, shared by the
// `nchains` chains of that rank.  A "virtual rank" here = nchains chains + one 624-word MT state, seeded
// iseed + r*r*10000 + 23*r.  The number of draws a chain step consumes never depends on the forward result, so
// per iteration one thread per virtual rank runs the serial proposal pass (draws, proposal, validity, the
// acceptance uniform), then ALL forward+likelihood evaluations run batched, then acceptance is parallel.
#include <vector>
#include <cstring>
#include "rfinv_handle.h"
#include "rfinv_pt.h"

namespace {

constexpr double PI2 = 2.0 * 3.1415926535897931;  // src/math.f90:37

// ---------------- mt19937 (src/mt19937.f90): state word i of stream r at mt[r*624 + i] ----------------
// Two ways to drive a stream: by one thread (init, swap) or by a whole warp in lock step (proposal pass): all lanes
// then execute the same draws on replicated scalars and the 624-word reload is done cooperatively.
struct Mt {
  uint32_t* mt;
  int mti;
  bool warp;   // true: called by all 32 lanes of a warp in lock step
  __device__ Mt(uint32_t* base, int r, int mti_, bool warp_ = false) : mt(base + (size_t)r * 624), mti(mti_), warp(warp_) {}
  // (measured: serving the draws of a warp from a register window of the next 32 state words -- one coalesced load per 32
  // draws, a shuffle per draw -- is slower than reading the word, which hits the L1: 867 vs 860 us per PT iteration)
  __device__ uint32_t& w(int i) { return mt[i]; }
  __device__ static uint32_t twist(uint32_t cur, uint32_t nxt, uint32_t far) {
    const uint32_t y = (cur & 0x80000000u) | (nxt & 0x7fffffffu);
    return far ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
  }
  __device__ void reload() {  // src/mt19937.f90:96-116
    if (!warp) {
      for (int kk = 0; kk < 624; ++kk) w(kk) = twist(w(kk), w(kk == 623 ? 0 : kk + 1), w(kk + 397 < 624 ? kk + 397 : kk - 227));
    } else {
      // new[kk] depends on old[kk], old[kk+1] and on old[kk+397] (kk < 227) or new[kk-227]: batches of <= 227
      // consecutive words are independent.  Read everything of a 32-word round first, then write.
      const int lane = threadIdx.x & 31;
      const int bounds[4] = {0, 227, 454, 623};
      for (int b = 0; b < 3; ++b)
        for (int base = bounds[b]; base < bounds[b + 1]; base += 32) {
          const int kk = base + lane;
          const bool act = kk < bounds[b + 1];
          uint32_t v = 0;
          if (act) v = twist(w(kk), w(kk + 1), w(kk + 397 < 624 ? kk + 397 : kk - 227));
          __syncwarp();
          if (act) w(kk) = v;
          __syncwarp();
        }
      const uint32_t last = twist(w(623), w(0), w(396));
      __syncwarp();
      if (lane == 0) w(623) = last;
      __syncwarp();
    }
    mti = 0;
  }
  __device__ static double temper(uint32_t y) {
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return (double)y * 2.3283064365386963e-10;  // y / 2^32 (src/mt19937.f90:125-129: [0,1)); a power of two: the product is the exact quotient
  }
  __device__ double grnd() {
    if (mti >= 624) reload();
    return temper(w(mti++));
  }
  __device__ double peek() {  // next output without consuming it
    if (mti >= 624) reload();
    return temper(w(mti));
  }
};

__device__ double gauss(Mt& g) {  // src/math.f90:34-50: cosine branch only, exactly two draws
  double v1 = g.grnd();
  const double v2 = g.grnd();
  if (v1 == 0.0) v1 = (double)1.0e-16f;
  return __dmul_rn(sqrt(__dmul_rn(-2.0, log(v1))), cos(__dmul_rn(PI2, v2)));
}

__device__ double laplace(Mt& g) {  // src/prior.f90:57-123; +,-,*,/ only: bit-exact without FMA contraction
  const double d = 0.69314718055994529;
  double u1 = g.grnd();
  const double u1p = __dmul_rn(2.0, u1);
  double u1pp, a = 0.0, w, val;
  int i_sign;
  if (u1p < 1.0) { i_sign = 1; u1pp = __dsub_rn(1.0, u1p); } else { i_sign = -1; u1pp = __dsub_rn(2.0, u1p); }
  for (;;) {
    const double u1ppp = __dmul_rn(2.0, u1pp);
    if (u1ppp >= 1.0) { u1 = __dsub_rn(u1ppp, 1.0); break; }
    a = __dadd_rn(a, d);
    u1pp = u1ppp;
  }
  for (;;) {
    w = __dmul_rn(d, u1);
    val = __dmul_rn((double)i_sign, __dadd_rn(a, w));
    int k = 1;
    for (;;) {
      const double u2 = g.grnd();
      if (u2 >= w) { u1 = __ddiv_rn(__dsub_rn(u2, w), __dsub_rn(1.0, w)); break; }
      w = u2;
      ++k;
    }
    if (k & 1) break;
  }
  return val;
}

__device__ double prior_draw(Mt& g, int prior_mode) { return prior_mode == 1 ? laplace(g) : gauss(g); }

__device__ double log_prior_ratio(double x_new, double x_old, double dev, int prior_mode) {  // src/prior.f90:36-53
  if (prior_mode == 1) return __ddiv_rn(-__dsub_rn(fabs(x_new), fabs(x_old)), dev);
  return __ddiv_rn(-__dsub_rn(__dmul_rn(x_new, x_new), __dmul_rn(x_old, x_old)), __dmul_rn(__dmul_rn(2.0, dev), dev));
}

// format_model's validity flag (src/model.f90:175-290) for one model held in thread-local arrays.
__device__ bool model_valid(const DevConfig& cfg, int k, const double* zin, const double* dvpin, const double* dvsin,
                            double dvp_half, double dvs_half) {
  double z[RFINV_MAX_K], dp[RFINV_MAX_K], ds[RFINV_MAX_K];
  for (int i = 0; i < k; ++i) { z[i] = zin[i]; dp[i] = dvpin[i]; ds[i] = dvsin[i]; }
  for (int i = 1; i < k; ++i) {
    const double a = z[i], b = dp[i], d = ds[i];
    int m = i - 1;
    while (m >= 0 && z[m] > a) { z[m + 1] = z[m]; dp[m + 1] = dp[m]; ds[m + 1] = ds[m]; --m; }
    z[m + 1] = a; dp[m + 1] = b; ds[m + 1] = d;
  }
  bool valid = true;
  for (int l = 0; l <= k; ++l) {
    double zc, h, dvs_l, dvp_l;
    if (l == 0) { zc = __dmul_rn(0.5, __dadd_rn(cfg.sdep, z[0])); h = __dsub_rn(z[0], cfg.sdep); dvs_l = ds[0]; dvp_l = dp[0]; }
    else if (l < k) { zc = __dmul_rn(0.5, __dadd_rn(z[l], z[l - 1])); h = __dsub_rn(z[l], z[l - 1]); dvs_l = ds[l]; dvp_l = dp[l]; }
    else { zc = __dmul_rn(0.5, __dadd_rn(cfg.z_max, z[k - 1])); h = 999.0; dvs_l = dvs_half; dvp_l = dvp_half; }
    double a, b;
    bool ok = layer_velocity(cfg, zc, dvs_l, dvp_l, a, b);
    if (l == 0) ok = ok && !(h < __dmul_rn(0.125, a));
    else if (l < k) ok = ok && !(h < cfg.h_min);
    valid = valid && ok;
  }
  return valid;
}

// ---------------- init: sgrnd + init_model + init_sig + temperatures, one thread per virtual rank ----------------
__global__ void pt_init_kernel(const DevConfig cfg, const PtDev p) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= p.G) return;
  const int km = cfg.k_max, Cl = p.Cl, T = cfg.ntrc;
  const uint32_t grank = (uint32_t)(p.rank_begin + r);
  Mt g(p.mt, r, 624);
  {  // sgrnd, src/mt19937.f90:78-90; seed src/rf_inv.f90:75 (wraps like default-integer arithmetic)
    uint32_t s = (uint32_t)p.iseed + grank * grank * 10000u + 23u * grank;
    g.w(0) = s;
    for (int i = 1; i < 624; ++i) { s = 69069u * s; g.w(i) = s; }
  }
  double z[RFINV_MAX_K], dvp[RFINV_MAX_K], dvs[RFINV_MAX_K];
  for (int ic = 0; ic < p.nchains; ++ic) {  // init_model, src/model.f90:62-95
    const int c = r * p.nchains + ic;
    int kk = 1;
    bool valid = false;
    // the reference zeroes z/dvp/dvs once (src/model.f90:59-61); entries written by a rejected draw stay in place
    for (int i = 0; i < km; ++i) { z[i] = 0.0; dvp[i] = 0.0; dvs[i] = 0.0; }
    while (!valid) {
      kk = cfg.k_min + (int)(g.grnd() * (double)(cfg.k_max - cfg.k_min));
      for (int i = 0; i < kk; ++i) z[i] = __dadd_rn(cfg.z_min, __dmul_rn(g.grnd(), __dsub_rn(cfg.z_max, cfg.z_min)));
      for (int i = 0; i < kk; ++i) {
        dvs[i] = __dmul_rn(prior_draw(g, cfg.prior_mode), p.dvs_prior);
        dvp[i] = __dmul_rn(prior_draw(g, cfg.prior_mode), p.dvp_prior);
      }
      dvs[km - 1] = __dmul_rn(prior_draw(g, cfg.prior_mode), p.dvs_prior);
      dvp[km - 1] = __dmul_rn(prior_draw(g, cfg.prior_mode), p.dvp_prior);
      valid = model_valid(cfg, kk, z, dvp, dvs, dvp[km - 1], dvs[km - 1]);
    }
    p.k[c] = kk;
    for (int i = 0; i < km - 1; ++i) p.z[(size_t)i * Cl + c] = z[i];
    for (int i = 0; i < km; ++i) { p.dvp[(size_t)i * Cl + c] = dvp[i]; p.dvs[(size_t)i * Cl + c] = dvs[i]; }
  }
  for (int ic = 0; ic < p.nchains; ++ic)  // init_sig, src/likelihood.f90:117-126
    for (int t = 0; t < T; ++t) {
      const int c = r * p.nchains + ic;
      p.sig[(size_t)t * Cl + c] = p.sig_mode[t]
          ? __dadd_rn(p.sig_min[t], __dmul_rn(g.grnd(), __dsub_rn(p.sig_max[t], p.sig_min[t]))) : p.sig_min[t];
    }
  for (int ic = 0; ic < p.nchains; ++ic) {  // src/pt_mcmc.f90:447-452
    const int c = r * p.nchains + ic;
    p.temps[c] = ic < p.ncool ? 1.0 : exp(__dmul_rn(g.grnd(), log(p.t_high)));
  }
  p.mti[r] = g.mti;
}

// Draws `n` deviates from the stream of local virtual rank r, advancing it: kind 0 = grnd() (src/mt19937.f90:92-130),
// kind 1 = gauss() (src/math.f90:34-50).  One thread: the stream is sequential.  make_syn's noise (src/make_syn.f90:80-110).
__global__ void pt_draw_kernel(const PtDev p, int r, int kind, int n, double* out) {
  Mt g(p.mt, r, p.mti[r]);
  for (int i = 0; i < n; ++i) out[i] = kind == 1 ? gauss(g) : g.grnd();
  p.mti[r] = g.mti;
}

// ---------------- proposal pass: mcmc, src/pt_mcmc.f90:77-169 + the draws of judge_mcmc :611-615 ----------------
// One WARP per virtual rank, chains of the rank in order (they share the stream).  All lanes execute the same draws
// on replicated scalars (no divergence); the model arrays are distributed: lane holds elements `lane` and `lane+32`.
__device__ __forceinline__ double lane_get(double v0, double v1, int idx) {  // element idx of a distributed array
  const double a = __shfl_sync(0xffffffffu, v0, idx & 31), b = __shfl_sync(0xffffffffu, v1, idx & 31);
  return idx < 32 ? a : b;
}
__device__ __forceinline__ void lane_set(double& v0, double& v1, int idx, double val, int lane) {
  if (lane == (idx & 31)) { if (idx < 32) v0 = val; else v1 = val; }
}

// format_model's validity flag (src/model.f90:175-290), warp-parallel: the layer below interface i is described by
// z_i and its predecessor (largest interface depth below z_i, or the sea floor), no sort needed.
__device__ bool model_valid_warp(const DevConfig& cfg, int k, double z0, double z1, double p0, double p1, double s0,
                                 double s1, double dvp_half, double dvs_half, int lane) {
  const int i0 = lane, i1 = lane + 32;
  double prev0 = -INFINITY, prev1 = -INFINITY, zmax = -INFINITY;
  for (int j = 0; j < k; ++j) {
    const double zj = lane_get(z0, z1, j);
    if (zj < z0 || (zj == z0 && j < i0)) prev0 = fmax(prev0, zj);
    if (zj < z1 || (zj == z1 && j < i1)) prev1 = fmax(prev1, zj);
    zmax = fmax(zmax, zj);
  }
  bool ok = true;
  for (int slot = 0; slot < 2; ++slot) {
    const int i = slot ? i1 : i0;
    if (i >= k) continue;
    const double zi = slot ? z1 : z0, prev = slot ? prev1 : prev0;
    const bool top = prev == -INFINITY;
    const double below = top ? cfg.sdep : prev;
    const double zc = __dmul_rn(0.5, top ? __dadd_rn(cfg.sdep, zi) : __dadd_rn(zi, prev));
    const double h = __dsub_rn(zi, below);
    double a, b;
    bool lok = layer_velocity(cfg, zc, slot ? s1 : s0, slot ? p1 : p0, a, b);
    if (top) lok = lok && !(h < __dmul_rn(0.125, a));
    else lok = lok && !(h < cfg.h_min);
    ok = ok && lok;
  }
  if (lane == 0) {  // half space
    double a, b;
    ok = layer_velocity(cfg, __dmul_rn(0.5, __dadd_rn(cfg.z_max, zmax)), dvs_half, dvp_half, a, b) && ok;
  }
  return __all_sync(0xffffffffu, ok);
}

// ---- peer-memory exchange (rfinv_pt.h, PtPeers) ----
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// (the arrays of PtPeers are only indexed by compile-time constants -- unrolled loops over RFINV_MAX_PEERS with a predicate -- or
// through own_gather / own_flag: a run-time index would make every thread copy the parameter block to local memory)
__device__ __forceinline__ unsigned long long* pt_pair_flag(unsigned long long* flag_base, int world) { return flag_base + world + 1; }
__device__ __forceinline__ double* pt_pair_slot(unsigned long long* flag_base, int world, int it) {   // slot of iteration `it`
  return reinterpret_cast<double*>(flag_base + world + 2) + 2 * (it & 3);
}
// waits until *f >= want (a flag a peer raises); bounded: a peer that never arrives -- it stopped on an error -- sets this
// process's error word instead of hanging the GPU (the host checks the word after the run)
__device__ __forceinline__ void pt_peer_wait(const PtPeers& px, const unsigned long long* f, unsigned long long want) {
  const long long t0 = clock64();
  while (ld_acquire_sys(f) < want) {
    if (clock64() - t0 > 40000000000LL) { px.own_flag[px.world] = 1ULL; break; }   // ~20 s
    __nanosleep(100);
  }
}
// the swap proposal of an iteration, from the pair drawn by virtual rank 0 (global chain indices)
struct SwapPlan { int i1, i2, own1, own2, l1, l2, rank1_local; };
__device__ __forceinline__ SwapPlan pt_swap_plan(const PtDev& p, double t1, double t2) {
  SwapPlan s;
  s.i1 = (int)t1; s.i2 = (int)t2;
  s.own1 = s.i1 / p.Cl; s.own2 = s.i2 / p.Cl;
  s.l1 = s.i1 - s.own1 * p.Cl; s.l2 = s.i2 - s.own2 * p.Cl;
  s.rank1_local = s.l1 / p.nchains;
  return s;
}

// ---- random-walk width tuning (rfinv_pt_set_step_tuning, DESIGN.md 7e) ----
// row of proposal type itype in the [4] of a (rank, level): 0 move z, 1 dVs, 2 dVp, 3 sigma; -1 birth and death
__device__ __forceinline__ int pt_step_type(const PtDev& p, int itype) {
  return itype == p.it_z ? 0 : itype == p.it_dvs ? 1 : itype == p.it_dvp ? 2 : itype == p.it_sig ? 3 : -1;
}
// the width chain c of local rank r proposes type tau with: the params.in width dev, times the scale of the chain's level
// when the tuning is on -- except for the two chains of the previous iteration's global swap, whose level may depend on that
// swap's acceptance and so on their own state (the pair rule).  The pair is loaded where it is needed, not held in registers
// across the proposal loop: PEER, while the swap is still to be applied (px.done[0] < iteration), from its pair slot -- rank 0's
// warp copies it to st_pair meanwhile, so st_pair is not read then --, otherwise from st_pair.  Never from the swap table,
// whose pair entries rank 0's warp overwrites during this kernel.
template <bool PEER>
__device__ __forceinline__ double pt_step_width(const PtDev& p, const PtPeers& px, double dev, int tau, int r, int c) {
  if (!p.st_on) return dev;
  int q1, q2;
  if (PEER && px.done[0] < *p.it_dev) {
    const double* pr = pt_pair_slot(px.own_flag, px.world, *p.it_dev - 1);
    q1 = (int)__ldcg(pr); q2 = (int)__ldcg(pr + 1);
  } else {
    q1 = p.st_pair[0]; q2 = p.st_pair[1];
  }
  const int gc = p.rank_begin * p.nchains + c;
  if (gc == q1 || gc == q2) return dev;
  return __dmul_rn(dev, p.st_scale[((size_t)r * p.nchains + p.st_lvl[c]) * 4 + tau]);
}

// STAGED: the states of the rank's chains are first brought into shared memory with coalesced loads (the chains of a rank
// are neighbours in the chain-fastest arrays: one 128-byte line serves 16 of them) and the proposals leave the same way --
// one memory latency per rank instead of one per chain, a third of the sectors.  Per warp: 2 x nchains x stride doubles
// (pt_propose_smem_doubles); ranks with too many chains for that use the direct variant.
__host__ __device__ inline int pt_propose_stride(int km, int T) { return (3 * km + T) | 1; }     // odd: conflict-free transposition
__host__ __device__ inline size_t pt_propose_smem_doubles(int km, int T, int nchains) { return (size_t)2 * nchains * pt_propose_stride(km, T); }
// PEER (several processes, peer-memory exchange): the warp first applies the stream shift of the previous iteration's swap --
// judge_pt's draw from the stream of rank1, known from the pair alone -- and the owner of virtual rank 0 publishes the pair it
// draws at the end to every process.
template <bool STAGED, bool PEER>
__global__ void __launch_bounds__(128) pt_propose_kernel(const DevConfig cfg, const PtDev p, double* __restrict__ table, const PtPeers px) {
  extern __shared__ __align__(16) double pp_smem[];
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= p.G) return;
  const int km = cfg.k_max, Cl = p.Cl, T = cfg.ntrc, nch = p.nchains;
  const int S = pt_propose_stride(km, T);
  double* s_in = pp_smem + (size_t)(threadIdx.x >> 5) * pt_propose_smem_doubles(km, T, nch);   // [nchains][S]: z | dvp | dvs | sig of a chain
  double* s_out = s_in + (size_t)nch * S;
  const int c0 = r * nch;
  // row `row` of the chain-fastest state (z: km-1 rows, dvp: km, dvs: km, sig: T) -> its array and its column in a staged chain
  auto state_row = [&](int row, const double* z, const double* dvp, const double* dvs, const double* sig, int& col) -> const double* {
    if (row < km - 1) { col = row; return z + (size_t)row * Cl; }
    if (row < 2 * km - 1) { col = km + row - (km - 1); return dvp + (size_t)(row - (km - 1)) * Cl; }
    if (row < 3 * km - 1) { col = 2 * km + row - (2 * km - 1); return dvs + (size_t)(row - (2 * km - 1)) * Cl; }
    col = 3 * km + row - (3 * km - 1);
    return sig + (size_t)(row - (3 * km - 1)) * Cl;
  };
  const int rows = 3 * km - 1 + T;
  // lane -> (chain, first row): whole rows of nch chains per warp instruction when nch divides 32, else element by element
  const bool even = nch <= 32 && 32 % nch == 0;
  const int st_ic = even ? lane % nch : 0, st_row0 = even ? lane / nch : 0, st_step = even ? 32 / nch : 1;
  if (STAGED) {
    if (even) {
      for (int row = st_row0; row < rows; row += 8 * st_step) {     // eight independent loads in flight per lane
        double v[8]; int col[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int rr = row + q * st_step;
          col[q] = 0; v[q] = 0.0;
          if (rr < rows) v[q] = state_row(rr, p.z, p.dvp, p.dvs, p.sig, col[q])[c0 + st_ic];
        }
#pragma unroll
        for (int q = 0; q < 8; ++q)
          if (row + q * st_step < rows) s_in[st_ic * S + col[q]] = v[q];
      }
    } else {
      for (int idx = lane; idx < rows * nch; idx += 32) {
        const int row = idx / nch, ic = idx - row * nch;
        int col;
        const double v = state_row(row, p.z, p.dvp, p.dvs, p.sig, col)[c0 + ic];
        s_in[ic * S + col] = v;
      }
    }
    for (int ic = lane; ic < nch; ic += 32) s_in[ic * S + km - 1] = 0.0;     // element km-1 of z does not exist
  }
  int shift = 0;
  const int it_now = PEER ? *p.it_dev : 0;
  if (PEER && p.nchains >= 2 && px.done[0] < it_now) {     // swap it_now - 1: its pair was published an iteration ago
    if (lane == 0) pt_peer_wait(px, pt_pair_flag(px.own_flag, px.world), (unsigned long long)it_now);
    __syncwarp();
    const double* pr = pt_pair_slot(px.own_flag, px.world, it_now - 1);
    const SwapPlan sp = pt_swap_plan(p, __ldcg(pr), __ldcg(pr + 1));
    if (sp.own1 == px.me && sp.rank1_local == r) shift = 1;   // the stream of rank1 consumed the judge_pt uniform
    // step tuning: the pair for pt_finish_kernel's counters and, at the end of a run, the next run (pt_drain_kernel otherwise)
    if (p.st_on && r == 0 && lane == 0) { p.st_pair[0] = sp.i1; p.st_pair[1] = sp.i2; }
  }
  if (PEER) table += (size_t)(it_now & 1) * (2 * Cl + p.G + 2);   // the local table alternates: the previous one is being pushed
  Mt g(p.mt, r, p.mti[r] + shift, /*warp=*/true);
  __syncwarp();
  const bool has1 = lane + 32 < km;
  // per-chain scalars of the proposals, kept by lane (ic & 31) until the coalesced store at the end (STAGED)
  int o_pk = 0, o_itype = 0, o_pflag = 0;
  double o_logr = 0.0, o_lp12 = 0.0;
  for (int ic = 0; ic < nch; ++ic) {
    const int c = c0 + ic;
    int pk = p.k[c];
    // current state, distributed (element km-1 of z does not exist: 0)
    double z0, z1, dp0, dp1, ds0, ds1, sg;
    if (STAGED) {
      const double* sc = s_in + ic * S;
      z0 = lane < km - 1 ? sc[lane] : 0.0; z1 = lane + 32 < km - 1 ? sc[lane + 32] : 0.0;
      dp0 = lane < km ? sc[km + lane] : 0.0; dp1 = has1 ? sc[km + lane + 32] : 0.0;
      ds0 = lane < km ? sc[2 * km + lane] : 0.0; ds1 = has1 ? sc[2 * km + lane + 32] : 0.0;
      sg = lane < T ? sc[3 * km + lane] : 0.0;
    } else {
      z0 = lane < km - 1 ? p.z[(size_t)lane * Cl + c] : 0.0;
      z1 = lane + 32 < km - 1 ? p.z[(size_t)(lane + 32) * Cl + c] : 0.0;
      dp0 = lane < km ? p.dvp[(size_t)lane * Cl + c] : 0.0; dp1 = has1 ? p.dvp[(size_t)(lane + 32) * Cl + c] : 0.0;
      ds0 = lane < km ? p.dvs[(size_t)lane * Cl + c] : 0.0; ds1 = has1 ? p.dvs[(size_t)(lane + 32) * Cl + c] : 0.0;
      sg = lane < T ? p.sig[(size_t)lane * Cl + c] : 0.0;
    }
    const double cz0 = z0, cz1 = z1, cdp0 = dp0, cdp1 = dp1, cds0 = ds0, cds1 = ds1;  // the chain's current values
    double log_prior12 = 0.0;
    bool null_flag = false;
    const int itype = (int)(g.grnd() * (double)p.ntype) + 1;
    if (itype == p.it_birth) {
      pk = pk + 1;
      if (pk < km) {
        const double nvp = __dmul_rn(prior_draw(g, cfg.prior_mode), p.dvp_prior);
        const double nvs = __dmul_rn(prior_draw(g, cfg.prior_mode), p.dvs_prior);
        const double nz = __dadd_rn(cfg.z_min, __dmul_rn(g.grnd(), __dsub_rn(cfg.z_max, cfg.z_min)));
        lane_set(dp0, dp1, pk - 1, nvp, lane);
        lane_set(ds0, ds1, pk - 1, nvs, lane);
        lane_set(z0, z1, pk - 1, nz, lane);
      } else null_flag = true;
    } else if (itype == p.it_death) {
      pk = pk - 1;
      if (pk >= cfg.k_min) {
        const int itarget = (int)(g.grnd() * (double)(pk + 1)) + 1;
        // prop(il) = cur(il+1) for il = itarget..pk (1-based); prop(pk+1) = 0
        // (all shuffles are executed by every lane; selection happens afterwards)
        const double dz0 = __shfl_down_sync(0xffffffffu, cz0, 1), nz0b = __shfl_sync(0xffffffffu, cz1, 0);
        const double dq0 = __shfl_down_sync(0xffffffffu, cdp0, 1), np0b = __shfl_sync(0xffffffffu, cdp1, 0);
        const double dr0 = __shfl_down_sync(0xffffffffu, cds0, 1), ns0b = __shfl_sync(0xffffffffu, cds1, 0);
        const double nz1 = __shfl_down_sync(0xffffffffu, cz1, 1), np1 = __shfl_down_sync(0xffffffffu, cdp1, 1);
        const double ns1 = __shfl_down_sync(0xffffffffu, cds1, 1);
        const double nz0 = dz0, np0 = dq0, ns0 = dr0;
        const int e0 = lane, e1 = lane + 32;  // 0-based element indices; shift range [itarget-1, pk-1], zero at pk
        if (e0 >= itarget - 1 && e0 <= pk - 1) { z0 = lane < 31 ? nz0 : nz0b; dp0 = lane < 31 ? np0 : np0b; ds0 = lane < 31 ? ns0 : ns0b; }
        if (e1 >= itarget - 1 && e1 <= pk - 1) { z1 = lane < 31 ? nz1 : 0.0; dp1 = lane < 31 ? np1 : 0.0; ds1 = lane < 31 ? ns1 : 0.0; }
        if (e0 == pk) { z0 = 0.0; dp0 = 0.0; ds0 = 0.0; }
        if (e1 == pk) { z1 = 0.0; dp1 = 0.0; ds1 = 0.0; }
      } else null_flag = true;
    } else if (itype == p.it_z) {
      const int itarget = (int)(g.grnd() * (double)pk) + 1;
      const double nz = __dadd_rn(lane_get(z0, z1, itarget - 1), __dmul_rn(gauss(g), pt_step_width<PEER>(p, px, p.dev_z, 0, r, c)));
      lane_set(z0, z1, itarget - 1, nz, lane);
      if (nz < cfg.z_min || nz > cfg.z_max) null_flag = true;
    } else if (itype == p.it_dvs) {
      int itarget = (int)(g.grnd() * (double)(pk + 1)) + 1;
      if (itarget == pk + 1) itarget = km;
      const double old = lane_get(ds0, ds1, itarget - 1);
      const double nv = __dadd_rn(old, __dmul_rn(gauss(g), pt_step_width<PEER>(p, px, p.dev_dvs, 1, r, c)));
      lane_set(ds0, ds1, itarget - 1, nv, lane);
      log_prior12 = log_prior_ratio(nv, old, p.dvs_prior, cfg.prior_mode);
    } else if (itype == p.it_dvp) {
      int itarget = (int)(g.grnd() * (double)(pk + 1)) + 1;
      if (itarget == pk + 1) itarget = km;
      const double old = lane_get(dp0, dp1, itarget - 1);
      const double nv = __dadd_rn(old, __dmul_rn(gauss(g), pt_step_width<PEER>(p, px, p.dev_dvp, 2, r, c)));
      lane_set(dp0, dp1, itarget - 1, nv, lane);
      log_prior12 = log_prior_ratio(nv, old, p.dvp_prior, cfg.prior_mode);
    } else if (itype == p.it_sig) {
      const int itarget = p.isig_trc[(int)(g.grnd() * (double)p.nsig_trc)];
      const double nv = __dadd_rn(__shfl_sync(0xffffffffu, sg, itarget), __dmul_rn(gauss(g), pt_step_width<PEER>(p, px, p.dev_sig, 3, r, c)));
      if (lane == itarget) sg = nv;
      if (nv < p.sig_min[itarget] || nv > p.sig_max[itarget]) null_flag = true;
    }
    if (!null_flag) {
      const double dvp_half = lane_get(dp0, dp1, km - 1), dvs_half = lane_get(ds0, ds1, km - 1);
      if (!model_valid_warp(cfg, pk, z0, z1, dp0, dp1, ds0, ds1, dvp_half, dvs_half, lane)) null_flag = true;
    }
    double log_r = 0.0;
    if (!null_flag) {  // judge_mcmc draws (src/pt_mcmc.f90:610-615): independent of the likelihood
      double rr;
      do { rr = g.grnd(); } while (!(rr >= 2.220446049250313e-16));
      log_r = log(rr);
    }
    const int flag = null_flag ? -1 : (itype == p.it_sig ? 2 : 1);  // 1: forward needed, 2: cached RF (fwd_flag false)
    if (STAGED) {
      double* so = s_out + ic * S;
      if (lane < km - 1) so[lane] = z0;
      if (lane + 32 < km - 1) so[lane + 32] = z1;
      if (lane < km) { so[km + lane] = dp0; so[2 * km + lane] = ds0; }
      if (has1) { so[km + lane + 32] = dp1; so[2 * km + lane + 32] = ds1; }
      if (lane < T) so[3 * km + lane] = sg;
      if (nch <= 32) {
        if (lane == ic) { o_pk = pk; o_itype = itype; o_pflag = flag; o_logr = log_r; o_lp12 = log_prior12; }
      } else if (lane == 0) {
        p.pk[c] = pk; p.itype[c] = (int8_t)itype; p.pflag[c] = (int8_t)flag; p.log_r[c] = log_r; p.log_prior12[c] = log_prior12;
      }
    } else {
      if (lane < km - 1) p.pz[(size_t)lane * Cl + c] = z0;
      if (lane + 32 < km - 1) p.pz[(size_t)(lane + 32) * Cl + c] = z1;
      if (lane < km) { p.pdvp[(size_t)lane * Cl + c] = dp0; p.pdvs[(size_t)lane * Cl + c] = ds0; }
      if (has1) { p.pdvp[(size_t)(lane + 32) * Cl + c] = dp1; p.pdvs[(size_t)(lane + 32) * Cl + c] = ds1; }
      if (lane < T) p.psig[(size_t)lane * Cl + c] = sg;
      if (lane == 0) {
        p.pk[c] = pk; p.itype[c] = (int8_t)itype; p.pflag[c] = (int8_t)flag; p.log_r[c] = log_r; p.log_prior12[c] = log_prior12;
      }
    }
  }
  // The rank's part of the swap table (src/pt_mcmc.f90:501-516), here because it is the rank's last use of its stream in the
  // iteration: the owner of virtual rank 0 draws the pair (consuming its stream), then every rank leaves the NEXT uniform of
  // its stream -- what judge_pt would draw if the rank turns out to be rank1 -- without consuming it (pt_swap_kernel does).
  if (r == 0) {
    double t1 = -1.0, t2 = -1.0;
    if (p.rank_begin == 0 && p.nchains >= 2) {
      const int n_all = p.nproc_total * p.nchains;
      const int i1 = (int)(g.grnd() * (double)n_all);
      int i2;
      do { i2 = (int)(g.grnd() * (double)n_all); } while (i2 == i1);
      t1 = i1; t2 = i2;
    }
    if (lane == 0) { table[2 * Cl + p.G] = t1; table[2 * Cl + p.G + 1] = t2; }   // (PEER: pt_pairpush_kernel takes it to the other processes)
  }
  {
    const double u = g.peek();   // may reload the state (mti 624 -> 0); nothing is consumed
    if (lane == 0) { table[2 * Cl + r] = u; p.mti[r] = g.mti; }
  }
  if (STAGED) {
    __syncwarp();
    if (even) {
      for (int row = st_row0; row < rows; row += st_step) {
        int col;
        double* dst = const_cast<double*>(state_row(row, p.pz, p.pdvp, p.pdvs, p.psig, col));
        dst[c0 + st_ic] = s_out[st_ic * S + col];
      }
    } else {
      for (int idx = lane; idx < rows * nch; idx += 32) {
        const int row = idx / nch, ic = idx - row * nch;
        int col;
        double* dst = const_cast<double*>(state_row(row, p.pz, p.pdvp, p.pdvs, p.psig, col));
        dst[c0 + ic] = s_out[ic * S + col];
      }
    }
    if (nch <= 32 && lane < nch) {
      const int c = c0 + lane;
      p.pk[c] = o_pk; p.itype[c] = (int8_t)o_itype; p.pflag[c] = (int8_t)o_pflag; p.log_r[c] = o_logr; p.log_prior12[c] = o_lp12;
    }
  }
  // List of the chains that need a forward evaluation (pflag == 1), built here: one atomicAdd per rank reserves the rank's
  // slots, its chains go in ascending order.  The order of the ranks in the list follows their arrival -- it only decides
  // which CTA evaluates which chain; every chain's result is computed on its own (no sum runs across rows of a block), so the
  // results do not depend on it.  *p.n_active was left at zero by the previous iteration's pt_swap_kernel.
  __syncwarp();
  for (int base = 0; base < nch; base += 32) {
    const int ic = base + lane;
    int f;
    if (STAGED && nch <= 32) f = lane < nch && o_pflag == 1;
    else f = ic < nch && __ldcg(reinterpret_cast<const signed char*>(p.pflag) + c0 + ic) == 1;   // written by lane 0 above
    const unsigned m = __ballot_sync(0xffffffffu, f);
    int pos = 0;
    if (lane == 0 && m) { pos = atomicAdd(p.n_active, __popc(m)); atomicAdd(p.n_eval, (unsigned long long)__popc(m)); }
    pos = __shfl_sync(0xffffffffu, pos, 0);
    if (f) p.active[pos + __popc(m & ((1u << lane) - 1u))] = c0 + ic;
  }
}


// ---------------- acceptance: src/pt_mcmc.f90:178-201, one thread per chain ----------------
// slot of the current iteration in the optional logs, or -1
__device__ __forceinline__ int pt_log_slot(const PtDev& p) {
  if (!p.log_flags) return -1;
  const int s = *p.it_dev - p.log_base;
  return (s >= 0 && s < p.log_cap) ? s : -1;
}

// judge_pt (src/pt_mcmc.f90:580-595) on the gathered swap tables (`world` tables of table_len doubles, process order; a
// single process: its own table); called by ONE thread.  Ends the iteration: advances the device-side iteration counter and
// empties the list of chains to evaluate.
__device__ void pt_swap_decide(const PtDev& p, const double* gathered, int world, int table_len) {
  const int log_slot = pt_log_slot(p);
  *p.it_dev += 1;                    // the iteration is complete
  *p.n_active = 0;                   // pt_propose_kernel of the next iteration appends to an empty list
  if (p.nchains < 2) return;
  const int G = p.G, Cl = p.Cl;
  const double* t0 = gathered;  // process 0 owns virtual rank 0
  const int i1 = (int)__ldcg(t0 + 2 * Cl + G), i2 = (int)__ldcg(t0 + 2 * Cl + G + 1);
  const int own1 = i1 / Cl, own2 = i2 / Cl, l1 = i1 - own1 * Cl, l2 = i2 - own2 * Cl;
  const double* ta = gathered + (size_t)own1 * table_len;
  const double* tb = gathered + (size_t)own2 * table_len;
  const double temp1 = __ldcg(ta + l1), temp2 = __ldcg(tb + l2), e1 = __ldcg(ta + Cl + l1), e2 = __ldcg(tb + Cl + l2);
  const int rank1_local = l1 / p.nchains;
  const double u = __ldcg(ta + 2 * Cl + rank1_local);
  const double del_s = __dmul_rn(__dsub_rn(e2, e1), __dsub_rn(__ddiv_rn(1.0, temp1), __ddiv_rn(1.0, temp2)));
  const int yn = log(u) <= del_s;
  if (p.st_on) { p.st_pair[0] = i1; p.st_pair[1] = i2; }   // the next iteration's pair rule (step tuning)
  const int me = p.rank_begin / G;
  if (me == own1) {
    p.mti[rank1_local] += 1;  // the stream of rank1 consumed the judge_pt uniform
    if (yn) p.temps[l1] = temp2;
  }
  if (me == own2 && yn) p.temps[l2] = temp1;
  if (log_slot >= 0) {
    p.log_swaps[3 * log_slot] = i1; p.log_swaps[3 * log_slot + 1] = i2; p.log_swaps[3 * log_slot + 2] = yn;
  }
}

// ---------------- the tail of an iteration in ONE kernel, one thread per chain ----------------
//   acceptance            src/pt_mcmc.f90:178-201 (judge_mcmc :600-621)
//   adoption              src/pt_mcmc.f90:186-194: the accepted proposal becomes the state (rows z | dvp | dvs | sig | phi)
//   likelihood_hist(it)   src/pt_mcmc.f90:199-200: tree sum per CTA; the CTA that arrives last adds the per-CTA sums in CTA order
//                         (the same value from run to run whatever the schedule)
//   swap table            [0,Cl) temps | [Cl,2Cl) logL | [2Cl,2Cl+G) next uniform of every local stream | itarget1, itarget2
//                         (the last G + 2 entries were left by pt_propose_kernel)
// PEER: every entry of the table also goes straight into slot `me` of every process's gather buffer (peer memory over
// NVLink) and the last CTA raises this process's flag on every process (rfinv_pt.h, PtPeers) -- the all-gather of the swap
// exchange (src/pt_mcmc.f90:518-571) fused into the kernel that produces its payload.
// SWAP (single process, no bookkeeping kernels in between): the last CTA also takes the swap decision.
// (Four kernels -- accept, adopt, likelihood history, table -- and a fifth for the swap until round 2: every boundary
// between two small dependent kernels costs more than the kernels themselves.)
constexpr int PT_FIN_THREADS = 128;   // 32 chains per CTA: warp 0 decides, the four warps share the rows of the adoption
constexpr int PT_FIN_CHAINS = 32;
template <bool PEER, bool SWAP>
__global__ void __launch_bounds__(PT_FIN_THREADS) pt_finish_kernel(const DevConfig cfg, const PtDev p, double* __restrict__ table,
                                                                   const PtPeers px, double* __restrict__ lhist,
                                                                   double* __restrict__ part, int* __restrict__ arrived) {
  __shared__ double s_sum[PT_FIN_THREADS / 32];
  __shared__ int s_code[PT_FIN_CHAINS];
  __shared__ int s_last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = blockIdx.x * PT_FIN_CHAINS + lane;
  const int km = cfg.k_max, Cl = p.Cl, T = cfg.ntrc;
  const int it = *p.it_dev;
  if (PEER) table += (size_t)(it & 1) * (2 * Cl + p.G + 2);   // pt_push_kernel takes it to the other processes during the next iteration
  auto put = [&](int idx, double v) { table[idx] = v; };
  double cold_logl = 0.0;
  if (warp == 0) {
    // PEER: the previous iteration's swap exchanges its two temperatures here, in front of their first reader (every CTA takes
    // the decision for itself from the tables that arrived during this iteration; the owners' threads adopt the new values)
    int sw_l1 = -1, sw_l2 = -1;
    double sw_t1 = 0.0, sw_t2 = 0.0;
    if (PEER && p.nchains >= 2 && px.done[1] < it) {
      if (lane < px.world) pt_peer_wait(px, px.own_flag + lane, (unsigned long long)it);
      __syncwarp();
      const double* pr = pt_pair_slot(px.own_flag, px.world, it - 1);
      const SwapPlan sp = pt_swap_plan(p, __ldcg(pr), __ldcg(pr + 1));
      const double* gathered = px.own_gather + (size_t)((it - 1) & 1) * px.world * px.table_len;
      const double* ta = gathered + (size_t)sp.own1 * px.table_len;
      const double* tb = gathered + (size_t)sp.own2 * px.table_len;
      const double temp1 = __ldcg(ta + sp.l1), temp2 = __ldcg(tb + sp.l2), e1 = __ldcg(ta + Cl + sp.l1), e2 = __ldcg(tb + Cl + sp.l2);
      const double u = __ldcg(ta + 2 * Cl + sp.rank1_local);
      const double del_s = __dmul_rn(__dsub_rn(e2, e1), __dsub_rn(__ddiv_rn(1.0, temp1), __ddiv_rn(1.0, temp2)));
      const int yn = log(u) <= del_s;
      if (yn) {
        if (sp.own1 == px.me) { sw_l1 = sp.l1; sw_t1 = temp2; }
        if (sp.own2 == px.me) { sw_l2 = sp.l2; sw_t2 = temp1; }
      }
      if (blockIdx.x == 0 && lane == 0 && p.log_flags) {
        const int ls = it - 1 - p.log_base;
        if (ls >= 0 && ls < p.log_cap) { p.log_swaps[3 * ls] = sp.i1; p.log_swaps[3 * ls + 1] = sp.i2; p.log_swaps[3 * ls + 2] = yn; }
      }
    }
    int code = 0;   // 3: adopt model and phi, 4: model only (sigma-only proposal), 0: nothing
    if (c < Cl) {
      const int flag = p.pflag[c];
      double temp = p.temps[c];
      if (PEER) {
        if (c == sw_l1) { temp = sw_t1; p.temps[c] = temp; }
        else if (c == sw_l2) { temp = sw_t2; p.temps[c] = temp; }
      }
      double logl = p.logl[c];
      int yn = 0;
      if (flag != -1) {
        double ll = 0.0;
        for (int t = 0; t < T; ++t) {  // src/likelihood.f90:94-96; sigma-only proposals reuse the cached phi (same rft, same obs)
          const double ph = flag == 1 ? p.pphi[(size_t)t * Cl + c] : p.phi[(size_t)t * Cl + c];
          const double sg = p.psig[(size_t)t * Cl + c];
          ll = __dsub_rn(__dsub_rn(ll, __ddiv_rn(__dmul_rn(0.5, ph), __dmul_rn(sg, sg))), __dmul_rn((double)cfg.nsmp, log(sg)));
        }
        const double del_s = __dadd_rn(__ddiv_rn(__dsub_rn(ll, logl), temp), p.log_prior12[c]);  // src/pt_mcmc.f90:608
        yn = p.log_r[c] <= del_s;
        if (yn) {
          logl = ll;
          p.logl[c] = ll;
          p.k[c] = p.pk[c];
          if (flag == 1) p.slot[c] ^= 1;  // the proposal's RF samples were written to the other slot
          code = flag == 1 ? 3 : 4;
        }
      }
      if (p.st_on) {   // step tuning: the proposal counts against (rank, level, type); lvl is a permutation in each rank
        const int tau = pt_step_type(p, p.itype[c]);
        const int gc = p.rank_begin * p.nchains + c;
        if (tau >= 0 && gc != p.st_pair[0] && gc != p.st_pair[1]) {
          const size_t row = ((size_t)(c - c % p.nchains) + p.st_lvl[c]) * 4 + tau;
          p.st_nprop[row] += 1ULL;
          p.st_nacc[row] += (unsigned long long)yn;
        }
      }
      const bool cold = temp <= 1.0 + (double)1.0e-6f;
      if (cold) {  // src/pt_mcmc.f90:196-201
        atomicAdd(&p.nprop[p.itype[c] - 1], 1ULL);
        if (yn) atomicAdd(&p.naccept[p.itype[c] - 1], 1ULL);
        cold_logl = logl;
      }
      const int log_slot = pt_log_slot(p);
      if (log_slot >= 0) {
        p.log_flags[(size_t)log_slot * Cl + c] = (int8_t)(flag == -1 ? -1 : yn);
        p.log_itypes[(size_t)log_slot * Cl + c] = p.itype[c];
      }
      put(c, temp);
      put(Cl + c, logl);
    }
    s_code[lane] = code;
    // likelihood history: fixed tree over the CTA's chains
    for (int o = 16; o > 0; o >>= 1) cold_logl += __shfl_down_sync(0xffffffffu, cold_logl, o);
    if (lane == 0) part[blockIdx.x] = cold_logl;
  }
  __syncthreads();
  {
    // the accepted proposals become the state (src/pt_mcmc.f90:186-194): rows z | dvp | dvs | sig | phi of the chain-fastest
    // arrays; lane <-> chain (coalesced), the four warps take every fourth row, eight independent copies in flight
    const int code = s_code[lane];
    if (code >= 3) {
      const int rows = 3 * km - 1 + T + (code == 3 ? T : 0);   // phi only when the forward model ran
      auto row_ptrs = [&](int row, const double*& src, double*& dst) {
        if (row < km - 1) { src = p.pz; dst = p.z; }
        else if ((row -= km - 1) < km) { src = p.pdvp; dst = p.dvp; }
        else if ((row -= km) < km) { src = p.pdvs; dst = p.dvs; }
        else if ((row -= km) < T) { src = p.psig; dst = p.sig; }
        else { row -= T; src = p.pphi; dst = p.phi; }
        src += (size_t)row * Cl + c; dst += (size_t)row * Cl + c;
      };
      for (int row0 = warp; row0 < rows; row0 += 8 * (PT_FIN_THREADS / 32)) {
        double v[8]; double* d[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int row = row0 + q * (PT_FIN_THREADS / 32);
          d[q] = nullptr;
          if (row < rows) { const double* sp; row_ptrs(row, sp, d[q]); v[q] = *sp; }
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) if (d[q]) *d[q] = v[q];
      }
    }
  }
  // the table entries (warp 0) are ordered before the arrival below; the adopted rows are only read by later kernels and
  // need no fence
  if (warp == 0) __threadfence();
  __syncthreads();
  if (tid == 0) s_last = atomicAdd(arrived, 1) == (int)gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  // the last CTA (every CTA's stores precede its arrival): the per-CTA sums in a fixed order -- thread t adds the sums of the
  // CTAs t, t + 128, ..., then the same tree as above -- with all loads in flight at once
  __threadfence();
  double tot = 0.0;
  for (unsigned b = tid; b < gridDim.x; b += PT_FIN_THREADS) tot += __ldcg(part + b);
  for (int o = 16; o > 0; o >>= 1) tot += __shfl_down_sync(0xffffffffu, tot, o);
  __syncthreads();              // (s_sum is being reused)
  if ((tid & 31) == 0) s_sum[tid >> 5] = tot;
  __syncthreads();
  if (tid == 0) {
    double acc = 0.0;
    for (int w = 0; w < PT_FIN_THREADS / 32; ++w) acc += s_sum[w];
    lhist[it] = acc;
    *arrived = 0;
    if (PEER) {
      px.done[0] = it; px.done[1] = it;   // the swaps of the iterations before this one are applied; this one's follows in the next
      *p.it_dev = it + 1;                 // the iteration is complete
      *p.n_active = 0;
    }
    if (SWAP) pt_swap_decide(p, table, 1, px.table_len);
  }
}

// judge_pt (src/pt_mcmc.f90:580-595) evaluated identically by every process from the gathered tables.
__global__ void pt_swap_kernel(const PtDev p, const double* gathered, int world, int table_len) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  pt_swap_decide(p, gathered, world, table_len);
}

// ---------------- even/odd temperature swaps inside every virtual rank (rfinv_pt_set_rank_swaps, DESIGN.md 7c) ----------------
// Philox4x64-10 (Salmon, Moraes, Dror & Shaw, SC 2011), output word 0: a counter-based generator without state, so the sweep
// leaves the mt19937 streams -- and with them every draw of the reference -- exactly as they are.
__device__ __forceinline__ uint64_t philox4x64_w0(uint64_t c0, uint64_t c1, uint64_t c2, uint64_t c3, uint64_t k0, uint64_t k1) {
  constexpr uint64_t M0 = 0xD2E7470EE14C6C93ULL, M1 = 0xCA5A826395121157ULL;
#pragma unroll
  for (int round = 0; round < 10; ++round) {
    if (round) { k0 += 0x9E3779B97F4A7C15ULL; k1 += 0xBB67AE8584CAA73BULL; }
    const uint64_t hi0 = __umul64hi(M0, c0), lo0 = M0 * c0, hi1 = __umul64hi(M1, c2), lo1 = M1 * c2;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
  }
  return c0;
}

// One WARP per virtual rank, after acceptance and bookkeeping, before the global swap.  Level of a chain = its place in the
// rank's chains sorted by (temperature, chain index), found by counting; levels l = i (mod 2) and l + 1 are proposed a swap
// with judge_pt's test (src/pt_mcmc.f90:580-595) and the Philox uniform of counter (i, global rank, l, 0).  Accepted pairs
// exchange their temperatures in temps and in the swap table.  peer: the peer-memory exchange, where pt_finish_kernel has
// already advanced *it_dev and the table alternates.  DECIDE (single process): the last CTA then takes the global swap
// decision that pt_finish_kernel<false, true> takes without the sweep.
// With the ladder tuning on (p.rs_tune), the iterations e - 1 of the tuning points e then retune every rank's ladder
// (pt_tune_ladder) before the global swap reads the table.  With the step tuning on (p.st_on), every iteration records the
// post-sweep levels (st_lvl) for the next iteration's proposals, and the tuning points' iterations tune the widths (pt_tune_steps).
constexpr int PT_RS_WARPS = 4;

// chain of the rank at each level: its place among the chains c0 .. c0 + n - 1 sorted by (temperature, chain index)
__device__ __forceinline__ void pt_rank_levels(const PtDev& p, int c0, int n, int lane, int* at) {
  for (int a = lane; a < n; a += 32) {
    const double ta = p.temps[c0 + a];
    int lvl = 0;
    for (int b = 0; b < n; ++b) { const double tb = p.temps[c0 + b]; lvl += tb < ta || (tb == ta && b < a); }
    at[lvl] = a;
  }
  __syncwarp();
}

// Ladder tuning of virtual rank r at tuning point e (DESIGN.md 7d; the C reference is lo_tune_rank in tests/ladder_oracle.c):
// the levels a+1 .. n-2 above the cold anchor a take the inverse temperatures that split the rank's rejection barrier
// Lambda -- the running sum of the per-pair rejection rates of the round [s, e) -- into equal parts, interpolated linearly in
// beta between the old levels.  One warp; the levels and the old ladder go to shared memory, lane 0 does the O(n) walk.
// Every operation is rounded on its own, as in the reference.
__device__ void pt_tune_ladder(const PtDev& p, double* __restrict__ table, int r, int e, int lane, int* at, double* lt) {
  const int n = p.nchains, c0 = r * n, nl = n - 1;
  pt_rank_levels(p, c0, n, lane, at);   // the sweep has just exchanged temperatures
  for (int l = lane; l < n; l += 32) lt[l] = p.temps[c0 + at[l]];
  __syncwarp();
  unsigned long long* acc = p.rs_nacc + (size_t)r * nl;
  unsigned long long* base = p.rs_base + (size_t)r * nl;
  if (lane == 0) {
    const double cold = 1.0 + (double)1.0e-6f;
    int c = 0;
    while (c < n && lt[c] <= cold) ++c;   // the cold chains are the lowest levels
    const int a = c > 0 ? c - 1 : 0, K = nl - a;
    if (K >= 2) {
      const int s = e == 64 ? 0 : e / 2;
      const double P = (double)((e - s) / 2);
      auto rho = [&](int l) {
        const double q = __ddiv_rn((double)(acc[l] - base[l]), P);
        const double x = __dsub_rn(1.0, q);
        return x < 0x1p-10 ? 0x1p-10 : x;
      };
      double LK = 0.0;
      for (int m = 0; m < K; ++m) LK = __dadd_rn(LK, rho(a + m));
      // pass 0 checks the guard, pass 1 writes; both walk the same ladder (the new T' are read from the old ladder lt only)
      for (int pass = 0; pass < 2; ++pass) {
        int m = 0;
        double Lm = 0.0, Lm1 = rho(a), prev = lt[a];
        bool ok = true;
        for (int k = 1; k < K; ++k) {
          const double lam = __ddiv_rn(__dmul_rn(LK, (double)k), (double)K);
          while (m < K - 1 && !(lam < Lm1)) { ++m; Lm = Lm1; Lm1 = __dadd_rn(Lm1, rho(a + m)); }
          const double f = __ddiv_rn(__dsub_rn(lam, Lm), __dsub_rn(Lm1, Lm));
          const double bm = __ddiv_rn(1.0, lt[a + m]), bm1 = __ddiv_rn(1.0, lt[a + m + 1]);
          const double t = __ddiv_rn(1.0, __dadd_rn(bm, __dmul_rn(f, __dsub_rn(bm1, bm))));
          if (pass == 0) { ok = ok && t > prev && t > cold; prev = t; }
          else { const int ch = c0 + at[a + k]; p.temps[ch] = t; table[ch] = t; }
        }
        if (pass == 0 && !(ok && lt[nl] > prev)) break;   // the guard: this rank keeps its ladder for this round
      }
    }
  }
  __syncwarp();
  for (int l = lane; l < nl; l += 32) base[l] = acc[l];
}

// Step tuning of virtual rank r at a tuning point (DESIGN.md 7e; the C reference is so_tune_rank in tests/step_oracle.c): every
// (level, type) the run proposes with at least 16 proposals in the round moves its scale by the factor (acceptance / target),
// clamped to [1/2, 2], the scale itself to [2^-8, 2^8]; every counter of the rank restarts at zero.  Lanes over the 4n entries.
__device__ void pt_tune_steps(const PtDev& p, int r, int lane) {
  const size_t base = (size_t)r * p.nchains * 4;
  for (int j = lane; j < 4 * p.nchains; j += 32) {
    const int tau = j & 3;
    const bool proposed = tau < 2 || (tau == 2 ? p.it_dvp > 0 : p.it_sig > 0);
    const unsigned long long P = p.st_nprop[base + j], A = p.st_nacc[base + j];
    if (proposed && P >= 16) {
      double f = __ddiv_rn(__ddiv_rn((double)A, (double)P), p.st_target);
      f = f < 0.5 ? 0.5 : (f > 2.0 ? 2.0 : f);
      double s = __dmul_rn(p.st_scale[base + j], f);
      s = s < 0x1p-8 ? 0x1p-8 : (s > 0x1p8 ? 0x1p8 : s);
      p.st_scale[base + j] = s;
    }
    p.st_nprop[base + j] = 0ULL;
    p.st_nacc[base + j] = 0ULL;
  }
}

template <bool DECIDE>
__global__ void __launch_bounds__(32 * PT_RS_WARPS) pt_rank_swap_kernel(const PtDev p, double* __restrict__ table, int table_len,
                                                                        int peer) {
  // [warps][nchains] chain at each level; with the ladder tuning on, [warps][nchains] doubles of the old ladder first
  extern __shared__ double rs_smem[];
  __shared__ int s_last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n = p.nchains;
  const int r = blockIdx.x * (blockDim.x >> 5) + warp;
  const int it = *p.it_dev - peer;
  if (peer) table += (size_t)(it & 1) * table_len;
  if (r < p.G) {
    int* at = (int*)(rs_smem + (p.rs_tune ? (size_t)(blockDim.x >> 5) * n : 0)) + (size_t)warp * n;
    const int c0 = r * n;
    pt_rank_levels(p, c0, n, lane, at);
    const uint64_t grank = (uint64_t)(p.rank_begin + r), key = (uint64_t)(uint32_t)p.iseed;
    for (int l = (it & 1) + 2 * lane; l + 1 < n; l += 64) {
      const int a = c0 + at[l], b = c0 + at[l + 1];
      const double ta = p.temps[a], tb = p.temps[b];
      const uint64_t w = philox4x64_w0((uint64_t)it, grank, (uint64_t)l, 0, key, 0);
      const double u = (double)(w >> 11) * 0x1p-53;
      const double del_s = __dmul_rn(__dsub_rn(p.logl[b], p.logl[a]), __dsub_rn(__ddiv_rn(1.0, ta), __ddiv_rn(1.0, tb)));
      const int yn = log(u) <= del_s;
      if (yn) { p.temps[a] = tb; p.temps[b] = ta; table[a] = tb; table[b] = ta; }
      p.rs_nacc[(size_t)r * (n - 1) + l] += (unsigned long long)yn;
    }
    if (r == 0 && lane == 0)
      for (int l = it & 1; l + 1 < n; l += 2) p.rs_nprop[l] += (unsigned long long)p.G;
    const int e = it + 1;   // the iteration count at the end of this iteration: a tuning point?
    const bool tune_point = e >= 64 && e <= p.nburn && (e & (e - 1)) == 0;
    if (p.rs_tune && tune_point) {
      __syncwarp();          // the sweep's exchanges and counts are visible to the whole warp
      pt_tune_ladder(p, table, r, e, lane, at, rs_smem + (size_t)warp * n);
    }
    if (p.st_on) {
      __syncwarp();          // the sweep's (and the ladder tuning's) exchanges are visible; `at` is free again
      pt_rank_levels(p, c0, n, lane, at);   // the post-sweep levels (the ladder tuning keeps their order)
      for (int l = lane; l < n; l += 32) p.st_lvl[c0 + at[l]] = l;
      if (tune_point) pt_tune_steps(p, r, lane);
    }
  }
  if (!DECIDE) return;
  __threadfence();   // this CTA's table entries are ordered before its arrival
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(p.rs_arrived, 1) == (int)gridDim.x - 1;
  __syncthreads();
  if (!s_last || threadIdx.x != 0) return;
  __threadfence();
  *p.rs_arrived = 0;
  pt_swap_decide(p, table, 1, table_len);
}

// Peer-memory exchange, side branch of the iteration (rfinv_pt.h).  pt_pairpush_kernel: one warp; the owner of virtual rank 0
// takes the pair pt_propose_kernel has just drawn (local table, parity it & 1) to every process.
__global__ void pt_pairpush_kernel(const PtDev p, const double* __restrict__ table, const PtPeers px) {
  if (p.rank_begin != 0 || p.nchains < 2 || threadIdx.x != 0) return;
  const int it = *p.it_dev;
  const double* tab = table + (size_t)(it & 1) * px.table_len + 2 * p.Cl + p.G;
  const double t1 = __ldcg(tab), t2 = __ldcg(tab + 1);
#pragma unroll
  for (int q = 0; q < RFINV_MAX_PEERS; ++q)
    if (q < px.world) { double* ps = pt_pair_slot(px.flag[q], px.world, it); ps[0] = t1; ps[1] = t2; }
  __threadfence_system();
#pragma unroll
  for (int q = 0; q < RFINV_MAX_PEERS; ++q)
    if (q < px.world) st_release_sys(pt_pair_flag(px.flag[q], px.world), (unsigned long long)it + 1ULL);
}

// pt_push_kernel: the swap table of the iteration before (local table, parity (it - 1) & 1) goes into slot `me` of every
// process's gather buffer; the last CTA raises this process's table flag everywhere.  Runs beside pt_propose_kernel of iteration
// `it` (and once more in front of pt_drain_kernel); a table is pushed once (done[2]).
constexpr int PT_PUSH_THREADS = 256;
__global__ void __launch_bounds__(PT_PUSH_THREADS) pt_push_kernel(const PtDev p, const double* __restrict__ table, const PtPeers px) {
  __shared__ int s_last;
  const int it = *p.it_dev;
  if (it < 1 || px.done[2] >= it) return;          // nothing to push (uniform over the grid: done[2] only changes at the very end)
  const int prev = it - 1;
  const double* tab = table + (size_t)(prev & 1) * px.table_len;
  const size_t slot = ((size_t)(prev & 1) * px.world + px.me) * px.table_len;
  for (int i = blockIdx.x * PT_PUSH_THREADS + threadIdx.x; i < px.table_len; i += gridDim.x * PT_PUSH_THREADS) {
    const double v = __ldcg(tab + i);
#pragma unroll
    for (int q = 0; q < RFINV_MAX_PEERS; ++q) if (q < px.world) px.gather[q][slot + i] = v;
  }
  __threadfence_system();     // this thread's stores into peer memory are ordered before the arrival below
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(px.done + 3, 1) == (int)gridDim.x - 1;
  __syncthreads();
  if (s_last && threadIdx.x == 0) {   // every CTA's stores precede its arrival: the table is complete everywhere
    __threadfence_system();
#pragma unroll
    for (int q = 0; q < RFINV_MAX_PEERS; ++q) if (q < px.world) st_release_sys(px.flag[q] + px.me, (unsigned long long)it);
    px.done[3] = 0;
    px.done[2] = it;
  }
}

// Peer-memory exchange: the swap of the LAST iteration of a run, in full (stream shift, temperatures, log) -- inside the
// run every swap is applied one iteration later by pt_propose_kernel / pt_finish_kernel.  One warp.
__global__ void pt_drain_kernel(const PtDev p, const PtPeers px) {
  const int lane = threadIdx.x & 31;
  const int it = *p.it_dev;                   // iterations completed; the pending swap is that of iteration it - 1
  if (p.nchains < 2 || it < 1 || px.done[1] >= it) return;
  if (lane < px.world) pt_peer_wait(px, px.own_flag + lane, (unsigned long long)it);
  if (lane == 0) pt_peer_wait(px, pt_pair_flag(px.own_flag, px.world), (unsigned long long)it);
  __syncwarp();
  if (lane != 0) return;
  const int Cl = p.Cl;
  const double* pr = pt_pair_slot(px.own_flag, px.world, it - 1);
  const SwapPlan sp = pt_swap_plan(p, __ldcg(pr), __ldcg(pr + 1));
  const double* gathered = px.own_gather + (size_t)((it - 1) & 1) * px.world * px.table_len;
  const double* ta = gathered + (size_t)sp.own1 * px.table_len;
  const double* tb = gathered + (size_t)sp.own2 * px.table_len;
  const double temp1 = __ldcg(ta + sp.l1), temp2 = __ldcg(tb + sp.l2), e1 = __ldcg(ta + Cl + sp.l1), e2 = __ldcg(tb + Cl + sp.l2);
  const double u = __ldcg(ta + 2 * Cl + sp.rank1_local);
  const double del_s = __dmul_rn(__dsub_rn(e2, e1), __dsub_rn(__ddiv_rn(1.0, temp1), __ddiv_rn(1.0, temp2)));
  const int yn = log(u) <= del_s;
  if (sp.own1 == px.me) {
    if (px.done[0] < it) p.mti[sp.rank1_local] += 1;
    if (yn) p.temps[sp.l1] = temp2;
  }
  if (sp.own2 == px.me && yn) p.temps[sp.l2] = temp1;
  if (p.st_on) { p.st_pair[0] = sp.i1; p.st_pair[1] = sp.i2; }   // for the next run's first iteration (step tuning)
  if (p.log_flags) {
    const int ls = it - 1 - p.log_base;
    if (ls >= 0 && ls < p.log_cap) { p.log_swaps[3 * ls] = sp.i1; p.log_swaps[3 * ls + 1] = sp.i2; p.log_swaps[3 * ls + 2] = yn; }
  }
  px.done[0] = it; px.done[1] = it;
}

// ordered numbering of the non-tempered chains (deterministic slot of each recorded model in all_models)
__global__ void pt_coldscan_kernel(const PtDev p) {
  __shared__ int s_cnt[1024];
  __shared__ int s_base;
  const int tid = threadIdx.x, nthr = blockDim.x;
  if (tid == 0) s_base = 0;
  __syncthreads();
  for (int start = 0; start < p.Cl; start += nthr) {
    const int c = start + tid;
    const int f = (c < p.Cl && p.temps[c] <= 1.0 + (double)1.0e-6f) ? 1 : 0;
    s_cnt[tid] = f;
    __syncthreads();
    for (int o = 1; o < nthr; o <<= 1) {
      const int v = tid >= o ? s_cnt[tid - o] : 0;
      __syncthreads();
      s_cnt[tid] += v;
      __syncthreads();
    }
    if (c < p.Cl) p.cold_ordinal[c] = f ? s_base + s_cnt[tid] - 1 : -1;
    __syncthreads();
    if (tid == nthr - 1) s_base += s_cnt[tid];
    __syncthreads();
  }
  if (tid == 0) *p.cold_count = s_base;
}

// Posterior bookkeeping of one non-tempered chain per CTA (src/pt_mcmc.f90:204-286).
__global__ void pt_record_kernel(const DevConfig cfg, const PtDev p) {
  const int c = blockIdx.x;
  const int ord = p.cold_ordinal[c];
  if (ord < 0) return;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int km = cfg.k_max, Cl = p.Cl, T = cfg.ntrc, S = cfg.nsmp;
  __shared__ double s_alpha[RFINV_MAX_LAY], s_beta[RFINV_MAX_LAY];
  __shared__ int s_iz1[RFINV_MAX_LAY + 1], s_nlay;
  const double dbin_amp = (p.amp_max - p.amp_min) / p.nbin_amp, dbin_vp = (cfg.vp_max - cfg.vp_min) / p.nbin_vp;
  const double dbin_vs = (cfg.vs_max - cfg.vs_min) / p.nbin_vs, dbin_z = (cfg.z_max - 0.0) / p.nbin_z;
  const double dbin_vpvs = (cfg.vpvs_max - cfg.vpvs_min) / p.nbin_vpvs;
  const int k = p.k[c];
  const long long imod = (long long)(*p.nmod) + ord;   // nmod is advanced by pt_record_finish_kernel
  if (tid == 0) {
    atomicAdd(&p.nk[k - 1], 1ULL);
    for (int t = 0; t < T; ++t)
      if (p.sig_mode[t]) {
        const double dbs = (p.sig_max[t] - p.sig_min[t]) / p.nbin_sig;
        const int ibin = (int)((p.sig[(size_t)t * Cl + c] - p.sig_min[t]) / dbs) + 1;
        if (ibin >= 1 && ibin <= p.nbin_sig) atomicAdd(&p.nsig[(size_t)t * p.nbin_sig + ibin - 1], 1ULL);
      }
    for (int il = 1; il <= k - 1; ++il) {  // first k-1 interfaces in stored order (src/pt_mcmc.f90:224-227)
      const int ibin = (int)((p.z[(size_t)(il - 1) * Cl + c] - cfg.z_min) / dbin_z) + 1;
      if (ibin >= 1 && ibin <= p.nbin_z) atomicAdd(&p.nz[ibin - 1], 1ULL);
    }
    // format_model (src/model.f90:175-290) of the current state
    double z[RFINV_MAX_K], dp[RFINV_MAX_K], ds[RFINV_MAX_K];
    for (int i = 0; i < k; ++i) { z[i] = p.z[(size_t)i * Cl + c]; dp[i] = p.dvp[(size_t)i * Cl + c]; ds[i] = p.dvs[(size_t)i * Cl + c]; }
    for (int i = 1; i < k; ++i) {
      const double a = z[i], b = dp[i], d = ds[i];
      int m = i - 1;
      while (m >= 0 && z[m] > a) { z[m + 1] = z[m]; dp[m + 1] = dp[m]; ds[m + 1] = ds[m]; --m; }
      z[m + 1] = a; dp[m + 1] = b; ds[m + 1] = d;
    }
    int n = 0;
    double tmpz = 0.0;
    if (cfg.sdep > 0.0) {
      s_alpha[n] = 1.5; s_beta[n] = -999.0; s_iz1[n] = (int)(tmpz / dbin_z) + 1;
      tmpz = __dadd_rn(tmpz, cfg.sdep); ++n;
    }
    for (int l = 0; l <= k; ++l) {
      double zc, h, dvs_l, dvp_l;
      if (l == 0) { zc = __dmul_rn(0.5, __dadd_rn(cfg.sdep, z[0])); h = __dsub_rn(z[0], cfg.sdep); dvs_l = ds[0]; dvp_l = dp[0]; }
      else if (l < k) { zc = __dmul_rn(0.5, __dadd_rn(z[l], z[l - 1])); h = __dsub_rn(z[l], z[l - 1]); dvs_l = ds[l]; dvp_l = dp[l]; }
      else { zc = __dmul_rn(0.5, __dadd_rn(cfg.z_max, z[k - 1])); h = 999.0;
             dvs_l = p.dvs[(size_t)(km - 1) * Cl + c]; dvp_l = p.dvp[(size_t)(km - 1) * Cl + c]; }
      double a, b;
      layer_velocity(cfg, zc, dvs_l, dvp_l, a, b);
      s_alpha[n] = a; s_beta[n] = b;
      s_iz1[n] = (int)(__ddiv_rn(tmpz, dbin_z)) + 1;
      tmpz = __dadd_rn(tmpz, h);
      ++n;
    }
    s_iz1[n] = p.nbin_z + 1;   // iz2 of the half space (src/pt_mcmc.f90:243)
    s_nlay = n;
  }
  __syncthreads();
  const int nlay = s_nlay;
  // each depth bin belongs to exactly one layer: iz1(l) <= iz < iz1(l+1)
  for (int iz = 1 + tid; iz <= p.nbin_z; iz += nthr) {
    int l = 0;
    while (l + 1 < nlay && iz >= s_iz1[l + 1]) ++l;
    if (iz < s_iz1[l]) continue;
    const double a = s_alpha[l], b = s_beta[l];
    int ivp = (int)((a - cfg.vp_min) / dbin_vp) + 1;
    int ivs = (int)((b - cfg.vs_min) / dbin_vs) + 1;
    if (ivs < 1) ivs = 1;
    int ivpvs = (int)(((a / b) - cfg.vpvs_min) / dbin_vpvs) + 1;
    if (ivpvs < 1) ivpvs = 1;
    if (ivpvs > p.nbin_vpvs) ivpvs = p.nbin_vpvs;
    if (ivp > p.nbin_vp) ivp = p.nbin_vp;    // the reference would write out of bounds
    if (ivp < 1) ivp = 1;
    if (ivs > p.nbin_vs) ivs = p.nbin_vs;
    atomicAdd(&p.nvpz[(size_t)(ivp - 1) * p.nbin_z + iz - 1], 1ULL);
    atomicAdd(&p.vp_mean[iz - 1], a);
    atomicAdd(&p.nvsz[(size_t)(ivs - 1) * p.nbin_z + iz - 1], 1ULL);
    atomicAdd(&p.nvpvsz[(size_t)(ivpvs - 1) * p.nbin_z + iz - 1], 1ULL);
    double vs_rec;
    if (b > 0.0) {
      atomicAdd(&p.vpvs_mean[iz - 1], a / b);
      atomicAdd(&p.vs_mean[iz - 1], b);
      vs_rec = b;
    } else {  // src/pt_mcmc.f90:260-263: assignment, not accumulation (ocean layer)
      p.vpvs_mean[iz - 1] = cfg.vpvs_min;
      p.vs_mean[iz - 1] = cfg.vs_min;
      p.ocean_bin[iz - 1] = 1;
      vs_rec = cfg.vs_min;
    }
    if (p.vp_model && imod < p.cap_models) {
      p.vp_model[(size_t)imod * p.nbin_z + iz - 1] = a;
      p.vs_model[(size_t)imod * p.nbin_z + iz - 1] = vs_rec;
    }
  }
  // RF amplitude histogram (src/pt_mcmc.f90:271-284) from the cached RF samples of the current state
  const double* rft = p.slot[c] ? p.rft_smp[1] : p.rft_smp[0];
  for (int i = tid; i < T * S; i += nthr) {
    const int t = i / S, it = i - t * S;
    int ibin = (int)((rft[((size_t)t * Cl + c) * S + it] - p.amp_min) / dbin_amp) + 1;
    if (ibin < 1) ibin = 1; else if (ibin > p.nbin_amp) ibin = p.nbin_amp;
    atomicAdd(&p.namp[((size_t)t * S + it) * p.nbin_amp + ibin - 1], 1ULL);
  }
}
__global__ void pt_record_finish_kernel(const PtDev p) { *p.nmod += (unsigned long long)*p.cold_count; }
// After the job-wide sum over processes (rfinv_pt_reduce_outputs): the bins the reference ASSIGNS instead of accumulating hold
// (processes that recorded) x the assigned value; they are set back to the value itself, so that the job-wide result does not
// depend on how many processes the virtual ranks were spread over (in the reference it does: DESIGN.md section 8).
__global__ void pt_fix_ocean_kernel(const DevConfig cfg, const PtDev p) {
  const int iz = blockIdx.x * blockDim.x + threadIdx.x;
  if (iz < p.nbin_z && p.ocean_bin[iz]) { p.vs_mean[iz] = cfg.vs_min; p.vpvs_mean[iz] = cfg.vpvs_min; }
}

template <typename T>
int dalloc(T** p, size_t n) {
  RFINV_CUDA_CHECK(cudaMalloc((void**)p, sizeof(T) * (n ? n : 1)));
  RFINV_CUDA_CHECK(cudaMemset(*p, 0, sizeof(T) * (n ? n : 1)));
  return RFINV_OK;
}

}  // namespace

int rfinv_pt_fix_assigned_bins(rfinv_handle* h) {
  PtDev& d = h->pt->dev;
  pt_fix_ocean_kernel<<<(d.nbin_z + 127) / 128, 128, 0, h->stream>>>(h->dc, d);
  RFINV_CUDA_CHECK(cudaGetLastError());
  return RFINV_OK;
}

// drops the captured iterations: something baked into their launches changed.  A new generation tells the groups the handle
// is in (rfinv_pt_group_run) to capture theirs again.
static void pt_drop_graphs(PtState* s) {
  for (cudaGraphExec_t& g : s->graph) { if (g) cudaGraphExecDestroy(g); g = nullptr; }
  s->generation = rfinv_pt_next_generation();
}

void rfinv_handle::invalidate_pt_graphs() {
  if (pt) pt_drop_graphs(pt);
}

void rfinv_handle::free_pt() {
  if (!pt) return;
  PtDev& d = pt->dev;
  cudaFree(d.mt); cudaFree(d.mti); cudaFree(d.k); cudaFree(d.z); cudaFree(d.dvp); cudaFree(d.dvs); cudaFree(d.sig);
  cudaFree(d.logl); cudaFree(d.temps); cudaFree(d.phi); cudaFree(d.slot); cudaFree(d.rft_smp[0]); cudaFree(d.rft_smp[1]);
  cudaFree(d.pk); cudaFree(d.pz); cudaFree(d.pdvp); cudaFree(d.pdvs); cudaFree(d.psig); cudaFree(d.pphi); cudaFree(d.log_r);
  cudaFree(d.log_prior12); cudaFree(d.itype); cudaFree(d.pflag); cudaFree(d.active); cudaFree(d.n_active);
  cudaFree(d.nprop); cudaFree(d.naccept); cudaFree(d.n_eval); cudaFree(d.rs_nprop); cudaFree(d.rs_nacc); cudaFree(d.rs_arrived);
  cudaFree(d.rs_base); cudaFree(d.st_scale); cudaFree(d.st_nprop); cudaFree(d.st_nacc); cudaFree(d.st_lvl); cudaFree(d.st_pair);
  cudaFree(d.log_flags); cudaFree(d.log_itypes); cudaFree(d.log_swaps);
  cudaFree(d.nk); cudaFree(d.nz); cudaFree(d.nsig); cudaFree(d.namp); cudaFree(d.nvpz); cudaFree(d.nvsz); cudaFree(d.nvpvsz); cudaFree(d.nmod);
  cudaFree(d.vp_mean); cudaFree(d.vs_mean); cudaFree(d.vpvs_mean); cudaFree(d.vp_model); cudaFree(d.vs_model); cudaFree(d.cold_ordinal); cudaFree(d.cold_count); cudaFree(d.ocean_bin);
  cudaFree(pt->d_lhist); cudaFree(pt->d_lh_part); cudaFree(pt->d_lh_cnt); cudaFree(pt->d_table); cudaFree(pt->d_gather); cudaFree(d.it_dev);
  if (pt->capture_stream) cudaStreamDestroy(pt->capture_stream);
  if (pt->side_stream) cudaStreamDestroy(pt->side_stream);
  for (cudaEvent_t e : pt->ev_side) if (e) cudaEventDestroy(e);
  for (cudaGraphExec_t g : pt->graph) if (g) cudaGraphExecDestroy(g);
  rfinv_comm_peer_release(this);
  delete pt;
  pt = nullptr;
}

static int pt_require(rfinv_handle* h, const char* who) {
  if (!h) { rfinv_set_error("%s: handle is NULL", who); return RFINV_ERR_ARG; }
  if (!h->pt) { rfinv_set_error("%s: call rfinv_pt_init first", who); return RFINV_ERR_STATE; }
  return RFINV_OK;
}

// forward + quadratic form for the chains in `active` (or all), proposal or current state
static int pt_eval(rfinv_handle* h, bool proposal, bool all) {
  PtState* s = h->pt;
  PtDev& d = s->dev;
  ModelBatch mb;
  mb.C = d.Cl;
  mb.k = proposal ? d.pk : d.k; mb.z = proposal ? d.pz : d.z; mb.dvp = proposal ? d.pdvp : d.dvp;
  mb.dvs = proposal ? d.pdvs : d.dvs; mb.sig = proposal ? d.psig : d.sig;
  mb.active = all ? nullptr : d.active; mb.n_active = all ? 0 : d.Cl; mb.n_active_dev = all ? nullptr : d.n_active;
  EvalOutputs out;
  out.misfit = h->d_misfit; out.rft_smp = d.rft_smp[0]; out.rft_smp_alt = d.rft_smp[1]; out.slot = d.slot;
  out.slot_invert = proposal ? 1 : 0; out.rft_full = nullptr; out.is_valid = nullptr;
  int st;
  if ((st = rfinv_launch_forward(h->dc, mb, out, h->d_scratch, h->stream)) != RFINV_OK) return st;
  return rfinv_launch_quadform(h->dc, d.Cl, h->d_misfit, proposal ? d.pphi : d.phi, h->d_qpart, h->d_qcnt, mb.active, mb.n_active, mb.n_active_dev,
                               h->stream);
}

extern "C" {

int32_t rfinv_pt_init(rfinv_handle* h, int32_t nproc_total, int32_t rank_begin, int32_t rank_count) {
  if (!h) { rfinv_set_error("rfinv_pt_init: handle is NULL"); return RFINV_ERR_ARG; }
  const rfinv_config& c = h->cfg;
  if (nproc_total < 1 || rank_begin < 0 || rank_count < 1 || rank_begin + rank_count > nproc_total ||
      (rank_begin % rank_count) != 0 || (nproc_total % rank_count) != 0) {
    rfinv_set_error("rfinv_pt_init: ranks must be split evenly: nproc_total=%d rank_begin=%d rank_count=%d", nproc_total,
                    rank_begin, rank_count);
    return RFINV_ERR_ARG;
  }
  if (c.nchains < 1 || c.ncool < 0 || c.ncool > c.nchains || (c.prior_mode != 1 && c.prior_mode != 2)) {
    rfinv_set_error("rfinv_pt_init: need 0 <= ncool <= nchains, nchains >= 1, prior_mode 1 or 2");
    return RFINV_ERR_ARG;
  }
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  h->free_pt();
  PtState* s = new PtState();
  h->pt = s;
  PtDev& d = s->dev;
  std::memset(&d, 0, sizeof(d));
  const int km = c.k_max, T = c.ntrc, S = c.nsmp;
  d.nproc_total = nproc_total; d.rank_begin = rank_begin; d.G = rank_count; d.nchains = c.nchains; d.Cl = rank_count * c.nchains;
  d.ncool = c.ncool; d.iseed = c.iseed; d.t_high = c.t_high;
  d.dev_z = c.dev_z; d.dev_dvs = c.dev_dvs; d.dev_dvp = c.dev_dvp; d.dev_sig = c.dev_sig;
  d.dvs_prior = c.dvs_prior; d.dvp_prior = c.dvp_prior;
  // proposal types, src/pt_mcmc.f90:311-365
  d.ntype = 4; d.it_birth = 1; d.it_death = 2; d.it_z = 3; d.it_dvs = 4;
  if (c.vp_mode == 1) { d.ntype++; d.it_dvp = d.ntype; } else d.it_dvp = -1;
  d.nsig_trc = 0;
  for (int t = 0; t < T; ++t) {
    d.sig_min[t] = c.sig_min[t]; d.sig_max[t] = c.sig_max[t];
    d.sig_mode[t] = (c.sig_max[t] - c.sig_min[t] > (double)1.0e-5f) ? 1 : 0;  // src/params.f90:262
    if (d.sig_mode[t]) d.isig_trc[d.nsig_trc++] = t;
  }
  if (d.nsig_trc > 0) { d.ntype++; d.it_sig = d.ntype; } else d.it_sig = -1;
  const size_t Cl = d.Cl, G = d.G;
  int st;
#define A(x) if ((st = (x)) != RFINV_OK) { h->free_pt(); return st; }
  A(dalloc(&d.mt, 624 * G)); A(dalloc(&d.mti, G));
  A(dalloc(&d.k, Cl)); A(dalloc(&d.z, Cl * (km - 1))); A(dalloc(&d.dvp, Cl * km)); A(dalloc(&d.dvs, Cl * km));
  A(dalloc(&d.sig, Cl * T)); A(dalloc(&d.logl, Cl)); A(dalloc(&d.temps, Cl)); A(dalloc(&d.phi, Cl * T)); A(dalloc(&d.slot, Cl));
  A(dalloc(&d.rft_smp[0], Cl * T * S)); A(dalloc(&d.rft_smp[1], Cl * T * S));
  A(dalloc(&d.pk, Cl)); A(dalloc(&d.pz, Cl * (km - 1))); A(dalloc(&d.pdvp, Cl * km)); A(dalloc(&d.pdvs, Cl * km));
  A(dalloc(&d.psig, Cl * T)); A(dalloc(&d.pphi, Cl * T)); A(dalloc(&d.log_r, Cl)); A(dalloc(&d.log_prior12, Cl));
  A(dalloc(&d.itype, Cl)); A(dalloc(&d.pflag, Cl)); A(dalloc(&d.active, Cl)); A(dalloc(&d.n_active, 1));
  A(dalloc(&d.nprop, 8)); A(dalloc(&d.naccept, 8)); A(dalloc(&d.n_eval, 1)); A(dalloc(&d.it_dev, 1));
  d.nburn = c.nburn; d.ncorr = c.ncorr > 0 ? c.ncorr : 1;
  d.nbin_z = c.nbin_z; d.nbin_vs = c.nbin_vs; d.nbin_vp = c.nbin_vp; d.nbin_vpvs = c.nbin_vpvs; d.nbin_sig = c.nbin_sig;
  d.nbin_amp = c.nbin_amp; d.amp_min = c.amp_min; d.amp_max = c.amp_max;
  s->record = c.nbin_z > 0 && c.nbin_vs > 0 && c.nbin_vp > 0 && c.nbin_vpvs > 0 && c.nbin_sig > 0 && c.nbin_amp > 0 && c.niter > 0;
  if (s->record) {
    A(dalloc(&d.nk, (size_t)km)); A(dalloc(&d.nz, (size_t)c.nbin_z)); A(dalloc(&d.nsig, (size_t)c.nbin_sig * T));
    A(dalloc(&d.namp, (size_t)c.nbin_amp * S * T)); A(dalloc(&d.nvpz, (size_t)c.nbin_z * c.nbin_vp));
    A(dalloc(&d.nvsz, (size_t)c.nbin_z * c.nbin_vs)); A(dalloc(&d.nvpvsz, (size_t)c.nbin_z * c.nbin_vpvs)); A(dalloc(&d.nmod, 1));
    A(dalloc(&d.vp_mean, (size_t)c.nbin_z)); A(dalloc(&d.vs_mean, (size_t)c.nbin_z)); A(dalloc(&d.vpvs_mean, (size_t)c.nbin_z));
    A(dalloc(&d.cold_ordinal, Cl)); A(dalloc(&d.cold_count, 1)); A(dalloc(&d.ocean_bin, (size_t)c.nbin_z));
    // all_models: the reference allocates nbin_z x (nchains*niter/ncorr) per rank (src/pt_mcmc.f90:405-406)
    const long long want = (long long)(c.niter / d.ncorr) * (long long)Cl;
    if (want > 0 && (double)want * c.nbin_z * 16.0 <= 8.0e9) {
      d.cap_models = want;
      A(dalloc(&d.vp_model, (size_t)want * c.nbin_z)); A(dalloc(&d.vs_model, (size_t)want * c.nbin_z));
    }
  }
  s->table_len = (int)(2 * Cl + G + 2);
  A(dalloc(&s->d_table, (size_t)2 * s->table_len));
  s->cap_lhist = c.nburn + c.niter > 0 ? c.nburn + c.niter : 1024;
  A(dalloc(&s->d_lhist, (size_t)s->cap_lhist));
  A(dalloc(&s->d_lh_part, (Cl + PT_FIN_CHAINS - 1) / PT_FIN_CHAINS)); A(dalloc(&s->d_lh_cnt, 1));
  A(h->ensure_capacity(d.Cl));
#undef A
  pt_init_kernel<<<(d.G + 63) / 64, 64, 0, h->stream>>>(h->dc, d);
  // init_rft, src/likelihood.f90:143-163: forward + likelihood of every initial model
  st = cudaGetLastError() == cudaSuccess ? RFINV_OK : RFINV_ERR_CUDA;
  if (st == RFINV_OK) st = pt_eval(h, /*proposal=*/false, /*all=*/true);
  if (st == RFINV_OK) st = rfinv_launch_loglik(h->dc, d.Cl, d.phi, d.sig, d.logl, h->stream);
  if (st == RFINV_OK) {
    const cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { rfinv_set_error("rfinv_pt_init: %s", cudaGetErrorString(e)); st = RFINV_ERR_CUDA; }
  } else if (st == RFINV_ERR_CUDA && !*rfinv_last_error()) {
    rfinv_set_error("rfinv_pt_init: kernel launch failed");
  }
  if (st != RFINV_OK) { h->free_pt(); return st; }
  s->it_done = 0;
  s->n_eval = d.Cl;
  return RFINV_OK;
}

int32_t rfinv_pt_draw(rfinv_handle* h, int32_t local_rank, int32_t kind, int32_t n, double* out) {
  int st = pt_require(h, "rfinv_pt_draw");
  if (st != RFINV_OK) return st;
  PtDev& d = h->pt->dev;
  if (local_rank < 0 || local_rank >= d.G || kind < 0 || kind > 1 || n < 0 || (n > 0 && !out)) {
    rfinv_set_error("rfinv_pt_draw: bad argument (local_rank %d of %d, kind %d, n %d)", local_rank, d.G, kind, n);
    return RFINV_ERR_ARG;
  }
  if (n == 0) return RFINV_OK;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  double* d_out = nullptr;
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_out, sizeof(double) * (size_t)n));
  pt_draw_kernel<<<1, 1, 0, h->stream>>>(d, local_rank, kind, n, d_out);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(d_out);
  if (e != cudaSuccess) { rfinv_set_error("rfinv_pt_draw: %s", cudaGetErrorString(e)); return RFINV_ERR_CUDA; }
  return RFINV_OK;
}

int32_t rfinv_pt_ntype(rfinv_handle* h) { return (h && h->pt) ? h->pt->dev.ntype : -1; }

int32_t rfinv_pt_set_logging(rfinv_handle* h, int32_t cap_iters) {
  int st = pt_require(h, "rfinv_pt_set_logging");
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  PtDev& d = s->dev;
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  pt_drop_graphs(s);   // the log pointers are baked into the captured launches
  cudaFree(d.log_flags); cudaFree(d.log_itypes); cudaFree(d.log_swaps);
  d.log_flags = nullptr; d.log_itypes = nullptr; d.log_swaps = nullptr;
  s->log_cap = 0; s->log_base = s->it_done;
  if (cap_iters > 0) {
    if ((st = dalloc(&d.log_flags, (size_t)cap_iters * d.Cl)) != RFINV_OK) return st;
    if ((st = dalloc(&d.log_itypes, (size_t)cap_iters * d.Cl)) != RFINV_OK) return st;
    if ((st = dalloc(&d.log_swaps, (size_t)cap_iters * 3)) != RFINV_OK) return st;
    s->log_cap = cap_iters;
  }
  d.log_cap = s->log_cap; d.log_base = s->log_base;
  return RFINV_OK;
}

int32_t rfinv_pt_set_rank_swaps(rfinv_handle* h, int32_t mode) {
  int st = pt_require(h, "rfinv_pt_set_rank_swaps");
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  PtDev& d = s->dev;
  if (mode != 0 && mode != 1) { rfinv_set_error("rfinv_pt_set_rank_swaps: mode %d (0: off, 1: even/odd swaps inside every rank)", mode); return RFINV_ERR_ARG; }
  if (s->step_pending) {
    rfinv_set_error("rfinv_pt_set_rank_swaps: an iteration is half done (rfinv_pt_local_step without rfinv_pt_apply_swap)");
    return RFINV_ERR_STATE;
  }
  if (s->reduced) { rfinv_set_error("rfinv_pt_set_rank_swaps: rfinv_pt_reduce_outputs has run"); return RFINV_ERR_STATE; }
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  if (mode == 1 && d.nchains >= 2 && !d.rs_nprop) {   // counters start at zero and survive later switches
    if ((st = dalloc(&d.rs_nprop, (size_t)d.nchains - 1)) != RFINV_OK) return st;
    if ((st = dalloc(&d.rs_nacc, (size_t)d.G * (d.nchains - 1))) != RFINV_OK) return st;
    if ((st = dalloc(&d.rs_arrived, 1)) != RFINV_OK) return st;
  }
  pt_drop_graphs(s);   // the captured launch sequence depends on the mode
  s->rank_swaps = mode;
  if (mode == 0 && d.rs_tune) {   // the ladder tuning works on the sweep's counters: it goes with it
    s->tune_points_off = pt_tuning_points(s->it_done, d.nburn);
    d.rs_tune = 0;
  }
  if (mode == 0 && d.st_on) {     // the step tuning works on the sweep's levels: likewise
    s->step_points_off = pt_tuning_points(s->it_done, d.nburn);
    d.st_on = 0;
  }
  return RFINV_OK;
}

int32_t rfinv_pt_set_step_tuning(rfinv_handle* h, int32_t on, double target) {
  static const char* who = "rfinv_pt_set_step_tuning";
  int st = pt_require(h, who);
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  PtDev& d = s->dev;
  if (on != 0 && on != 1) { rfinv_set_error("%s: %d (0: off, 1: tune the random-walk widths during the burn-in)", who, on); return RFINV_ERR_ARG; }
  if (!(target > 0.0 && target < 1.0)) { rfinv_set_error("%s: target %g is outside (0, 1)", who, target); return RFINV_ERR_ARG; }
  if (s->step_pending) {
    rfinv_set_error("%s: an iteration is half done (rfinv_pt_local_step without rfinv_pt_apply_swap)", who);
    return RFINV_ERR_STATE;
  }
  if (s->reduced) { rfinv_set_error("%s: rfinv_pt_reduce_outputs has run", who); return RFINV_ERR_STATE; }
  if (on) {
    if (s->it_done > 0) {
      rfinv_set_error("%s: %d iterations have run; the tuning starts with the run (before its first iteration or a restore)", who, s->it_done);
      return RFINV_ERR_STATE;
    }
    if (d.nchains < 2) { rfinv_set_error("%s: nchains = %d: the tuning needs levels, at least two chains per rank", who, d.nchains); return RFINV_ERR_ARG; }
    if (s->rank_swaps != 1) { rfinv_set_error("%s: the tuning needs the rank swaps on (rfinv_pt_set_rank_swaps(h, 1) first)", who); return RFINV_ERR_STATE; }
  }
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  if (on) {   // a fresh start: scales 1, counters zero, no pair yet, the levels of the initial temperatures
    const size_t rows = (size_t)d.G * d.nchains * 4;
    if (!d.st_scale) {
      if ((st = dalloc(&d.st_scale, rows)) != RFINV_OK) return st;
      if ((st = dalloc(&d.st_nprop, rows)) != RFINV_OK) return st;
      if ((st = dalloc(&d.st_nacc, rows)) != RFINV_OK) return st;
      if ((st = dalloc(&d.st_lvl, (size_t)d.Cl)) != RFINV_OK) return st;
      if ((st = dalloc(&d.st_pair, 2)) != RFINV_OK) return st;
    }
    const std::vector<double> ones(rows, 1.0);
    RFINV_CUDA_CHECK(cudaMemcpy(d.st_scale, ones.data(), sizeof(double) * rows, cudaMemcpyHostToDevice));
    RFINV_CUDA_CHECK(cudaMemset(d.st_nprop, 0, sizeof(unsigned long long) * rows));
    RFINV_CUDA_CHECK(cudaMemset(d.st_nacc, 0, sizeof(unsigned long long) * rows));
    const int none[2] = {-1, -1};
    RFINV_CUDA_CHECK(cudaMemcpy(d.st_pair, none, sizeof(none), cudaMemcpyHostToDevice));
    std::vector<double> t((size_t)d.Cl);
    RFINV_CUDA_CHECK(cudaMemcpy(t.data(), d.temps, sizeof(double) * t.size(), cudaMemcpyDeviceToHost));
    std::vector<int> lvl((size_t)d.Cl);
    for (int c0 = 0; c0 < d.Cl; c0 += d.nchains)   // (temperature, chain index) order within each rank
      for (int a = 0; a < d.nchains; ++a) {
        int l = 0;
        for (int b = 0; b < d.nchains; ++b) l += t[c0 + b] < t[c0 + a] || (t[c0 + b] == t[c0 + a] && b < a);
        lvl[c0 + a] = l;
      }
    RFINV_CUDA_CHECK(cudaMemcpy(d.st_lvl, lvl.data(), sizeof(int) * lvl.size(), cudaMemcpyHostToDevice));
  }
  if (!on && d.st_on) s->step_points_off = pt_tuning_points(s->it_done, d.nburn);
  pt_drop_graphs(s);   // the captured launches carry the flag and the target
  d.st_on = on;
  if (on) d.st_target = target;
  return RFINV_OK;
}

int32_t rfinv_pt_get_step_tuning(rfinv_handle* h, int32_t* on, double* target, int32_t* n_points, double* widths,
                                 int64_t* n_prop, int64_t* n_acc) {
  int st = pt_require(h, "rfinv_pt_get_step_tuning");
  if (st != RFINV_OK) return st;
  const PtState* s = h->pt;
  const PtDev& d = s->dev;
  if (on) *on = d.st_on;
  if (target) *target = d.st_target;
  if (n_points) *n_points = d.st_on ? pt_tuning_points(s->it_done, d.nburn) : s->step_points_off;
  const size_t rows = (size_t)d.G * d.nchains * 4;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  if (widths) {   // off: the params.in widths
    const double dev[4] = {d.dev_z, d.dev_dvs, d.dev_dvp, d.dev_sig};
    std::vector<double> sc(rows, 1.0);
    if (d.st_on) RFINV_CUDA_CHECK(cudaMemcpy(sc.data(), d.st_scale, sizeof(double) * rows, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < rows; ++i) widths[i] = dev[i & 3] * sc[i];
  }
  for (int k = 0; k < 2; ++k) {
    int64_t* out = k ? n_acc : n_prop;
    if (!out) continue;
    if (d.st_scale) RFINV_CUDA_CHECK(cudaMemcpy(out, k ? d.st_nacc : d.st_nprop, sizeof(int64_t) * rows, cudaMemcpyDeviceToHost));
    else std::memset(out, 0, sizeof(int64_t) * rows);
  }
  return RFINV_OK;
}

int32_t rfinv_pt_set_ladder_tuning(rfinv_handle* h, int32_t on) {
  static const char* who = "rfinv_pt_set_ladder_tuning";
  int st = pt_require(h, who);
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  PtDev& d = s->dev;
  if (on != 0 && on != 1) { rfinv_set_error("%s: %d (0: off, 1: tune the ladders during the burn-in)", who, on); return RFINV_ERR_ARG; }
  if (s->step_pending) {
    rfinv_set_error("%s: an iteration is half done (rfinv_pt_local_step without rfinv_pt_apply_swap)", who);
    return RFINV_ERR_STATE;
  }
  if (s->reduced) { rfinv_set_error("%s: rfinv_pt_reduce_outputs has run", who); return RFINV_ERR_STATE; }
  if (on && !d.rs_tune) {
    if (s->it_done > 0) {
      rfinv_set_error("%s: %d iterations have run; the tuning starts with the run (before its first iteration or a restore)", who, s->it_done);
      return RFINV_ERR_STATE;
    }
    if (s->rank_swaps != 1) { rfinv_set_error("%s: the tuning needs the rank swaps on (rfinv_pt_set_rank_swaps(h, 1) first)", who); return RFINV_ERR_STATE; }
    // the kernel keeps a rank's ladder and its levels in shared memory
    if ((sizeof(int) + sizeof(double)) * (size_t)d.nchains > 200 * 1024) {
      rfinv_set_error("%s: nchains = %d is beyond the %d chains per rank the tuning supports", who, d.nchains, (int)(200 * 1024 / 12));
      return RFINV_ERR_ARG;
    }
  }
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  if (on && d.nchains >= 2 && !d.rs_base)
    if ((st = dalloc(&d.rs_base, (size_t)d.G * (d.nchains - 1))) != RFINV_OK) return st;
  if (!on && d.rs_tune) s->tune_points_off = pt_tuning_points(s->it_done, d.nburn);
  pt_drop_graphs(s);   // the captured launches carry the flag
  d.rs_tune = on;
  return RFINV_OK;
}

int32_t rfinv_pt_get_ladder_tuning(rfinv_handle* h, int32_t* on, int32_t* n_points) {
  int st = pt_require(h, "rfinv_pt_get_ladder_tuning");
  if (st != RFINV_OK) return st;
  const PtState* s = h->pt;
  if (on) *on = s->dev.rs_tune;
  if (n_points) *n_points = s->dev.rs_tune ? pt_tuning_points(s->it_done, s->dev.nburn) : s->tune_points_off;
  return RFINV_OK;
}

int32_t rfinv_pt_get_rank_swaps(rfinv_handle* h, int32_t* mode, int64_t* n_prop, int64_t* n_acc) {
  int st = pt_require(h, "rfinv_pt_get_rank_swaps");
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  PtDev& d = s->dev;
  if (mode) *mode = s->rank_swaps;
  const int nl = d.nchains - 1;
  if (nl < 1) return RFINV_OK;
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  std::vector<unsigned long long> prop(nl, 0ULL), rows((size_t)d.G * nl, 0ULL);
  if (d.rs_nprop) {
    RFINV_CUDA_CHECK(cudaMemcpy(prop.data(), d.rs_nprop, sizeof(unsigned long long) * nl, cudaMemcpyDeviceToHost));
    RFINV_CUDA_CHECK(cudaMemcpy(rows.data(), d.rs_nacc, sizeof(unsigned long long) * rows.size(), cudaMemcpyDeviceToHost));
  }
  for (int l = 0; l < nl; ++l) {
    unsigned long long acc = 0ULL;
    for (int r = 0; r < d.G; ++r) acc += rows[(size_t)r * nl + l];
    if (n_prop) n_prop[l] = (int64_t)prop[l];
    if (n_acc) n_acc[l] = (int64_t)acc;
  }
  return RFINV_OK;
}

// room in the likelihood history for iterations [0, upto); never called while a launch sequence is being captured
static int pt_reserve_lhist(rfinv_handle* h, int upto) {
  PtState* s = h->pt;
  if (upto <= s->cap_lhist) return RFINV_OK;
  int ncap = s->cap_lhist;
  while (ncap < upto) ncap *= 2;
  double* nl = nullptr;
  int st;
  if ((st = dalloc(&nl, (size_t)ncap)) != RFINV_OK) return st;
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  RFINV_CUDA_CHECK(cudaMemcpy(nl, s->d_lhist, sizeof(double) * s->cap_lhist, cudaMemcpyDeviceToDevice));
  cudaFree(s->d_lhist);
  s->d_lhist = nl; s->cap_lhist = ncap;
  pt_drop_graphs(s);   // the history pointer is baked into the captured launches
  return RFINV_OK;
}

// The launches of one iteration except the swap decision: proposal pass, batched evaluation, acceptance, likelihood
// history, (posterior bookkeeping,) and this process's swap table.  Nothing here depends on the host's iteration counter.
// fuse_swap: a single process -- the swap decision is taken by the last CTA of pt_finish_kernel (unless bookkeeping kernels
// have to run in between) or, with the rank sweep on, by the last CTA of pt_rank_swap_kernel
static int pt_enqueue_local(rfinv_handle* h, bool record, bool peer_exchange = false, bool fuse_swap = false) {
  PtState* s = h->pt;
  PtDev& d = s->dev;
  cudaStream_t q = h->stream;
  int st;
  const bool peer_side = s->peer_state == 1 && peer_exchange;
  if (peer_side) {   // side branch of the iteration: the previous iteration's table goes to the other processes beside the proposal pass
    RFINV_CUDA_CHECK(cudaEventRecord(s->ev_side[0], q));
    RFINV_CUDA_CHECK(cudaStreamWaitEvent(s->side_stream, s->ev_side[0], 0));
    const int nbp = (s->table_len + PT_PUSH_THREADS - 1) / PT_PUSH_THREADS;
    pt_push_kernel<<<nbp < 64 ? nbp : 64, PT_PUSH_THREADS, 0, s->side_stream>>>(d, s->d_table, s->peers);
  }
  {
    // staged variant while a warp's share of shared memory stays below 48 KB; 1, 2 or 4 warps per CTA accordingly
    const size_t per_warp = sizeof(double) * pt_propose_smem_doubles(h->dc.k_max, h->dc.ntrc, d.nchains);
    if (per_warp <= 48 * 1024) {
      const int warps = per_warp <= 12 * 1024 ? 4 : (per_warp <= 24 * 1024 ? 2 : 1);
      RFINV_CUDA_CHECK(rfinv_raise_smem_limit((const void*)pt_propose_kernel<true, false>, per_warp * warps));
      const bool peer = s->peer_state == 1 && peer_exchange;
      RFINV_CUDA_CHECK(rfinv_raise_smem_limit((const void*)pt_propose_kernel<true, true>, per_warp * warps));
      if (peer) pt_propose_kernel<true, true><<<(d.G + warps - 1) / warps, 32 * warps, per_warp * warps, q>>>(h->dc, d, s->d_table, s->peers);
      else pt_propose_kernel<true, false><<<(d.G + warps - 1) / warps, 32 * warps, per_warp * warps, q>>>(h->dc, d, s->d_table, s->peers);
    } else {
      if (s->peer_state == 1 && peer_exchange) pt_propose_kernel<false, true><<<(d.G * 32 + 127) / 128, 128, 0, q>>>(h->dc, d, s->d_table, s->peers);
      else pt_propose_kernel<false, false><<<(d.G * 32 + 127) / 128, 128, 0, q>>>(h->dc, d, s->d_table, s->peers);
    }
  }
  RFINV_CUDA_CHECK(cudaGetLastError());
  if (peer_side) {   // the pair just drawn goes to the other processes beside the evaluation
    RFINV_CUDA_CHECK(cudaEventRecord(s->ev_side[1], q));
    RFINV_CUDA_CHECK(cudaStreamWaitEvent(s->side_stream, s->ev_side[1], 0));
    pt_pairpush_kernel<<<1, 32, 0, s->side_stream>>>(d, s->d_table, s->peers);
    RFINV_CUDA_CHECK(cudaEventRecord(s->ev_side[2], s->side_stream));
  }
  if ((st = pt_eval(h, /*proposal=*/true, /*all=*/false)) != RFINV_OK) return st;
  if (peer_side) RFINV_CUDA_CHECK(cudaStreamWaitEvent(q, s->ev_side[2], 0));   // the side branch joins in front of pt_finish_kernel
  const bool peer = s->peer_state == 1 && peer_exchange;
  const bool sweep = pt_sweeps(s);
  {
    const unsigned nb = (unsigned)((d.Cl + PT_FIN_CHAINS - 1) / PT_FIN_CHAINS);
    if (peer) pt_finish_kernel<true, false><<<nb, PT_FIN_THREADS, 0, q>>>(h->dc, d, s->d_table, s->peers, s->d_lhist, s->d_lh_part, s->d_lh_cnt);
    else if (fuse_swap && !record && !sweep) pt_finish_kernel<false, true><<<nb, PT_FIN_THREADS, 0, q>>>(h->dc, d, s->d_table, s->peers, s->d_lhist, s->d_lh_part, s->d_lh_cnt);
    else pt_finish_kernel<false, false><<<nb, PT_FIN_THREADS, 0, q>>>(h->dc, d, s->d_table, s->peers, s->d_lhist, s->d_lh_part, s->d_lh_cnt);
  }
  if (record) {   // posterior bookkeeping of the state after acceptance, before the swap (src/pt_mcmc.f90:204-286)
    pt_coldscan_kernel<<<1, 1024, 0, q>>>(d);
    pt_record_kernel<<<d.Cl, 128, 0, q>>>(h->dc, d);
    pt_record_finish_kernel<<<1, 1, 0, q>>>(d);
  }
  if (sweep) {   // after the bookkeeping (it sees the temperatures at acceptance), before the global swap reads the table
    const int warps = d.nchains <= 3072 ? PT_RS_WARPS : 1;
    const size_t smem = (sizeof(int) + (d.rs_tune ? sizeof(double) : 0)) * (size_t)d.nchains * warps;
    const unsigned nb = (unsigned)((d.G + warps - 1) / warps);
    if (fuse_swap && !peer) {
      RFINV_CUDA_CHECK(rfinv_raise_smem_limit((const void*)pt_rank_swap_kernel<true>, smem));
      pt_rank_swap_kernel<true><<<nb, 32 * warps, smem, q>>>(d, s->d_table, s->table_len, 0);
    } else {
      RFINV_CUDA_CHECK(rfinv_raise_smem_limit((const void*)pt_rank_swap_kernel<false>, smem));
      pt_rank_swap_kernel<false><<<nb, 32 * warps, smem, q>>>(d, s->d_table, s->table_len, peer ? 1 : 0);
    }
  }
  RFINV_CUDA_CHECK(cudaGetLastError());
  return RFINV_OK;
}

// does iteration number it_done + 1 record the posterior bookkeeping?  (src/pt_mcmc.f90:204-205)
static bool pt_records(const PtState* s) {
  const int it = s->it_done + 1;
  return s->record && it > s->dev.nburn && it % s->dev.ncorr == 0;
}

int32_t rfinv_pt_local_step(rfinv_handle* h) {
  int st = pt_require(h, "rfinv_pt_local_step");
  if (st != RFINV_OK) return st;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  if ((st = pt_reserve_lhist(h, h->pt->it_done + 1)) != RFINV_OK) return st;
  if ((st = pt_enqueue_local(h, pt_records(h->pt))) != RFINV_OK) return st;
  h->pt->step_pending = true;
  return RFINV_OK;
}

int32_t rfinv_pt_swap_table(rfinv_handle* h, uint64_t* dev_ptr, int32_t* n_doubles) {
  int st = pt_require(h, "rfinv_pt_swap_table");
  if (st != RFINV_OK) return st;
  if (dev_ptr) *dev_ptr = reinterpret_cast<uint64_t>(h->pt->d_table);
  if (n_doubles) *n_doubles = h->pt->table_len;
  return RFINV_OK;
}

// gathered: `world` tables back to back, in process order (process q owns virtual ranks [q*G, (q+1)*G))
int32_t rfinv_pt_apply_swap(rfinv_handle* h, uint64_t gathered_dev_ptr, int32_t world) {
  int st = pt_require(h, "rfinv_pt_apply_swap");
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  if (world * s->dev.G != s->dev.nproc_total) {
    rfinv_set_error("rfinv_pt_apply_swap: world=%d inconsistent with nproc_total=%d, rank_count=%d", world, s->dev.nproc_total, s->dev.G);
    return RFINV_ERR_ARG;
  }
  pt_swap_kernel<<<1, 32, 0, h->stream>>>(s->dev, reinterpret_cast<const double*>(gathered_dev_ptr), world, s->table_len);
  RFINV_CUDA_CHECK(cudaGetLastError());
  s->it_done++;
  s->step_pending = false;
  return RFINV_OK;
}

// One whole iteration on the handle's stream: local step, (all-gather of the swap tables over the handle's communicator,)
// swap decision.  world == 1: the own table is the gathered table.
static int pt_enqueue_iteration(rfinv_handle* h, int world, bool record) {
  PtState* s = h->pt;
  int st;
  const bool peer = world > 1 && s->peer_state == 1;
  if ((st = pt_enqueue_local(h, record, peer, world == 1)) != RFINV_OK) return st;
  if (world == 1 && (!record || pt_sweeps(s))) return RFINV_OK;   // pt_finish_kernel or pt_rank_swap_kernel took the swap decision
  if (peer) return RFINV_OK;   // pair and table went to every process from inside the kernels; the swap is applied an iteration later
  const double* gathered = s->d_table;
  if (world > 1) {
    if ((st = rfinv_comm_allgather(h, s->d_table, s->d_gather, (size_t)s->table_len, h->stream)) != RFINV_OK) return st;
    gathered = s->d_gather;
  }
  pt_swap_kernel<<<1, 32, 0, h->stream>>>(s->dev, gathered, world, s->table_len);
  RFINV_CUDA_CHECK(cudaGetLastError());
  return RFINV_OK;
}

// RFINV_PT_GRAPH=0: plain launches instead of replaying captured iterations
static bool pt_use_graph() {
  static const bool use = !(getenv("RFINV_PT_GRAPH") && atoi(getenv("RFINV_PT_GRAPH")) == 0);
  return use;
}

// pt_control's loop (src/pt_mcmc.f90:488-572) for n_iter iterations over `world` processes.  The launch sequence of an
// iteration -- five kernels; with several processes also the two kernels of the peer-memory exchange on a side branch, or one
// ncclAllGather and the swap kernel -- is captured once per variant (with / without the bookkeeping kernels) in a CUDA graph and
// replayed: one launch per iteration (RFINV_PT_GRAPH=0: plain launches).
static int pt_iterate(rfinv_handle* h, int n_iter, int world) {
  PtState* s = h->pt;
  int st;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  if ((st = pt_reserve_lhist(h, s->it_done + n_iter)) != RFINV_OK) return st;
  if (world > 1 && s->peer_state == 0) {   // first distributed run since rfinv_pt_init: try the peer-memory exchange (collective)
    if ((st = rfinv_comm_peer_setup(h)) != RFINV_OK) return st;
    pt_drop_graphs(s);
  }
  if (world > 1 && s->peer_state != 1 && s->cap_gather < world * s->table_len) {
    cudaFree(s->d_gather); s->d_gather = nullptr; s->cap_gather = 0;
    if ((st = dalloc(&s->d_gather, (size_t)world * s->table_len)) != RFINV_OK) return st;
    s->cap_gather = world * s->table_len;
    pt_drop_graphs(s);
  }
  if (world > 1 && s->peer_state == 1) {
    // every run ends with pt_drain_kernel, so at this point every swap of the iterations done so far is applied -- also when
    // some of them were driven through rfinv_pt_local_step / rfinv_pt_apply_swap in between
    const int applied[3] = {s->it_done, s->it_done, s->it_done};
    RFINV_CUDA_CHECK(cudaMemcpyAsync(s->peers.done, applied, sizeof(applied), cudaMemcpyHostToDevice, h->stream));
    RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  }
  if (world > 1 && s->peer_state == 1 && !s->side_stream) {   // (created outside any capture)
    RFINV_CUDA_CHECK(cudaStreamCreateWithFlags(&s->side_stream, cudaStreamNonBlocking));
    for (cudaEvent_t& e : s->ev_side) RFINV_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  const bool use_graph = pt_use_graph();
  if (s->graph_world != world) { pt_drop_graphs(s); s->graph_world = world; }
  for (int it = 0; it < n_iter; ++it) {
    const bool record = pt_records(s);
    if (use_graph) {
      cudaGraphExec_t& g = s->graph[record ? 1 : 0];
      if (!g) {
        // captured on a stream of its own (the caller's may be the legacy default stream, which cannot capture); replayed on
        // the handle's stream
        cudaGraph_t graph = nullptr;
        if (!s->capture_stream) RFINV_CUDA_CHECK(cudaStreamCreateWithFlags(&s->capture_stream, cudaStreamNonBlocking));
        cudaStream_t user_stream = h->stream;
        RFINV_CUDA_CHECK(cudaStreamSynchronize(user_stream));
        h->stream = s->capture_stream;
        cudaError_t e = cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal);
        if (e != cudaSuccess) { h->stream = user_stream; rfinv_set_error("cudaStreamBeginCapture: %s", cudaGetErrorString(e)); return RFINV_ERR_CUDA; }
        st = pt_enqueue_iteration(h, world, record);
        e = cudaStreamEndCapture(h->stream, &graph);
        h->stream = user_stream;
        if (st != RFINV_OK) { if (graph) cudaGraphDestroy(graph); return st; }
        if (e != cudaSuccess) { rfinv_set_error("cudaStreamEndCapture: %s", cudaGetErrorString(e)); return RFINV_ERR_CUDA; }
        e = cudaGraphInstantiate(&g, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) { g = nullptr; rfinv_set_error("cudaGraphInstantiate: %s", cudaGetErrorString(e)); return RFINV_ERR_CUDA; }
      }
      RFINV_CUDA_CHECK(cudaGraphLaunch(g, h->stream));
    } else if ((st = pt_enqueue_iteration(h, world, record)) != RFINV_OK) {
      return st;
    }
    s->it_done++;
  }
  if (world > 1 && s->peer_state == 1) {   // the last table and the last swap of this run (inside the run every swap is applied an iteration later)
    const int nbp = (s->table_len + PT_PUSH_THREADS - 1) / PT_PUSH_THREADS;
    pt_push_kernel<<<nbp < 64 ? nbp : 64, PT_PUSH_THREADS, 0, h->stream>>>(s->dev, s->d_table, s->peers);
    pt_drain_kernel<<<1, 32, 0, h->stream>>>(s->dev, s->peers);
    RFINV_CUDA_CHECK(cudaGetLastError());
  }
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  if (world > 1 && s->peer_state == 1) {
    unsigned long long err = 0ULL;
    RFINV_CUDA_CHECK(cudaMemcpy(&err, s->d_peer_flags + world, sizeof(err), cudaMemcpyDeviceToHost));
    if (err) { rfinv_set_error("rfinv_pt_run_distributed: a process never delivered its swap table (peer-memory exchange timed out)"); return RFINV_ERR_STATE; }
  }
  return RFINV_OK;
}

// single-process run
int32_t rfinv_pt_run(rfinv_handle* h, int32_t n_iter) {
  int st = pt_require(h, "rfinv_pt_run");
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  if (s->dev.G != s->dev.nproc_total) {
    rfinv_set_error("rfinv_pt_run: this handle holds %d of %d ranks; use rfinv_pt_run_distributed (or rfinv_pt_local_step / apply_swap)",
                    s->dev.G, s->dev.nproc_total);
    return RFINV_ERR_STATE;
  }
  return pt_iterate(h, n_iter, 1);
}

int32_t rfinv_pt_exchange_mode(rfinv_handle* h) {
  if (!h || !h->pt || !h->comm || h->comm_world < 2) return 0;
  return h->pt->peer_state == 1 ? 1 : (h->pt->peer_state == -1 ? 2 : 0);
}

// one process per GPU: the handle's communicator (rfinv_comm_init) carries the per-iteration exchange
int32_t rfinv_pt_run_distributed(rfinv_handle* h, int32_t n_iter) {
  int st = pt_require(h, "rfinv_pt_run_distributed");
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  const int world = h->comm ? h->comm_world : 1;
  if (world * s->dev.G != s->dev.nproc_total || s->dev.rank_begin != (h->comm ? h->comm_rank : 0) * s->dev.G) {
    rfinv_set_error("rfinv_pt_run_distributed: process %d of %d must own the virtual ranks [%d, %d) of %d (rfinv_pt_init), it owns [%d, %d)",
                    h->comm ? h->comm_rank : 0, world, (h->comm ? h->comm_rank : 0) * s->dev.G, ((h->comm ? h->comm_rank : 0) + 1) * s->dev.G,
                    s->dev.nproc_total, s->dev.rank_begin, s->dev.rank_begin + s->dev.G);
    return RFINV_ERR_STATE;
  }
  return pt_iterate(h, n_iter, world);
}

int32_t rfinv_pt_get_state(rfinv_handle* h, int32_t* k, double* z, double* dvp, double* dvs, double* sig, double* logl,
                           double* temps) {
  int st = pt_require(h, "rfinv_pt_get_state");
  if (st != RFINV_OK) return st;
  PtDev& d = h->pt->dev;
  const int km = h->cfg.k_max, T = h->cfg.ntrc, Cl = d.Cl;
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  std::vector<double> tmp;
  auto fetch = [&](const double* src, double* dst, int len) -> int {  // device [len][Cl] -> host [Cl][len]
    if (!dst) return RFINV_OK;
    tmp.resize((size_t)len * Cl);
    RFINV_CUDA_CHECK(cudaMemcpy(tmp.data(), src, sizeof(double) * tmp.size(), cudaMemcpyDeviceToHost));
    for (int i = 0; i < len; ++i)
      for (int c = 0; c < Cl; ++c) dst[(size_t)c * len + i] = tmp[(size_t)i * Cl + c];
    return RFINV_OK;
  };
  if (k) RFINV_CUDA_CHECK(cudaMemcpy(k, d.k, sizeof(int) * Cl, cudaMemcpyDeviceToHost));
  if ((st = fetch(d.z, z, km - 1)) != RFINV_OK) return st;
  if ((st = fetch(d.dvp, dvp, km)) != RFINV_OK) return st;
  if ((st = fetch(d.dvs, dvs, km)) != RFINV_OK) return st;
  if ((st = fetch(d.sig, sig, T)) != RFINV_OK) return st;
  if (logl) RFINV_CUDA_CHECK(cudaMemcpy(logl, d.logl, sizeof(double) * Cl, cudaMemcpyDeviceToHost));
  if (temps) RFINV_CUDA_CHECK(cudaMemcpy(temps, d.temps, sizeof(double) * Cl, cudaMemcpyDeviceToHost));
  return RFINV_OK;
}

int32_t rfinv_pt_get_counters(rfinv_handle* h, int64_t* nprop, int64_t* naccept, double* likelihood_hist, int32_t n_hist,
                              int64_t* n_eval) {
  int st = pt_require(h, "rfinv_pt_get_counters");
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  if (nprop) RFINV_CUDA_CHECK(cudaMemcpy(nprop, s->dev.nprop, sizeof(int64_t) * s->dev.ntype, cudaMemcpyDeviceToHost));
  if (naccept) RFINV_CUDA_CHECK(cudaMemcpy(naccept, s->dev.naccept, sizeof(int64_t) * s->dev.ntype, cudaMemcpyDeviceToHost));
  if (likelihood_hist && n_hist > 0) {
    const int n = n_hist < s->it_done ? n_hist : s->it_done;
    RFINV_CUDA_CHECK(cudaMemcpy(likelihood_hist, s->d_lhist, sizeof(double) * n, cudaMemcpyDeviceToHost));
  }
  if (n_eval) {
    unsigned long long ne = 0;
    RFINV_CUDA_CHECK(cudaMemcpy(&ne, s->dev.n_eval, sizeof(ne), cudaMemcpyDeviceToHost));
    *n_eval = s->n_eval + (long long)ne;
  }
  return RFINV_OK;
}

int32_t rfinv_pt_get_hist(rfinv_handle* h, int64_t* nmod, int64_t* nk, int64_t* nz, int64_t* nsig, int64_t* namp,
                          int64_t* nvpz, int64_t* nvsz, int64_t* nvpvsz, double* vp_mean, double* vs_mean,
                          double* vpvs_mean) {
  int st = pt_require(h, "rfinv_pt_get_hist");
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  if (!s->record) { rfinv_set_error("rfinv_pt_get_hist: bookkeeping disabled (needs niter > 0 and all nbin_* > 0)"); return RFINV_ERR_STATE; }
  const rfinv_config& c = h->cfg;
  PtDev& d = s->dev;
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
#define G64(dst, src, n) if (dst) RFINV_CUDA_CHECK(cudaMemcpy(dst, src, sizeof(int64_t) * (size_t)(n), cudaMemcpyDeviceToHost))
#define GD(dst, src, n) if (dst) RFINV_CUDA_CHECK(cudaMemcpy(dst, src, sizeof(double) * (size_t)(n), cudaMemcpyDeviceToHost))
  G64(nmod, d.nmod, 1); G64(nk, d.nk, c.k_max); G64(nz, d.nz, c.nbin_z); G64(nsig, d.nsig, c.nbin_sig * c.ntrc);
  G64(namp, d.namp, (size_t)c.nbin_amp * c.nsmp * c.ntrc); G64(nvpz, d.nvpz, c.nbin_z * c.nbin_vp);
  G64(nvsz, d.nvsz, c.nbin_z * c.nbin_vs); G64(nvpvsz, d.nvpvsz, c.nbin_z * c.nbin_vpvs);
  GD(vp_mean, d.vp_mean, c.nbin_z); GD(vs_mean, d.vs_mean, c.nbin_z); GD(vpvs_mean, d.vpvs_mean, c.nbin_z);
#undef G64
#undef GD
  return RFINV_OK;
}

// recorded models (all_models): vp_model/vs_model [n_models][nbin_z]; n_models = min(nmod, capacity)
int32_t rfinv_pt_get_models(rfinv_handle* h, int64_t max_models, double* vp_model, double* vs_model, int64_t* n_models) {
  int st = pt_require(h, "rfinv_pt_get_models");
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  PtDev& d = s->dev;
  if (!s->record || !d.vp_model) { if (n_models) *n_models = 0; return RFINV_OK; }
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  unsigned long long nm = 0;
  RFINV_CUDA_CHECK(cudaMemcpy(&nm, d.nmod, sizeof(nm), cudaMemcpyDeviceToHost));
  long long n = (long long)nm < d.cap_models ? (long long)nm : d.cap_models;
  if (n > max_models) n = max_models;
  if (n > 0 && vp_model) RFINV_CUDA_CHECK(cudaMemcpy(vp_model, d.vp_model, sizeof(double) * (size_t)n * d.nbin_z, cudaMemcpyDeviceToHost));
  if (n > 0 && vs_model) RFINV_CUDA_CHECK(cudaMemcpy(vs_model, d.vs_model, sizeof(double) * (size_t)n * d.nbin_z, cudaMemcpyDeviceToHost));
  if (n_models) *n_models = n;
  return RFINV_OK;
}

int32_t rfinv_pt_iterations_done(rfinv_handle* h) { return (h && h->pt) ? h->pt->it_done : -1; }

int32_t rfinv_pt_get_log(rfinv_handle* h, int8_t* flags, int8_t* itypes, int32_t* swaps, int32_t* n_logged) {
  int st = pt_require(h, "rfinv_pt_get_log");
  if (st != RFINV_OK) return st;
  PtState* s = h->pt;
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  int log_used = s->it_done - s->log_base;
  log_used = log_used < 0 ? 0 : (log_used > s->log_cap ? s->log_cap : log_used);
  const size_t n = (size_t)log_used * s->dev.Cl;
  if (flags && n) RFINV_CUDA_CHECK(cudaMemcpy(flags, s->dev.log_flags, n, cudaMemcpyDeviceToHost));
  if (itypes && n) RFINV_CUDA_CHECK(cudaMemcpy(itypes, s->dev.log_itypes, n, cudaMemcpyDeviceToHost));
  if (swaps && log_used) RFINV_CUDA_CHECK(cudaMemcpy(swaps, s->dev.log_swaps, sizeof(int32_t) * 3 * log_used, cudaMemcpyDeviceToHost));
  if (n_logged) *n_logged = log_used;
  return RFINV_OK;
}

}  // extern "C"

int rfinv_pt_reserve_lhist(rfinv_handle* h, int upto) { return pt_reserve_lhist(h, upto); }

// ---------------- several single-process runs advanced together (rfinv_pt_group_*) ----------------
// One iteration of every member is ONE graph: the group's stream forks to the members' capture streams, each member's own
// launch sequence (pt_enqueue_iteration) is captured on its branch, and the branches join again.  The members' kernels then
// run side by side, so many small runs fill the GPU that one of them leaves mostly idle.  Variant [0]: nobody records the
// posterior bookkeeping in this iteration, [1]: the members with the bookkeeping on record (equal nburn / ncorr /
// iterations_done make that decision the same for all of them).
struct rfinv_pt_group {
  std::vector<rfinv_handle*> h;
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr;
  std::vector<cudaEvent_t> join;
  cudaGraphExec_t graph[2] = {nullptr, nullptr};
  // per member: the PtState and its generation the graphs were captured with (a new one, or a new generation, means the
  // member's buffers may have moved: capture again)
  std::vector<PtState*> cap_state;
  std::vector<uint64_t> cap_gen;
};

static void group_drop_graphs(rfinv_pt_group* g) {
  for (cudaGraphExec_t& e : g->graph) { if (e) cudaGraphExecDestroy(e); e = nullptr; }
}

// the members' iterations of variant `v` as one fork-join graph on the group's stream
static int group_capture(rfinv_pt_group* g, cudaGraphExec_t* out) {
  const int n = (int)g->h.size();
  for (rfinv_handle* h : g->h)   // (created outside the capture)
    if (!h->pt->capture_stream) RFINV_CUDA_CHECK(cudaStreamCreateWithFlags(&h->pt->capture_stream, cudaStreamNonBlocking));
  cudaGraph_t graph = nullptr;
  cudaError_t e = cudaStreamBeginCapture(g->stream, cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) { rfinv_set_error("rfinv_pt_group_run: cudaStreamBeginCapture: %s", cudaGetErrorString(e)); return RFINV_ERR_CUDA; }
  int st = RFINV_OK;
  e = cudaEventRecord(g->fork, g->stream);
  for (int i = 0; i < n && e == cudaSuccess && st == RFINV_OK; ++i) {
    rfinv_handle* h = g->h[i];
    PtState* s = h->pt;
    e = cudaStreamWaitEvent(s->capture_stream, g->fork, 0);
    if (e != cudaSuccess) break;
    cudaStream_t user_stream = h->stream;   // the member's launch code enqueues on h->stream: its branch of the capture
    h->stream = s->capture_stream;
    st = pt_enqueue_iteration(h, 1, pt_records(s));
    h->stream = user_stream;
    if (st != RFINV_OK) break;
    e = cudaEventRecord(g->join[i], s->capture_stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(g->stream, g->join[i], 0);
  }
  const cudaError_t e_end = cudaStreamEndCapture(g->stream, &graph);
  if (st != RFINV_OK) { if (graph) cudaGraphDestroy(graph); return st; }
  if (e == cudaSuccess) e = e_end;
  if (e != cudaSuccess) {
    if (graph) cudaGraphDestroy(graph);
    rfinv_set_error("rfinv_pt_group_run: capture of the group's iteration: %s", cudaGetErrorString(e));
    return RFINV_ERR_CUDA;
  }
  e = cudaGraphInstantiate(out, graph, 0);
  cudaGraphDestroy(graph);
  if (e != cudaSuccess) { *out = nullptr; rfinv_set_error("rfinv_pt_group_run: cudaGraphInstantiate: %s", cudaGetErrorString(e)); return RFINV_ERR_CUDA; }
  return RFINV_OK;
}

extern "C" {

int32_t rfinv_pt_group_create(rfinv_handle* const* handles, int32_t n, rfinv_pt_group** out) {
  static const char* who = "rfinv_pt_group_create";
  if (!out) { rfinv_set_error("%s: out is NULL", who); return RFINV_ERR_ARG; }
  *out = nullptr;
  if (!handles || n < 1) { rfinv_set_error("%s: need at least one handle (n = %d)", who, n); return RFINV_ERR_ARG; }
  for (int i = 0; i < n; ++i) {
    rfinv_handle* h = handles[i];
    if (!h) { rfinv_set_error("%s: member %d is NULL", who, i); return RFINV_ERR_ARG; }
    for (int j = 0; j < i; ++j)
      if (handles[j] == h) { rfinv_set_error("%s: member %d is the same handle as member %d", who, i, j); return RFINV_ERR_ARG; }
    if (!h->pt) { rfinv_set_error("%s: member %d: call rfinv_pt_init first", who, i); return RFINV_ERR_STATE; }
    if (h->pt->dev.G != h->pt->dev.nproc_total) {
      rfinv_set_error("%s: member %d holds %d of %d ranks (a distributed layout); a group advances single-process runs", who, i,
                      h->pt->dev.G, h->pt->dev.nproc_total);
      return RFINV_ERR_STATE;
    }
    if (h->device != handles[0]->device) {
      rfinv_set_error("%s: member %d is on device %d, member 0 on device %d", who, i, h->device, handles[0]->device);
      return RFINV_ERR_ARG;
    }
  }
  RFINV_CUDA_CHECK(cudaSetDevice(handles[0]->device));
  rfinv_pt_group* g = new rfinv_pt_group();
  g->h.assign(handles, handles + n);
  g->device = handles[0]->device;
  g->join.assign(n, nullptr);
  g->cap_state.assign(n, nullptr);
  g->cap_gen.assign(n, 0);
  cudaError_t e = cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g->fork, cudaEventDisableTiming);
  for (int i = 0; i < n && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&g->join[i], cudaEventDisableTiming);
  if (e != cudaSuccess) {
    rfinv_set_error("%s: %s", who, cudaGetErrorString(e));
    rfinv_pt_group_destroy(g);
    return RFINV_ERR_CUDA;
  }
  *out = g;
  return RFINV_OK;
}

int32_t rfinv_pt_group_run(rfinv_pt_group* g, int32_t n_iter) {
  static const char* who = "rfinv_pt_group_run";
  if (!g) { rfinv_set_error("%s: group is NULL", who); return RFINV_ERR_ARG; }
  if (n_iter < 0) { rfinv_set_error("%s: n_iter = %d", who, n_iter); return RFINV_ERR_ARG; }
  const int n = (int)g->h.size();
  for (int i = 0; i < n; ++i) {
    rfinv_handle* h = g->h[i];
    const PtState* s = h->pt;
    if (!s) { rfinv_set_error("%s: member %d: call rfinv_pt_init first", who, i); return RFINV_ERR_STATE; }
    if (s->dev.G != s->dev.nproc_total) {
      rfinv_set_error("%s: member %d holds %d of %d ranks (a distributed layout)", who, i, s->dev.G, s->dev.nproc_total);
      return RFINV_ERR_STATE;
    }
    if (s->step_pending) {
      rfinv_set_error("%s: member %d is between rfinv_pt_local_step and rfinv_pt_apply_swap", who, i);
      return RFINV_ERR_STATE;
    }
    if (s->reduced) { rfinv_set_error("%s: member %d: rfinv_pt_reduce_outputs has run", who, i); return RFINV_ERR_STATE; }
    const PtState* s0 = g->h[0]->pt;
    if (s->dev.nburn != s0->dev.nburn || s->dev.ncorr != s0->dev.ncorr || s->it_done != s0->it_done) {
      rfinv_set_error("%s: member %d has nburn %d, ncorr %d and %d iterations done, member 0 has %d, %d and %d: the members must "
                      "agree on all three", who, i, s->dev.nburn, s->dev.ncorr, s->it_done, s0->dev.nburn, s0->dev.ncorr, s0->it_done);
      return RFINV_ERR_STATE;
    }
  }
  if (n_iter == 0) return RFINV_OK;
  int st;
  RFINV_CUDA_CHECK(cudaSetDevice(g->device));
  for (rfinv_handle* h : g->h) {
    RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));   // the caller may have queued work on the member's own stream
    if ((st = pt_reserve_lhist(h, h->pt->it_done + n_iter)) != RFINV_OK) return st;
  }
  const bool use_graph = pt_use_graph();
  if (use_graph) {
    bool stale = false;
    for (int i = 0; i < n; ++i) stale = stale || g->cap_state[i] != g->h[i]->pt || g->cap_gen[i] != g->h[i]->pt->generation;
    if (stale) {
      group_drop_graphs(g);
      for (int i = 0; i < n; ++i) { g->cap_state[i] = g->h[i]->pt; g->cap_gen[i] = g->h[i]->pt->generation; }
    }
  }
  for (int it = 0; it < n_iter; ++it) {
    const PtState* s0 = g->h[0]->pt;
    const int next = s0->it_done + 1;   // pt_records without a member's bookkeeping switch
    const int variant = next > s0->dev.nburn && next % s0->dev.ncorr == 0 ? 1 : 0;
    if (use_graph) {
      cudaGraphExec_t& ge = g->graph[variant];
      if (!ge && (st = group_capture(g, &ge)) != RFINV_OK) return st;
      RFINV_CUDA_CHECK(cudaGraphLaunch(ge, g->stream));
    } else {
      for (rfinv_handle* h : g->h)   // round robin over the members' own streams
        if ((st = pt_enqueue_iteration(h, 1, pt_records(h->pt))) != RFINV_OK) return st;
    }
    for (rfinv_handle* h : g->h) h->pt->it_done++;
  }
  if (use_graph) RFINV_CUDA_CHECK(cudaStreamSynchronize(g->stream));
  else for (rfinv_handle* h : g->h) RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  return RFINV_OK;
}

void rfinv_pt_group_destroy(rfinv_pt_group* g) {
  if (!g) return;
  cudaSetDevice(g->device);
  if (g->stream) cudaStreamSynchronize(g->stream);
  group_drop_graphs(g);
  for (cudaEvent_t e : g->join) if (e) cudaEventDestroy(e);
  if (g->fork) cudaEventDestroy(g->fork);
  if (g->stream) cudaStreamDestroy(g->stream);
  delete g;
}

}  // extern "C"
