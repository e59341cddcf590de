// Fused forward kernel: format_model -> layered-medium propagator response -> Gaussian filter ->
// shared-memory inverse FFT -> time shift / normalisation -> misfit.  One CTA per (model, ray).
//
// Replaces, for a whole batch of chains at once (paths relative to the reference checkout):
//   format_model      src/model.f90:175-290
//   calc_seis         src/forward.f90:212-344   (e_inverse :350-380, layer_matrix_sol :385-421,
//                                                layer_matrix_liq :424-442)
//   calc_rf           src/forward.f90:123-208   (water_level_decon :447-470, direct_arrival :474-491)
//   FFTW c2r          src/fftw.f90:44, executed at src/forward.f90:172,200
//   misfit            src/likelihood.f90:87
//
// Arithmetic re-design (DESIGN.md section 4).  The reference multiplies dense complex 4x4 layer
// matrices P_l and then E^-1 * prod(P_l); only rows 3,4 x columns 1,2 (and 4 with a water layer) of the
// result are used.  P_l has a fixed checkerboard real/imaginary structure: P = D S B S^-1 D^-1 with
// D = diag(1,i,1,i), S = diag(1,1,w,w) (w = angular frequency) and B REAL and free of explicit w, so two
// REAL 4-vectors (column e1 and the free-surface / water-layer combination of e2,e4) are propagated from
// the top layer down.  B_l itself is never formed: B_l = V_l R_l V_l^-1, with R_l two plane rotations by
// (w xi h, w eta h) -- the standing P and S waves of the layer -- and V_l frequency independent with two
// decoupled 2x2 blocks (components {1,4} and {2,3}).  The vectors are carried in wave coordinates
// w = V_l^-1 y; a layer is "rotate both pairs", an interface is "apply the two 2x2 blocks of
// V_{l+1}^-1 V_l", and the free per-layer scale of the P and S coordinates is chosen so that the {1,4}
// block has a unit diagonal.  Per layer and frequency: 2 x 14 FP64 instructions for the two vectors plus
// 8 to advance the two (cos, sin) pairs.  The trigonometric values come from two-level rotation tables
// per layer, advanced across the thread's J frequencies by a fixed rotation (equally spaced bins).
#include <cstdlib>
#include "rfinv_common.cuh"

#if defined(RFINV_PHASE_TIMING) && !defined(RFINV_FWD_GENERAL_TU)
// Debug build only (tools/phase_timing.py): per-phase cycle totals of forward_kernel, summed over CTAs.
__device__ unsigned long long g_phase[16];
#define PHASE_MARK(i)                                                            \
  do {                                                                           \
    if (tid == 0) {                                                              \
      const long long now__ = clock64();                                         \
      atomicAdd(&g_phase[i], (unsigned long long)(now__ - t_phase__));           \
      t_phase__ = now__;                                                         \
    }                                                                            \
  } while (0)
#define PHASE_INIT() long long t_phase__ = clock64(); if (tid == 0) atomicAdd(&g_phase[15], 1ULL)
extern "C" int rfinv_debug_get_phases(unsigned long long* out) {
  cudaError_t e = cudaMemcpyFromSymbol(out, g_phase, sizeof(g_phase));
  unsigned long long zero[16] = {0};
  cudaMemcpyToSymbol(g_phase, zero, sizeof(zero));
  return e == cudaSuccess ? 0 : 2;
}
// prep_kernel phases (lane 0 of every warp), slots 8..14
#define PREP_MARK(i)                                                             \
  do {                                                                           \
    if (lane == 0) {                                                             \
      const long long now__ = clock64();                                         \
      atomicAdd(&g_phase[8 + (i)], (unsigned long long)(now__ - tp_phase__));    \
      tp_phase__ = now__;                                                        \
    }                                                                            \
  } while (0)
#define PREP_INIT() long long tp_phase__ = clock64()
#else
#define PHASE_MARK(i) do { } while (0)
#define PHASE_INIT() do { } while (0)
#define PREP_MARK(i) do { } while (0)
#define PREP_INIT() do { } while (0)
#endif

namespace {

// Per (model, ray, solid layer) constants, written by prep_kernel.
struct LayerConst {
  double c1x, s1x, c1e, s1e;      // cos, sin of thx = domg*xi*h and the = domg*eta*h: the phase advance per frequency bin
  double c16x, s16x, c16e, s16e;  // cos, sin of 16 thx, 16 the (seeds of the two table levels of forward_kernel)
  double cbx, sbx, cbe, sbe;  // rotation by B*thx, B*the (B = threads per CTA = frequency stride of a thread)
  double t12, t21;            // interface to the next layer, {1,4} block [[1, t12], [t21, 1]] on (P, S) coordinates
  double u11, u12, u21, u22;  // interface to the next layer, {2,3} block
  double cb2x, cb2e;          // 2 cbx, 2 cbe: third and later bins of a thread by cos((m+1)b + t) = 2 cos b cos(mb + t) - cos((m-1)b + t)
};
constexpr int LC_DOUBLES = sizeof(LayerConst) / sizeof(double);  // 20
static_assert(LC_DOUBLES % 2 == 0, "LayerConst is moved in 16-byte pieces");

// The rays one forward_kernel launch works on: every ray of the configuration, or -- when the traces have different
// band limits -- the traces of one band-limit group, so that each group runs the kernel variant built for its width.
// (trace indices packed four bits each: a kernel parameter array indexed at run time would be copied to local memory)
struct TraceSel {
  int n;
  unsigned long long packed;
  __host__ __device__ int t(int i) const { return (int)((packed >> (4 * i)) & 15ULL); }
  __host__ void push(int trace) { packed |= (unsigned long long)trace << (4 * n); ++n; }
};
static_assert(RFINV_MAX_TRC <= 16, "TraceSel packs trace indices in four bits");

// Per (model, ray) constants written by prep_kernel.
struct RayConst {
  double h14[4], h23[4];      // rows 3,4 of E^-1 (1/w factors removed) times the last solid layer's basis, per block
  double a1, b1;              // start vector e1 in the wave coordinates of the top solid layer
  double q1a, q1b, q2a, q2b;  // start vector (0, cw, 0, -rw sw): (a1,b1) = sw*(q1a,q1b), (a2,b2) = cw*(q2a,q2b)
  double thw, cbw, sbw;       // water layer: phase per bin, stride rotation
  double wseed[4];            // cos, sin of thw and of 16 thw: seeds of the water-layer phase table
  double tp;                  // direct-arrival delay (src/forward.f90:474-491)
  double2 edge[4];            // fr, fv at the DC pseudo-frequency and at Nyquist
  double sta[4];              // buried station: displacement rows of the scaled basis of the layer above it,
                              // y1 = sta0 a1 + sta1 b1, y2 = sta2 a2 + sta3 b2 (wave coordinates after that layer's rotation)
  int k, valid;               // k: solid layers above the bottom boundary condition (model layers + the split at a buried station)
  int npre, l_sta;            // nint((-t_start -/+ tp)/delta): circular shift of the trace (src/forward.f90:177, 186);
                              // index of the (sub)layer whose bottom is the buried station, -1 = station at the surface
};
constexpr int RC_DOUBLES = sizeof(RayConst) / sizeof(double);
static_assert(sizeof(RayConst) % 16 == 0, "RayConst is moved in 16-byte pieces");

__device__ __forceinline__ void rot(double& c, double& s, double cb, double sb) {
  double c2 = c * cb - s * sb;
  double s2 = s * cb + c * sb;
  c = c2;
  s = s2;
}

// One vector in wave coordinates: (a1, a2) the standing P wave, (b1, b2) the standing S wave of the layer.
// Physical components {1,4} depend on (a1, b1) only, components {2,3} on (a2, b2) only.
struct Wave { double a1, a2, b1, b2; };

// the layer itself: rotate the P pair by w xi h = (c1,s1) and the S pair by w eta h = (c2,s2)
__device__ __forceinline__ void wave_rotate(Wave& w, double c1, double s1, double c2, double s2) {
  const double a1 = fma(-s1, w.a2, c1 * w.a1);
  const double a2 = fma(s1, w.a1, c1 * w.a2);
  const double b1 = fma(-s2, w.b2, c2 * w.b1);
  const double b2 = fma(s2, w.b1, c2 * w.b2);
  w.a1 = a1; w.a2 = a2; w.b1 = b1; w.b2 = b2;
}

// the interface below it: coordinates of the same displacement-stress vector in the next layer's basis
__device__ __forceinline__ void wave_interface(Wave& w, double t12, double t21, double u11, double u12, double u21,
                                               double u22) {
  const double a1 = fma(t12, w.b1, w.a1);
  const double b1 = fma(t21, w.a1, w.b1);
  const double a2 = fma(u12, w.b2, u11 * w.a2);
  const double b2 = fma(u22, w.b2, u21 * w.a2);
  w.a1 = a1; w.a2 = a2; w.b1 = b1; w.b2 = b2;
}

__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
  return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

// Boundary conditions (src/forward.f90:267-287) in the scaled real basis, then the sign conventions of
// calc_rf (src/forward.f90:145-146): fr = conj(ur), fv = -conj(uz).  (A3, A4) / (B3, B4) are rows 3,4 of
// E^-1 prod(P) applied to the two propagated vectors: real parts from the {1,4} block, imaginary parts from {2,3}.
// `gain` multiplies both results (the Gaussian filter weight of the bin: folded into the reciprocal of the determinant).
__device__ __forceinline__ void surface_response(const double* h14, const double* h23, const Wave& wa, const Wave& wb,
                                                 double cw, int ipha, double2& fr, double2& fv, double gain = 1.0) {
  const double2 A3 = make_double2(fma(h14[0], wa.a1, h14[1] * wa.b1), fma(h23[0], wa.a2, h23[1] * wa.b2));
  const double2 A4 = make_double2(fma(h14[2], wa.a1, h14[3] * wa.b1), fma(h23[2], wa.a2, h23[3] * wa.b2));
  const double2 B3 = make_double2(fma(h14[0], wb.a1, h14[1] * wb.b1), fma(h23[0], wb.a2, h23[1] * wb.b2));
  const double2 B4 = make_double2(fma(h14[2], wb.a1, h14[3] * wb.b1), fma(h23[2], wb.a2, h23[3] * wb.b2));
  const double2 p = cmul(A3, B4), q = cmul(B3, A4);
  const double2 dl = make_double2(p.x - q.x, p.y - q.y);
  const double rn = gain / (dl.x * dl.x + dl.y * dl.y);
  const double2 inv = make_double2(dl.x * rn, -dl.y * rn);
  double2 ur, uz;
  if (ipha >= 0) {
    ur = cmul(B4, inv);
    const double2 w = cmul(A4, inv);  // uz = -i * A4/Delta * cos_w
    uz = make_double2(w.y * cw, -w.x * cw);
  } else {
    const double2 w0 = cmul(B3, inv);
    ur = make_double2(-w0.x, -w0.y);
    const double2 w = cmul(A3, inv);  // uz = +i * A3/Delta * cos_w
    uz = make_double2(-w.y * cw, w.x * cw);
  }
  fr = make_double2(ur.x, -ur.y);
  fv = make_double2(-uz.x, uz.y);
}

// Buried station (src/forward.f90:289-338, commented out in the reference): the surface vector (ur, uz, 0, s4) is the
// combination alpha * e1 + beta * (0, cw, 0, -rw sw) of the two start vectors, alpha = ur, beta = -i uz / cw, so the
// displacement at depth is the same combination of the two propagated vectors there.  (ya1, ya2) / (yb1, yb2): their
// displacement components at the station in the scaled real basis (component 2 carries the factor i of D).
__device__ __forceinline__ void surface_response_buried(const double* h14, const double* h23, const Wave& wa, const Wave& wb,
                                                        int ipha, double2 ya, double2 yb, double2& fr, double2& fv) {
  const double2 A3 = make_double2(fma(h14[0], wa.a1, h14[1] * wa.b1), fma(h23[0], wa.a2, h23[1] * wa.b2));
  const double2 A4 = make_double2(fma(h14[2], wa.a1, h14[3] * wa.b1), fma(h23[2], wa.a2, h23[3] * wa.b2));
  const double2 B3 = make_double2(fma(h14[0], wb.a1, h14[1] * wb.b1), fma(h23[0], wb.a2, h23[1] * wb.b2));
  const double2 B4 = make_double2(fma(h14[2], wb.a1, h14[3] * wb.b1), fma(h23[2], wb.a2, h23[3] * wb.b2));
  const double2 p = cmul(A3, B4), q = cmul(B3, A4);
  const double2 dl = make_double2(p.x - q.x, p.y - q.y);
  const double rn = 1.0 / (dl.x * dl.x + dl.y * dl.y);
  const double2 inv = make_double2(dl.x * rn, -dl.y * rn);
  double2 al, be;
  if (ipha >= 0) {       // ur = B4/Delta, uz = -i cw A4/Delta
    al = cmul(B4, inv);
    const double2 w = cmul(A4, inv);
    be = make_double2(-w.x, -w.y);
  } else {               // ur = -B3/Delta, uz = +i cw A3/Delta
    const double2 w0 = cmul(B3, inv);
    al = make_double2(-w0.x, -w0.y);
    be = cmul(A3, inv);
  }
  const double2 ur = make_double2(fma(al.x, ya.x, be.x * yb.x), fma(al.y, ya.x, be.y * yb.x));
  const double2 s = make_double2(fma(al.x, ya.y, be.x * yb.y), fma(al.y, ya.y, be.y * yb.y));
  const double2 uz = make_double2(-s.y, s.x);   // i * s
  fr = make_double2(ur.x, -ur.y);
  fv = make_double2(-uz.x, uz.y);
}

// 2x2 helpers, row-major m[4] = {m11, m12, m21, m22}
__device__ __forceinline__ void mat2_mul(const double* a, const double* b, double* c) {
  const double c0 = fma(a[0], b[0], a[1] * b[2]), c1 = fma(a[0], b[1], a[1] * b[3]);
  const double c2 = fma(a[2], b[0], a[3] * b[2]), c3 = fma(a[2], b[1], a[3] * b[3]);
  c[0] = c0; c[1] = c1; c[2] = c2; c[3] = c3;
}

// ------------------------------------------------------------------------------------------------
// prep_kernel: one CTA per MODEL, one warp per ray, lane <-> layer.  format_model (src/model.f90:175-290) once per
// model, then per ray the per-layer constants of the wave-coordinate propagator (rotation angles, interface blocks),
// half-space / water-layer constants, the direct-arrival delay, and the two bins that do not fit the regular
// frequency grid of forward_kernel: the DC pseudo-frequency omega = 1.0e-5 (src/forward.f90:246-248) and Nyquist.
//
// Basis of a solid layer (columns = standing P wave, standing S wave; rows = components {1,4} / {2,3}):
//   V14 = [[p, 1], [rho bp, -2 rho beta^2 p]],          V14^-1 = [[2 beta^2 p, 1/rho], [bp, -p/rho]]
//   V23 = [[xi, -p/eta], [-2 rho beta^2 p xi, -rho bp/eta]],   V23^-1 = [[bp/xi, -p/(rho xi)], [-2 beta^2 p eta, -eta/rho]]
// with bp = 1 - 2 beta^2 p^2; B_l = V R V^-1 reproduces layer_matrix_sol (src/forward.f90:385-421).
// The basis of layer l is scaled by (sP_l, sS_l) on its (P, S) columns so that T14_l = V14_l^-1 V14_{l-1} has a
// unit diagonal: with tau = (unscaled V_l^-1)(unscaled V_{l-1}), sP_l = prod tau14[0][0], sS_l = prod tau14[1][1]
// (warp prefix products), and the interface constants only need the ratio r = sS/sP of the layer above.
//
// Phases: (A) warp 0: rank sort of the interfaces, then everything of a layer that does not depend on the ray --
// reference-velocity lookup, validity, density, 1/alpha^2, 1/beta^2 -- one layer per lane, left in shared memory for
// the other warps; (B) every warp, for its ray: per-layer physics with all transcendental functions, prefix products
// and interface constants, ray constants; (C) the only serial part, once per model: the four edge-bin vectors
// (a | b) x (DC | Nyquist) of EVERY ray go down the stack side by side, four lanes per ray, next to the lanes that sum
// the delays in the reference's order; (D) the finished RayConst records leave through one coalesced copy.
// ------------------------------------------------------------------------------------------------
struct PrepBasis {   // per (ray, layer), shared memory
  double v14[4], v23[4];   // unscaled basis blocks of this layer
  double i14[4], i23[4];   // their inverses (closed form)
};
struct PrepSerial {  // per (ray, layer): what the serial pass reads
  double tr[8];            // cos, sin of (w xi h), (w eta h) at the DC pseudo-frequency, then at Nyquist
  double ic[6];            // t12, t21, u11, u12, u21, u22 of the interface below this layer
  double tpterm, pad;
};
struct PrepShared {  // per layer of the propagation: independent of the ray
  double h, rho, irho, beta2, inv_b2, inv_a2, a, b;
};
constexpr int PB_DOUBLES = sizeof(PrepBasis) / sizeof(double), PS_DOUBLES = sizeof(PrepSerial) / sizeof(double);
constexpr int PSH_DOUBLES = sizeof(PrepShared) / sizeof(double);
constexpr int PREP_RAYS_PER_PASS = 6;   // rays of one serial pass: 4 vector lanes + 1 delay lane each
constexpr int PREP_MISC_DOUBLES = 8;    // k, ls, valid (ints) and h_part
// shared memory of a prep_kernel CTA, in doubles: [model part | per-ray part x rays]
__host__ __device__ inline size_t prep_sorted_doubles(int km) { return ((size_t)3 * km + 1) & ~(size_t)1; }   // zs | dps | dss, 16-byte granular
__host__ __device__ inline size_t prep_smem_model_doubles(int km) { return prep_sorted_doubles(km) + (size_t)(km + 2) * PSH_DOUBLES + PREP_MISC_DOUBLES; }
__host__ __device__ inline size_t prep_smem_ray_doubles(int km) { return (size_t)(km + 1) * PB_DOUBLES + (size_t)km * PS_DOUBLES + RC_DOUBLES + 8; }

// sin, cos of a small argument (|x| < 0.01: Taylor remainder < 3e-21); falls back to sincos otherwise
__device__ __forceinline__ void small_sincos(double x, double* sn, double* cs) {
  if (fabs(x) < 0.01) {
    const double x2 = x * x;
    *cs = fma(x2, fma(x2, fma(x2, -1.0 / 720.0, 1.0 / 24.0), -0.5), 1.0);
    *sn = x * fma(x2, fma(x2, fma(x2, -1.0 / 5040.0, 1.0 / 120.0), -1.0 / 6.0), 1.0);
  } else {
    sincos(x, sn, cs);
  }
}

__device__ __forceinline__ double warp_scan_mul(double x, int lane) {   // inclusive prefix product, fixed order
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x *= y;
  }
  return x;
}

// HOSTLAYOUT: the batch of rfinv_eval_batch (chain-slowest arrays, possibly still arriving piece by piece); the
// device-resident variants carry none of that
template <bool BURIED, bool HOSTLAYOUT>
__global__ void __maxnreg__(80) prep_kernel(const DevConfig cfg, const ModelBatch mb, double* __restrict__ lc_out,
                                                                 double* __restrict__ rc_out, uint8_t* __restrict__ is_valid,
                                                                 int* __restrict__ counter, int n_models, int ntr_eff, int nthr_fwd,
                                                                 int rays_per_cta, int m_begin) {
  extern __shared__ __align__(16) double prep_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // a model with many rays is spread over several CTAs (shared memory): group g works on rays [t_first, t_first + nr_cta)
  const int n_groups = (ntr_eff + rays_per_cta - 1) / rays_per_cta;
  const int bm = blockIdx.x / n_groups, t_first = (blockIdx.x - bm * n_groups) * rays_per_cta;
  const int ci = m_begin + bm;                 // this launch covers the models [m_begin, n_models) of the batch (host path: one piece)
  const int nr_cta = min(rays_per_cta, ntr_eff - t_first);
  pdl_trigger();   // forward_kernel may take the SM slots this kernel's last wave frees (it waits for our results: pdl_wait)
  if (blockIdx.x == 0 && m_begin == 0 && threadIdx.x < RFINV_MAX_TRC) counter[threadIdx.x] = 0;   // work counters of the forward_kernel launches that follow on the same stream
  if (ci >= n_models) return;
  if (mb.n_active_dev && ci >= *mb.n_active_dev) return;
  const int c = mb.active ? mb.active[ci] : ci;
  const int km = cfg.k_max, C = mb.C;
  const bool has_ray = warp < nr_cta;          // (a short last group leaves warps without a ray: they only keep the barriers)
  const int t0 = t_first + (has_ray ? warp : 0);   // the ray of this warp
  const size_t item = (size_t)ci * ntr_eff + t0;
  // ---- shared memory ----
  double* zs = prep_smem;                      // sorted interfaces and their perturbations
  double *dps = zs + km, *dss = dps + km;
  PrepShared* LA = reinterpret_cast<PrepShared*>(zs + prep_sorted_doubles(km));   // [km + 2]
  double* s_misc = reinterpret_cast<double*>(LA + km + 2);
  int* s_int = reinterpret_cast<int*>(s_misc + 1);                               // k, ls, valid
  double* ray0 = s_misc + PREP_MISC_DOUBLES;
  const size_t ray_stride = prep_smem_ray_doubles(km);
  auto ray_basis = [&](int t) { return reinterpret_cast<PrepBasis*>(ray0 + (size_t)t * ray_stride); };                  // [km + 1]
  auto ray_serial = [&](int t) { return reinterpret_cast<PrepSerial*>(ray0 + (size_t)t * ray_stride + (size_t)(km + 1) * PB_DOUBLES); };   // [km]
  auto ray_const = [&](int t) { return reinterpret_cast<RayConst*>(ray0 + (size_t)t * ray_stride + (size_t)(km + 1) * PB_DOUBLES + (size_t)km * PS_DOUBLES); };
  auto ray_water = [&](int t) { return reinterpret_cast<double*>(ray_const(t)) + RC_DOUBLES; };   // cw0, sw0, cw1, sw1 | xi, eta, bp of the half space
  constexpr bool buried = BURIED;   // cfg.bdep > 0

  PREP_INIT();
  if (warp == 0) {
    // The layer count and the model arrays are requested together (one memory latency instead of two): every lane loads
    // its elements whether or not they lie below k -- the arrays are k_max long -- and drops the rest.
    int k = mb.k[c];
    double zr[2] = {0.0, 0.0}, dr[2] = {0.0, 0.0}, sr[2] = {0.0, 0.0};
    static_assert(RFINV_MAX_K <= 64, "two elements per lane");
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int i = lane + 32 * q;
      if (i < km - 1) {
        if (HOSTLAYOUT) {
          zr[q] = mb.z[(size_t)c * (km - 1) + i]; sr[q] = mb.dvs[(size_t)c * km + i];
          if (cfg.vp_mode == 1) dr[q] = mb.dvp[(size_t)c * km + i];   // not uploaded at vp_mode 0 (format_model never reads it)
        } else {
          zr[q] = mb.z[(size_t)i * C + c]; dr[q] = mb.dvp[(size_t)i * C + c]; sr[q] = mb.dvs[(size_t)i * C + c];
        }
      }
    }
    double dvs_half, dvp_half = 0.0;              // perturbations of the half space: element k_max of the arrays
    if (HOSTLAYOUT) { dvs_half = mb.dvs[(size_t)c * km + km - 1]; if (cfg.vp_mode == 1) dvp_half = mb.dvp[(size_t)c * km + km - 1]; }
    else { dvs_half = mb.dvs[(size_t)(km - 1) * C + c]; dvp_half = mb.dvp[(size_t)(km - 1) * C + c]; }
    k = k < 1 ? 1 : (k > km - 1 ? km - 1 : k);
    // ---- sort the k interfaces by depth with their perturbations (src/sort.f90:34-68; ties keep their order) ----
    double* zu = reinterpret_cast<double*>(ray_basis(0));   // unsorted z, dvp, dvs: the region is rewritten in phase B
    double *du = zu + km, *su = du + km;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int i = lane + 32 * q;
      if (i < k) { zu[i] = zr[q]; du[i] = dr[q]; su[i] = sr[q]; }
    }
    __syncwarp();
    for (int i = lane; i < k; i += 32) {
      const double zi = zu[i];
      int rank = 0;
      for (int j = 0; j < k; ++j) { const double zj = zu[j]; rank += (zj < zi || (zj == zi && j < i)) ? 1 : 0; }
      zs[rank] = zi; dps[rank] = du[i]; dss[rank] = su[i];
    }
    __syncwarp();

    // ---- buried station (src/forward.f90:308-334, commented out in the reference): the layer that holds it is split at the
    // station depth into two sublayers of the same material, so the station sits on a (transparent) interface of the
    // propagation; a station below the last interface adds a layer of half-space material on top of the half space.
    // ls = model layer with the station (k = half space), h_part = its thickness above the station; same running sum
    // as the reference (z_tmp = z_tmp + h(ilay); z_tmp < bdep continues).
    int ls = -1;
    double h_part = 0.0;
    if (buried) {
      double z_tmp = 0.0;
      ls = k;
      for (int l = 0; l < k; ++l) {
        const double hl = l == 0 ? __dsub_rn(zs[0], cfg.sdep) : __dsub_rn(zs[l], zs[l - 1]);
        z_tmp = __dadd_rn(z_tmp, hl);
        if (!(z_tmp < cfg.bdep)) { ls = l; h_part = __dsub_rn(__dadd_rn(cfg.bdep, hl), z_tmp); break; }
      }
      if (ls == k) h_part = __dsub_rn(cfg.bdep, z_tmp);
    }
    const int ka = buried ? k + 1 : k;    // solid layers of the propagation
    PREP_MARK(0);
    // ---- what a layer has that does not depend on the ray, one layer per lane ----
    bool valid = true;
    for (int la = lane; la <= ka; la += 32) {
      const int l = (buried && la > ls) ? la - 1 : la;       // model layer behind propagation layer la
      double zc, h, dvs_l, dvp_l;
      if (l == 0) { zc = __dmul_rn(0.5, __dadd_rn(cfg.sdep, zs[0])); h = __dsub_rn(zs[0], cfg.sdep); dvs_l = dss[0]; dvp_l = dps[0]; }
      else if (l < k) { zc = __dmul_rn(0.5, __dadd_rn(zs[l], zs[l - 1])); h = __dsub_rn(zs[l], zs[l - 1]); dvs_l = dss[l]; dvp_l = dps[l]; }
      else { zc = __dmul_rn(0.5, __dadd_rn(cfg.z_max, zs[k - 1])); h = 999.0; dvs_l = dvs_half; dvp_l = dvp_half; }
      double a, b;
      bool ok = layer_velocity(cfg, zc, dvs_l, dvp_l, a, b);
      if (l == 0) ok = ok && !(h < __dmul_rn(0.125, a));     // src/model.f90:229
      else if (l < k) ok = ok && !(h < cfg.h_min);           // src/model.f90:257
      valid = valid && ok;
      if (buried) {
        if (la == ls) h = h_part;                                        // above the station
        else if (la == ls + 1 && ls < k) h = __dsub_rn(h, h_part);       // rest of the split layer
      }
      PrepShared S;
      S.h = h; S.a = a; S.b = b;
      S.rho = vp_to_rho(a);
      S.irho = 1.0 / S.rho;
      S.beta2 = __dmul_rn(b, b);
      S.inv_b2 = __ddiv_rn(1.0, S.beta2);                     // src/forward.f90:395
      S.inv_a2 = __ddiv_rn(1.0, __dmul_rn(a, a));             // src/forward.f90:396
      LA[la] = S;
    }
    valid = __all_sync(0xffffffffu, valid);
    if (lane == 0) { s_int[0] = k; s_int[1] = ls; s_int[2] = valid ? 1 : 0; s_misc[0] = h_part; }
    PREP_MARK(1);
  }
  __syncthreads();

  const int k = s_int[0], ls = s_int[1];
  const bool valid = s_int[2] != 0;
  const int ka = buried ? k + 1 : k;
  // Layers above the bottom boundary condition.  A station in the half space does not move it: the incident wave keeps
  // its phase reference at the last model interface (src/forward.f90:250-264), the extra layer only carries the
  // vectors on to the station.
  const int kb = (buried && ls == k) ? k : ka;
  PrepBasis* PB = ray_basis(warp);
  PrepSerial* PS = ray_serial(warp);
  if (has_ray) {

  // ---- (B) per-layer physics of this ray, one layer per lane ----
  const double p = cfg.rayp[t0];
  const int ipha = cfg.ipha[t0];
  const double p2 = __dmul_rn(p, p);
  const double nyq = (double)(cfg.nfft / 2);
  int nyq_doublings = 0;
  while ((nthr_fwd << nyq_doublings) < cfg.nfft_p2 / 2) ++nyq_doublings;   // nfft/2 = nthr_fwd * 2^d (nfft a power of two)
  for (int la = lane; la <= ka; la += 32) {
    const PrepShared S = LA[la];
    const double h = S.h, rho = S.rho, beta2 = S.beta2;
    double tp_sign = 1.0;                                  // direct-arrival delay counts from the station down
    if (buried) {
      if (la == ls) tp_sign = ls == k ? -1.0 : 0.0;        // above the station (in the half space: negative)
      else if (la < ls) tp_sign = 0.0;
    }
    const double bp = 1.0 - 2.0 * beta2 * p2;
    const double eta = sqrt(__dsub_rn(S.inv_b2, p2));      // src/forward.f90:395
    const double xi = sqrt(__dsub_rn(S.inv_a2, p2));       // src/forward.f90:396
    if (la < ka) {
      PrepBasis& Q = PB[la];
      PrepSerial& Z = PS[la];
      const double g2 = 2.0 * beta2 * p;   // 2 beta^2 p
      const double ieta = 1.0 / eta, irho = S.irho, ixi = 1.0 / xi;
      Q.v14[0] = p; Q.v14[1] = 1.0; Q.v14[2] = rho * bp; Q.v14[3] = -rho * g2;
      Q.v23[0] = xi; Q.v23[1] = -p * ieta; Q.v23[2] = -rho * g2 * xi; Q.v23[3] = -rho * bp * ieta;
      Q.i14[0] = g2; Q.i14[1] = irho; Q.i14[2] = bp; Q.i14[3] = -p * irho;
      Q.i23[0] = bp * ixi; Q.i23[1] = -p * irho * ixi; Q.i23[2] = -g2 * eta; Q.i23[3] = -eta * irho;
      Z.tpterm = cfg.deconv_mode == 0 ? __dmul_rn(tp_sign, __dmul_rn(h, ipha == 1 ? xi : eta)) : 0.0;   // src/forward.f90:489-491
      LayerConst* L = reinterpret_cast<LayerConst*>(lc_out) + item * km + la;
      // All transcendental functions of the layer: the phase advance per bin; 16 times it (forward_kernel builds its
      // two-level rotation tables from these two seeds by angle addition alone) and the stride rotation B = 16 * 2^d follow
      // by angle doubling (4 + d <= 8 doublings: a phase error of at most 2^8 ulp = 3e-14, against a tolerance of 1e-9).
      const double thx = cfg.domg * xi * h, the = cfg.domg * eta * h;
      double snx, csx, sne, cse;
      sincos(thx, &snx, &csx); L->c1x = csx; L->s1x = snx;
      sincos(the, &sne, &cse); L->c1e = cse; L->s1e = sne;
#pragma unroll
      for (int d = 0; d < 4; ++d) {
        const double c2 = fma(csx, csx, -snx * snx), s2 = 2.0 * csx * snx; csx = c2; snx = s2;
        const double c3 = fma(cse, cse, -sne * sne), s3 = 2.0 * cse * sne; cse = c3; sne = s3;
      }
      L->c16x = csx; L->s16x = snx; L->c16e = cse; L->s16e = sne;
      for (int b = 16; b < nthr_fwd; b <<= 1) {
        const double c2 = fma(csx, csx, -snx * snx), s2 = 2.0 * csx * snx; csx = c2; snx = s2;
        const double c3 = fma(cse, cse, -sne * sne), s3 = 2.0 * cse * sne; cse = c3; sne = s3;
      }
      L->cbx = csx; L->sbx = snx; L->cbe = cse; L->sbe = sne;
      L->cb2x = csx + csx; L->cb2e = cse + cse;
      small_sincos((double)1.0e-5f * xi * h, &Z.tr[1], &Z.tr[0]);   // (omega*xi)*z with omega = 1.0e-5 (single precision literal)
      small_sincos((double)1.0e-5f * eta * h, &Z.tr[3], &Z.tr[2]);
      // Nyquist = (nfft/2) bins = nyq_doublings doublings of the stride rotation; its bin carries the smallest
      // filter weight of the whole spectrum, so the doubled rounding error is immaterial
      double cn = csx, sn2 = snx, ce = cse, se = sne;
      if (cfg.fft_general) {   // nfft/2 is not the stride times a power of two: straight from the angle
        sincos(nyq * thx, &sn2, &cn);
        sincos(nyq * the, &se, &ce);
      } else {
        for (int d = 0; d < nyq_doublings; ++d) {
          const double c2 = fma(cn, cn, -sn2 * sn2), s2 = 2.0 * cn * sn2; cn = c2; sn2 = s2;
          const double c3 = fma(ce, ce, -se * se), s3 = 2.0 * ce * se; ce = c3; se = s3;
        }
      }
      Z.tr[4] = cn; Z.tr[5] = sn2; Z.tr[6] = ce; Z.tr[7] = se;
    } else {   // half space: its ray-dependent quantities go to the ray constants through shared memory
      double* W = ray_water(warp);
      W[4] = xi; W[5] = eta; W[6] = bp;
    }
  }
  __syncwarp();

  PREP_MARK(2);
  // ---- interfaces l-1 -> l (l = 1..k-1): tau = V_l^-1 V_{l-1} unscaled, prefix products of its {1,4} diagonal ----
  double carryP = 1.0, carryS = 1.0;      // scale products of the slots already done
  double sP_last = 1.0, sS_last = 1.0;    // scales of the last solid layer above the half space (kb-1)
  double sP_sta = 1.0, sS_sta = 1.0;      // scales of the layer above a buried station
  for (int base = 0; base < ka; base += 32) {
    const int l = base + lane;
    double t14[4] = {1.0, 0.0, 0.0, 1.0}, t23[4] = {1.0, 0.0, 0.0, 1.0};
    if (l >= 1 && l < ka) {
      mat2_mul(PB[l].i14, PB[l - 1].v14, t14);
      mat2_mul(PB[l].i23, PB[l - 1].v23, t23);
    }
    const double sP = carryP * warp_scan_mul(t14[0], lane), sS = carryS * warp_scan_mul(t14[3], lane);   // scales of layer l
    double sPp = __shfl_up_sync(0xffffffffu, sP, 1), sSp = __shfl_up_sync(0xffffffffu, sS, 1);           // scales of layer l-1
    if (lane == 0) { sPp = carryP; sSp = carryS; }
    if (l >= 1 && l < ka) {
      double* ic = PS[l - 1].ic;
      const double rP = 1.0 / sP, rS = 1.0 / sS;
      const double pp = sPp * rP, sp = sSp * rP, ps = sPp * rS, ss = sSp * rS;
      ic[0] = t14[1] * sp; ic[1] = t14[2] * ps;
      ic[2] = t23[0] * pp; ic[3] = t23[1] * sp; ic[4] = t23[2] * ps; ic[5] = t23[3] * ss;
      LayerConst* L = reinterpret_cast<LayerConst*>(lc_out) + item * km + (l - 1);
      L->t12 = ic[0]; L->t21 = ic[1]; L->u11 = ic[2]; L->u12 = ic[3]; L->u21 = ic[4]; L->u22 = ic[5];
    }
    const int last_lane = (ka - 1 - base) < 31 ? (ka - 1 - base) : 31;   // highest lane of this slot holding a solid layer
    if (buried && ls >= base && ls < base + 32) { sP_sta = __shfl_sync(0xffffffffu, sP, ls - base); sS_sta = __shfl_sync(0xffffffffu, sS, ls - base); }
    if (kb - 1 >= base && kb - 1 < base + 32) { sP_last = __shfl_sync(0xffffffffu, sP, kb - 1 - base); sS_last = __shfl_sync(0xffffffffu, sS, kb - 1 - base); }
    carryP = __shfl_sync(0xffffffffu, sP, last_lane);
    carryS = __shfl_sync(0xffffffffu, sS, last_lane);
  }
  if (lane == 0) {   // the last solid layer has no in-loop interface: the half space follows
    LayerConst* L = reinterpret_cast<LayerConst*>(lc_out) + item * km + (ka - 1);
    L->t12 = 0.0; L->t21 = 0.0; L->u11 = 1.0; L->u12 = 0.0; L->u21 = 0.0; L->u22 = 1.0;
    double* ic = PS[ka - 1].ic;
    ic[0] = 0.0; ic[1] = 0.0; ic[2] = 1.0; ic[3] = 0.0; ic[4] = 0.0; ic[5] = 1.0;
  }
  __syncwarp();

  PREP_MARK(3);
  // ---- ray constants: half space, water layer, start vectors ----
  {
    RayConst R;
    double cw0 = 1.0, sw0 = 0.0, cw1 = 1.0, sw1 = 0.0, rw = 0.0;
    if (cfg.sdep > 0.0) {   // water layer (src/model.f90:201-207, src/forward.f90:424-442)
      const double aw = 1.5, rhow = 1.0, hw = cfg.sdep;
      const double xiw = sqrt(1.0 / (aw * aw) - p * p);
      R.thw = cfg.domg * xiw * hw;
      sincos(R.thw, &R.wseed[1], &R.wseed[0]);
      R.cbw = R.wseed[0]; R.sbw = R.wseed[1];
#pragma unroll
      for (int d = 0; d < 4; ++d) { const double c2 = fma(R.cbw, R.cbw, -R.sbw * R.sbw), s2 = 2.0 * R.cbw * R.sbw; R.cbw = c2; R.sbw = s2; }
      R.wseed[2] = R.cbw; R.wseed[3] = R.sbw;
      for (int b = 16; b < nthr_fwd; b <<= 1) { const double c2 = fma(R.cbw, R.cbw, -R.sbw * R.sbw), s2 = 2.0 * R.cbw * R.sbw; R.cbw = c2; R.sbw = s2; }
      rw = rhow / xiw;
      small_sincos((double)1.0e-5f * xiw * hw, &sw0, &cw0);
      sincos(nyq * R.thw, &sw1, &cw1);
    } else {
      R.thw = 0.0; R.cbw = 1.0; R.sbw = 0.0;
      R.wseed[0] = R.wseed[2] = 1.0; R.wseed[1] = R.wseed[3] = 0.0;
    }
    {
      // half space: rows 3,4 of E^-1 (src/forward.f90:350-380) without their 1/omega factors, times the scaled basis of
      // the last solid layer
      const PrepShared& H = LA[ka];
      const double* W = ray_water(warp);
      const double a = H.a, b = H.b, rho = H.rho, beta2 = H.beta2, xi = W[4], eta = W[5], bp = W[6];
      const double r1 = 1.0 / (2.0 * rho * a * xi), r2 = 1.0 / (2.0 * rho * b * eta);
      const double e11 = beta2 * p * (2.0 * rho * xi) * r1, e12 = bp * rho * r1, e13 = p * r1, e14 = xi * r1;
      const double e21 = bp * rho * r2, e22 = b * p, e23 = eta * r2, e24 = p * r2;
      const double r14[4] = {e11, e14, e21, -e24};
      const double r23[4] = {-e12, e13, e22, e23};
      const PrepBasis& Q = PB[kb - 1];
      const double v14[4] = {Q.v14[0] * sP_last, Q.v14[1] * sS_last, Q.v14[2] * sP_last, Q.v14[3] * sS_last};
      const double v23[4] = {Q.v23[0] * sP_last, Q.v23[1] * sS_last, Q.v23[2] * sP_last, Q.v23[3] * sS_last};
      mat2_mul(r14, v14, R.h14);
      mat2_mul(r23, v23, R.h23);
    }
    {
      // start vectors in layer 0's coordinates (scale 1): e1, and (0, cw, 0, -rw sw) for a free / water-loaded surface
      const PrepBasis& Q = PB[0];
      R.a1 = Q.i14[0]; R.b1 = Q.i14[2];                   // V14^-1 (1, 0)^T
      R.q1a = -rw * Q.i14[1]; R.q1b = -rw * Q.i14[3];     // -rw V14^-1 (0, 1)^T
      R.q2a = Q.i23[0]; R.q2b = Q.i23[2];                 // V23^-1 (1, 0)^T
    }
    R.l_sta = -1;
    R.sta[0] = R.sta[1] = R.sta[2] = R.sta[3] = 0.0;
    if (buried) {   // displacement rows of V14 / V23 of the layer above the station, with that layer's scales
      const PrepBasis& Q = PB[ls];
      R.l_sta = ls;
      R.sta[0] = Q.v14[0] * sP_sta; R.sta[1] = Q.v14[1] * sS_sta;
      R.sta[2] = Q.v23[0] * sP_sta; R.sta[3] = Q.v23[1] * sS_sta;
    }
    R.k = kb;
    R.valid = valid;
    R.tp = 0.0; R.npre = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) R.edge[i] = make_double2(0.0, 0.0);
    if (lane == 0) {   // staged in shared memory; the serial pass completes it
      *ray_const(warp) = R;
      double* W = ray_water(warp);
      W[0] = cw0; W[1] = sw0; W[2] = cw1; W[3] = sw1;
    }
  }
  PREP_MARK(4);
  }   // has_ray
  __syncthreads();

  // ---- (C) serial part, once per model: four lanes per ray carry (vector a | b) x (DC | Nyquist) down the stack; one more
  // lane per ray sums the delay in the reference's order.  Up to PREP_RAYS_PER_PASS rays per warp. ----
  for (int r0 = warp * PREP_RAYS_PER_PASS; r0 < nr_cta; r0 += (int)(blockDim.x >> 5) * PREP_RAYS_PER_PASS) {   // r0: ray index inside the CTA
    const int nr = min(PREP_RAYS_PER_PASS, nr_cta - r0);
    const bool vec_lane = lane < 4 * nr, tp_lane = lane >= 4 * nr && lane < 5 * nr;
    const int tr_ray = r0 + (vec_lane ? (lane >> 2) : (tp_lane ? lane - 4 * nr : 0));   // the ray this lane works for
    const RayConst* Rr = ray_const(tr_ray);
    const double* Wr = ray_water(tr_ray);
    const PrepSerial* Zr = ray_serial(tr_ray);
    const bool is_b = lane & 1, is_nyq = (lane >> 1) & 1;
    Wave w;
    double2 y_sta = make_double2(0.0, 0.0);   // displacement components of this lane's vector at a buried station
    double tp = 0.0;
    {
      const double cw = is_nyq ? Wr[2] : Wr[0], sw = is_nyq ? Wr[3] : Wr[1];
      if (!is_b) { w.a1 = Rr->a1; w.b1 = Rr->b1; w.a2 = 0.0; w.b2 = 0.0; }
      else { w.a1 = sw * Rr->q1a; w.b1 = sw * Rr->q1b; w.a2 = cw * Rr->q2a; w.b2 = cw * Rr->q2b; }
    }
    if (vec_lane) {
      const int o = is_nyq ? 4 : 0;
      const double st0 = Rr->sta[0], st1 = Rr->sta[1], st2 = Rr->sta[2], st3 = Rr->sta[3];
      Wave w_bc = w;
      for (int l = 0; l < ka; ++l) {
        const PrepSerial& Q = Zr[l];
        wave_rotate(w, Q.tr[o], Q.tr[o + 1], Q.tr[o + 2], Q.tr[o + 3]);
        if (buried && l == ls) { y_sta.x = fma(st0, w.a1, st1 * w.b1); y_sta.y = fma(st2, w.a2, st3 * w.b2); }
        if (l == kb - 1) w_bc = w;   // what the bottom boundary condition sees
        if (l + 1 < ka) wave_interface(w, Q.ic[0], Q.ic[1], Q.ic[2], Q.ic[3], Q.ic[4], Q.ic[5]);
      }
      w = w_bc;
    } else if (tp_lane) {
      for (int l = 0; l < ka; ++l) tp = __dadd_rn(tp, Zr[l].tpterm);
      RayConst* Rw = ray_const(tr_ray);
      const int iph = cfg.ipha[t_first + tr_ray];
      Rw->tp = tp;
      Rw->npre = iph == 1 ? f_nint((-cfg.t_start - tp) / cfg.delta)    // src/forward.f90:177
                          : f_nint((-cfg.t_start + tp) / cfg.delta);   // src/forward.f90:186
    }
    PREP_MARK(5);
    // lanes 2r + e finish edge bin e (0 = DC, 1 = Nyquist) of ray r: vectors a, b of that bin sit in lanes 4r + 2e, 4r + 2e + 1
    {
      const int rr = lane >> 1, e = lane & 1;
      const bool fin = lane < 2 * nr;
      const int src_a = fin ? 4 * rr + 2 * e : 0, src_b = src_a + 1;
      Wave ea, eb;
      ea.a1 = __shfl_sync(0xffffffffu, w.a1, src_a); ea.a2 = __shfl_sync(0xffffffffu, w.a2, src_a);
      ea.b1 = __shfl_sync(0xffffffffu, w.b1, src_a); ea.b2 = __shfl_sync(0xffffffffu, w.b2, src_a);
      eb.a1 = __shfl_sync(0xffffffffu, w.a1, src_b); eb.a2 = __shfl_sync(0xffffffffu, w.a2, src_b);
      eb.b1 = __shfl_sync(0xffffffffu, w.b1, src_b); eb.b2 = __shfl_sync(0xffffffffu, w.b2, src_b);
      const double2 ya = make_double2(__shfl_sync(0xffffffffu, y_sta.x, src_a), __shfl_sync(0xffffffffu, y_sta.y, src_a));
      const double2 yb = make_double2(__shfl_sync(0xffffffffu, y_sta.x, src_b), __shfl_sync(0xffffffffu, y_sta.y, src_b));
      if (fin) {
        RayConst* Rf = ray_const(r0 + rr);
        const double* Wf = ray_water(r0 + rr);
        double h14[4], h23[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { h14[i] = Rf->h14[i]; h23[i] = Rf->h23[i]; }
        double2 fr, fv;
        if (!buried) surface_response(h14, h23, ea, eb, e ? Wf[2] : Wf[0], cfg.ipha[t_first + r0 + rr], fr, fv);
        else surface_response_buried(h14, h23, ea, eb, cfg.ipha[t_first + r0 + rr], ya, yb, fr, fv);
        Rf->edge[2 * e] = fr; Rf->edge[2 * e + 1] = fv;
      }
    }
  }
  __syncthreads();
  // ---- (D) the RayConst records of this model: one contiguous, coalesced copy ----
  {
    double2* dst = reinterpret_cast<double2*>(rc_out + ((size_t)ci * ntr_eff + t_first) * RC_DOUBLES);
    for (int i = threadIdx.x; i < nr_cta * (RC_DOUBLES / 2); i += blockDim.x) {
      const int t = i / (RC_DOUBLES / 2), j = i - t * (RC_DOUBLES / 2);
      dst[i] = reinterpret_cast<const double2*>(ray_const(t))[j];
    }
    if (is_valid && threadIdx.x == 0 && t_first == 0) is_valid[c] = (uint8_t)valid;
  }
  PREP_MARK(6);
}

// Twiddles of the radix-8 DIF stages, one table per stage laid out [q-1][o] (q = 1..7 output index of the butterfly,
// o < N/8 its offset inside the sub-transform of length N): entry = exp(+2 pi i q o / N).  Consecutive threads read
// consecutive entries (no bank conflicts, no quadrant logic).  Stages with N = 8 need none.
__host__ __device__ inline size_t fft_twiddle_entries(size_t n) {
  size_t e = 0;
  for (size_t N = n; N > 8; N >>= 3) e += 7 * (N >> 3);
  return e;
}
// fills the tables from the full-circle table tw[m] = exp(+2 pi i m / n) in global memory (once per CTA)
__device__ __forceinline__ void fill_fft_twiddles(double2* s_tw, const double2* __restrict__ tw, int n, int tid, int nthr) {
  int off = 0;
  for (int N = n; N > 8; N >>= 3) {
    const int stride = N >> 3, tmul = n / N;
    for (int i = tid; i < 7 * stride; i += nthr) {
      const int q = i / stride + 1, o = i - (q - 1) * stride;
      s_tw[off + i] = tw[q * o * tmul];
    }
    off += 7 * stride;
  }
}

// Position of logical element p in the padded FFT buffer: one pad element per 8 -- "8 consecutive elements per thread"
// (last radix-8 stage) and "consecutive elements across threads" are both conflict free -- plus, for n >= 512, one per
// n/8: the transform leaves element f at bit-reversed position, so the consecutive samples the output phase reads differ
// in the TOP bits of the position, which this term folds into the bank index (28 -> 5 wavefronts per warp-wide read at
// n = 1024; sh = log2(n) - 3, or 31 = no second term for the short transforms run by 32 / 64 threads).
__host__ __device__ __forceinline__ int fft_pad_shift(int log2n) { return log2n >= 9 ? log2n - 3 : 31; }
__device__ __forceinline__ int fpad(int p, int sh) { return p + (p >> 3) + (p >> sh); }
__device__ __forceinline__ unsigned fpad(unsigned p, int sh) { return p + (p >> 3) + (p >> sh); }
__host__ __device__ inline size_t fft_buf_elems(size_t n) { return n + (n >> 3) + 9; }

// 8-point inverse DFT in registers: v[q] <- sum_r v[r] exp(+2 pi i q r / 8).  Z = bit mask of inputs known to be zero (legs of
// the first FFT stage that lie above the band limit): their additions are dropped, not executed with a zero operand.
template <bool ZA, bool ZB>
__device__ __forceinline__ double2 zadd(double2 a, double2 b) {
  if constexpr (ZA && ZB) return make_double2(0.0, 0.0);
  else if constexpr (ZB) return a;
  else if constexpr (ZA) return b;
  else return make_double2(a.x + b.x, a.y + b.y);
}
template <bool ZA, bool ZB>
__device__ __forceinline__ double2 zsub(double2 a, double2 b) {
  if constexpr (ZA && ZB) return make_double2(0.0, 0.0);
  else if constexpr (ZB) return a;
  else if constexpr (ZA) return make_double2(-b.x, -b.y);
  else return make_double2(a.x - b.x, a.y - b.y);
}
template <unsigned Z = 0u>
__device__ __forceinline__ void dft8(double2* v) {
  const double hs = 0.70710678118654752440;
  constexpr bool z0 = Z & 1u, z1 = Z & 2u, z2 = Z & 4u, z3 = Z & 8u, z4 = Z & 16u, z5 = Z & 32u, z6 = Z & 64u, z7 = Z & 128u;
  double2 e0, e1, e2, e3, o0, o1, o2, o3;
  {
    const double2 a = zadd<z0, z4>(v[0], v[4]), b = zsub<z0, z4>(v[0], v[4]);
    const double2 c = zadd<z2, z6>(v[2], v[6]), dd = zsub<z2, z6>(v[2], v[6]), d = make_double2(-dd.y, dd.x);
    e0 = make_double2(a.x + c.x, a.y + c.y); e1 = make_double2(b.x + d.x, b.y + d.y);
    e2 = make_double2(a.x - c.x, a.y - c.y); e3 = make_double2(b.x - d.x, b.y - d.y);
  }
  {
    const double2 a = zadd<z1, z5>(v[1], v[5]), b = zsub<z1, z5>(v[1], v[5]);
    const double2 c = zadd<z3, z7>(v[3], v[7]), dd = zsub<z3, z7>(v[3], v[7]), d = make_double2(-dd.y, dd.x);
    o0 = make_double2(a.x + c.x, a.y + c.y);
    const double2 t1 = make_double2(b.x + d.x, b.y + d.y), t2 = make_double2(a.x - c.x, a.y - c.y);
    const double2 t3 = make_double2(b.x - d.x, b.y - d.y);
    o1 = make_double2((t1.x - t1.y) * hs, (t1.x + t1.y) * hs);     // * (1 + i)/sqrt 2
    o2 = make_double2(-t2.y, t2.x);                                // * i
    o3 = make_double2(-(t3.x + t3.y) * hs, (t3.x - t3.y) * hs);    // * (-1 + i)/sqrt 2
  }
  v[0] = make_double2(e0.x + o0.x, e0.y + o0.y); v[4] = make_double2(e0.x - o0.x, e0.y - o0.y);
  v[1] = make_double2(e1.x + o1.x, e1.y + o1.y); v[5] = make_double2(e1.x - o1.x, e1.y - o1.y);
  v[2] = make_double2(e2.x + o2.x, e2.y + o2.y); v[6] = make_double2(e2.x - o2.x, e2.y - o2.y);
  v[3] = make_double2(e3.x + o3.x, e3.y + o3.y); v[7] = make_double2(e3.x - o3.x, e3.y - o3.y);
}

// In-place decimation-in-frequency inverse FFT (sign +, unnormalised) of n complex points in the padded shared
// buffer: radix-8 stages while the sub-transform length N >= 8, then one radix-4 or radix-2 stage.  Every stage
// stores output q of a butterfly at bit-reversed digit position, so element f of the result ends up at logical
// position bitreverse(f).  One barrier per stage.  Returns the maximum imaginary part over all n outputs (the
// vertical trace rides in the imaginary part); the block reduction shares the last stage's barrier.
struct CtaSync { __device__ __forceinline__ void operator()() const { __syncthreads(); } };
// warp maximum -> s_red[warp]; the caller's next barrier publishes it to the CTA
__device__ __forceinline__ void publish_max(double v, double* s_red, int tid) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  if ((tid & 31) == 0) s_red[tid >> 5] = v;
}

// One radix-8 stage of sub-transform length N (compile time): strides, pad offsets and the twiddle table offset are
// constants; TW = twiddles follow the butterfly (every stage but N == 8), LAST = collect the maximum imaginary part.
// PLO..PHI (first stage only; empty when PLO > PHI): legs of every butterfly that hold zeros because their bins lie above the
// band limit of the trace (bins [J NT, n - J NT] except Nyquist): not loaded, not added.  The one exception is the
// butterfly with offset 0 (thread 0), whose leg 4 is the Nyquist bin: its contribution (+-X on the 8 outputs) is added back.
// WL (warp-local later stages): with exactly one butterfly per thread and stage (n = 8 nthr) the butterflies of a warp cover,
// from the second stage on, the same 256 consecutive elements in every stage -- after the first stage the warps no longer
// exchange data until the transform is complete, so those stages are separated by __syncwarp instead of a CTA barrier (no
// warp waits for the slowest one four times per transform).
template <int LOG2N, int N, class Sync, int PLO = 8, int PHI = -1, bool WL = false>
__device__ __forceinline__ void fft_stage8(double2* buf, const double2* __restrict__ stw, double& vmax, double* s_red, int tid,
                                           int nthr, Sync sync) {
  constexpr unsigned n = 1u << LOG2N, stride = N >> 3;
  constexpr bool prune = PLO <= PHI;
  constexpr unsigned zmask = prune ? (((1u << (PHI + 1)) - 1u) & ~((1u << PLO) - 1u)) : 0u;
  constexpr int PSH = LOG2N >= 9 ? LOG2N - 3 : 31;
  constexpr bool last = (N == 8);
  for (unsigned j = tid; j < (n >> 3); j += nthr) {
    const unsigned o = j & (stride - 1), base = ((j - o) << 3) + o;
    double2 v[8];
    unsigned pos[8];
    // base + r * stride never carries into bit PSH (a butterfly stays inside one block of n/8 elements, or, in the first
    // stage, moves by whole blocks): with whole groups of 8 between the legs the padded positions are one address plus
    // constant offsets
    if (stride % 8 == 0) {
      const unsigned p0 = fpad(base, PSH);
      constexpr unsigned step = stride + (stride >> 3) + (PSH < 31 ? (stride >> PSH) : 0u);
#pragma unroll
      for (int r = 0; r < 8; ++r) pos[r] = p0 + r * step;
    } else {
#pragma unroll
      for (int r = 0; r < 8; ++r) pos[r] = fpad(base + r * stride, PSH);
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) if (!((zmask >> r) & 1u)) v[r] = buf[pos[r]];
    if (!last) {
      double2 w[7];
#pragma unroll
      for (int q = 1; q < 8; ++q) w[q - 1] = stw[(q - 1) * stride + o];
      dft8<zmask>(v);
      if (prune && o == 0) {     // leg 4 of this butterfly is the Nyquist bin
        const double2 x = buf[pos[4]];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = (q & 1) ? make_double2(v[q].x - x.x, v[q].y - x.y) : make_double2(v[q].x + x.x, v[q].y + x.y);
      }
#pragma unroll
      for (int q = 1; q < 8; ++q) v[q] = cmul(v[q], w[q - 1]);
    } else {
      dft8(v);
#pragma unroll
      for (int q = 0; q < 8; ++q) vmax = fmax(vmax, v[q].y);
    }
    buf[pos[0]] = v[0]; buf[pos[4]] = v[1]; buf[pos[2]] = v[2]; buf[pos[6]] = v[3];
    buf[pos[1]] = v[4]; buf[pos[5]] = v[5]; buf[pos[3]] = v[6]; buf[pos[7]] = v[7];
  }
  if (last) publish_max(vmax, s_red, tid);   // N == 8: no stage follows
  if constexpr (WL && N < (1 << LOG2N) && !(last && LOG2N % 3 == 0)) __syncwarp();   // (the barrier that ends the transform stays)
  else sync();
  if constexpr (N >= 64) fft_stage8<LOG2N, (N >> 3), Sync, 8, -1, WL>(buf, stw + 7 * stride, vmax, s_red, tid, nthr, sync);
}

// JP, NT (optional): the spectrum is zero in bins [JP NT, n - JP NT] except Nyquist (band limit of forward_kernel)
template <int LOG2N, class Sync, int JP = 0, int NT = 1>
__device__ __forceinline__ double fft_inverse_dif_n(double2* buf, const double2* twq, double* s_red, int tid, int nthr, Sync sync) {
  constexpr unsigned n = 1u << LOG2N;
#ifdef RFINV_NO_FFT_PRUNE
  constexpr int PLO = 8, PHI = -1;
#else
  constexpr int jfull = (1 << (LOG2N - 1)) / NT;                          // bin groups of the full band
  constexpr int PLO = (JP > 0 && LOG2N >= 6) ? (4 * JP + jfull - 1) / jfull : 8, PHI = 7 - PLO;   // leg r covers bins [r n/8, (r+1) n/8)
#endif
  constexpr int PSH = LOG2N >= 9 ? LOG2N - 3 : 31;
  constexpr int REM = LOG2N % 3;          // what is left after the radix-8 stages: 1 (N = 1), 2 or 4
#ifdef RFINV_NO_FFT_WARPLOCAL
  constexpr bool WL = false;
#else
  constexpr bool WL = NT >= 32 && (NT << 3) == (1 << LOG2N) && LOG2N >= 9;   // one butterfly per thread and stage, whole warps
#endif
  double vmax = -INFINITY;
  fft_stage8<LOG2N, (1 << LOG2N), Sync, PLO, PHI, WL>(buf, twq, vmax, s_red, tid, nthr, sync);
  if (REM == 2) {
    // WL: the 64 quads of the warp's own 256 elements (two per lane) instead of quads tid, tid + nthr
    for (unsigned jj = tid; jj < (n >> 2); jj += nthr) {
      const unsigned j = WL ? (((unsigned)tid >> 5) << 6) + ((unsigned)tid & 31u) + ((jj >= (unsigned)nthr) ? 32u : 0u) : jj;
      const unsigned p0 = fpad(j << 2, PSH);     // the four elements share a pad group
      const double2 v0 = buf[p0], v1 = buf[p0 + 1], v2 = buf[p0 + 2], v3 = buf[p0 + 3];
      const double2 a0 = make_double2(v0.x + v2.x, v0.y + v2.y), a1 = make_double2(v0.x - v2.x, v0.y - v2.y);
      const double2 a2 = make_double2(v1.x + v3.x, v1.y + v3.y), a3 = make_double2(-(v1.y - v3.y), v1.x - v3.x);
      const double2 r0 = make_double2(a0.x + a2.x, a0.y + a2.y), r1 = make_double2(a1.x + a3.x, a1.y + a3.y);
      const double2 r2 = make_double2(a0.x - a2.x, a0.y - a2.y), r3 = make_double2(a1.x - a3.x, a1.y - a3.y);
      vmax = fmax(fmax(vmax, r0.y), fmax(fmax(r1.y, r2.y), r3.y));
      buf[p0] = r0; buf[p0 + 2] = r1; buf[p0 + 1] = r2; buf[p0 + 3] = r3;
    }
    publish_max(vmax, s_red, tid);
    sync();
  } else if (REM == 1) {
    // WL: the 128 pairs of the warp's own 256 elements (four per lane) instead of pairs tid + i nthr
    for (unsigned jj = tid, i = 0; jj < (n >> 1); jj += nthr, ++i) {
      const unsigned j = WL ? (((unsigned)tid >> 5) << 7) + ((unsigned)tid & 31u) + 32u * i : jj;
      const unsigned p0 = fpad(j << 1, PSH);     // both elements share a pad group
      const double2 a = buf[p0], b = buf[p0 + 1];
      const double2 r0 = make_double2(a.x + b.x, a.y + b.y), r1 = make_double2(a.x - b.x, a.y - b.y);
      vmax = fmax(vmax, fmax(r0.y, r1.y));
      buf[p0] = r0; buf[p0 + 1] = r1;
    }
    publish_max(vmax, s_red, tid);
    sync();
  }
  const int nw = (nthr + 31) >> 5;
  double r = s_red[0];
  for (int i = 1; i < nw; ++i) r = fmax(r, s_red[i]);
  return r;
}

// run-time length -> compile-time instantiation (nfft is a power of two in [64, 4096]); LO..HI = the lengths the caller
// can see (a kernel variant is tied to a thread count, hence to one or two transform lengths)
template <int LO, int HI, class Sync, int JP = 0, int NT = 1>
__device__ __forceinline__ double fft_inverse_dif(double2* buf, int n, const double2* twq, double* s_red, int tid, int nthr, Sync sync) {
  if constexpr (LO == HI) {
    return fft_inverse_dif_n<LO, Sync, JP, NT>(buf, twq, s_red, tid, nthr, sync);
  } else {
    if (n == (1 << LO)) return fft_inverse_dif_n<LO, Sync, JP, NT>(buf, twq, s_red, tid, nthr, sync);
    return fft_inverse_dif<LO + 1, HI, Sync, JP, NT>(buf, n, twq, s_red, tid, nthr, sync);
  }
}

// ---- transform lengths that are not a power of two (FFTW accepts any, src/fftw.f90:43-45): Bluestein's chirp-z form ----
// x[t] = sum_f Z[f] exp(+2 pi i f t / n) with f t = (f^2 + t^2 - (t - f)^2) / 2 is a convolution,
//   x[t] = w[t] * sum_f (Z[f] w[f]) conj(w[t - f]),   w[m] = exp(+i pi m^2 / n),
// evaluated as a circular convolution of length M = cfg.fft_len (a power of two >= 2n) by the power-of-two transform above:
// the caller has stored conj(Z[f] w[f]) at logical position f < n and zeros in [n, M); the forward transform is the
// conjugate of the inverse one; cfg.chirp_b = FFT_M(conj(w) wrapped around M) / M comes from the host.  The transforms
// leave element m at bit-reversed position, so the two element-wise passes in between are pair swaps (p, brev p): each
// thread reads both members and writes both, no second buffer.  On return x[t] sits at logical position t (natural
// order) for t < n.  Returns the maximum imaginary part over t < n like fft_inverse_dif.
template <int LOG2M, class Sync>
__device__ __forceinline__ double bluestein_inverse_m(double2* buf, int n, const double2* __restrict__ chirp,
                                                      const double2* __restrict__ chirp_b, const double2* twq, double* s_red,
                                                      int tid, int nthr, Sync sync) {
  constexpr unsigned M = 1u << LOG2M;
  constexpr int PSH = LOG2M >= 9 ? LOG2M - 3 : 31;
  fft_inverse_dif_n<LOG2M, Sync>(buf, twq, s_red, tid, nthr, sync);       // conj(A[m]) at position brev(m)
  for (unsigned p = tid; p < M; p += nthr) {
    const unsigned q = __brev(p) >> (32 - LOG2M);
    if (p > q) continue;
    const double2 u = buf[fpad(p, PSH)], v = buf[fpad(q, PSH)];           // u = conj(A[q]), v = conj(A[p])
    const double2 bq = chirp_b[q], bp = chirp_b[p];
    buf[fpad(q, PSH)] = cmul(make_double2(u.x, -u.y), bq);                // natural order: position m <- A[m] B[m]
    if (p != q) buf[fpad(p, PSH)] = cmul(make_double2(v.x, -v.y), bp);
  }
  sync();
  fft_inverse_dif_n<LOG2M, Sync>(buf, twq, s_red, tid, nthr, sync);       // c[t] (the 1/M is in chirp_b) at position brev(t)
  double vmax = -INFINITY;
  for (unsigned p = tid; p < M; p += nthr) {
    const unsigned q = __brev(p) >> (32 - LOG2M);
    if (p > q) continue;
    const double2 u = buf[fpad(p, PSH)], v = buf[fpad(q, PSH)];           // u = c[q], v = c[p]
    if (q < (unsigned)n) { const double2 x = cmul(u, chirp[q]); buf[fpad(q, PSH)] = x; vmax = fmax(vmax, x.y); }
    if (p != q && p < (unsigned)n) { const double2 x = cmul(v, chirp[p]); buf[fpad(p, PSH)] = x; vmax = fmax(vmax, x.y); }
  }
  publish_max(vmax, s_red + 32, tid);   // (second half of s_red: the first one may still be read by a slower warp)
  sync();
  const int nw = (nthr + 31) >> 5;
  double r = s_red[32];
  for (int i = 1; i < nw; ++i) r = fmax(r, s_red[32 + i]);
  return r;
}
template <int LO, int HI, class Sync>
__device__ __forceinline__ double bluestein_inverse(double2* buf, const DevConfig& cfg, const double2* twq, double* s_red, int tid,
                                                    int nthr, Sync sync) {
  if constexpr (LO == HI) {
    return bluestein_inverse_m<LO, Sync>(buf, cfg.nfft, cfg.chirp, cfg.chirp_b, twq, s_red, tid, nthr, sync);
  } else {
    if (cfg.log2n == LO) return bluestein_inverse_m<LO, Sync>(buf, cfg.nfft, cfg.chirp, cfg.chirp_b, twq, s_red, tid, nthr, sync);
    return bluestein_inverse<LO + 1, HI, Sync>(buf, cfg, twq, s_red, tid, nthr, sync);
  }
}

template <class Sync>
__device__ __forceinline__ double block_max(double v, double* scratch, int tid, int nthr, Sync sync) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  sync();
  if ((tid & 31) == 0) scratch[tid >> 5] = v;
  sync();
  const int nw = (nthr + 31) >> 5;
  double r = scratch[0];
  for (int i = 1; i < nw; ++i) r = fmax(r, scratch[i]);
  return r;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src));
}

// Two-level rotation tables of one item: cos/sin(t*theta) = rot(lo[t & 15], hi[t >> 4]) for t < 16*n_hi.
// Layout [row][column]: rows 0..15 = lo level (multiples 0..15 of theta), rows 16..16+n_hi-1 = hi level (multiples of
// 16 theta); column 2l + which (which = 0: xi, 1: eta) for layer l; row stride 2 k_max + 1 entries.  Consecutive tasks of
// a level write consecutive columns of a row and the 16 rows a warp reads in the layer loop start in different banks
// (odd stride): no bank conflicts on either side (the layer-major layout of the first version cost 24 wavefronts per
// store instead of 3).
// One thread per (layer, angle, level): the seed (cos, sin)(theta) or (cos, sin)(16 theta) comes from prep_kernel, then angle
// doubling e[len+j] = rot(e[j], e[len]) -- log depth, independent rotations inside a level (error ~1e-16 * log2(16)).
__host__ __device__ inline size_t trig_table_entries(size_t km, size_t nthr) { return (16 + (nthr >> 4)) * (2 * km + 1); }
template <int NT>
__device__ __forceinline__ void build_trig_tables(double2* s_tab, const LayerConst* s_lc, int k, int km, int tid) {
  constexpr int n_hi = NT >> 4;
  const int ts = 2 * km + 1;
  for (int task = tid; task < 4 * k; task += NT) {
    const int level = task >= 2 * k ? 1 : 0, idx = task - level * 2 * k;
    const int l = idx >> 1, which = idx & 1;
    double2* dst = s_tab + (level ? 16 * ts : 0) + idx;
    double2 e[16];
    e[0] = make_double2(1.0, 0.0);
    e[1] = reinterpret_cast<const double2*>(&s_lc[l].c1x)[2 * level + which];   // (c1x,s1x) (c1e,s1e) (c16x,s16x) (c16e,s16e)
#pragma unroll
    for (int len = 2; len < 16; len <<= 1) {
      e[len] = e[len >> 1];
      rot(e[len].x, e[len].y, e[len >> 1].x, e[len >> 1].y);
#pragma unroll
      for (int j = 1; j < len; ++j) {
        e[len + j] = e[j];
        rot(e[len + j].x, e[len + j].y, e[len].x, e[len].y);
      }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (i < n_hi || !level) dst[i * ts] = e[i];
  }
}

// Water layer: cos / sin of (tid * thw) -- the phase of the thread's first bin -- from a two-level table like the layers'
// (s_tabw: lo[16] | hi[n_hi], built once per item by two otherwise idle threads from prep_kernel's seeds).
__device__ __forceinline__ void build_water_table(double2* s_tabw, const RayConst* s_rc, int n_hi, int tid, int nthr) {
  const int level = nthr - 1 - tid;          // the last thread builds the lo level, the one before it the hi level
  if (level > 1 || s_rc->thw == 0.0) return;
  const int cnt = level ? n_hi : 16;
  double2 e[16];
  e[0] = make_double2(1.0, 0.0);
  e[1] = make_double2(s_rc->wseed[2 * level], s_rc->wseed[2 * level + 1]);
#pragma unroll
  for (int len = 2; len < 16; len <<= 1) {
    e[len] = e[len >> 1];
    rot(e[len].x, e[len].y, e[len >> 1].x, e[len >> 1].y);
#pragma unroll
    for (int j = 1; j < len; ++j) {
      e[len + j] = e[j];
      rot(e[len + j].x, e[len + j].y, e[len].x, e[len].y);
    }
  }
#pragma unroll
  for (int i = 0; i < 16; ++i)
    if (i < cnt) s_tabw[level * 16 + i] = e[i];
}
__device__ __forceinline__ void water_phase(const double2* s_tabw, double thw, int tid, double& cw, double& sw) {
  cw = 1.0; sw = 0.0;
  if (thw != 0.0) {
    const double2 a = s_tabw[tid & 15], b = s_tabw[16 + (tid >> 4)];
    cw = a.x; sw = a.y;
    rot(cw, sw, b.x, b.y);
  }
}

// Propagator product over the k solid layers, top down, in wave coordinates, for the J bins tid + m*NT of this thread.
// The (cos, sin) pairs of the thread's first bin come from the two-level tables, those of its second bin by the stride
// rotation, from the third on by the three-term recurrence with 2 cos(stride) (one FMA per value instead of two instructions).
template <int J, int NT>
__device__ __forceinline__ void propagate(const RayConst* s_rc, const LayerConst* s_lc, const double2* s_tab, const double2* s_tabw,
                                          int k, int km, int tid, Wave* wa, Wave* wb) {
  {
    const double thw = s_rc->thw, cbw = s_rc->cbw, sbw = s_rc->sbw;
    const double a1 = s_rc->a1, b1 = s_rc->b1, q1a = s_rc->q1a, q1b = s_rc->q1b, q2a = s_rc->q2a, q2b = s_rc->q2b;
    double cw, sw;
    water_phase(s_tabw, thw, tid, cw, sw);
#pragma unroll
    for (int m = 0; m < J; ++m) {
      wa[m].a1 = a1; wa[m].a2 = 0.0; wa[m].b1 = b1; wa[m].b2 = 0.0;
      wb[m].a1 = sw * q1a; wb[m].b1 = sw * q1b; wb[m].a2 = cw * q2a; wb[m].b2 = cw * q2b;
      rot(cw, sw, cbw, sbw);
    }
  }
  const int ts = 2 * km + 1;
  const double2* p_lo = s_tab + (tid & 15) * ts;            // rows of this thread in the two table levels
  const double2* p_hi = s_tab + (16 + (tid >> 4)) * ts;
  double c1, s1, c2, s2;                                    // the pairs of the thread's first bin in the current layer
  {
    const double2 a = p_lo[0], cc = p_lo[1], b = p_hi[0], d = p_hi[1];
    c1 = a.x; s1 = a.y; rot(c1, s1, b.x, b.y);
    c2 = cc.x; s2 = cc.y; rot(c2, s2, d.x, d.y);
  }
  for (int l = 0; l < k; ++l) {
    const LayerConst& L = s_lc[l];
    const int ln = l + 1 < k ? l + 1 : l;
    double2 na, ncc, nb, nd;                             // table entries of the next layer: fetched while the last bin of
                                                         // this one is computed, so no warp waits for them at the layer top
    double pc1 = 0.0, ps1 = 0.0, pc2 = 0.0, ps2 = 0.0;   // the pairs of the previous bin (recurrence)
    auto advance = [&](int m) {
      if (m == 0) {
        pc1 = c1; ps1 = s1; pc2 = c2; ps2 = s2;
        rot(c1, s1, L.cbx, L.sbx);
        rot(c2, s2, L.cbe, L.sbe);
      } else {
        const double cb2x = L.cb2x, cb2e = L.cb2e;
        const double n1 = fma(cb2x, c1, -pc1), m1 = fma(cb2x, s1, -ps1), n2 = fma(cb2e, c2, -pc2), m2 = fma(cb2e, s2, -ps2);
        pc1 = c1; ps1 = s1; pc2 = c2; ps2 = s2;
        c1 = n1; s1 = m1; c2 = n2; s2 = m2;
      }
    };
    if (l + 1 < k) {
      const double t12 = L.t12, t21 = L.t21, u11 = L.u11, u12 = L.u12, u21 = L.u21, u22 = L.u22;
#pragma unroll
      for (int m = 0; m < J; ++m) {
#ifndef RFINV_NO_TABPREFETCH
        if (m == J - 1) { na = p_lo[2 * ln]; ncc = p_lo[2 * ln + 1]; nb = p_hi[2 * ln]; nd = p_hi[2 * ln + 1]; }
#endif
        wave_rotate(wa[m], c1, s1, c2, s2);
        wave_rotate(wb[m], c1, s1, c2, s2);
        wave_interface(wa[m], t12, t21, u11, u12, u21, u22);
        wave_interface(wb[m], t12, t21, u11, u12, u21, u22);
        if (m + 1 < J) advance(m);
      }
#ifdef RFINV_NO_TABPREFETCH
      na = p_lo[2 * ln]; ncc = p_lo[2 * ln + 1]; nb = p_hi[2 * ln]; nd = p_hi[2 * ln + 1];
#endif
      c1 = na.x; s1 = na.y; rot(c1, s1, nb.x, nb.y);
      c2 = ncc.x; s2 = ncc.y; rot(c2, s2, nd.x, nd.y);
    } else {   // last solid layer: the half space follows (rows 3,4 of E^-1 are applied by surface_response)
#pragma unroll
      for (int m = 0; m < J; ++m) {
        wave_rotate(wa[m], c1, s1, c2, s2);
        wave_rotate(wb[m], c1, s1, c2, s2);
        if (m + 1 < J) advance(m);
      }
    }
  }
}

// Runs the layer loop for the first jm (<= JB) bin groups of the thread; jm takes the values band_limits() hands out.
template <int JB, int NT, bool MIXED>
__device__ __forceinline__ void propagate_groups(int jm, const RayConst* s_rc, const LayerConst* s_lc, const double2* s_tab,
                                                 const double2* s_tabw, int k, int km, int tid, Wave* wa, Wave* wb) {
  if (!MIXED || jm >= JB) { propagate<JB, NT>(s_rc, s_lc, s_tab, s_tabw, k, km, tid, wa, wb); return; }
  if constexpr (MIXED) {
  if constexpr (JB > 6) if (jm == 6) { propagate<6, NT>(s_rc, s_lc, s_tab, s_tabw, k, km, tid, wa, wb); return; }
  if constexpr (JB > 4) if (jm == 4) { propagate<4, NT>(s_rc, s_lc, s_tab, s_tabw, k, km, tid, wa, wb); return; }
  if constexpr (JB > 3) if (jm == 3) { propagate<3, NT>(s_rc, s_lc, s_tab, s_tabw, k, km, tid, wa, wb); return; }
  if constexpr (JB > 2) if (jm == 2) { propagate<2, NT>(s_rc, s_lc, s_tab, s_tabw, k, km, tid, wa, wb); return; }
  if constexpr (JB > 1) propagate<1, NT>(s_rc, s_lc, s_tab, s_tabw, k, km, tid, wa, wb);
  }
}

// Surface response of the thread's first J bin groups (the groups above them are zero filled).  STAGE = false: straight into the packed, filtered spectrum
// Z = X_r + i X_v with Hermitian extension (src/forward.f90:168, 199) in the padded FFT buffer; STAGE = true: the
// unfiltered spectra go to s_fr / s_fv (common rays, water-level deconvolution).  Thread 0 adds the two edge bins.
// GEN (nfft not a power of two, Bluestein): bins from jtop on do not exist (the thread grid is laid out for the next power of
// two); position f of the buffer takes conj(Z[f] w[f]) with the chirp w, w[n - f] = (-1)^n w[f]; zeros in [n, fft_len).
template <int J, bool STAGE, bool GEN>
__device__ __forceinline__ void surface_and_pack(const RayConst* s_rc, const Wave* wa, const Wave* wb, int jfull, int ipha,
                                                 int n, int nh, int tid, int nthr, const double* __restrict__ flt, double2* s_buf,
                                                 double2* s_fr, double2* s_fv, bool buried, const double2* s_tabw, int psh,
                                                 const double2* __restrict__ chirp = nullptr, int fft_len = 0) {
  const bool odd = GEN && (n & 1);
  const int jtop = odd ? nh : nh - 1;     // regular bins: [1, jtop); an even length has its Nyquist bin at nh - 1 (prep_kernel)
  const double wsgn = odd ? -1.0 : 1.0;
  double h14[4], h23[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { h14[i] = s_rc->h14[i]; h23[i] = s_rc->h23[i]; }
  const double thw = s_rc->thw, cbw = s_rc->cbw, sbw = s_rc->sbw;
  double cw, sw;
  water_phase(s_tabw, thw, tid, cw, sw);
#pragma unroll
  for (int m = 0; m < J; ++m) {
    const int j = tid + m * nthr;
    double2 fr, fv;
    const bool live = !GEN || j < jtop;
    if (STAGE && buried) { if (live) surface_response_buried(h14, h23, wa[m], wb[m], ipha, s_fr[j], s_fv[j], fr, fv); }   // station pass left them there
    else surface_response(h14, h23, wa[m], wb[m], cw, ipha, fr, fv, STAGE ? 1.0 : (live ? flt[j] : 0.0));   // filtered on the way out
    rot(cw, sw, cbw, sbw);
    if (STAGE) {
      if (j > 0 && live) { s_fr[j] = fr; s_fv[j] = fv; }
    } else if (GEN) {
      if (j > 0 && live) {
        const double2 xv = fv;
        const double2 xr = ipha == 1 ? fr : xv;
        const double2 w = chirp[j];
        const double2 a = cmul(make_double2(xr.x - xv.y, xr.y + xv.x), w);
        const double2 b = cmul(make_double2(xr.x + xv.y, xv.x - xr.y), w);
        s_buf[fpad(j, psh)] = make_double2(a.x, -a.y);
        s_buf[fpad(n - j, psh)] = make_double2(wsgn * b.x, -wsgn * b.y);
      }
    } else if (j > 0) {
      const double2 xv = fv;
      const double2 xr = ipha == 1 ? fr : xv;
      s_buf[fpad(j, psh)] = make_double2(xr.x - xv.y, xr.y + xv.x);
      s_buf[fpad(n - j, psh)] = make_double2(xr.x + xv.y, xv.x - xr.y);
    }
  }
  for (int m = J; m < jfull; ++m) {    // bins above the band limit of this trace (band_limits(), capi.cu)
    const int j = tid + m * nthr;
    if (GEN && j >= jtop) continue;
    if (STAGE) { s_fr[j] = make_double2(0.0, 0.0); s_fv[j] = make_double2(0.0, 0.0); }
    else { s_buf[fpad(j, psh)] = make_double2(0.0, 0.0); s_buf[fpad(n - j, psh)] = make_double2(0.0, 0.0); }
  }
  if (GEN && !STAGE) for (int f = n + tid; f < fft_len; f += nthr) s_buf[fpad(f, psh)] = make_double2(0.0, 0.0);
  if (!GEN && !STAGE && tid == 0 && 2 * jfull * nthr < n) {
    // pruned first FFT stage (jfull = the kernel variant's bin groups): the butterfly with offset 0 still reads its leg
    // n - jfull*nthr, the mirror of the first bin above the band limit
    s_buf[fpad(jfull * nthr, psh)] = make_double2(0.0, 0.0);
    s_buf[fpad(n - jfull * nthr, psh)] = make_double2(0.0, 0.0);
  }
  if (tid == 0) {  // the two bins off the regular grid
    if (STAGE) {
      s_fr[0] = s_rc->edge[0]; s_fv[0] = s_rc->edge[1];
      if (!odd) { s_fr[nh - 1] = s_rc->edge[2]; s_fv[nh - 1] = s_rc->edge[3]; }
    } else {       // c2r ignores the imaginary parts of DC and Nyquist
      const double f0 = flt[0], f1 = flt[nh - 1];
      const double2 r0 = ipha == 1 ? s_rc->edge[0] : s_rc->edge[1], r1 = ipha == 1 ? s_rc->edge[2] : s_rc->edge[3];
      if (GEN) {
        s_buf[fpad(0, psh)] = make_double2(r0.x * f0, -s_rc->edge[1].x * f0);     // w[0] = 1
        if (!odd) {
          const double2 a = cmul(make_double2(r1.x * f1, s_rc->edge[3].x * f1), chirp[nh - 1]);
          s_buf[fpad(nh - 1, psh)] = make_double2(a.x, -a.y);
        }
      } else {
        s_buf[fpad(0, psh)] = make_double2(r0.x * f0, s_rc->edge[1].x * f0);
        s_buf[fpad(nh - 1, psh)] = make_double2(r1.x * f1, s_rc->edge[3].x * f1);
      }
    }
  }
}

// Shift / sign / normalise the transformed trace (src/forward.f90:176-203) and write misfit, cached samples and
// (optionally) the complete RF.  Element f of the transform sits at bit-reversed position (n is a power of two).
// Misfit row layout: m_i = rft(i) - obs(i) in [0, nsmp), or with DevConfig::qf_split the sums s_i = m_i + m_{S-1-i} in
// [0, Sp/2) (the centre sample of an odd window at i = S/2) and the differences a_i = m_i - m_{S-1-i} in [Sp/2, Sp):
// what the split quadratic form contracts (capi.cu).  The padding of the row is written (zeros) on every call: the
// rows move when the batch size changes and a stale NaN would survive the multiplication by a zero of R^-1 / W.
constexpr int OBS_PRE = 4;   // observed samples per thread fetched before the FFT
// index of the q-th observed sample thread `tid` needs (write_outputs below): the left (q even) or right (q odd) member
// of its pair p = tid + (q>>1)*nthr of samples (p, S-1-p)
__device__ __forceinline__ int obs_pre_index(int S, int q, int tid, int nthr) {
  const int pr = tid + (q >> 1) * nthr;
  return pr < (S >> 1) ? ((q & 1) ? S - 1 - pr : pr) : S;   // S = nothing to fetch
}
template <bool GEN>
__device__ __forceinline__ void write_outputs(const DevConfig& cfg, const EvalOutputs& out, const double2* s_buf, int C, int c,
                                              int t, int ipha, int npre, double scale, const double* obs_pre, int tid, int nthr) {
  const int n = cfg.nfft, S = cfg.nsmp, Sp = cfg.nsmp_pad, nmask = n - 1, brev_shift = 32 - cfg.log2n, psh = fft_pad_shift(cfg.log2n);
  double* __restrict__ mis = out.misfit + ((size_t)t * C + c) * Sp;
  double* smp_base = out.rft_smp;
  if (out.slot && ((out.slot[c] ^ out.slot_invert) & 1)) smp_base = out.rft_smp_alt;
  double* __restrict__ smp = smp_base ? smp_base + ((size_t)t * C + c) * S : nullptr;
  const double* __restrict__ obs = cfg.obs + (size_t)t * S;
  auto sample = [&](int i) {
    if constexpr (GEN) {   // Bluestein leaves the trace in natural order; the circular shift is a true modulo
      int f = (ipha == 1 ? i - npre : npre - i - 1) % n;
      if (f < 0) f += n;
      const double v = s_buf[fpad(f, psh)].x * scale;
      return ipha == 1 ? v : -v;
    }
    const int f = ipha == 1 ? ((i - npre) & nmask)            // src/forward.f90:178-184
                            : ((npre - i - 1) & nmask);       // src/forward.f90:187-193
    const double v = s_buf[fpad((int)(__brev((unsigned)f) >> brev_shift), psh)].x * scale;
    return ipha == 1 ? v : -v;
  };
  // every thread handles pairs (p, S-1-p) of samples: both layouts come out of the same loop
  const bool split = cfg.qf_split[t] != 0;
  const int ha = S >> 1, half = Sp >> 1;
  auto emit = [&](int pr, double o1, double o2) {
    const double v1 = sample(pr), v2 = sample(S - 1 - pr);
    const double d1 = v1 - o1, d2 = v2 - o2;
    mis[pr] = split ? d1 + d2 : d1;
    mis[split ? half + pr : S - 1 - pr] = split ? d1 - d2 : d2;
    if (smp) { smp[pr] = v1; smp[S - 1 - pr] = v2; }
  };
#pragma unroll
  for (int q = 0; q < OBS_PRE / 2; ++q) {
    const int pr = tid + q * nthr;
    if (pr < ha) emit(pr, obs_pre[2 * q], obs_pre[2 * q + 1]);
  }
  for (int pr = tid + (OBS_PRE / 2) * nthr; pr < ha; pr += nthr) emit(pr, __ldg(obs + pr), __ldg(obs + S - 1 - pr));
  if ((S & 1) && tid == 0) {                  // centre sample of an odd window: a coordinate of its own in both layouts
    const double v = sample(ha);
    mis[ha] = v - __ldg(obs + ha);
    if (smp) smp[ha] = v;
  }
  if (split) {
    for (int i = S - ha + tid; i < half; i += nthr) mis[i] = 0.0;
    for (int i = half + ha + tid; i < Sp; i += nthr) mis[i] = 0.0;
  } else {
    for (int i = S + tid; i < Sp; i += nthr) mis[i] = 0.0;
  }
  if (out.rft_full) {
    double* __restrict__ full = out.rft_full + ((size_t)c * cfg.ntrc + t) * n;
    for (int i = tid; i < n; i += nthr) full[i] = sample(i);
  }
}

template <int JB, bool STAGE, bool MIXED, bool GEN>
__device__ __forceinline__ void surface_groups(int jm, const RayConst* s_rc, const Wave* wa, const Wave* wb, int jfull, int ipha, int n,
                                               int nh, int tid, int nthr, const double* __restrict__ flt, double2* s_buf,
                                               double2* s_fr, double2* s_fv, bool buried, const double2* s_tabw, int psh,
                                               const double2* __restrict__ chirp, int fft_len) {
#define SURF(JM) surface_and_pack<JM, STAGE, GEN>(s_rc, wa, wb, jfull, ipha, n, nh, tid, nthr, flt, s_buf, s_fr, s_fv, buried, s_tabw, psh, chirp, fft_len)
  if (!MIXED || jm >= JB) { SURF(JB); return; }
  if constexpr (MIXED) {
  if constexpr (JB > 6) if (jm == 6) { SURF(6); return; }
  if constexpr (JB > 4) if (jm == 4) { SURF(4); return; }
  if constexpr (JB > 3) if (jm == 3) { SURF(3); return; }
  if constexpr (JB > 2) if (jm == 2) { SURF(2); return; }
  if constexpr (JB > 1) SURF(1);
  }
#undef SURF
}

// ------------------------------------------------------------------------------------------------
// forward_kernel: persistent CTAs, one (model, ray) item at a time, items handed out by an atomic counter
// (the work per item is proportional to its layer count).  The constants of the next item are fetched with
// cp.async while the current one is computed.  Thread `tid` owns frequency bins j = tid + m*B, m < nfft/2/B
// (B = blockDim.x), of which only the first cfg.jbins[trace] <= J groups carry signal through the Gaussian filter
// (band_limits(), capi.cu) and are propagated.  Bins 0 (DC) and nfft/2 (Nyquist) come from prep_kernel.
// Shared memory: one region that first holds the trigonometric tables of the layer loop and then the padded
// in-place FFT buffer; the unfiltered spectra only when they must outlive one FFT (common rays) or feed the
// water-level deconvolution; two sets of layer / ray constants; quarter-wave twiddles.
// ------------------------------------------------------------------------------------------------
template <int J, int BMAX, int MINB, bool MIXED, bool BURIED, bool GEN = false>
__global__ void __launch_bounds__(BMAX, MINB) forward_kernel(const DevConfig cfg, const ModelBatch mb, const EvalOutputs out,
                                                             const double* __restrict__ lc_in,
                                                             const double* __restrict__ rc_in, int* __restrict__ counter,
                                                             const TraceSel sel) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_next;
  const int tid = threadIdx.x;
  constexpr int nthr = BMAX;       // threads per CTA (launch_forward_t launches exactly BMAX): addressing and loop bounds fold
  const int n = cfg.nfft, nh = cfg.nh, km = cfg.k_max, C = mb.C, psh = fft_pad_shift(cfg.log2n);
  const int ntr_eff = cfg.ray_common ? 1 : cfg.ntrc;   // rays per model in the scratch arrays prep_kernel filled
  // items of this launch: (model, ray) for the rays in `sel` (all of them, or the traces of one band-limit group)
  constexpr bool buried = BURIED;   // cfg.bdep > 0: a kernel variant of its own, the surface-station variants carry none of it
  const bool general = cfg.ray_common || cfg.deconv_mode == 1 || buried;   // spectra staged in shared memory

  constexpr int n_hi = nthr >> 4;                     // table split: tid = 16*hi + lo
  const int nf = GEN ? cfg.fft_len : n;             // points of the shared-memory transform
  const size_t tab_entries = trig_table_entries(km, nthr);
  const size_t region0 = tab_entries > fft_buf_elems(nf) ? tab_entries : fft_buf_elems(nf);
  double2* s_buf = reinterpret_cast<double2*>(smem_raw);
  double2* s_tab = s_buf;                             // dead before the FFT buffer is first written
  double2* s_fr = s_buf + region0;                    // [nh+1] unfiltered radial spectrum (or deconvolved RF spectrum)
  double2* s_fv = s_fr + (nh + 1);                    // [nh+1] unfiltered vertical spectrum
  double2* s_twq_sm = s_fr + (general ? 2 * (nh + 1) : 0);   // per-stage FFT twiddle tables (GEN: read from global memory instead --
  const double2* s_twq = GEN ? cfg.twq : s_twq_sm;           //  the two transforms of twice the length need the room for their buffer)
  double* s_red = reinterpret_cast<double*>(s_twq_sm + (GEN ? 0 : fft_twiddle_entries(nf)));   // [64]
  RayConst* s_rc2 = reinterpret_cast<RayConst*>(s_red + 64);     // [2]
  LayerConst* s_lc2 = reinterpret_cast<LayerConst*>(s_rc2 + 2);  // [2][km]
  double2* s_tabw = reinterpret_cast<double2*>(s_lc2 + 2 * (size_t)km);   // [16 + n_hi] water-layer phase table (not aliased)

  // item / sel.n without an integer division per item: multiply-high by ceil(2^32 / n), exact for item < 2^32 / n
  const unsigned sel_magic = sel.n > 1 ? (unsigned)((0x100000000ULL + (unsigned)sel.n - 1u) / (unsigned)sel.n) : 0u;
  auto div_sel = [&](int x) { return sel.n > 1 ? (int)__umulhi((unsigned)x, sel_magic) : x; };
  auto prefetch = [&](int item_sel, int slot) {
    const int ci_ = div_sel(item_sel);
    const size_t item = (size_t)ci_ * ntr_eff + sel.t(item_sel - ci_ * sel.n);   // index into prep_kernel's arrays
    const double2* src = reinterpret_cast<const double2*>(rc_in + (size_t)item * RC_DOUBLES);
    double2* dst = reinterpret_cast<double2*>(s_rc2 + slot);
    for (int i = tid; i < RC_DOUBLES / 2; i += nthr) cp_async16(dst + i, src + i);
    const double2* src2 = reinterpret_cast<const double2*>(lc_in + (size_t)item * km * LC_DOUBLES);
    double2* dst2 = reinterpret_cast<double2*>(s_lc2 + (size_t)slot * km);
    for (int i = tid; i < km * (LC_DOUBLES / 2); i += nthr) cp_async16(dst2 + i, src2 + i);   // all k_max layers: k is not known yet
  };

  // Three items in flight per CTA: `item` is computed, the constants of `next` are being fetched, and the index
  // after that is on its way back from the atomic counter (thread 0 holds it in a register until the end of the
  // iteration, so nobody waits for the round trip).
  int item = blockIdx.x, slot = 0;
  pdl_trigger();                               // quadform_kernel may queue up behind this grid
  if (!GEN) fill_fft_twiddles(s_twq_sm, cfg.tw, nf, tid, nthr);   // (nothing of prep_kernel is touched before pdl_wait)
  pdl_wait();                                  // prep_kernel (and everything before it on the stream) is complete
  const int n_items = (mb.n_active_dev ? *mb.n_active_dev : (mb.active ? mb.n_active : C)) * sel.n;
  if (item >= n_items) return;
  prefetch(item, 0);
  asm volatile("cp.async.commit_group;\n" ::);
  if (tid == 0) s_next = (int)gridDim.x + atomicAdd(counter, 1);
  asm volatile("cp.async.wait_all;\n" ::);
  __syncthreads();   // constants of the first item and the twiddles have landed; s_next is visible

  while (item < n_items) {
    PHASE_INIT();
    // the constants of `item` and s_next were published by the barrier that closed the previous iteration
    const int next = s_next;
    if (next < n_items) prefetch(next, slot ^ 1);
    asm volatile("cp.async.commit_group;\n" ::);
    int next2 = 0;
    if (tid == 0) next2 = atomicAdd(counter, 1);   // consumed at the end of the iteration: nobody waits for the round trip
    const RayConst* s_rc = s_rc2 + slot;
    const LayerConst* s_lc = s_lc2 + (size_t)slot * km;
    const int ci = div_sel(item), t0 = sel.t(item - ci * sel.n);
    const int c = mb.active ? mb.active[ci] : ci;
    const int k = s_rc->k;
    const int ipha = cfg.ipha[t0];
    PHASE_MARK(0);
    build_trig_tables<nthr>(s_tab, s_lc, buried ? max(k, s_rc->l_sta + 1) : k, km, tid);
    build_water_table(s_tabw, s_rc, n_hi, tid, nthr);
    __syncthreads();
    PHASE_MARK(1);

    const int jm = MIXED ? cfg.jbins[t0] : J;   // bin groups with signal for this trace (<= J; MIXED: it varies by trace)
    Wave wa[J], wb[J];
    // Buried station: a first pass down to the station leaves the displacement components of both vectors there in the
    // spectrum staging arrays (same thread, same bins as the surface response that combines them); then the full stack.
    for (int pass = buried ? 0 : 1; pass < 2; ++pass) {
      propagate_groups<J, nthr, MIXED>(jm, s_rc, s_lc, s_tab, s_tabw, pass == 0 ? s_rc->l_sta + 1 : k, km, tid, wa, wb);
      if (pass == 0) {
        const double c0 = s_rc->sta[0], c1 = s_rc->sta[1], c2 = s_rc->sta[2], c3 = s_rc->sta[3];
#pragma unroll
        for (int m = 0; m < J; ++m) {
          const int j = tid + m * nthr;
          if (m < jm && (!GEN || j < nh)) {
            s_fr[j] = make_double2(fma(c0, wa[m].a1, c1 * wa[m].b1), fma(c2, wa[m].a2, c3 * wa[m].b2));
            s_fv[j] = make_double2(fma(c0, wb[m].a1, c1 * wb[m].b1), fma(c2, wb[m].a2, c3 * wb[m].b2));
          }
        }
      }
    }
    PHASE_MARK(2);
    __syncthreads();   // the trigonometric tables are dead: their region becomes the FFT buffer

    // ---- surface response per bin; straight into the packed, filtered spectrum when no staging is needed ----
    const int jfull = (cfg.nfft_p2 >> 1) / nthr;
#ifdef RFINV_NO_FFT_PRUNE
    constexpr bool kPruned = false;
#else
    constexpr bool kPruned = !GEN;   // the first FFT stage skips the bin groups from J on: nobody has to zero them
#endif
    if (general) surface_groups<J, true, MIXED, GEN>(jm, s_rc, wa, wb, jfull, ipha, n, nh, tid, nthr, nullptr, s_buf, s_fr, s_fv, buried, s_tabw, psh, cfg.chirp, nf);
    else surface_groups<J, false, MIXED, GEN>(jm, s_rc, wa, wb, kPruned ? J : jfull, ipha, n, nh, tid, nthr, cfg.flt + (size_t)t0 * nh, s_buf, s_fr, s_fv, false, s_tabw, psh, cfg.chirp, nf);
    if constexpr (kPruned && (J & 1) && nthr == 256) {
      // The pruned first FFT stage skips only the legs of n/8 bins that lie wholly above the band limit.  J NT is a leg
      // boundary at every shape but one: an odd J of 256 threads at nfft 4096 (legs of 512 bins) ends inside leg 1, whose
      // bins from J NT + 1 to the leg boundary and their mirrors nobody else writes (bin J NT itself: surface_and_pack).
      const int top = (J * nthr + (n >> 3) - 1) & ~((n >> 3) - 1);
      if (!general)
        for (int j = J * nthr + 1 + tid; j <= top; j += nthr) {
          s_buf[fpad(j, psh)] = make_double2(0.0, 0.0);
          s_buf[fpad(n - j, psh)] = make_double2(0.0, 0.0);
        }
    }
    __syncthreads();
    PHASE_MARK(3);

    // ---- water-level deconvolution (src/forward.f90:148-153, 447-470): overwrites s_fr with rff ----
    if (cfg.deconv_mode == 1) {
      const double2* xs = ipha == 1 ? s_fv : s_fr;  // denominator spectrum
      const double2* ys = ipha == 1 ? s_fr : s_fv;
      double mx = -INFINITY;
      for (int j = tid; j < nh; j += nthr) mx = fmax(mx, xs[j].x * xs[j].x + xs[j].y * xs[j].y);
      mx = block_max(mx, s_red, tid, nthr, CtaSync());
      const double wlvl = 0.001 * mx;
      double2 keep[J + 1];
#pragma unroll
      for (int q = 0; q < J + 1; ++q) {
        const int j = tid + q * nthr;
        if (j < nh) {
          const double2 x = xs[j], y = ys[j];
          const double amp = x.x * x.x + x.y * x.y;
          const double d = fmax(amp, wlvl);
          keep[q] = make_double2((y.x * x.x + y.y * x.y) / d, (y.y * x.x - y.x * x.y) / d);
        }
      }
      __syncthreads();
#pragma unroll
      for (int q = 0; q < J + 1; ++q) {
        const int j = tid + q * nthr;
        if (j < nh) s_fr[j] = keep[q];
      }
      __syncthreads();
    }

    // ---- per trace: filter -> inverse FFT -> shift / normalise -> outputs ----
    const int t_begin = cfg.ray_common ? 0 : t0, t_end = cfg.ray_common ? cfg.ntrc : t0 + 1;
    for (int t = t_begin; t < t_end; ++t) {
      if (general) {
        const double* __restrict__ flt = cfg.flt + (size_t)t * nh;
        const double2* src_r = (cfg.deconv_mode == 1 || ipha == 1) ? s_fr : s_fv;  // rff
        for (int j = tid; j < nh; j += nthr) {
          const double f = flt[j];
          const double2 xr = make_double2(src_r[j].x * f, src_r[j].y * f);
          double2 xv = make_double2(0.0, 0.0);
          if (cfg.deconv_mode == 0) xv = make_double2(s_fv[j].x * f, s_fv[j].y * f);
          const bool edge_bin = j == 0 || (j == nh - 1 && !(GEN && (n & 1)));   // DC, Nyquist of an even length: real
          if constexpr (GEN) {   // Bluestein: conj(Z[f] w[f]), w[n - f] = (-1)^n w[f]
            const double2 w = cfg.chirp[j];
            if (edge_bin) {
              const double2 a = cmul(make_double2(xr.x, xv.x), w);
              s_buf[fpad(j, psh)] = make_double2(a.x, -a.y);
            } else {
              const double sg = (n & 1) ? -1.0 : 1.0;
              const double2 a = cmul(make_double2(xr.x - xv.y, xr.y + xv.x), w), b = cmul(make_double2(xr.x + xv.y, xv.x - xr.y), w);
              s_buf[fpad(j, psh)] = make_double2(a.x, -a.y);
              s_buf[fpad(n - j, psh)] = make_double2(sg * b.x, -sg * b.y);
            }
          } else if (edge_bin) {
            s_buf[fpad(j, psh)] = make_double2(xr.x, xv.x);
          } else {
            s_buf[fpad(j, psh)] = make_double2(xr.x - xv.y, xr.y + xv.x);
            s_buf[fpad(n - j, psh)] = make_double2(xr.x + xv.y, xv.x - xr.y);
          }
        }
        if constexpr (GEN) for (int f = n + tid; f < nf; f += nthr) s_buf[fpad(f, psh)] = make_double2(0.0, 0.0);
        __syncthreads();
      }
      PHASE_MARK(4);
      double obs_pre[OBS_PRE];
      const double* __restrict__ obs_t = cfg.obs + (size_t)t * cfg.nsmp;
#pragma unroll
      for (int q = 0; q < OBS_PRE; ++q) {   // observed samples of this thread's outputs: in flight during the FFT
        const int i = obs_pre_index(cfg.nsmp, q, tid, nthr);
        obs_pre[q] = i < cfg.nsmp ? __ldg(obs_t + i) : 0.0;
      }
      // threads per CTA fix the transform length: 32 -> 64/128, 64 -> 256/512, 128 -> 1024, 256 -> 2048/4096
      constexpr int FLO = BMAX <= 32 ? 6 : (BMAX <= 64 ? 8 : (BMAX <= 128 ? 10 : 11));
      constexpr int FHI = BMAX <= 32 ? 7 : (BMAX <= 64 ? 9 : (BMAX <= 128 ? 10 : 12));
      double mx;
      if constexpr (GEN) mx = bluestein_inverse<FLO + 1, (FHI + 1 > 12 ? 12 : FHI + 1), CtaSync>(s_buf, cfg, s_twq, s_red, tid, nthr, CtaSync());
      else mx = fft_inverse_dif<FLO, FHI, CtaSync, J, nthr>(s_buf, n, s_twq, s_red, tid, nthr, CtaSync());
      PHASE_MARK(5);
      const double scale = cfg.deconv_mode == 0 ? 1.0 / mx : 1.0;   // src/forward.f90:197-203
      write_outputs<GEN>(cfg, out, s_buf, C, c, t, ipha, s_rc->npre, scale, obs_pre, tid, nthr);
      if (tid == 0 && t + 1 == t_end) s_next = (int)gridDim.x + next2;
      asm volatile("cp.async.wait_all;\n" ::);   // the next item's constants, in flight since the top of this iteration
      __syncthreads();   // the buffer is rewritten by the next trace / the next item's tables; constants and s_next published
      PHASE_MARK(6);
    }
    item = next;
    slot ^= 1;
  }
}

// ------------------------------------------------------------------------------------------------
// filter_traces_kernel: y = c2r( r2c(x) * flt(:, trace) ), both transforms unnormalised like FFTW's -- the noise
// shaping of make_syn (src/make_syn.f90:96-100; plans src/fftw.f90:44-45).  One CTA per series.  For real x the
// forward transform is the conjugate of the inverse one, so both directions run through fft_inverse_dif.
// ------------------------------------------------------------------------------------------------
template <bool GEN>
__global__ void __launch_bounds__(128) filter_traces_kernel(const DevConfig cfg, const double* __restrict__ in,
                                                           const int* __restrict__ trace_of, double* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, nthr = blockDim.x, n = cfg.nfft, nh = cfg.nh, brev_shift = 32 - cfg.log2n, psh = fft_pad_shift(cfg.log2n);
  const int nf = cfg.fft_len;
  double2* b0 = reinterpret_cast<double2*>(smem_raw);
  double2* b1 = b0 + fft_buf_elems(nf);
  double2* s_tw_sm = b1 + fft_buf_elems(nf);
  const double2* s_tw = GEN ? cfg.twq : s_tw_sm;      // GEN: twiddle tables from global memory
  double* s_red = reinterpret_cast<double*>(s_tw_sm + (GEN ? 0 : fft_twiddle_entries(nf)));   // [64]
  const double* x = in + (size_t)blockIdx.x * n;
  const double* __restrict__ flt = cfg.flt + (size_t)trace_of[blockIdx.x] * nh;
  if (!GEN) fill_fft_twiddles(s_tw_sm, cfg.tw, nf, tid, nthr);
  if constexpr (GEN) {
    // any length (Bluestein): both transforms leave their result in natural order
    const bool odd = n & 1;
    for (int i = tid; i < nf; i += nthr) {
      double2 v = make_double2(0.0, 0.0);
      if (i < n) { const double2 w = cfg.chirp[i]; const double xi = x[i]; v = make_double2(xi * w.x, -xi * w.y); }   // conj(x w)
      b0[fpad(i, psh)] = v;
      if (i >= n) b1[fpad(i, psh)] = v;
    }
    __syncthreads();
    bluestein_inverse<7, 12>(b0, cfg, s_tw, s_red, tid, nthr, CtaSync());
    for (int f = tid; f < nh; f += nthr) {
      const double2 v = b0[fpad(f, psh)];
      const double g = flt[f];
      const double2 w = cfg.chirp[f];
      const bool edge_bin = f == 0 || (f == nh - 1 && !odd);
      double2 y = make_double2(v.x * g, -v.y * g);                // r2c bin f (conjugate), filtered
      if (edge_bin) y.y = 0.0;                                    // c2r ignores these imaginary parts
      const double2 a = cmul(y, w);
      b1[fpad(f, psh)] = make_double2(a.x, -a.y);
      if (!edge_bin) {
        const double sg = odd ? -1.0 : 1.0;
        const double2 b = cmul(make_double2(y.x, -y.y), w);
        b1[fpad(n - f, psh)] = make_double2(sg * b.x, -sg * b.y);
      }
    }
    __syncthreads();
    bluestein_inverse<7, 12>(b1, cfg, s_tw, s_red, tid, nthr, CtaSync());
    for (int i = tid; i < n; i += nthr) out[(size_t)blockIdx.x * n + i] = b1[fpad(i, psh)].x;
  } else {
  for (int i = tid; i < n; i += nthr) b0[fpad(i, psh)] = make_double2(x[i], 0.0);
  __syncthreads();
  fft_inverse_dif<6, 12>(b0, n, s_tw, s_red, tid, nthr, CtaSync());
  for (int f = tid; f < nh; f += nthr) {
    const double2 v = b0[fpad((int)(__brev((unsigned)f) >> brev_shift), psh)];
    const double w = flt[f];
    const double2 y = make_double2(v.x * w, -v.y * w);          // r2c bin f (conjugate), filtered
    if (f == 0 || f == nh - 1) {
      b1[fpad(f, psh)] = make_double2(y.x, 0.0);                     // c2r ignores these imaginary parts
    } else {
      b1[fpad(f, psh)] = y;
      b1[fpad(n - f, psh)] = make_double2(y.x, -y.y);
    }
  }
  __syncthreads();
  fft_inverse_dif<6, 12>(b1, n, s_tw, s_red, tid, nthr, CtaSync());
  for (int i = tid; i < n; i += nthr) out[(size_t)blockIdx.x * n + i] = b1[fpad((int)(__brev((unsigned)i) >> brev_shift), psh)].x;
  }
}

__global__ void format_model_kernel(const DevConfig cfg, const ModelBatch mb, int* nlay_out, double* alpha,
                                    double* beta, double* rho, double* h, uint8_t* is_valid) {
  // One thread per model; used by rfinv_format_model_batch (host diagnostics / parity tests).
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= mb.C) return;
  const int km = cfg.k_max, C = mb.C, k = mb.k[c], stride = km + 1;
  double z[RFINV_MAX_K], dp[RFINV_MAX_K], ds[RFINV_MAX_K];
  for (int i = 0; i < k; ++i) {
    z[i] = mb.z[(size_t)i * C + c]; dp[i] = mb.dvp[(size_t)i * C + c]; ds[i] = mb.dvs[(size_t)i * C + c];
  }
  for (int i = 1; i < k; ++i) {
    const double a = z[i], b = dp[i], d = ds[i];
    int m = i - 1;
    while (m >= 0 && z[m] > a) { z[m + 1] = z[m]; dp[m + 1] = dp[m]; ds[m + 1] = ds[m]; --m; }
    z[m + 1] = a; dp[m + 1] = b; ds[m + 1] = d;
  }
  int i = 0;
  bool valid = true;
  double* A = alpha + (size_t)c * stride; double* Bt = beta + (size_t)c * stride;
  double* R = rho + (size_t)c * stride; double* H = h + (size_t)c * stride;
  if (cfg.sdep > 0.0) { A[i] = 1.5; Bt[i] = -999.0; R[i] = 1.0; H[i] = cfg.sdep; ++i; }
  for (int l = 0; l <= k; ++l) {
    double zc, hh, dvs_l, dvp_l;
    if (l == 0) { zc = __dmul_rn(0.5, __dadd_rn(cfg.sdep, z[0])); hh = __dsub_rn(z[0], cfg.sdep); dvs_l = ds[0]; dvp_l = dp[0]; }
    else if (l < k) { zc = __dmul_rn(0.5, __dadd_rn(z[l], z[l - 1])); hh = __dsub_rn(z[l], z[l - 1]); dvs_l = ds[l]; dvp_l = dp[l]; }
    else { zc = __dmul_rn(0.5, __dadd_rn(cfg.z_max, z[k - 1])); hh = 999.0;
           dvs_l = mb.dvs[(size_t)(km - 1) * C + c]; dvp_l = mb.dvp[(size_t)(km - 1) * C + c]; }
    double a, b;
    bool ok = layer_velocity(cfg, zc, dvs_l, dvp_l, a, b);
    if (l == 0) ok = ok && !(hh < __dmul_rn(0.125, a));
    else if (l < k) ok = ok && !(hh < cfg.h_min);
    valid = valid && ok;
    if (i < stride) { A[i] = a; Bt[i] = b; R[i] = vp_to_rho(a); H[i] = hh; }
    ++i;
  }
  nlay_out[c] = i;
  is_valid[c] = (uint8_t)valid;
}

size_t forward_smem_bytes(const DevConfig& cfg, int nthr) {
  const size_t n = cfg.fft_len, nh = cfg.nh, km = cfg.k_max;
  const size_t tab_entries = trig_table_entries(km, nthr);
  const size_t region0 = tab_entries > fft_buf_elems(n) ? tab_entries : fft_buf_elems(n);
  const bool general = cfg.ray_common || cfg.deconv_mode == 1 || cfg.bdep > 0.0;
  const size_t spectra = general ? 2 * (nh + 1) : 0;
  return sizeof(double2) * (region0 + spectra + (cfg.fft_general ? 0 : fft_twiddle_entries(n))) + sizeof(double) * 64 + 2 * sizeof(RayConst) +
         2 * sizeof(LayerConst) * km + sizeof(double2) * (16 + (nthr >> 4));
}

template <int J, int BMAX, int MINB, bool MIXED, bool BURIED, bool GEN = false>
int launch_forward_t(const DevConfig& cfg, const ModelBatch& mb, const EvalOutputs& out, const double* lc,
                     const double* rc, int* counter, int nthr, cudaStream_t stream, const TraceSel& sel) {
  static const size_t extra = getenv("RFINV_FWD_EXTRA_SMEM") ? (size_t)atoi(getenv("RFINV_FWD_EXTRA_SMEM")) : 0;  // occupancy experiments
  const size_t smem = forward_smem_bytes(cfg, nthr) + extra;
  if (nthr != BMAX) { rfinv_set_error("forward_kernel<%d,%d>: launched with %d threads", J, BMAX, nthr); return RFINV_ERR_ARG; }
  RFINV_CUDA_CHECK(rfinv_raise_smem_limit((const void*)forward_kernel<J, BMAX, MINB, MIXED, BURIED, GEN>, smem));
  int dev = 0, n_sm = 0, per_sm = 0;
  RFINV_CUDA_CHECK(cudaGetDevice(&dev));
  RFINV_CUDA_CHECK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  RFINV_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, forward_kernel<J, BMAX, MINB, MIXED, BURIED, GEN>, nthr, smem));
  if (per_sm < 1) { rfinv_set_error("forward_kernel does not fit on an SM (%zu bytes of shared memory)", smem); return RFINV_ERR_CUDA; }
  const int n_models = mb.active ? mb.n_active : mb.C;
  const long long items = (long long)n_models * sel.n;
  const long long resident = (long long)n_sm * per_sm;   // persistent CTAs: one wave, items handed out dynamically
  const unsigned grid = (unsigned)(items < resident ? items : resident);
  RFINV_CUDA_CHECK(rfinv_launch_pdl(1, forward_kernel<J, BMAX, MINB, MIXED, BURIED, GEN>, dim3(grid), dim3(nthr), smem, stream, cfg, mb, out, lc, rc, counter, sel));
  return RFINV_OK;
}

// kernel variant for a group of traces that keep JB bin groups: <bin groups per thread that are propagated (band limit),
// upper bound of threads per CTA, CTAs per SM, MIXED = the variant is wider than the group>
#ifndef RFINV_FWD_GENERAL_TU
}  // namespace
// the variants for transform lengths that are not powers of two are compiled in forward_general.cu
int rfinv_launch_forward_group_general(const DevConfig& cfg, const ModelBatch& mb, const EvalOutputs& out, const double* lc,
                                       const double* rc, int* counter, int nthr, cudaStream_t stream, int sel_n,
                                       unsigned long long sel_packed);
namespace {
int launch_forward_group(const DevConfig& cfg, const ModelBatch& mb, const EvalOutputs& out, const double* lc, const double* rc,
                         int* counter, int nthr, cudaStream_t stream, const TraceSel& sel, int JB) {
  if (cfg.fft_general) return rfinv_launch_forward_group_general(cfg, mb, out, lc, rc, counter, nthr, stream, sel.n, sel.packed);
#define FWD(JJ, BB, MM)                                                                                   \
  do {                                                                                                    \
    if (cfg.bdep > 0.0) return launch_forward_t<JJ, BB, MM, true, true>(cfg, mb, out, lc, rc, counter, nthr, stream, sel); \
    if (JJ != JB) return launch_forward_t<JJ, BB, MM, true, false>(cfg, mb, out, lc, rc, counter, nthr, stream, sel); \
    return launch_forward_t<JJ, BB, MM, false, false>(cfg, mb, out, lc, rc, counter, nthr, stream, sel);  \
  } while (0)
  if (nthr <= 32) { if (JB <= 1) FWD(1, 32, 8); FWD(2, 32, 8); }
  if (nthr <= 64) { if (JB <= 2) FWD(2, 64, 6); FWD(4, 64, 6); }
  if (nthr <= 128) {
    if (JB <= 2) FWD(2, 128, 6);
    static const int minb3 = getenv("RFINV_FWD_MINB3") ? atoi(getenv("RFINV_FWD_MINB3")) : 4;   // tuning knob
    if (JB <= 3) { if (minb3 == 5) FWD(3, 128, 5); FWD(3, 128, 4); }
    FWD(4, 128, 4);
  }
  if (JB <= 3) FWD(3, 256, 2);
  if (JB <= 4) FWD(4, 256, 2);
  if (JB <= 6) FWD(6, 256, 1);
  FWD(8, 256, 1);
#undef FWD
}
#endif   // !RFINV_FWD_GENERAL_TU

}  // namespace

#ifdef RFINV_FWD_GENERAL_TU
// Any transform length (Bluestein): one variant per thread count, the widest bin-group count of that thread count with the
// band limit of the trace read at run time (MIXED).
int rfinv_launch_forward_group_general(const DevConfig& cfg, const ModelBatch& mb, const EvalOutputs& out, const double* lc,
                                       const double* rc, int* counter, int nthr, cudaStream_t stream, int sel_n,
                                       unsigned long long sel_packed) {
  TraceSel sel;
  sel.n = sel_n; sel.packed = sel_packed;
#define FWDG(JJ, BB, MM)                                                                                                \
  do {                                                                                                                  \
    if (cfg.bdep > 0.0) return launch_forward_t<JJ, BB, MM, true, true, true>(cfg, mb, out, lc, rc, counter, nthr, stream, sel); \
    return launch_forward_t<JJ, BB, MM, true, false, true>(cfg, mb, out, lc, rc, counter, nthr, stream, sel);           \
  } while (0)
  if (nthr <= 32) FWDG(2, 32, 8);
  if (nthr <= 64) FWDG(4, 64, 6);
  if (nthr <= 128) FWDG(4, 128, 4);
  FWDG(4, 256, 2);
#undef FWDG
}
#else

int rfinv_forward_bins_per_thread(int nfft) {
  if (nfft <= 64) return 1;
  if (nfft <= 256) return 2;
  if (nfft <= 2048) return 4;   // 2048: 256 threads x 4 bins (8 bins per thread would need ~250 registers)
  return 8;
}

size_t rfinv_forward_scratch_doubles(const DevConfig& cfg, long long n_models) {
  const long long ntr_eff = cfg.ray_common ? 1 : cfg.ntrc;
  return (size_t)(n_models * ntr_eff) * ((size_t)cfg.k_max * LC_DOUBLES + RC_DOUBLES) + RFINV_MAX_TRC / 2;   // + the work counters
}

// prep_kernel for the models [m_begin, m_begin + m_count) of the batch; scratch as in rfinv_launch_forward
int rfinv_launch_prep(const DevConfig& cfg, const ModelBatch& mb, uint8_t* is_valid, double* scratch, cudaStream_t stream,
                      int m_begin, int m_count) {
  const int nthr = rfinv_forward_threads(cfg);
  const int n_models = mb.active ? mb.n_active : mb.C;
  const int ntr_eff = cfg.ray_common ? 1 : cfg.ntrc;
  const long long n_items = (long long)n_models * ntr_eff;
  if (m_count <= 0) return RFINV_OK;
  double* lc = scratch;
  double* rc = scratch + (size_t)n_items * cfg.k_max * LC_DOUBLES;
  int* counter = reinterpret_cast<int*>(rc + (size_t)n_items * RC_DOUBLES);
  // one CTA per model, one warp per ray (rays per CTA: all of them while the shared memory stays below ~96 KB, else the
  // model is spread over several CTAs)
  int n_groups = 1;
  while (sizeof(double) * (prep_smem_model_doubles(cfg.k_max) + (size_t)((ntr_eff + n_groups - 1) / n_groups) * prep_smem_ray_doubles(cfg.k_max)) > 96 * 1024 &&
         n_groups < ntr_eff) ++n_groups;
  const int rays_per_cta = (ntr_eff + n_groups - 1) / n_groups;
  n_groups = (ntr_eff + rays_per_cta - 1) / rays_per_cta;
  const size_t prep_smem = sizeof(double) * (prep_smem_model_doubles(cfg.k_max) + (size_t)rays_per_cta * prep_smem_ray_doubles(cfg.k_max));
#define PREP(BUR, HOST)                                                                                                    \
  do {                                                                                                                     \
    RFINV_CUDA_CHECK(rfinv_raise_smem_limit((const void*)prep_kernel<BUR, HOST>, prep_smem));                                \
    prep_kernel<BUR, HOST><<<(unsigned)m_count * n_groups, 32 * rays_per_cta, prep_smem, stream>>>(cfg, mb, lc, rc, is_valid, counter, m_begin + m_count, ntr_eff, nthr, rays_per_cta, m_begin); \
  } while (0)
  if (cfg.bdep > 0.0) { if (mb.chain_major) PREP(true, true); else PREP(true, false); }
  else { if (mb.chain_major) PREP(false, true); else PREP(false, false); }
#undef PREP
  RFINV_CUDA_CHECK(cudaGetLastError());
  return RFINV_OK;
}

// scratch: rfinv_forward_scratch_doubles(cfg, n_models) doubles of device memory
int rfinv_launch_forward(const DevConfig& cfg, const ModelBatch& mb, const EvalOutputs& out, double* scratch,
                         cudaStream_t stream, int* n_kernels, bool prep_done) {
  const int nthr = rfinv_forward_threads(cfg);
  const int n_models = mb.active ? mb.n_active : mb.C;
  const int ntr_eff = cfg.ray_common ? 1 : cfg.ntrc;
  const long long n_items = (long long)n_models * ntr_eff;
  if (n_items == 0) { if (n_kernels) *n_kernels = 0; return RFINV_OK; }
  double* lc = scratch;
  double* rc = scratch + (size_t)n_items * cfg.k_max * LC_DOUBLES;
  int* counter = reinterpret_cast<int*>(rc + (size_t)n_items * RC_DOUBLES);
  if (!prep_done) {
    const int st = rfinv_launch_prep(cfg, mb, out.is_valid, scratch, stream, 0, n_models);
    if (st != RFINV_OK) return st;
  }
  // One launch per band-limit group: traces whose Gaussian filters keep the same number of bin groups share a launch of
  // the kernel variant built for exactly that many (different widths in one launch would have to run the widest
  // variant for every item: more registers, spills in the layer loop).  Common rays: one launch, one ray.
  int n_launch = 0;
  for (int g = 8; g >= 1; --g) {           // widest group first
    TraceSel sel;
    sel.n = 0; sel.packed = 0ULL;
    if (cfg.ray_common) { if (g == cfg.jb_max) sel.push(0); }
    else for (int t = 0; t < cfg.ntrc; ++t) if (cfg.jbins[t] == g) sel.push(t);
    if (sel.n == 0) continue;
    const int st = launch_forward_group(cfg, mb, out, lc, rc, counter + n_launch, nthr, stream, sel, g);
    if (st != RFINV_OK) return st;
    ++n_launch;
  }
  if (n_kernels) *n_kernels = (prep_done ? 0 : 1) + n_launch;   // prep_kernel + one forward_kernel per band-limit group
  return RFINV_OK;
}

// in / out: [n_series][nfft] in HBM, trace_of[n_series]: which trace's filter shapes the series
int rfinv_launch_filter_traces(const DevConfig& cfg, int n_series, const double* in, const int* trace_of, double* out,
                               cudaStream_t stream) {
  if (n_series == 0) return RFINV_OK;
  const size_t smem = sizeof(double2) * (2 * fft_buf_elems(cfg.fft_len) + (cfg.fft_general ? 0 : fft_twiddle_entries(cfg.fft_len))) + sizeof(double) * 64;
  const int nthr = cfg.fft_len / 8 < 32 ? 32 : (cfg.fft_len / 8 > 128 ? 128 : cfg.fft_len / 8);
  if (cfg.fft_general) {
    RFINV_CUDA_CHECK(rfinv_raise_smem_limit((const void*)filter_traces_kernel<true>, smem));
    filter_traces_kernel<true><<<n_series, nthr, smem, stream>>>(cfg, in, trace_of, out);
  } else {
    RFINV_CUDA_CHECK(rfinv_raise_smem_limit((const void*)filter_traces_kernel<false>, smem));
    filter_traces_kernel<false><<<n_series, nthr, smem, stream>>>(cfg, in, trace_of, out);
  }
  RFINV_CUDA_CHECK(cudaGetLastError());
  return RFINV_OK;
}

int rfinv_launch_format_model(const DevConfig& cfg, const ModelBatch& mb, int* nlay, double* alpha, double* beta,
                              double* rho, double* h, uint8_t* is_valid, cudaStream_t stream) {
  if (mb.C == 0) return RFINV_OK;
  format_model_kernel<<<(mb.C + 127) / 128, 128, 0, stream>>>(cfg, mb, nlay, alpha, beta, rho, h, is_valid);
  RFINV_CUDA_CHECK(cudaGetLastError());
  return RFINV_OK;
}
#endif   // !RFINV_FWD_GENERAL_TU
