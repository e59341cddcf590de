// Checkpoint and resume of the device-resident parallel-tempering state (rfinv_pt_save / rfinv_pt_restore).
//
// A checkpoint is an exact image of everything the rest of a run and its outputs depend on: the mt19937 streams, the chain
// state and both RF sample buffers, the swap table, counters, iteration counters, the likelihood history and -- when the
// posterior bookkeeping is on -- the histograms, means and recorded models.  Restoring it into a handle freshly set up by
// rfinv_pt_init with the same arguments continues the run bit for bit: run(N1); save; restore in a new process; run(N2) gives
// what run(N1 + N2) gives.  Per-iteration scratch (proposals, the active list, partial sums, arrival counters) is not held:
// every iteration leaves it empty or rewrites it before reading it.
//
// File (little-endian): CkHeader | sections (CkSection + count * elem_size bytes each) | XXH64 of everything before it.
// The header carries the rank layout, the shape and one fingerprint per group of configuration inputs, so that restore can
// name what differs.  The writer goes to path + ".tmp", fsyncs and renames: a crash leaves the previous checkpoint intact.
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <cerrno>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>
#include "rfinv_handle.h"
#include "rfinv_pt.h"

namespace {

constexpr char CK_MAGIC[8] = {'R', 'F', 'I', 'N', 'V', 'P', 'T', '\0'};
constexpr uint32_t CK_FORMAT = 1;

// fingerprint groups, in the order restore checks them
enum { FP_SCALARS, FP_TRACES, FP_OBS, FP_RINV, FP_REF, FP_SIG, FP_SWITCHES, FP_COUNT };
const char* const FP_NAMES[FP_COUNT] = {
    "configuration scalars", "rayps / a_gus / ipha", "observed traces (obs)", "R^-1 in use", "reference model",
    "sig_min / sig_max", "arithmetic switches (RFINV_FULL_BAND, RFINV_QF_DENSE, RFINV_QF_NOSPLIT)"};

struct CkHeader {
  char magic[8];
  uint32_t format_version, abi_version;
  int32_t nproc_total, rank_begin, rank_count, nchains;
  int32_t ntrc, nsmp, k_max, niter;
  int32_t it_done, record;
  int64_t n_eval_host;     // evaluations counted on the host (rfinv_pt_init's batch); the device counter is a section
  int64_t cap_models;      // rows of all_models the saving handle could hold
  uint64_t fp[FP_COUNT];
  uint32_t n_sections, reserved;
};
static_assert(sizeof(CkHeader) == 8 + 8 + 40 + 16 + 8 * FP_COUNT + 8, "CkHeader must have no padding");

struct CkSection {
  char name[16];
  uint32_t elem_size, reserved;
  uint64_t count;
};
static_assert(sizeof(CkSection) == 32, "CkSection must have no padding");

// ---- XXH64 (seed 0) ----------------------------------------------------------------------------------------------------
constexpr uint64_t P1 = 0x9E3779B185EBCA87ULL, P2 = 0xC2B2AE3D27D4EB4FULL, P3 = 0x165667B19E3779F9ULL,
                   P4 = 0x85EBCA77C2B2AE63ULL, P5 = 0x27D4EB2F165667C5ULL;
inline uint64_t rotl(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
inline uint64_t rd64(const uint8_t* p) { uint64_t v; std::memcpy(&v, p, 8); return v; }
inline uint32_t rd32(const uint8_t* p) { uint32_t v; std::memcpy(&v, p, 4); return v; }
inline uint64_t xround(uint64_t acc, uint64_t in) { return rotl(acc + in * P2, 31) * P1; }
inline uint64_t xmerge(uint64_t acc, uint64_t v) { return (acc ^ xround(0, v)) * P1 + P4; }

uint64_t xxh64(const void* data, size_t len) {
  const uint8_t* p = static_cast<const uint8_t*>(data);
  const uint8_t* end = p + len;
  uint64_t h;
  if (len >= 32) {
    uint64_t v1 = P1 + P2, v2 = P2, v3 = 0, v4 = 0 - P1;
    for (; p + 32 <= end; p += 32) {
      v1 = xround(v1, rd64(p)); v2 = xround(v2, rd64(p + 8)); v3 = xround(v3, rd64(p + 16)); v4 = xround(v4, rd64(p + 24));
    }
    h = rotl(v1, 1) + rotl(v2, 7) + rotl(v3, 12) + rotl(v4, 18);
    h = xmerge(h, v1); h = xmerge(h, v2); h = xmerge(h, v3); h = xmerge(h, v4);
  } else {
    h = P5;
  }
  h += (uint64_t)len;
  for (; p + 8 <= end; p += 8) h = rotl(h ^ xround(0, rd64(p)), 27) * P1 + P4;
  if (p + 4 <= end) { h = rotl(h ^ ((uint64_t)rd32(p) * P1), 23) * P2 + P3; p += 4; }
  for (; p < end; ++p) h = rotl(h ^ ((uint64_t)*p * P5), 11) * P1;
  h ^= h >> 33; h *= P2; h ^= h >> 29; h *= P3; h ^= h >> 32;
  return h;
}

// values hashed one by one, by value (never struct bytes: the configuration holds pointers and padding)
struct Fp {
  std::vector<uint8_t> b;
  void i(int64_t v) { const uint8_t* p = reinterpret_cast<const uint8_t*>(&v); b.insert(b.end(), p, p + 8); }
  void d(double v) { const uint8_t* p = reinterpret_cast<const uint8_t*>(&v); b.insert(b.end(), p, p + 8); }
  void dv(const double* v, size_t n) { i((int64_t)n); for (size_t k = 0; k < n; ++k) d(v[k]); }
  uint64_t done() const { return xxh64(b.data(), b.size()); }
};

void fingerprints(const rfinv_handle* h, uint64_t fp[FP_COUNT]) {
  const rfinv_config& c = h->cfg;
  const size_t T = c.ntrc, S = c.nsmp;
  {  // every scalar of rfinv_config except niter, which may grow between save and restore (see rfinv_pt_restore)
    Fp f;
    for (int64_t v : {c.ntrc, c.nfft, c.nsmp, c.deconv_mode, c.nref, c.vp_mode, c.k_min, c.k_max, c.prior_mode, c.nburn,
                      c.ncorr, c.nchains, c.ncool, c.iseed, c.nbin_z, c.nbin_vs, c.nbin_vp, c.nbin_vpvs, c.nbin_sig, c.nbin_amp})
      f.i(v);
    for (double v : {c.delta, c.t_start, c.sdep, c.z_ref_min, c.dz_ref, c.z_min, c.z_max, c.h_min, c.dvs_prior, c.dvp_prior,
                     c.vp_min, c.vp_max, c.vs_min, c.vs_max, c.vpvs_min, c.vpvs_max, c.dev_z, c.dev_dvs, c.dev_dvp, c.dev_sig,
                     c.t_high, c.amp_min, c.amp_max, c.bdep})
      f.d(v);
    fp[FP_SCALARS] = f.done();
  }
  { Fp f; f.dv(c.rayps, T); f.dv(c.a_gus, T); for (size_t t = 0; t < T; ++t) f.i(c.ipha[t]); fp[FP_TRACES] = f.done(); }
  { Fp f; f.dv(c.obs, T * S); fp[FP_OBS] = f.done(); }
  { Fp f; f.dv(h->h_r_inv.data(), h->h_r_inv.size()); fp[FP_RINV] = f.done(); }
  { Fp f; f.i(c.nref); f.d(c.z_ref_min); f.d(c.dz_ref); f.dv(c.vp_ref, c.nref); f.dv(c.vs_ref, c.nref); fp[FP_REF] = f.done(); }
  { Fp f; f.dv(c.sig_min, T); f.dv(c.sig_max, T); fp[FP_SIG] = f.done(); }
  { Fp f; f.i(rfinv_arith_switches()); fp[FP_SWITCHES] = f.done(); }
}

struct Part {
  const char* name;
  void* dev;           // device array
  uint32_t elem;
  uint64_t count;
};

// The sections of a checkpoint, in file order.  it_done: length of the likelihood history; n_models: recorded rows.
std::vector<Part> parts(rfinv_handle* h, int it_done, long long n_models) {
  PtState* s = h->pt;
  PtDev& d = s->dev;
  const rfinv_config& c = h->cfg;
  const uint64_t Cl = d.Cl, G = d.G, km = c.k_max, T = c.ntrc, S = c.nsmp;
  std::vector<Part> v = {
      {"mt", d.mt, 4, 624 * G}, {"mti", d.mti, 4, G},
      {"k", d.k, 4, Cl}, {"z", d.z, 8, Cl * (km - 1)}, {"dvp", d.dvp, 8, Cl * km}, {"dvs", d.dvs, 8, Cl * km},
      {"sig", d.sig, 8, Cl * T}, {"logl", d.logl, 8, Cl}, {"temps", d.temps, 8, Cl}, {"phi", d.phi, 8, Cl * T},
      {"slot", d.slot, 1, Cl}, {"rft_smp0", d.rft_smp[0], 8, Cl * T * S}, {"rft_smp1", d.rft_smp[1], 8, Cl * T * S},
      {"swap_table", s->d_table, 8, 2 * (uint64_t)s->table_len},
      {"nprop", d.nprop, 8, 8}, {"naccept", d.naccept, 8, 8}, {"n_eval", d.n_eval, 8, 1}, {"it_dev", d.it_dev, 4, 1},
      {"lhist", s->d_lhist, 8, (uint64_t)it_done}};
  if (s->record) {
    const uint64_t nz = c.nbin_z;
    v.insert(v.end(), {{"nk", d.nk, 8, km}, {"nz", d.nz, 8, nz}, {"nsig", d.nsig, 8, (uint64_t)c.nbin_sig * T},
                       {"namp", d.namp, 8, (uint64_t)c.nbin_amp * S * T}, {"nvpz", d.nvpz, 8, nz * c.nbin_vp},
                       {"nvsz", d.nvsz, 8, nz * c.nbin_vs}, {"nvpvsz", d.nvpvsz, 8, nz * c.nbin_vpvs}, {"nmod", d.nmod, 8, 1},
                       {"vp_mean", d.vp_mean, 8, nz}, {"vs_mean", d.vs_mean, 8, nz}, {"vpvs_mean", d.vpvs_mean, 8, nz},
                       // set by the recording kernel for the bins inside the sea layer (pt_record_kernel): held like the sums
                       {"ocean_bin", d.ocean_bin, 1, nz},
                       {"vp_model", d.vp_model, 8, (uint64_t)n_models * nz}, {"vs_model", d.vs_model, 8, (uint64_t)n_models * nz}});
  }
  if (d.st_on) {   // the step tuning (rfinv_pt_set_step_tuning), only with it on: a file without it keeps its sections
    const uint64_t rows = G * d.nchains * 4;
    v.insert(v.end(), {{"step_scale", d.st_scale, 8, rows}, {"step_nprop", d.st_nprop, 8, rows}, {"step_nacc", d.st_nacc, 8, rows},
                       {"step_lvl", d.st_lvl, 4, Cl}, {"step_pair", d.st_pair, 4, 2}});
  }
  if (d.dg_on) {   // the diagnostics (rfinv_pt_set_diagnostics), only with them on: the samples recorded so far
    long long ns = pt_diag_samples(it_done, d.nburn, d.ncorr);
    if (ns > d.dg_cap) ns = d.dg_cap;
    v.insert(v.end(), {{"diag_trace", d.dg_trace, 8, (uint64_t)ns * G * d.dg_nq}, {"diag_t0", d.dg_t0, 8, (uint64_t)ns * G},
                       {"diag_trip_st", d.dg_trip_st, 1, Cl}, {"diag_trips", d.dg_trips, 8, 2 * G}});
  }
  return v;
}

// The rank sweep's section (rfinv_pt_set_rank_swaps), written only in mode 1 -- a file written in mode 0 has the sections of
// a library without the sweep: int64 [mode | n_prop per level | n_acc per level, summed over the ranks]
constexpr const char* RS_SECTION = "rank_swaps";
// The ladder tuning's section (rfinv_pt_set_ladder_tuning), written only with the tuning on: int64 [on | per local rank and
// level pair, the acceptances since the last tuning point].  The rank_swaps section keeps only sums over the ranks, so the
// restore rebuilds the snapshot rows as (restored rows) - (acceptances of the round): the next tuning point sees the counts
// of an uninterrupted run.
constexpr const char* LT_SECTION = "ladder_tuning";
// The step tuning's setting, written only with it on: double [target].  Its device arrays are sections of parts().
constexpr const char* ST_SECTION = "step_tuning";
// The diagnostics' setting, written only with them on: int64 [number of depth bins | the bins, padded to 16 | trace capacity
// of the saving handle].  Their device arrays are sections of parts().
constexpr const char* DG_SECTION = "diagnostics";
constexpr int DG_WORDS = 1 + 16 + 1;

// The sections of the opt-in settings above, in file order after those of parts().  Each is in a file exactly when the
// handle that wrote it had the setting on.
struct Setting {
  const char* name;        // the section; the setting's setter is rfinv_pt_set_<name>
  uint32_t elem;
  uint64_t count;
  bool on;                 // this handle has the setting on: save writes the section, restore needs it
  const char* what;        // for restore's message: "... written with <what> <state>, this handle has <them> <state>"
  const char* them;
  const char* state[2];    // off, on
};
enum { SET_RS, SET_LT, SET_ST, SET_DG, SET_COUNT };

std::vector<Setting> settings(const rfinv_handle* h) {
  const PtState* s = h->pt;
  const PtDev& d = s->dev;
  const uint64_t nl = d.nchains > 1 ? d.nchains - 1 : 0;
  return {{RS_SECTION, sizeof(int64_t), 1 + 2 * nl, s->rank_swaps == 1, "the rank swaps", "them", {"off (mode 0)", "on (mode 1)"}},
          {LT_SECTION, sizeof(int64_t), 1 + d.G * nl, d.rs_tune != 0, "the ladder tuning", "it", {"off", "on"}},
          {ST_SECTION, sizeof(double), 1, d.st_on != 0, "the step tuning", "it", {"off", "on"}},
          {DG_SECTION, sizeof(int64_t), DG_WORDS, d.dg_on != 0, "the diagnostics", "them", {"off", "on"}}};
}

// writes a section header at buf + off and advances off past it
void put_section(uint8_t* buf, size_t& off, const char* name, uint32_t elem, uint64_t count) {
  CkSection sc;
  std::memset(&sc, 0, sizeof(sc));
  std::snprintf(sc.name, sizeof(sc.name), "%s", name);
  sc.elem_size = elem; sc.count = count;
  std::memcpy(buf + off, &sc, sizeof(sc)); off += sizeof(sc);
}

int io_error(const char* who, const std::string& path, const char* what) {
  rfinv_set_error("%s: %s: %s", who, path.c_str(), what);
  return RFINV_ERR_IO;
}

}  // namespace

extern "C" {

int32_t rfinv_pt_save(rfinv_handle* h, const char* path) {
  static const char* who = "rfinv_pt_save";
  if (!h || !path || !*path) { rfinv_set_error("%s: handle or path is NULL", who); return RFINV_ERR_ARG; }
  if (!h->pt) { rfinv_set_error("%s: call rfinv_pt_init first", who); return RFINV_ERR_STATE; }
  PtState* s = h->pt;
  int st;
  if ((st = pt_require_settled(s, who)) != RFINV_OK) return st;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  PtDev& d = s->dev;
  long long n_models = 0;
  if (s->record && d.vp_model) {
    unsigned long long nm = 0;
    RFINV_CUDA_CHECK(cudaMemcpy(&nm, d.nmod, sizeof(nm), cudaMemcpyDeviceToHost));
    n_models = (long long)nm < d.cap_models ? (long long)nm : d.cap_models;
  }
  const std::vector<Part> ps = parts(h, s->it_done, n_models);
  CkHeader hd;
  std::memset(&hd, 0, sizeof(hd));
  std::memcpy(hd.magic, CK_MAGIC, sizeof(CK_MAGIC));
  hd.format_version = CK_FORMAT; hd.abi_version = RFINV_ABI_VERSION;
  hd.nproc_total = d.nproc_total; hd.rank_begin = d.rank_begin; hd.rank_count = d.G; hd.nchains = d.nchains;
  hd.ntrc = h->cfg.ntrc; hd.nsmp = h->cfg.nsmp; hd.k_max = h->cfg.k_max; hd.niter = h->cfg.niter;
  hd.it_done = s->it_done; hd.record = s->record ? 1 : 0; hd.n_eval_host = s->n_eval; hd.cap_models = d.vp_model ? d.cap_models : 0;
  fingerprints(h, hd.fp);
  // the payloads of the settings' sections that are on, in the order of settings()
  const std::vector<Setting> ss = settings(h);
  std::vector<int64_t> rs, lt, dg;
  if (ss[SET_RS].on) {
    rs.assign(ss[SET_RS].count, 0);
    const size_t nl = (rs.size() - 1) / 2;
    int32_t mode = 0;
    if ((st = rfinv_pt_get_rank_swaps(h, &mode, rs.data() + 1, rs.data() + 1 + nl)) != RFINV_OK) return st;
    rs[0] = mode;
  }
  if (ss[SET_LT].on) {
    lt.assign(ss[SET_LT].count, 0);
    lt[0] = 1;
    const size_t nr = lt.size() - 1;
    if (nr) {
      std::vector<unsigned long long> acc(nr), base(nr);
      RFINV_CUDA_CHECK(cudaMemcpy(acc.data(), d.rs_nacc, sizeof(unsigned long long) * nr, cudaMemcpyDeviceToHost));
      RFINV_CUDA_CHECK(cudaMemcpy(base.data(), d.rs_base, sizeof(unsigned long long) * nr, cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < nr; ++i) lt[1 + i] = (int64_t)(acc[i] - base[i]);
    }
  }
  if (ss[SET_DG].on) {
    dg.assign(DG_WORDS, 0);
    dg[0] = d.dg_nbins;
    std::vector<int32_t> bins(16, 0);
    if (d.dg_nbins) RFINV_CUDA_CHECK(cudaMemcpy(bins.data(), d.dg_bins, sizeof(int32_t) * d.dg_nbins, cudaMemcpyDeviceToHost));
    for (int j = 0; j < 16; ++j) dg[1 + j] = bins[j];
    dg[17] = d.dg_cap;
  }
  const void* const payload[SET_COUNT] = {rs.data(), lt.data(), &d.st_target, dg.data()};
  hd.n_sections = (uint32_t)ps.size();
  size_t total = sizeof(CkHeader) + sizeof(uint64_t);
  for (const Part& p : ps) total += sizeof(CkSection) + (size_t)p.elem * p.count;
  for (const Setting& x : ss)
    if (x.on) { ++hd.n_sections; total += sizeof(CkSection) + (size_t)x.elem * x.count; }
  std::unique_ptr<uint8_t[]> buf(new (std::nothrow) uint8_t[total]);
  if (!buf) { rfinv_set_error("%s: cannot allocate %zu bytes of host memory", who, total); return RFINV_ERR_IO; }
  size_t off = 0;
  std::memcpy(buf.get(), &hd, sizeof(hd)); off += sizeof(hd);
  for (const Part& p : ps) {
    put_section(buf.get(), off, p.name, p.elem, p.count);
    const size_t n = (size_t)p.elem * p.count;
    if (n) RFINV_CUDA_CHECK(cudaMemcpy(buf.get() + off, p.dev, n, cudaMemcpyDeviceToHost));
    off += n;
  }
  for (int i = 0; i < SET_COUNT; ++i) {
    if (!ss[i].on) continue;
    put_section(buf.get(), off, ss[i].name, ss[i].elem, ss[i].count);
    const size_t n = (size_t)ss[i].elem * ss[i].count;
    std::memcpy(buf.get() + off, payload[i], n); off += n;
  }
  const uint64_t sum = xxh64(buf.get(), off);
  std::memcpy(buf.get() + off, &sum, sizeof(sum));
  // atomically: the temporary file is complete and on disk before it replaces `path`
  const std::string tmp = std::string(path) + ".tmp";
  const int fd = open(tmp.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644);
  if (fd < 0) return io_error(who, tmp, std::strerror(errno));
  for (size_t w = 0; w < total;) {
    const ssize_t r = write(fd, buf.get() + w, total - w);
    if (r < 0 && errno == EINTR) continue;
    if (r <= 0) { const int e = errno; close(fd); unlink(tmp.c_str()); return io_error(who, tmp, std::strerror(e)); }
    w += (size_t)r;
  }
  if (fsync(fd) != 0) { const int e = errno; close(fd); unlink(tmp.c_str()); return io_error(who, tmp, std::strerror(e)); }
  if (close(fd) != 0) { unlink(tmp.c_str()); return io_error(who, tmp, std::strerror(errno)); }
  if (rename(tmp.c_str(), path) != 0) { const int e = errno; unlink(tmp.c_str()); return io_error(who, path, std::strerror(e)); }
  return RFINV_OK;
}

int32_t rfinv_pt_restore(rfinv_handle* h, const char* path) {
  static const char* who = "rfinv_pt_restore";
  if (!h || !path || !*path) { rfinv_set_error("%s: handle or path is NULL", who); return RFINV_ERR_ARG; }
  if (!h->pt) { rfinv_set_error("%s: call rfinv_pt_init first", who); return RFINV_ERR_STATE; }
  PtState* s = h->pt;
  PtDev& d = s->dev;
  if (s->it_done != 0 || s->step_pending || s->reduced) {
    rfinv_set_error("%s: restore needs a handle fresh from rfinv_pt_init (%d iterations have run on it)", who, s->it_done);
    return RFINV_ERR_STATE;
  }
  const std::string file(path);
  // ---- read and check the file as a whole before anything on the device changes ----
  std::vector<uint8_t> buf;
  {
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return io_error(who, file, std::strerror(errno));
    struct stat st;
    if (fstat(fd, &st) != 0) { const int e = errno; close(fd); return io_error(who, file, std::strerror(e)); }
    buf.resize((size_t)st.st_size);
    for (size_t r = 0; r < buf.size();) {
      const ssize_t n = read(fd, buf.data() + r, buf.size() - r);
      if (n < 0 && errno == EINTR) continue;
      if (n <= 0) { const int e = n < 0 ? errno : EIO; close(fd); return io_error(who, file, std::strerror(e)); }
      r += (size_t)n;
    }
    close(fd);
  }
  if (buf.size() < sizeof(CkHeader) + sizeof(uint64_t)) return io_error(who, file, "file is short (no complete header)");
  CkHeader hd;
  std::memcpy(&hd, buf.data(), sizeof(hd));
  if (std::memcmp(hd.magic, CK_MAGIC, sizeof(CK_MAGIC)) != 0) return io_error(who, file, "not a parallel-tempering checkpoint (bad magic)");
  if (hd.format_version != CK_FORMAT) {
    rfinv_set_error("%s: %s: unknown checkpoint format version %u (this library reads %u)", who, path, hd.format_version, CK_FORMAT);
    return RFINV_ERR_IO;
  }
  const size_t body = buf.size() - sizeof(uint64_t);
  std::map<std::string, std::pair<size_t, CkSection>> found;   // name -> (offset of the data, section header)
  {
    size_t off = sizeof(CkHeader);
    for (uint32_t i = 0; i < hd.n_sections; ++i) {
      if (off + sizeof(CkSection) > body) {
        rfinv_set_error("%s: %s: file is short: section %u of %u is missing", who, path, i + 1, hd.n_sections);
        return RFINV_ERR_IO;
      }
      CkSection sc;
      std::memcpy(&sc, buf.data() + off, sizeof(sc));
      sc.name[sizeof(sc.name) - 1] = '\0';
      off += sizeof(sc);
      const size_t n = (size_t)sc.elem_size * sc.count;
      if (sc.elem_size == 0 || n / sc.elem_size != sc.count || n > body - off) {
        rfinv_set_error("%s: %s: file is short: section '%s' needs %llu elements of %u bytes, %zu bytes are left", who, path,
                        sc.name, (unsigned long long)sc.count, sc.elem_size, body - off);
        return RFINV_ERR_IO;
      }
      found[sc.name] = {off, sc};
      off += n;
    }
    if (off != body) return io_error(who, file, "trailing bytes after the last section");
  }
  uint64_t sum;
  std::memcpy(&sum, buf.data() + body, sizeof(sum));
  if (sum != xxh64(buf.data(), body)) return io_error(who, file, "checksum mismatch (the file is damaged)");
  // ---- does it fit this handle? ----
  const rfinv_config& c = h->cfg;
  if (hd.nproc_total != d.nproc_total || hd.rank_begin != d.rank_begin || hd.rank_count != d.G) {
    rfinv_set_error("%s: %s holds virtual ranks [%d, %d) of %d, this handle owns [%d, %d) of %d (rfinv_pt_init)", who, path,
                    hd.rank_begin, hd.rank_begin + hd.rank_count, hd.nproc_total, d.rank_begin, d.rank_begin + d.G, d.nproc_total);
    return RFINV_ERR_ARG;
  }
  if (hd.nchains != d.nchains) {
    rfinv_set_error("%s: %s has nchains = %d, this configuration %d", who, path, hd.nchains, d.nchains);
    return RFINV_ERR_ARG;
  }
  if (hd.ntrc != c.ntrc || hd.nsmp != c.nsmp || hd.k_max != c.k_max) {
    rfinv_set_error("%s: %s has ntrc / nsmp / k_max = %d / %d / %d, this configuration %d / %d / %d", who, path, hd.ntrc,
                    hd.nsmp, hd.k_max, c.ntrc, c.nsmp, c.k_max);
    return RFINV_ERR_ARG;
  }
  if (hd.niter > c.niter) {
    rfinv_set_error("%s: %s was written with niter = %d; niter may only grow (this configuration: %d)", who, path, hd.niter, c.niter);
    return RFINV_ERR_ARG;
  }
  if ((hd.record != 0) != s->record) {
    rfinv_set_error("%s: %s was written with the posterior bookkeeping %s, this configuration has it %s", who, path,
                    hd.record ? "on" : "off", s->record ? "on" : "off");
    return RFINV_ERR_ARG;
  }
  uint64_t fp[FP_COUNT];
  fingerprints(h, fp);
  for (int g = 0; g < FP_COUNT; ++g)
    if (fp[g] != hd.fp[g]) {
      rfinv_set_error("%s: %s: the %s differ from those the checkpoint was written with", who, path, FP_NAMES[g]);
      return RFINV_ERR_ARG;
    }
  // recorded models: rows [0, min(nmod, cap)) of the saving handle; they must all fit here, and a larger niter must not
  // open rows the saving handle had no room for (they would be missing)
  long long n_models = 0;
  if (s->record) {
    auto it = found.find("nmod");
    if (it == found.end() || it->second.second.elem_size != 8 || it->second.second.count != 1)
      return io_error(who, file, "section 'nmod' is missing or malformed");
    unsigned long long nm = 0;
    std::memcpy(&nm, buf.data() + it->second.first, sizeof(nm));
    n_models = (long long)nm < hd.cap_models ? (long long)nm : hd.cap_models;
    const long long cap_here = d.vp_model ? d.cap_models : 0;
    if (n_models > cap_here || ((long long)nm > hd.cap_models && cap_here > hd.cap_models)) {
      rfinv_set_error("%s: %s: %llu models were recorded, the checkpoint holds %lld of them and this configuration has room "
                      "for %lld: the recorded models would differ from an uninterrupted run", who, path, nm, n_models, cap_here);
      return RFINV_ERR_ARG;
    }
  }
  // the settings are part of the run: each is on in the file exactly when it is on here (set with its setter before restoring)
  for (const Setting& x : settings(h)) {
    const auto it = found.find(x.name);
    const bool in_file = it != found.end();
    if (in_file != x.on) {
      rfinv_set_error("%s: %s was written with %s %s, this handle has %s %s (rfinv_pt_set_%s before restore)", who, path, x.what,
                      x.state[in_file], x.them, x.state[x.on], x.name);
      return RFINV_ERR_ARG;
    }
    if (in_file && (it->second.second.elem_size != x.elem || it->second.second.count != x.count))
      return io_error(who, file, ("section '" + std::string(x.name) + "' is malformed").c_str());
  }
  const int nl = d.nchains > 1 ? d.nchains - 1 : 0;
  if (d.st_on) {   // with the same target
    double target;
    std::memcpy(&target, buf.data() + found[ST_SECTION].first, sizeof(double));
    if (target != d.st_target) {
      rfinv_set_error("%s: %s was written with the step tuning's target %.17g, this handle has %.17g", who, path, target, d.st_target);
      return RFINV_ERR_ARG;
    }
  }
  if (d.dg_on) {   // with the same depth bins
    int64_t dg[DG_WORDS];
    std::memcpy(dg, buf.data() + found[DG_SECTION].first, sizeof(dg));
    std::vector<int32_t> bins(16, 0);
    if (d.dg_nbins) RFINV_CUDA_CHECK(cudaMemcpy(bins.data(), d.dg_bins, sizeof(int32_t) * d.dg_nbins, cudaMemcpyDeviceToHost));
    bool same = dg[0] == d.dg_nbins;
    for (int j = 0; j < 16; ++j) same = same && dg[1 + j] == bins[j];
    if (!same) {
      rfinv_set_error("%s: %s was written with %lld diagnostic depth bins that differ from this handle's %d", who, path,
                      (long long)dg[0], d.dg_nbins);
      return RFINV_ERR_ARG;
    }
    // as for the recorded models: a larger capacity must not open samples the saving handle had no room for
    if (hd.it_done >= 0 && pt_diag_samples(hd.it_done, d.nburn, d.ncorr) > dg[17] && d.dg_cap > dg[17]) {
      rfinv_set_error("%s: %s: its trace was full at %lld samples and this configuration has room for %lld: the trace would "
                      "differ from an uninterrupted run", who, path, (long long)dg[17], d.dg_cap);
      return RFINV_ERR_ARG;
    }
  }
  if (hd.it_done < 0) return io_error(who, file, "negative iteration count");
  const std::vector<Part> ps = parts(h, hd.it_done, n_models);
  for (const Part& p : ps) {
    auto it = found.find(p.name);
    if (it == found.end()) { rfinv_set_error("%s: %s: section '%s' is missing", who, path, p.name); return RFINV_ERR_IO; }
    const CkSection& sc = it->second.second;
    if (sc.elem_size != p.elem || sc.count != p.count) {
      rfinv_set_error("%s: %s: section '%s' holds %llu elements of %u bytes, this handle needs %llu of %u", who, path, p.name,
                      (unsigned long long)sc.count, sc.elem_size, (unsigned long long)p.count, p.elem);
      return RFINV_ERR_IO;
    }
  }
  // ---- overwrite the state rfinv_pt_init left ----
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  RFINV_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  int st;
  if ((st = rfinv_pt_reserve_lhist(h, hd.it_done)) != RFINV_OK) return st;
  const std::vector<Part> dst = parts(h, hd.it_done, n_models);   // (the history may have moved)
  for (const Part& p : dst) {
    const size_t n = (size_t)p.elem * p.count;
    if (n) RFINV_CUDA_CHECK(cudaMemcpy(p.dev, buf.data() + found[p.name].first, n, cudaMemcpyHostToDevice));
  }
  if (s->rank_swaps == 1 && nl > 0) {   // the per-level sums go into the row of local rank 0, the other rows start at zero
    std::vector<int64_t> rs(1 + 2 * (size_t)nl);
    std::memcpy(rs.data(), buf.data() + found[RS_SECTION].first, sizeof(int64_t) * rs.size());
    std::vector<int64_t> rows((size_t)d.G * nl, 0);
    std::memcpy(rows.data(), rs.data() + 1 + nl, sizeof(int64_t) * nl);
    RFINV_CUDA_CHECK(cudaMemcpy(d.rs_nprop, rs.data() + 1, sizeof(int64_t) * nl, cudaMemcpyHostToDevice));
    RFINV_CUDA_CHECK(cudaMemcpy(d.rs_nacc, rows.data(), sizeof(int64_t) * rows.size(), cudaMemcpyHostToDevice));
    if (d.rs_tune) {   // snapshot = restored row - acceptances of the round (modulo 2^64)
      std::vector<int64_t> round((size_t)d.G * nl);
      std::memcpy(round.data(), buf.data() + found[LT_SECTION].first + sizeof(int64_t), sizeof(int64_t) * round.size());
      std::vector<unsigned long long> base(round.size());
      for (size_t i = 0; i < base.size(); ++i) base[i] = (unsigned long long)rows[i] - (unsigned long long)round[i];
      RFINV_CUDA_CHECK(cudaMemcpy(d.rs_base, base.data(), sizeof(unsigned long long) * base.size(), cudaMemcpyHostToDevice));
    }
  }
  s->it_done = hd.it_done;
  s->n_eval = hd.n_eval_host;
  h->invalidate_pt_graphs();
  return rfinv_pt_set_logging(h, 0);   // logs restart empty at the restored iteration
}

}  // extern "C"
