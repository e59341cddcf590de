// The collectives of the parallel-tempering driver, inside the library: a NCCL communicator per handle.
//
// Replaces the reference's MPI traffic on this path (paths relative to the reference checkout):
//   pt_control's swap exchange      src/pt_mcmc.f90:518-571  (mpi_bcast of the pair, mpi_send / mpi_recv of temperature and
//                                   likelihood between the two ranks)   ->  stores into peer memory (rfinv_pt.h: PtPeers), or
//                                                                           ONE ncclAllGather of the swap tables per iteration
//   output_results' 14 reduces      src/mcmc_out.f90:52-79   ->  ncclReduce of the device-resident bookkeeping arrays to process 0
//   output_results' 2 gathers       src/mcmc_out.f90:86-93   ->  ncclSend / ncclRecv of the recorded models to process 0
// NCCL is bound at run time (dlopen of libnccl.so.2: the copy the host process already loaded, e.g. torch's, or the system
// one); a build without NCCL still loads, and rfinv_comm_* then fail with a clear message.  The unique id is created on one
// process and handed to the others by the host (MPI_Bcast in a Fortran host, torch.distributed / a file in the Python one).
#include <dlfcn.h>
#include <cstring>
#include <vector>
#include "rfinv_handle.h"
#include "rfinv_pt.h"

namespace {

// the part of nccl.h this file needs (types only: no link-time dependency)
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclInt8 = 0, ncclInt32 = 2, ncclUint64 = 5, ncclFloat64 = 8 };
enum { ncclSum = 0 };

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Reduce)(const void*, void*, size_t, int, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*GetVersion)(int*) = nullptr;
};

NcclApi* nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (tried) return api.lib ? &api : nullptr;
  tried = true;
  const char* names[] = {getenv("RFINV_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    if (!n || !*n) continue;
    api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (api.lib) break;
  }
  if (!api.lib) return nullptr;
#define SYM(field, name) *(void**)(&api.field) = dlsym(api.lib, name); if (!api.field) { dlclose(api.lib); api.lib = nullptr; return nullptr; }
  SYM(GetUniqueId, "ncclGetUniqueId") SYM(CommInitRank, "ncclCommInitRank") SYM(CommDestroy, "ncclCommDestroy")
  SYM(GetErrorString, "ncclGetErrorString") SYM(AllGather, "ncclAllGather") SYM(Reduce, "ncclReduce") SYM(Send, "ncclSend")
  SYM(Recv, "ncclRecv") SYM(GroupStart, "ncclGroupStart") SYM(GroupEnd, "ncclGroupEnd") SYM(GetVersion, "ncclGetVersion")
#undef SYM
  return &api;
}

#define RFINV_NCCL_CHECK(api, expr)                                                                \
  do {                                                                                             \
    ncclResult_t r__ = (expr);                                                                     \
    if (r__ != 0) { rfinv_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, (api)->GetErrorString(r__)); return RFINV_ERR_CUDA; } \
  } while (0)

}  // namespace

// all-gather of `count` doubles per process on stream s (capturable in a CUDA graph)
int rfinv_comm_allgather(rfinv_handle* h, const double* send, double* recv, size_t count, cudaStream_t s) {
  NcclApi* api = nccl_api();
  if (!api || !h->comm) { rfinv_set_error("no communicator: call rfinv_comm_init first"); return RFINV_ERR_STATE; }
  RFINV_NCCL_CHECK(api, api->AllGather(send, recv, count, ncclFloat64, (ncclComm_t)h->comm, s));
  return RFINV_OK;
}

// ---- swap exchange over peer memory (rfinv_pt.h: PtPeers) ---------------------------------------------------------
// Collective over the handle's communicator, outside any capture: every process allocates its gather buffer and flag
// words (one allocation), exports it through CUDA IPC, the 64-byte handles travel by ncclAllGather, every process maps its peers'
// buffers (cudaIpcMemLazyEnablePeerAccess: NVLink peer access) and the outcome is agreed on by a second all-gather -- one
// process that cannot map a peer (no peer access, another node, IPC forbidden by the container) keeps the NCCL all-gather
// for everybody.  RFINV_PT_EXCHANGE=nccl forces that.  The all-gathers double as the barrier between "my flags are zero"
// and "a peer raises one".
int rfinv_comm_peer_setup(rfinv_handle* h) {
  PtState* s = h->pt;
  NcclApi* api = nccl_api();
  if (!s || !api || !h->comm) { rfinv_set_error("rfinv_comm_peer_setup: no communicator"); return RFINV_ERR_STATE; }
  const int world = h->comm_world, me = h->comm_rank;
  ncclComm_t comm = (ncclComm_t)h->comm;
  cudaStream_t q = h->stream;
  s->peer_state = -1;
  const char* mode = getenv("RFINV_PT_EXCHANGE");
  int want = !(mode && std::strcmp(mode, "nccl") == 0) && world <= RFINV_MAX_PEERS;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  struct Blob { cudaIpcMemHandle_t mem; int ok; int pad[3]; };
  Blob mine;
  std::memset(&mine, 0, sizeof(mine));
  const size_t n_gather = (size_t)2 * world * s->table_len;
  if (want) {
    // one allocation (one IPC handle): [2][world][table_len] doubles, then the flag words and pair slots (rfinv_pt.h)
    if (cudaMalloc((void**)&s->d_peer_gather, sizeof(double) * (n_gather + pt_peer_tail_words(world))) != cudaSuccess ||
        cudaMalloc((void**)&s->peers.done, 4 * sizeof(int)) != cudaSuccess) want = 0;
  }
  if (want) {
    s->d_peer_flags = reinterpret_cast<unsigned long long*>(s->d_peer_gather + n_gather);
    cudaMemset(s->d_peer_gather, 0, sizeof(double) * (n_gather + pt_peer_tail_words(world)));
    const int applied[4] = {s->it_done, s->it_done, s->it_done, 0};   // every swap of the iterations run so far has been applied in full
    cudaMemcpy(s->peers.done, applied, sizeof(applied), cudaMemcpyHostToDevice);
    if (cudaIpcGetMemHandle(&mine.mem, s->d_peer_gather) != cudaSuccess) want = 0;
    cudaDeviceSynchronize();
  }
  cudaGetLastError();
  mine.ok = want;
  // exchange the blobs
  std::vector<Blob> all(world);
  char* d_blobs = nullptr;
  RFINV_CUDA_CHECK(cudaMalloc((void**)&d_blobs, sizeof(Blob) * (world + 1)));
  RFINV_CUDA_CHECK(cudaMemcpyAsync(d_blobs + sizeof(Blob) * world, &mine, sizeof(Blob), cudaMemcpyHostToDevice, q));
  RFINV_NCCL_CHECK(api, api->AllGather(d_blobs + sizeof(Blob) * world, d_blobs, sizeof(Blob), ncclInt8, comm, q));
  RFINV_CUDA_CHECK(cudaMemcpyAsync(all.data(), d_blobs, sizeof(Blob) * world, cudaMemcpyDeviceToHost, q));
  RFINV_CUDA_CHECK(cudaStreamSynchronize(q));
  int ok = 1;
  for (int r = 0; r < world; ++r) ok &= all[r].ok;
  PtPeers& px = s->peers;
  px.world = world; px.me = me; px.table_len = s->table_len;
  if (ok) {
    for (int r = 0; r < world && ok; ++r) {
      if (r == me) { px.gather[r] = s->d_peer_gather; px.flag[r] = s->d_peer_flags; px.own_gather = s->d_peer_gather; px.own_flag = s->d_peer_flags; continue; }
      void* g = nullptr;
      if (cudaIpcOpenMemHandle(&g, all[r].mem, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; g = nullptr; }
      px.gather[r] = (double*)g;
      px.flag[r] = g ? reinterpret_cast<unsigned long long*>((double*)g + n_gather) : nullptr;
    }
    cudaGetLastError();
  }
  // agree on the outcome
  int* d_ok = reinterpret_cast<int*>(d_blobs);
  std::vector<int> oks(world, 0);
  RFINV_CUDA_CHECK(cudaMemcpyAsync(d_ok + world, &ok, sizeof(int), cudaMemcpyHostToDevice, q));
  RFINV_NCCL_CHECK(api, api->AllGather(d_ok + world, d_ok, 1, ncclInt32, comm, q));
  RFINV_CUDA_CHECK(cudaMemcpyAsync(oks.data(), d_ok, sizeof(int) * world, cudaMemcpyDeviceToHost, q));
  RFINV_CUDA_CHECK(cudaStreamSynchronize(q));
  cudaFree(d_blobs);
  int all_ok = 1;
  for (int r = 0; r < world; ++r) all_ok &= oks[r];
  if (all_ok) { s->peer_state = 1; return RFINV_OK; }
  rfinv_comm_peer_release(h);
  s->peer_state = -1;
  return RFINV_OK;
}

void rfinv_comm_peer_release(rfinv_handle* h) {
  PtState* s = h->pt;
  if (!s) return;
  PtPeers& px = s->peers;
  for (int r = 0; r < px.world && r < RFINV_MAX_PEERS; ++r) {
    if (r == px.me) continue;
    if (px.gather[r]) cudaIpcCloseMemHandle(px.gather[r]);
  }
  cudaFree(s->d_peer_gather); cudaFree(px.done);   // (the flag words live in the gather allocation)
  s->d_peer_gather = nullptr; s->d_peer_flags = nullptr;
  std::memset(&px, 0, sizeof(px));
  s->peer_state = 0;
  cudaGetLastError();
}

extern "C" {

int32_t rfinv_comm_id_bytes(void) { return (int32_t)sizeof(ncclUniqueId); }

int32_t rfinv_comm_create_id(void* id_out) {
  if (!id_out) { rfinv_set_error("rfinv_comm_create_id: NULL argument"); return RFINV_ERR_ARG; }
  NcclApi* api = nccl_api();
  if (!api) { rfinv_set_error("rfinv_comm_create_id: libnccl.so.2 not found (set RFINV_NCCL_LIB)"); return RFINV_ERR_STATE; }
  ncclUniqueId id;
  RFINV_NCCL_CHECK(api, api->GetUniqueId(&id));
  std::memcpy(id_out, &id, sizeof(id));
  return RFINV_OK;
}

int32_t rfinv_comm_init(rfinv_handle* h, const void* id, int32_t world, int32_t rank) {
  if (!h || !id || world < 1 || rank < 0 || rank >= world) { rfinv_set_error("rfinv_comm_init: bad argument"); return RFINV_ERR_ARG; }
  NcclApi* api = nccl_api();
  if (!api) { rfinv_set_error("rfinv_comm_init: libnccl.so.2 not found (set RFINV_NCCL_LIB)"); return RFINV_ERR_STATE; }
  if (h->comm) { rfinv_set_error("rfinv_comm_init: the handle already has a communicator"); return RFINV_ERR_STATE; }
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  ncclUniqueId uid;
  std::memcpy(&uid, id, sizeof(uid));
  ncclComm_t c = nullptr;
  RFINV_NCCL_CHECK(api, api->CommInitRank(&c, world, uid, rank));
  h->comm = c; h->comm_world = world; h->comm_rank = rank;
  return RFINV_OK;
}

int32_t rfinv_comm_destroy(rfinv_handle* h) {
  if (!h || !h->comm) return RFINV_OK;
  NcclApi* api = nccl_api();
  cudaSetDevice(h->device);
  h->invalidate_pt_graphs();   // graphs with captured collectives keep the communicator alive: ncclCommDestroy would wait for them
  if (h->stream) cudaStreamSynchronize(h->stream);
  cudaDeviceSynchronize();
  if (api) api->CommDestroy((ncclComm_t)h->comm);
  h->comm = nullptr; h->comm_world = 1; h->comm_rank = 0;
  return RFINV_OK;
}

int32_t rfinv_comm_info(rfinv_handle* h, int32_t* world, int32_t* rank, int32_t* nccl_version) {
  if (!h) { rfinv_set_error("rfinv_comm_info: handle is NULL"); return RFINV_ERR_ARG; }
  if (world) *world = h->comm ? h->comm_world : 1;
  if (rank) *rank = h->comm ? h->comm_rank : 0;
  if (nccl_version) { *nccl_version = 0; NcclApi* api = nccl_api(); if (api) { int v = 0; api->GetVersion(&v); *nccl_version = v; } }
  return RFINV_OK;
}

// output_results' reductions (src/mcmc_out.f90:52-79) on the device-resident bookkeeping: afterwards process 0 holds the
// job-wide sums of nmod, nprop, naccept, nk, namp, nvpz, nvsz, nvpvsz, nz, nsig, likelihood_hist, vp/vs/vpvs_mean (the getters
// rfinv_pt_get_hist / _get_counters then return what mpi_reduce delivers on rank 0; with the rank sweep on, also its counters) and, like mpi_gather (:86-93), the
// recorded models of every process in process order (rfinv_pt_get_models).  Collective; call once, after the last iteration.
int32_t rfinv_pt_reduce_outputs(rfinv_handle* h) {
  if (!h || !h->pt) { rfinv_set_error("rfinv_pt_reduce_outputs: call rfinv_pt_init first"); return RFINV_ERR_STATE; }
  h->pt->reduced = true;
  if (!h->comm || h->comm_world == 1) return RFINV_OK;   // a single process already holds the job-wide sums
  NcclApi* api = nccl_api();
  PtState* s = h->pt;
  PtDev& d = s->dev;
  const rfinv_config& c = h->cfg;
  ncclComm_t comm = (ncclComm_t)h->comm;
  cudaStream_t q = h->stream;
  RFINV_CUDA_CHECK(cudaSetDevice(h->device));
  struct Arr { void* p; size_t n; int type; };
  std::vector<Arr> arrs = {{d.nprop, (size_t)d.ntype, ncclUint64}, {d.naccept, (size_t)d.ntype, ncclUint64},
                           {s->d_lhist, (size_t)s->it_done, ncclFloat64}};
  if (s->rank_swaps == 1 && d.rs_nprop)   // every process holds G rows of the same shape: their sum sums over all ranks
    arrs.insert(arrs.end(), {{d.rs_nprop, (size_t)d.nchains - 1, ncclUint64}, {d.rs_nacc, (size_t)d.G * (d.nchains - 1), ncclUint64}});
  if (s->record) {
    const size_t T = c.ntrc, S = c.nsmp;
    arrs.insert(arrs.end(), {{d.nk, (size_t)c.k_max, ncclUint64}, {d.nz, (size_t)c.nbin_z, ncclUint64}, {d.nsig, (size_t)c.nbin_sig * T, ncclUint64},
                             {d.namp, (size_t)c.nbin_amp * S * T, ncclUint64}, {d.nvpz, (size_t)c.nbin_z * c.nbin_vp, ncclUint64},
                             {d.nvsz, (size_t)c.nbin_z * c.nbin_vs, ncclUint64}, {d.nvpvsz, (size_t)c.nbin_z * c.nbin_vpvs, ncclUint64},
                             {d.vp_mean, (size_t)c.nbin_z, ncclFloat64}, {d.vs_mean, (size_t)c.nbin_z, ncclFloat64},
                             {d.vpvs_mean, (size_t)c.nbin_z, ncclFloat64}});
  }
  // recorded models: counts first (all-gather of nmod), then the models themselves point to point into process 0
  std::vector<unsigned long long> counts(h->comm_world, 0ULL);
  unsigned long long* d_counts = nullptr;
  if (s->record) {
    RFINV_CUDA_CHECK(cudaMalloc((void**)&d_counts, sizeof(unsigned long long) * h->comm_world));
    RFINV_NCCL_CHECK(api, api->AllGather(d.nmod, d_counts, 1, ncclUint64, comm, q));
    RFINV_CUDA_CHECK(cudaMemcpyAsync(counts.data(), d_counts, sizeof(unsigned long long) * h->comm_world, cudaMemcpyDeviceToHost, q));
    RFINV_CUDA_CHECK(cudaStreamSynchronize(q));
    cudaFree(d_counts);
  }
  RFINV_NCCL_CHECK(api, api->GroupStart());
  for (const Arr& a : arrs)
    if (a.p && a.n) RFINV_NCCL_CHECK(api, api->Reduce(a.p, a.p, a.n, a.type, ncclSum, 0, comm, q));
  RFINV_NCCL_CHECK(api, api->GroupEnd());
  if (s->record) {
    RFINV_NCCL_CHECK(api, api->Reduce(d.nmod, d.nmod, 1, ncclUint64, ncclSum, 0, comm, q));
    if (d.vp_model) {
      // every process keeps min(nmod, cap_models) models; process 0 needs room for all of them
      std::vector<long long> kept(h->comm_world);
      long long total = 0;
      for (int r = 0; r < h->comm_world; ++r) { kept[r] = (long long)counts[r] < d.cap_models ? (long long)counts[r] : d.cap_models; total += kept[r]; }
      const size_t row = (size_t)c.nbin_z;
      if (h->comm_rank == 0) {
        if (total > d.cap_models) {   // grow rank 0's buffers, keeping its own models in front
          double *nvp = nullptr, *nvs = nullptr;
          RFINV_CUDA_CHECK(cudaMalloc((void**)&nvp, sizeof(double) * (size_t)total * row));
          RFINV_CUDA_CHECK(cudaMalloc((void**)&nvs, sizeof(double) * (size_t)total * row));
          RFINV_CUDA_CHECK(cudaMemcpyAsync(nvp, d.vp_model, sizeof(double) * (size_t)kept[0] * row, cudaMemcpyDeviceToDevice, q));
          RFINV_CUDA_CHECK(cudaMemcpyAsync(nvs, d.vs_model, sizeof(double) * (size_t)kept[0] * row, cudaMemcpyDeviceToDevice, q));
          RFINV_CUDA_CHECK(cudaStreamSynchronize(q));
          cudaFree(d.vp_model); cudaFree(d.vs_model);
          d.vp_model = nvp; d.vs_model = nvs; d.cap_models = total;
        }
        RFINV_NCCL_CHECK(api, api->GroupStart());
        long long off = kept[0];
        for (int r = 1; r < h->comm_world; ++r) {
          if (kept[r] > 0) {
            RFINV_NCCL_CHECK(api, api->Recv(d.vp_model + (size_t)off * row, (size_t)kept[r] * row, ncclFloat64, r, comm, q));
            RFINV_NCCL_CHECK(api, api->Recv(d.vs_model + (size_t)off * row, (size_t)kept[r] * row, ncclFloat64, r, comm, q));
          }
          off += kept[r];
        }
        RFINV_NCCL_CHECK(api, api->GroupEnd());
      } else if (kept[h->comm_rank] > 0) {
        RFINV_NCCL_CHECK(api, api->GroupStart());
        RFINV_NCCL_CHECK(api, api->Send(d.vp_model, (size_t)kept[h->comm_rank] * row, ncclFloat64, 0, comm, q));
        RFINV_NCCL_CHECK(api, api->Send(d.vs_model, (size_t)kept[h->comm_rank] * row, ncclFloat64, 0, comm, q));
        RFINV_NCCL_CHECK(api, api->GroupEnd());
      }
    }
  }
  if (s->record && h->comm_rank == 0) {
    const int st = rfinv_pt_fix_assigned_bins(h);
    if (st != RFINV_OK) return st;
  }
  if (d.dg_on) {
    // convergence diagnostics: every process's per-rank rows (computed from its own trace) and round-trip counters go to
    // process 0 in process order, i.e. global rank order; the trace itself stays where it is
    const size_t row = (size_t)d.dg_nq * PT_DG_ROW, G = d.G;
    double* rows = nullptr;
    unsigned long long* trips = d.dg_trips;
    if (h->comm_rank == 0) {
      cudaFree(s->dg_job_rows); cudaFree(s->dg_job_trips);
      RFINV_CUDA_CHECK(cudaMalloc((void**)&s->dg_job_rows, sizeof(double) * row * d.nproc_total));
      RFINV_CUDA_CHECK(cudaMalloc((void**)&s->dg_job_trips, sizeof(unsigned long long) * 2 * d.nproc_total));
      rows = s->dg_job_rows;
      trips = s->dg_job_trips;
      RFINV_CUDA_CHECK(cudaMemcpyAsync(trips, d.dg_trips, sizeof(unsigned long long) * 2 * G, cudaMemcpyDeviceToDevice, q));
    } else {
      RFINV_CUDA_CHECK(cudaMalloc((void**)&rows, sizeof(double) * row * G));
    }
    int st = rfinv_pt_diag_rows(h, rows);
    if (st == RFINV_OK) {
      RFINV_NCCL_CHECK(api, api->GroupStart());
      if (h->comm_rank == 0) {
        for (int r = 1; r < h->comm_world; ++r) {
          RFINV_NCCL_CHECK(api, api->Recv(rows + (size_t)r * G * row, G * row, ncclFloat64, r, comm, q));
          RFINV_NCCL_CHECK(api, api->Recv(trips + (size_t)r * G * 2, G * 2, ncclUint64, r, comm, q));
        }
      } else {
        RFINV_NCCL_CHECK(api, api->Send(rows, G * row, ncclFloat64, 0, comm, q));
        RFINV_NCCL_CHECK(api, api->Send(d.dg_trips, G * 2, ncclUint64, 0, comm, q));
      }
      RFINV_NCCL_CHECK(api, api->GroupEnd());
    }
    if (h->comm_rank != 0) {
      const cudaError_t e = cudaStreamSynchronize(q);
      cudaFree(rows);
      if (st == RFINV_OK && e != cudaSuccess) { rfinv_set_error("rfinv_pt_reduce_outputs: %s", cudaGetErrorString(e)); st = RFINV_ERR_CUDA; }
    }
    if (st != RFINV_OK) return st;
  }
  RFINV_CUDA_CHECK(cudaStreamSynchronize(q));
  return RFINV_OK;
}

}  // extern "C"
