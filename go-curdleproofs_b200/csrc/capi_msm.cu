// C ABI of the large-MSM path (include/curdle_b200.h, "large MSM / multi-GPU"):
// host- and device-pointer forms of (*G1Jac).MultiExp for one big MSM, raw device
// buffers so that point vectors can stay resident in HBM between calls, and the
// window-partitioned multi-GPU form whose only exchange is an NCCL all-gather of
// one partial sum per rank.  NCCL is bound at run time (dlopen), so the library
// loads on hosts without it.
#include <dlfcn.h>
#if __has_include(<nccl.h>)
#include <nccl.h>
#else
// the five entry points used below, declared locally (NCCL's ABI: 128-byte unique id, opaque
// communicator, ncclChar = 0, ncclSuccess = 0); the library itself is bound with dlopen
#include <cuda_runtime.h>
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef enum { ncclSuccess = 0 } ncclResult_t;
typedef enum { ncclChar = 0 } ncclDataType_t;
#endif

#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "../../include/curdle_b200.h"
#include "context.cuh"
#include "host/engine.hpp"
#include "launch.h"

using namespace cdl;

namespace {

struct NcclApi {
  void* h = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string err;
};

NcclApi* nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    // RTLD_NOLOAD first: reuse the copy the host process already mapped (e.g. torch's bundled NCCL)
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      api.h = dlopen(nm, RTLD_NOW | RTLD_NOLOAD);
      if (api.h) break;
    }
    if (!api.h) {
      const char* env = getenv("CDL_NCCL_LIB");
      if (env) api.h = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
      for (const char* nm : names) {
        if (api.h) break;
        api.h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      }
    }
    if (!api.h) {
      api.err = "libnccl.so.2 not found (set CDL_NCCL_LIB)";
      return;
    }
    api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.h, "ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.h, "ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.h, "ncclCommDestroy");
    api.AllGather = (decltype(api.AllGather))dlsym(api.h, "ncclAllGather");
    api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.h, "ncclGetErrorString");
    if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllGather || !api.GetErrorString)
      api.err = "libnccl is missing a required symbol";
  });
  return &api;
}

// Terms per device slot from which cdl_g1_msm of host vectors is split by points over the slots of a
// multi-device context: max(1, min(D, n / kMsmSlotTerms)) slots.  Derived from the one-GPU sweep
// (profiles/r3_msm_sweep_1gpu.txt: 1.84 ms at 2^16 terms, 2.24 ms at 2^17), so that each block of a split call
// is still an MSM the Pippenger path runs near its best per-term rate.  Derived, not tuned: the split's own
// cost (the partials' round trip and k_big_combine) and its gain have not been measured.
constexpr size_t kMsmSlotTerms = 65536;

// the window width and batch-affine rounds of the root context (a lane's MSM follows its root's settings)
int pick_c(cdl_ctx* c, size_t n) {
  const int o = c->root()->msm_c_override;
  if (o >= 2 && o <= 18) return o;
  return big_msm_pick_c(n);
}

// partial (or whole) MSM on device buffers; result left in d_out (device), not synchronised
int32_t big_msm_on_device(cdl_ctx* c, const G1Affine* d_pts, const Fr* d_sc, size_t n, uint32_t part, uint32_t parts,
                          int normalize, G1Jac* d_out) {
  if (n >= ((size_t)1 << 30)) return c->fail(CDL_ERR_TOO_LARGE, "msm: %zu terms exceed 2^30 - 1", n);
  BigMsmDims d = big_msm_dims(n, pick_c(c, n), (int)part, (int)parts, c->root()->msm_ba_override);
  // the batch-affine rounds keep two generations of pair sums and the prefix products (~ 100 B per
  // sorted entry): beyond this budget the XYZZ-only path (36 B per entry less) runs instead
  constexpr size_t kBaScratchBudget = (size_t)48 << 30;
  if (d.R > 0 && big_msm_scratch_bytes(d) > kBaScratchBudget) d = big_msm_dims(n, d.c, (int)part, (int)parts, 0);
  // bucket counts, scan prefixes and entry offsets are 32-bit: 2 * n * (windows owned) entries must fit
  if (big_msm_entries(d) >= ((uint64_t)1 << 32))
    return c->fail(CDL_ERR_TOO_LARGE, "msm: %zu terms x %d windows exceed 2^32 - 1 sorted entries; use more ranks or a wider window",
                   n, d.nlocal);
  if (!c->msm_scratch.grow(big_msm_scratch_bytes(d), c->stream))
    return c->fail(CDL_ERR_CUDA, "msm scratch allocation of %zu bytes failed", big_msm_scratch_bytes(d));
  cudaError_t e = launch_big_msm(d_pts, d_sc, d, normalize, c->msm_scratch.d(), c->sm_count, d_out, c->stream);
  if (e != cudaSuccess) return c->fail(CDL_ERR_CUDA, "large-MSM launch failed: %s", cudaGetErrorString(e));
  return CDL_OK;
}

// An MSM of host vectors: the points and scalars go to the context's input buffers, `msm(d_pts, d_sc, d_out)`
// leaves the result in its output buffer, and that G1Jac is downloaded to `out`.  Caller holds the context mutex.
template <class Msm>
int32_t msm_of_host_vectors(cdl_ctx* c, const cdl_g1_affine* points, const cdl_fr* scalars, size_t n, cdl_g1_jac* out,
                            Msm&& msm) {
  if (!c->in.grow(n * sizeof(G1Affine), c->stream) || !c->in2.grow(n * sizeof(Fr), c->stream) ||
      !c->out.grow(sizeof(G1Jac), c->stream))
    return c->fail(CDL_ERR_CUDA, "device allocation failed");
  CDL_CUDA(c, cudaMemcpyAsync(c->in.d(), points, n * sizeof(G1Affine), cudaMemcpyHostToDevice, c->stream));
  CDL_CUDA(c, cudaMemcpyAsync(c->in2.d(), scalars, n * sizeof(Fr), cudaMemcpyHostToDevice, c->stream));
  int32_t rc = msm((const G1Affine*)c->in.d(), (const Fr*)c->in2.d(), (G1Jac*)c->out.d());
  if (rc) return rc;
  CDL_CUDA(c, cudaMemcpyAsync(out, c->out.d(), sizeof(G1Jac), cudaMemcpyDeviceToHost, c->stream));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  return CDL_OK;
}

// The MSM of host vectors on a root context of several slots, split by points: slot s of the D slots in use
// sums its block shard_bounds(n, D, s) on lane (s, 0) (own input buffers, scratch and stream, nothing
// normalised), and the D partial sums (144 bytes each, through the host) are added and normalised by
// k_big_combine on the root stream.  The root's mutex is held across the pieces and the combine.
int32_t big_msm_split(cdl_ctx* c, const cdl_g1_affine* points, const cdl_fr* scalars, size_t n, size_t D,
                      cdl_g1_jac* out) {
  std::lock_guard<std::mutex> lk(c->mu);
  // the whole call's limit, before any input is read (the per-device limits apply to every block)
  if (n >= ((size_t)1 << 30)) return c->fail(CDL_ERR_TOO_LARGE, "msm: %zu terms exceed 2^30 - 1", n);
  std::vector<cdl_g1_jac> part(D);
  int32_t rc = cdlh::run_split_locked(c, n, [&](cdl_ctx* l, size_t lo, size_t hi) -> int32_t {
    // l's buffers and stream without l's own mutex: every use of a lane happens under its root's mutex, held here
    CDL_CUDA(l, cudaSetDevice(l->device));
    return msm_of_host_vectors(l, points + lo, scalars + lo, hi - lo, &part[l->dev_slot],
                               [&](const G1Affine* d_pts, const Fr* d_sc, G1Jac* d_out) {
                                 return big_msm_on_device(l, d_pts, d_sc, hi - lo, 0, 1, 0, d_out);
                               });
  }, false, 1, kMsmSlotTerms);
  if (rc) return rc;
  CDL_CUDA(c, cudaSetDevice(c->device));
  if (!c->partials.grow(D * sizeof(G1Jac), c->stream) || !c->out.grow(sizeof(G1Jac), c->stream))
    return c->fail(CDL_ERR_CUDA, "device allocation failed");
  cdl_g1_jac sum;
  CDL_CUDA(c, cudaMemcpyAsync(c->partials.d(), part.data(), D * sizeof(G1Jac), cudaMemcpyHostToDevice, c->stream));
  launch_big_combine((const G1Jac*)c->partials.d(), (int)D, (G1Jac*)c->out.d(), c->stream);
  CDL_CUDA(c, cudaGetLastError());
  CDL_CUDA(c, cudaMemcpyAsync(&sum, c->out.d(), sizeof(G1Jac), cudaMemcpyDeviceToHost, c->stream));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  *out = sum;
  return CDL_OK;
}

}  // namespace

// cdl_g1_msm (capi.cu) above kBigMsmThreshold terms: split over the device slots from 2 * kMsmSlotTerms terms,
// else on the context's own device and buffers
extern "C" int32_t cdl_big_msm_host_(cdl_ctx* c, const cdl_g1_affine* points, const cdl_fr* scalars, size_t n, cdl_g1_jac* out) {
  const size_t D = cdlh::slots_for(c, n, kMsmSlotTerms);
  if (D > 1) return big_msm_split(c, points, scalars, n, D, out);
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  return msm_of_host_vectors(c, points, scalars, n, out, [&](const G1Affine* d_pts, const Fr* d_sc, G1Jac* d_out) {
    return big_msm_on_device(c, d_pts, d_sc, n, 0, 1, 1, d_out);
  });
}

extern "C" {

int32_t cdl_set_msm_window(cdl_ctx* c, int32_t window_bits) {
  if (!c || window_bits < 0 || window_bits > 18 || window_bits == 1) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  c->msm_c_override = window_bits;
  return CDL_OK;
}

int32_t cdl_set_msm_batch_affine(cdl_ctx* c, int32_t rounds) {
  if (!c || rounds < -1 || rounds > kBigMaxBaRounds) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  c->msm_ba_override = rounds;
  return CDL_OK;
}

// ---- raw device buffers -------------------------------------------------
int32_t cdl_dev_alloc(cdl_ctx* c, size_t bytes, void** d_ptr) {
  if (!c || !d_ptr) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  CDL_CUDA(c, cudaMalloc(d_ptr, bytes ? bytes : 16));
  return CDL_OK;
}
int32_t cdl_dev_free(cdl_ctx* c, void* d_ptr) {
  if (!c) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  CDL_CUDA(c, cudaFree(d_ptr));
  return CDL_OK;
}
int32_t cdl_dev_upload(cdl_ctx* c, void* d_dst, const void* h_src, size_t bytes) {
  if (!c || (bytes && (!d_dst || !h_src))) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  CDL_CUDA(c, cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, c->stream));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  return CDL_OK;
}
int32_t cdl_dev_download(cdl_ctx* c, void* h_dst, const void* d_src, size_t bytes) {
  if (!c || (bytes && (!h_dst || !d_src))) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  CDL_CUDA(c, cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, c->stream));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  return CDL_OK;
}

// out[i] = s[i*stride] * in[i] on device buffers (in-place allowed)
int32_t cdl_g1_scalar_mul_affine_device(cdl_ctx* c, const cdl_g1_affine* d_in, const cdl_fr* d_s, size_t n,
                                        size_t scalar_stride, cdl_g1_affine* d_out) {
  if (!c || (n && (!d_in || !d_s || !d_out)) || scalar_stride > 1 || n >= ((size_t)1 << 31)) return CDL_ERR_INVALID_ARG;
  if (!n) return CDL_OK;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  launch_scalar_mul((const G1Affine*)d_in, (const Fr*)d_s, (int)scalar_stride, nullptr, (G1Affine*)d_out, (int)n, c->stream);
  CDL_CUDA(c, cudaGetLastError());
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  return CDL_OK;
}

// L[i] += x * R[i] on device vectors (innerproductargument.go:155-166 with the bases resident in HBM)
int32_t cdl_g1_fold_device(cdl_ctx* c, cdl_g1_affine* d_L, const cdl_g1_affine* d_R, const cdl_fr* d_x, size_t n) {
  if (!c || (n && (!d_L || !d_R || !d_x)) || n >= ((size_t)1 << 31)) return CDL_ERR_INVALID_ARG;
  if (!n) return CDL_OK;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  launch_scalar_mul((const G1Affine*)d_R, (const Fr*)d_x, 0, (const G1Affine*)d_L, (G1Affine*)d_L, (int)n, c->stream);
  CDL_CUDA(c, cudaGetLastError());
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  return CDL_OK;
}

int32_t cdl_g1_msm_device(cdl_ctx* c, const cdl_g1_affine* d_points, const cdl_fr* d_scalars, size_t n,
                          uint32_t part_index, uint32_t part_count, int32_t normalize, cdl_g1_jac* d_out,
                          float* kernel_ms) {
  if (!c || !d_out || part_count == 0 || part_index >= part_count || (n && (!d_points || !d_scalars)))
    return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  CDL_CUDA(c, cudaEventRecord(c->ev0, c->stream));
  int32_t rc = big_msm_on_device(c, (const G1Affine*)d_points, (const Fr*)d_scalars, n, part_index, part_count,
                                 normalize, (G1Jac*)d_out);
  if (rc) return rc;
  CDL_CUDA(c, cudaEventRecord(c->ev1, c->stream));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  CDL_CUDA(c, cudaGetLastError());
  if (kernel_ms) cudaEventElapsedTime(kernel_ms, c->ev0, c->ev1);
  return CDL_OK;
}

// ---- multi-GPU ------------------------------------------------------------
int32_t cdl_comm_unique_id(uint8_t* id128) {
  if (!id128) return CDL_ERR_INVALID_ARG;
  NcclApi* a = nccl_api();
  if (!a->err.empty()) return CDL_ERR_NO_DEVICE;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  ncclUniqueId id;
  if (a->GetUniqueId(&id) != ncclSuccess) return CDL_ERR_CUDA;
  memcpy(id128, &id, 128);
  return CDL_OK;
}

int32_t cdl_comm_init(cdl_ctx* c, const uint8_t* id128, int32_t rank, int32_t world) {
  if (!c || !id128 || world < 1 || rank < 0 || rank >= world) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  // the sharded MSM runs one process (one single-device context) per GPU
  if (c->root()->slots.size() > 1)
    return c->fail(CDL_ERR_INVALID_ARG, "comm_init: a context with %zu device slots cannot join a communicator",
                   c->root()->slots.size());
  NcclApi* a = nccl_api();
  if (!a->err.empty()) return c->fail(CDL_ERR_NO_DEVICE, "NCCL unavailable: %s", a->err.c_str());
  CDL_CUDA(c, cudaSetDevice(c->device));
  if (c->nccl_comm) { a->CommDestroy((ncclComm_t)c->nccl_comm); c->nccl_comm = nullptr; }
  ncclUniqueId id;
  memcpy(&id, id128, 128);
  ncclComm_t comm;
  ncclResult_t r = a->CommInitRank(&comm, world, id, rank);
  if (r != ncclSuccess) return c->fail(CDL_ERR_CUDA, "ncclCommInitRank: %s", a->GetErrorString(r));
  c->nccl_comm = comm;
  c->comm_rank = rank;
  c->comm_world = world;
  return CDL_OK;
}

int32_t cdl_comm_destroy(cdl_ctx* c) {
  if (!c) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  if (c->nccl_comm) {
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    nccl_api()->CommDestroy((ncclComm_t)c->nccl_comm);
    c->nccl_comm = nullptr;
  }
  c->comm_rank = 0;
  c->comm_world = 1;
  return CDL_OK;
}

void cdl_comm_partition(size_t n, int32_t world, int32_t rank, int32_t window_bits, int32_t* first_window,
                        int32_t* window_step, int32_t* n_windows, int32_t* my_windows) {
  if (world < 1 || rank < 0 || rank >= world) {  // no partition exists: report zero windows
    if (first_window) *first_window = 0;
    if (window_step) *window_step = 0;
    if (n_windows) *n_windows = 0;
    if (my_windows) *my_windows = 0;
    return;
  }
  int c = window_bits >= 2 ? window_bits : big_msm_pick_c(n);
  BigMsmDims d = big_msm_dims(n, c, rank, world);
  if (first_window) *first_window = d.wfirst;
  if (window_step) *window_step = d.wstep;
  if (n_windows) *n_windows = d.W;
  if (my_windows) *my_windows = d.nlocal;
}

// every rank holds the full point/scalar vectors (device resident); rank r sums the
// windows r, r + world, ...; one all-gather of the partial sums; every rank gets the result
// caller holds c->mu
static int32_t msm_sharded_device_locked(cdl_ctx* c, const cdl_g1_affine* d_points, const cdl_fr* d_scalars, size_t n,
                                         cdl_g1_jac* d_out, float* kernel_ms) {
  CDL_CUDA(c, cudaSetDevice(c->device));
  const int world = c->comm_world, rank = c->comm_rank;
  if (world > 1 && !c->nccl_comm) return c->fail(CDL_ERR_INVALID_ARG, "cdl_comm_init has not been called");
  if (!c->partials.grow((size_t)(world + 1) * sizeof(G1Jac), c->stream)) return c->fail(CDL_ERR_CUDA, "device allocation failed");
  G1Jac* d_part = (G1Jac*)c->partials.d();
  CDL_CUDA(c, cudaEventRecord(c->ev0, c->stream));
  if (world == 1) {
    int32_t rc = big_msm_on_device(c, (const G1Affine*)d_points, (const Fr*)d_scalars, n, 0, 1, 1, (G1Jac*)d_out);
    if (rc) return rc;
  } else {
    G1Jac* mine = d_part + world;
    // Two ways to split one MSM over the ranks (SURVEY.md §8e).  Windows: rank r sums the windows r,
    // r + world, .. of every term (the digit passes and the sort still visit all n terms on every
    // rank).  Points: rank r runs a complete MSM over its n / world terms.  Windows are dealt while
    // every rank gets at least four of them; with fewer (W = 8 windows at c = 16: four ranks or more)
    // the per-rank fixed passes and the serial tail dominate and the points are partitioned instead.
    // Either way the exchange is one all-gather of one partial sum per rank.
    static const int forced = [] {
      const char* e = getenv("CDL_MSM_PARTITION");
      return !e ? 0 : e[0] == 'p' ? 1 : e[0] == 'w' ? 2 : 0;
    }();
    const BigMsmDims whole = big_msm_dims(n, pick_c(c, n), 0, 1);
    const bool by_points = forced ? forced == 1 : whole.W < 4 * world;
    int32_t rc;
    if (by_points) {
      const size_t lo = n * (size_t)rank / (size_t)world, hi = n * (size_t)(rank + 1) / (size_t)world;
      rc = big_msm_on_device(c, (const G1Affine*)d_points + lo, (const Fr*)d_scalars + lo, hi - lo, 0, 1, 0, mine);
    } else {
      rc = big_msm_on_device(c, (const G1Affine*)d_points, (const Fr*)d_scalars, n, (uint32_t)rank, (uint32_t)world, 0, mine);
    }
    // A rank that failed before the collective must still enter it (the others would wait for ever): it
    // contributes the point at infinity and returns its error afterwards; every size / allocation failure
    // above depends only on (n, world), so in practice all ranks fail alike.
    if (rc) cudaMemsetAsync(mine, 0, sizeof(G1Jac), c->stream);
    const int32_t local_rc = rc;
    NcclApi* a = nccl_api();
    ncclResult_t r = a->AllGather(mine, d_part, sizeof(G1Jac), ncclChar, (ncclComm_t)c->nccl_comm, c->stream);
    if (r != ncclSuccess) return c->fail(CDL_ERR_CUDA, "ncclAllGather: %s", a->GetErrorString(r));
    launch_big_combine(d_part, world, (G1Jac*)d_out, c->stream);
    if (local_rc) {
      cudaStreamSynchronize(c->stream);
      return local_rc;
    }
  }
  CDL_CUDA(c, cudaEventRecord(c->ev1, c->stream));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  CDL_CUDA(c, cudaGetLastError());
  if (kernel_ms) cudaEventElapsedTime(kernel_ms, c->ev0, c->ev1);
  return CDL_OK;
}

int32_t cdl_g1_msm_sharded_device(cdl_ctx* c, const cdl_g1_affine* d_points, const cdl_fr* d_scalars, size_t n,
                                  cdl_g1_jac* d_out, float* kernel_ms) {
  if (!c || !d_out || (n && (!d_points || !d_scalars))) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  return msm_sharded_device_locked(c, d_points, d_scalars, n, d_out, kernel_ms);
}

int32_t cdl_g1_msm_sharded(cdl_ctx* c, const cdl_g1_affine* points, const cdl_fr* scalars, size_t n, cdl_g1_jac* out) {
  if (!c || !out || (n && (!points || !scalars))) return CDL_ERR_INVALID_ARG;
  // one lock across staging, MSM and download: the staging slots belong to the context
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  return msm_of_host_vectors(c, points, scalars, n, out, [&](const G1Affine* d_pts, const Fr* d_sc, G1Jac* d_out) {
    return msm_sharded_device_locked(c, (const cdl_g1_affine*)d_pts, (const cdl_fr*)d_sc, n, (cdl_g1_jac*)d_out, nullptr);
  });
}

}  // extern "C"
