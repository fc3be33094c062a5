// Library context: a CUDA device, one stream, grow-only device scratch buffers.
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdio>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/curdle_b200.h"
#include "scratch.cuh"

struct cdl_ctx {
  int device = 0;
  int sm_count = 0;
  int clock_khz = 0;
  std::string name;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t ev_sync = nullptr;  // cudaEventBlockingSync: waiting host threads sleep instead of spinning
  // Wait for everything queued on the stream.  Lanes and ranks share the host cores with the
  // Fiat-Shamir work, so a waiting thread must not burn one (cudaStreamSynchronize spins).
  // A call that serves one proof at a time is a chain of ~50 dependent stages: there the wake-up latency of
  // a sleeping wait (tens of microseconds per stage) is on the critical path and the thread spins instead.
  bool spin_wait = false;
  cudaError_t sync_stream() {
    if (spin_wait) return cudaStreamSynchronize(stream);
    if (!ev_sync && cudaEventCreateWithFlags(&ev_sync, cudaEventBlockingSync | cudaEventDisableTiming) != cudaSuccess)
      return cudaStreamSynchronize(stream);
    cudaError_t e = cudaEventRecord(ev_sync, stream);
    if (e != cudaSuccess) return e;
    return cudaEventSynchronize(ev_sync);
  }
  std::mutex mu;
  std::string err;
  void* engine = nullptr;  // cdlh::Engine, created on first protocol-level call
  // multi-GPU communicator (capi_msm.cu): NCCL is dlopen'ed on first use
  void* nccl_comm = nullptr;
  int comm_rank = 0, comm_world = 1;
  int msm_c_override = 0;  // CDL_MSM_C / cdl_set_msm_window: 0 = pick by size
  int fixed_min_batch = -1;  // cdl_set_fixed_base_min_batch: instances per (lane) call from which the CRS fixed-base tables are used; -1 = CDL_FIXED_BASE_MINB or 64, 0 = never
  int batch_verify_min = -1;  // cdl_set_batch_verify_min: proofs per (lane) verification from which one combined MSM checks the batch first; -1 = default, 0 = never
  int msm_ba_override = -1;  // cdl_set_msm_batch_affine: batch-affine rounds of the large MSM, -1 = pick by bucket load
  // Batched protocol calls are cut into up to n_lanes sub-batches that advance
  // concurrently, each on its own lane context (own stream, engine, staging): one
  // lane's host-side Fiat-Shamir work overlaps the other lanes' kernels, and their
  // latency-bound kernels overlap each other.  A root context has one device slot per
  // entry of its device list (cdl_create_devices); every slot has its own lanes on its
  // device, and slot 0 is the root context's own device.
  struct Slot {
    int device = 0;
    cudaEvent_t base_ev = nullptr;  // origin of the slot's kernel-interval timeline (busy-time accounting)
    std::vector<cdl_ctx*> lanes;
  };
  cdl_ctx* parent = nullptr;
  std::vector<Slot> slots;       // root only
  size_t dev_slot = 0;           // lanes: the slot of root()->slots they belong to
  int n_lanes = 4;               // CDL_LANES / cdl_set_lanes: lanes per slot
  cdl_ctx* root() { return parent ? parent : this; }
  // device scratch of the host-pointer calls (capi.cu, capi_msm.cu), freed with the context
  DeviceScratch in;           // first input
  DeviceScratch in2;          // second input, or the scalars
  DeviceScratch addend;
  DeviceScratch status;       // per-point decode status
  DeviceScratch out;
  DeviceScratch partials;     // the sharded MSM's per-rank partial sums
  DeviceScratch msm_scratch;  // the large MSM's working memory
  int32_t fail(int32_t code, const char* fmt, ...) {
    char tmp[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(tmp, sizeof tmp, fmt, ap);
    va_end(ap);
    err = tmp;
    return code;
  }
};

// On failure the error is also taken off the thread's last-error slot: a call made after this one checks
// cudaGetLastError() after its launches and must not report this call's error (a sticky error still fails it).
#define CDL_CUDA(ctx, call)                                                                     \
  do {                                                                                          \
    cudaError_t e__ = (call);                                                                   \
    if (e__ != cudaSuccess) {                                                                   \
      cudaGetLastError();                                                                       \
      return (ctx)->fail(CDL_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                         __FILE__, __LINE__);                                                   \
    }                                                                                           \
  } while (0)
