// C ABI of libcurdle_b200.so (include/curdle_b200.h): context, device buffers,
// host-pointer entry points that mirror the gnark-crypto calls of the reference.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/curdle_b200.h"
#include "context.cuh"
#include "host/engine.hpp"
#include "launch.h"

using namespace cdl;

static_assert(sizeof(Fp) == sizeof(cdl_fp), "fp layout");
static_assert(sizeof(Fr) == sizeof(cdl_fr), "fr layout");
static_assert(sizeof(G1Affine) == sizeof(cdl_g1_affine), "affine layout");
static_assert(sizeof(G1Jac) == sizeof(cdl_g1_jac), "jac layout");

// the MSM stage's tasks for offsets[0..k], result j to pool slot j; false when the offsets are not monotone
static bool msm_tasks(const uint32_t* offsets, size_t k, std::vector<MsmTask>& tasks) {
  tasks.resize(k);
  for (size_t j = 0; j < k; j++) {
    if (offsets[j + 1] < offsets[j]) return false;
    tasks[j] = MsmTask{offsets[j], offsets[j + 1] - offsets[j], (uint32_t)j, 0};
  }
  return true;
}

// Terms per device slot from which cdl_g1_msm_batch is split over the slots of a multi-device context: the value
// of kMsmSlotTerms (capi_msm.cu), not measured for this call.
constexpr size_t kMsmBatchSlotTerms = 65536;

// The MSM blocks of cdl_g1_msm_batch on c (offsets monotone): slot s of the D' = slots_for(c, terms,
// kMsmBatchSlotTerms) slots takes MSMs [cut[s], cut[s + 1]), cut at the MSM boundary nearest to the term at which
// shard_bounds(terms, D', s) starts, so the blocks balance terms, not MSMs.  Equal offsets cut before the first
// of them, and trailing empty MSMs join the last block, so every non-empty block holds terms.  Empty when fewer
// than two blocks hold terms (one MSM holding every term, a lane, a small call): the call does not split.
static std::vector<size_t> msm_batch_cuts(cdl_ctx* c, const uint32_t* offsets, size_t k) {
  const size_t first = offsets[0], terms = offsets[k] - first;
  const size_t D = cdlh::slots_for(c, terms, kMsmBatchSlotTerms);
  std::vector<size_t> cut(D + 1, k);
  cut[0] = 0;
  size_t busy = 0;
  for (size_t s = 1; s <= D; s++) {
    if (s < D) {
      const size_t t = first + cdlh::shard_lo(terms, D, s);
      const uint32_t* hi = std::lower_bound(offsets, offsets + k + 1, t);  // offsets[k] >= t
      const uint32_t v = hi > offsets && t - hi[-1] < hi[0] - t ? hi[-1] : hi[0];
      cut[s] = v == offsets[k] ? k : (size_t)(std::lower_bound(offsets, offsets + k + 1, v) - offsets);
    }
    busy += offsets[cut[s]] > offsets[cut[s - 1]];
  }
  if (busy < 2) cut.clear();
  return cut;
}

extern "C" {

uint32_t cdl_abi_version(void) { return (1u << 16) | 11u; }

void cdl_destroy(cdl_ctx* c);

int32_t cdl_create_devices(const int32_t* devices, size_t n, cdl_ctx** out) {
  if (!out) return CDL_ERR_INVALID_ARG;
  *out = nullptr;
  if (!devices || n == 0 || n > 16) return CDL_ERR_INVALID_ARG;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) return CDL_ERR_NO_DEVICE;
  for (size_t s = 0; s < n; s++)
    if (devices[s] < 0 || devices[s] >= count) return CDL_ERR_INVALID_ARG;
  const int device = devices[0];
  cdl_ctx* c = new cdl_ctx();
  c->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete c;
    return CDL_ERR_CUDA;
  }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  c->sm_count = prop.multiProcessorCount;
  c->clock_khz = prop.clockRate;
  c->name = prop.name;
  cudaEventCreate(&c->ev0);
  cudaEventCreate(&c->ev1);
  c->slots.resize(n);
  for (size_t s = 0; s < n; s++) {
    cdl_ctx::Slot& sl = c->slots[s];
    sl.device = devices[s];
    if (cudaSetDevice(sl.device) != cudaSuccess || cudaEventCreate(&sl.base_ev) != cudaSuccess) {
      cdl_destroy(c);
      return CDL_ERR_CUDA;
    }
    // slot 0's timeline starts on the root stream; the others on their device's default stream
    cudaEventRecord(sl.base_ev, s == 0 ? c->stream : 0);
    cudaEventSynchronize(sl.base_ev);
    // the small-MSM kernel stages up to ~6000 terms in shared memory (a per-device kernel attribute)
    msm_small_init();
  }
  cudaSetDevice(device);
  if (const char* e = getenv("CDL_MSM_C")) c->msm_c_override = atoi(e);
  if (const char* e = getenv("CDL_LANES")) { int v = atoi(e); if (v >= 1 && v <= 16) c->n_lanes = v; }
  *out = c;
  return CDL_OK;
}

int32_t cdl_create(int device, cdl_ctx** out) {
  const int32_t d = device;
  return cdl_create_devices(&d, 1, out);
}

int32_t cdl_context_devices(cdl_ctx* c, int32_t* devices, size_t cap, size_t* n) {
  if (!c || !n || (cap && !devices)) return CDL_ERR_INVALID_ARG;
  const std::vector<cdl_ctx::Slot>& sl = c->root()->slots;
  *n = sl.size();
  for (size_t s = 0; s < sl.size() && s < cap; s++) devices[s] = sl[s].device;
  return CDL_OK;
}

// lane context `i` of slot `slot` of a root context (created on first use; caller holds the root's mutex)
cdl_ctx* cdl_lane_(cdl_ctx* root, size_t slot, size_t i) {
  cdl_ctx::Slot& sl = root->slots[slot];
  while (sl.lanes.size() <= i) {
    cdl_ctx* l = new cdl_ctx();
    l->device = sl.device;
    l->dev_slot = slot;
    l->clock_khz = root->clock_khz;
    l->name = root->name;
    l->parent = root;
    l->n_lanes = 1;
    cudaDeviceGetAttribute(&l->sm_count, cudaDevAttrMultiProcessorCount, l->device);
    if (cudaSetDevice(l->device) != cudaSuccess ||
        cudaStreamCreateWithFlags(&l->stream, cudaStreamNonBlocking) != cudaSuccess) {
      delete l;
      return nullptr;
    }
    cudaEventCreate(&l->ev0);
    cudaEventCreate(&l->ev1);
    sl.lanes.push_back(l);
  }
  return sl.lanes[i];
}

int32_t cdl_set_lanes(cdl_ctx* c, int32_t lanes) {
  if (!c || lanes < 1 || lanes > 16) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  c->n_lanes = lanes;
  return CDL_OK;
}

void cdl_engine_free_(void* engine);  // capi_protocol.cu
int32_t cdl_big_msm_host_(cdl_ctx* c, const cdl_g1_affine* points, const cdl_fr* scalars, size_t n, cdl_g1_jac* out);  // capi_msm.cu, takes the mutex

void cdl_destroy(cdl_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cdl_comm_destroy(c);
  for (cdl_ctx::Slot& sl : c->slots) {
    for (cdl_ctx* l : sl.lanes) cdl_destroy(l);
    sl.lanes.clear();
    cudaSetDevice(sl.device);
    if (sl.base_ev) cudaEventDestroy(sl.base_ev);
  }
  cudaSetDevice(c->device);
  if (c->engine) cdl_engine_free_(c->engine);
  cudaEventDestroy(c->ev0);
  cudaEventDestroy(c->ev1);
  if (c->ev_sync) cudaEventDestroy(c->ev_sync);
  cudaStreamDestroy(c->stream);
  delete c;
}

const char* cdl_last_error(cdl_ctx* c) { return c ? c->err.c_str() : "null context"; }

int32_t cdl_device_info(cdl_ctx* c, int32_t* sm_count, int32_t* clock_khz, char* name, size_t cap) {
  if (!c) return CDL_ERR_INVALID_ARG;
  if (sm_count) *sm_count = c->sm_count;
  if (clock_khz) *clock_khz = c->clock_khz;
  if (name && cap) { strncpy(name, c->name.c_str(), cap - 1); name[cap - 1] = 0; }
  return CDL_OK;
}

// --------------------------------------------------------------------- MSM
// The batched MSMs run as one MSM stage of the context's engine (Engine::run_msm picks the kernels and
// the chunking); MSM j of a call writes its result to engine-pool slot j.
int32_t cdl_g1_msm_batch(cdl_ctx* c, const cdl_g1_affine* points, const cdl_fr* scalars,
                         const uint32_t* offsets, size_t k, cdl_g1_affine* out) {
  if (!c || !offsets || !out || (k && offsets[k] && (!points || !scalars))) return CDL_ERR_INVALID_ARG;
  if (k == 0) return CDL_OK;
  std::lock_guard<std::mutex> lk(c->mu);
  const size_t total = offsets[k];
  cdlh::MsmStage st;
  if (!msm_tasks(offsets, k, st.tasks)) return c->fail(CDL_ERR_INVALID_ARG, "msm_batch: offsets not monotone");
  // the bases go to pool slots [k, k + total); pool indices are 30 bits (bit 31 negates, bit 30 is the kernels' flag)
  if (k + total >= (1u << 30))
    return c->fail(CDL_ERR_INVALID_ARG, "msm_batch: %zu MSMs of %zu terms exceed the 2^30-point pool", k, total);
  // on several slots, whole MSMs per slot with rebased offsets (the checks above ran on the whole call)
  const std::vector<size_t> cut = msm_batch_cuts(c, offsets, k);
  if (!cut.empty())
    return cdlh::run_blocks_locked(c, cut, [&](cdl_ctx* l, size_t j0, size_t j1) {
      std::vector<uint32_t> offs(j1 - j0 + 1);
      for (size_t j = j0; j <= j1; j++) offs[j - j0] = offsets[j] - offsets[j0];
      return cdl_g1_msm_batch(l, points + offsets[j0], scalars + offsets[j0], offs.data(), j1 - j0, out + j0);
    }, false);
  CDL_CUDA(c, cudaSetDevice(c->device));
  c->spin_wait = true;  // latency regime, as for small protocol batches: see cdl_ctx::sync_stream
  cdlh::Engine* E = cdlh::engine_of(c);
  st.idx.resize(total);
  for (size_t t = 0; t < total; t++) st.idx[t] = (uint32_t)(k + t);
  st.sc.assign(reinterpret_cast<const cdlh::Fr*>(scalars), reinterpret_cast<const cdlh::Fr*>(scalars) + total);
  int32_t rc;
  if ((rc = E->ensure_pool(k + total)) || (rc = E->upload_points((uint32_t)k, points, total)) || (rc = E->run_msm(st)))
    return rc;
  return E->download_points(0, out, k);
}

// Batched MSM over a DEVICE-RESIDENT pool of bases: term t of MSM j is scalars[t] * d_pool[idx[t]]
// (bit 31 of idx[t] negates the base), t in [offsets[j], offsets[j+1]).  Indices, scalars and offsets are
// host arrays (what a Go-hosted orchestration computes between rounds); the bases - e.g. the folded
// vectors of innerproductargument.go:100-172, kept in HBM with cdl_g1_fold_device - never leave the
// device.  Result j goes to d_pool[out_slot[j]] (when out_slot != NULL; later MSMs / folds can use
// it as a base), to out[j] in gnark's affine layout (when out != NULL) and to out48 + 48*j as the
// compressed encoding the transcript hashes (when out48 != NULL).
int32_t cdl_g1_msm_batch_device(cdl_ctx* c, cdl_g1_affine* d_pool, const uint32_t* idx, const cdl_fr* scalars,
                                const uint32_t* offsets, size_t k, const uint32_t* out_slot, cdl_g1_affine* out,
                                uint8_t* out48) {
  if (!c || !d_pool || !offsets || (k && offsets[k] && (!idx || !scalars))) return CDL_ERR_INVALID_ARG;
  if (k == 0) return CDL_OK;
  std::lock_guard<std::mutex> lk(c->mu);
  const size_t total = offsets[k];
  cdlh::MsmStage st;
  if (!msm_tasks(offsets, k, st.tasks)) return c->fail(CDL_ERR_INVALID_ARG, "msm_batch_device: offsets not monotone");
  // pool indices are 30 bits: bit 31 negates, bit 30 is the kernels' own flag
  for (size_t t = 0; t < total; t++)
    if (idx[t] & 0x40000000u) return c->fail(CDL_ERR_INVALID_ARG, "msm_batch_device: pool index of term %zu exceeds 2^30 - 1", t);
  CDL_CUDA(c, cudaSetDevice(c->device));
  c->spin_wait = true;  // latency regime, as for small protocol batches: see cdl_ctx::sync_stream
  cdlh::Engine* E = cdlh::engine_of(c);
  st.idx.assign(idx, idx + total);
  st.sc.assign(reinterpret_cast<const cdlh::Fr*>(scalars), reinterpret_cast<const cdlh::Fr*>(scalars) + total);
  int32_t rc;
  if ((rc = E->ensure_pool(k)) || (rc = E->run_msm(st, nullptr, reinterpret_cast<const G1Affine*>(d_pool)))) return rc;
  if (out48) memcpy(out48, st.out48.data(), k * 48);
  if (out_slot) {  // scatter the results into their pool slots (k small copies on the stream)
    for (size_t j = 0; j < k; j++)
      CDL_CUDA(c, cudaMemcpyAsync(reinterpret_cast<G1Affine*>(d_pool) + out_slot[j], E->d_pool() + j, sizeof(G1Affine),
                                  cudaMemcpyDeviceToDevice, c->stream));
  }
  if (out) return E->download_points(0, out, k);  // its wait covers the scatter
  CDL_CUDA(c, c->sync_stream());
  return CDL_OK;
}

int32_t cdl_g1_msm(cdl_ctx* c, const cdl_g1_affine* points, const cdl_fr* scalars, size_t n, cdl_g1_jac* out) {
  if (!c || !out || (n && (!points || !scalars))) return CDL_ERR_INVALID_ARG;
  // Pippenger path (k_msm_big.cu), split over the device slots when large enough; the small-MSM kernels
  // serve Prove/Verify sizes
  if (n > kBigMsmThreshold) return cdl_big_msm_host_(c, points, scalars, n, out);
  uint32_t offs[2] = {0, (uint32_t)n};
  cdl_g1_affine a;
  int32_t rc = cdl_g1_msm_batch(c, points, scalars, offs, 1, &a);
  if (rc != CDL_OK) return rc;
  cdlh::affine_to_jac(out, a);
  return CDL_OK;
}

int32_t cdl_g1_sum_affine(cdl_ctx* c, const cdl_g1_affine* in, size_t n, cdl_g1_affine* out) {
  if (!c || !out || (n && !in)) return CDL_ERR_INVALID_ARG;
  const std::vector<cdlh::Fr> one_v(n, cdlh::FR_ONE);
  const cdl_fr* ones = reinterpret_cast<const cdl_fr*>(one_v.data());
  if (n > kBigMsmThreshold) {
    cdl_g1_jac j;
    int32_t rc = cdl_g1_msm(c, in, ones, n, &j);
    if (rc != CDL_OK) return rc;
    bool inf = true;
    for (int i = 0; i < 6; i++) inf = inf && j.z.l[i] == 0;
    if (inf) memset(out, 0, sizeof *out);
    else { out->x = j.x; out->y = j.y; }  // normalised: Z = 1
    return CDL_OK;
  }
  uint32_t offs[2] = {0, (uint32_t)n};
  return cdl_g1_msm_batch(c, in, ones, offs, 1, out);
}

// --------------------------------------------------------------------- elementwise
static int32_t scalar_mul_impl(cdl_ctx* c, const cdl_g1_affine* in, const cdl_fr* s, size_t n, size_t stride,
                               const cdl_g1_affine* addend, cdl_g1_affine* out) {
  if (n == 0) return CDL_OK;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  size_t ns = stride ? n : 1;
  if (!c->in.grow(n * sizeof(G1Affine), c->stream) || !c->in2.grow(ns * sizeof(Fr), c->stream) ||
      (addend && !c->addend.grow(n * sizeof(G1Affine), c->stream)) || !c->out.grow(n * sizeof(G1Affine), c->stream))
    return c->fail(CDL_ERR_CUDA, "device allocation failed");
  G1Affine* d_in = (G1Affine*)c->in.d();
  Fr* d_s = (Fr*)c->in2.d();
  G1Affine* d_add = addend ? (G1Affine*)c->addend.d() : nullptr;
  G1Affine* d_out = (G1Affine*)c->out.d();
  CDL_CUDA(c, cudaMemcpyAsync(d_in, in, n * sizeof(G1Affine), cudaMemcpyHostToDevice, c->stream));
  CDL_CUDA(c, cudaMemcpyAsync(d_s, s, ns * sizeof(Fr), cudaMemcpyHostToDevice, c->stream));
  if (addend) CDL_CUDA(c, cudaMemcpyAsync(d_add, addend, n * sizeof(G1Affine), cudaMemcpyHostToDevice, c->stream));
  launch_scalar_mul(d_in, d_s, stride ? 1 : 0, d_add, d_out, (int)n, c->stream);
  CDL_CUDA(c, cudaGetLastError());
  CDL_CUDA(c, cudaMemcpyAsync(out, d_out, n * sizeof(G1Affine), cudaMemcpyDeviceToHost, c->stream));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  return CDL_OK;
}

// Points per device slot from which cdl_g1_scalar_mul_affine is split over the slots of a multi-device context,
// every slot running its block on its lane 0.  Measured on one B200 (tools/primitive_sweep.py,
// profiles/r10_primitive_slot_sweep.txt): from blocks of 4 096 points, halving a call takes more kernel time off
// it than a call's fixed cost (uploads, launch, wait and download: 0.11 ms); below, the GLV kernel is latency-bound.
constexpr size_t kScalarMulSlotPoints = 4096;

int32_t cdl_g1_scalar_mul_affine(cdl_ctx* c, const cdl_g1_affine* in, const cdl_fr* s, size_t n,
                                 size_t scalar_stride, cdl_g1_affine* out) {
  if (!c || (n && (!in || !s || !out)) || scalar_stride > 1) return CDL_ERR_INVALID_ARG;
  if (cdlh::slots_for(c, n, kScalarMulSlotPoints) > 1)  // a broadcast scalar goes to every block
    return cdlh::run_split(c, n, [&](cdl_ctx* l, size_t lo, size_t hi) {
      return cdl_g1_scalar_mul_affine(l, in + lo, s + scalar_stride * lo, hi - lo, scalar_stride, out + lo);
    }, false, 1, kScalarMulSlotPoints);
  return scalar_mul_impl(c, in, s, n, scalar_stride, nullptr, out);
}

// Points per device slot from which cdl_g1_fold is split, measured as for kScalarMulSlotPoints (the same kernel
// with an addend): halving a call saves 0.004 ms of kernel time at blocks of 2 048 points and 0.29 ms at 4 096,
// against a fixed cost of 0.03 ms
constexpr size_t kFoldSlotPoints = 4096;

int32_t cdl_g1_fold(cdl_ctx* c, cdl_g1_affine* L, const cdl_g1_affine* R, const cdl_fr* x, size_t n) {
  if (!c || (n && (!L || !R || !x))) return CDL_ERR_INVALID_ARG;
  if (cdlh::slots_for(c, n, kFoldSlotPoints) > 1)
    return cdlh::run_split(c, n, [&](cdl_ctx* l, size_t lo, size_t hi) {
      return cdl_g1_fold(l, L + lo, R + lo, x, hi - lo);
    }, false, 1, kFoldSlotPoints);
  return scalar_mul_impl(c, R, x, n, 0, L, L);
}

// Points per device slot from which cdl_g1_batch_to_affine is split, measured as for kScalarMulSlotPoints: the
// kernel time halving a call saves reaches the fixed cost (0.027 ms) from blocks of 32 768 points
constexpr size_t kToAffineSlotPoints = 32768;

int32_t cdl_g1_batch_to_affine(cdl_ctx* c, const cdl_g1_jac* in, size_t n, cdl_g1_affine* out) {
  if (!c || (n && (!in || !out))) return CDL_ERR_INVALID_ARG;
  if (n == 0) return CDL_OK;
  if (cdlh::slots_for(c, n, kToAffineSlotPoints) > 1)
    return cdlh::run_split(c, n, [&](cdl_ctx* l, size_t lo, size_t hi) {
      return cdl_g1_batch_to_affine(l, in + lo, hi - lo, out + lo);
    }, false, 1, kToAffineSlotPoints);
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  if (!c->in.grow(n * sizeof(G1Jac), c->stream) || !c->out.grow(n * sizeof(G1Affine), c->stream))
    return c->fail(CDL_ERR_CUDA, "device allocation failed");
  G1Jac* d_in = (G1Jac*)c->in.d();
  G1Affine* d_out = (G1Affine*)c->out.d();
  CDL_CUDA(c, cudaMemcpyAsync(d_in, in, n * sizeof(G1Jac), cudaMemcpyHostToDevice, c->stream));
  launch_jac_to_affine(d_in, d_out, (int)n, c->stream);
  CDL_CUDA(c, cudaGetLastError());
  CDL_CUDA(c, cudaMemcpyAsync(out, d_out, n * sizeof(G1Affine), cudaMemcpyDeviceToHost, c->stream));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  return CDL_OK;
}

// --------------------------------------------------------------------- codecs
// Points per device slot from which cdl_g1_compress is split, measured as for kScalarMulSlotPoints: the kernel
// time halving a call saves reaches the fixed cost (0.019 ms) from blocks of 131 072 points
constexpr size_t kCompressSlotPoints = 131072;

int32_t cdl_g1_compress(cdl_ctx* c, const cdl_g1_affine* in, size_t n, uint8_t* out48) {
  if (!c || (n && (!in || !out48))) return CDL_ERR_INVALID_ARG;
  if (n == 0) return CDL_OK;
  if (cdlh::slots_for(c, n, kCompressSlotPoints) > 1)
    return cdlh::run_split(c, n, [&](cdl_ctx* l, size_t lo, size_t hi) {
      return cdl_g1_compress(l, in + lo, hi - lo, out48 + 48 * lo);
    }, false, 1, kCompressSlotPoints);
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  if (!c->in.grow(n * sizeof(G1Affine), c->stream) || !c->out.grow(n * 48, c->stream))
    return c->fail(CDL_ERR_CUDA, "device allocation failed");
  G1Affine* d_in = (G1Affine*)c->in.d();
  uint8_t* d_out = (uint8_t*)c->out.d();
  CDL_CUDA(c, cudaMemcpyAsync(d_in, in, n * sizeof(G1Affine), cudaMemcpyHostToDevice, c->stream));
  launch_compress(d_in, d_out, (int)n, c->stream);
  CDL_CUDA(c, cudaGetLastError());
  CDL_CUDA(c, cudaMemcpyAsync(out48, d_out, n * 48, cudaMemcpyDeviceToHost, c->stream));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  return CDL_OK;
}

// CDL_ERR_DECODE naming the first rejected point of status[0 .. n), else CDL_OK
static int32_t decode_verdict(cdl_ctx* c, const uint8_t* status, size_t n) {
  for (size_t i = 0; i < n; i++)
    if (status[i]) return c->fail(CDL_ERR_DECODE, "g1 decompress: point %zu rejected (reason %u)", i, (unsigned)status[i]);
  return CDL_OK;
}

// Points per device slot from which cdl_g1_decompress is split, measured as for kScalarMulSlotPoints: the kernel
// time halving a call saves reaches the fixed cost (0.034 ms) from blocks of 16 384 points
constexpr size_t kDecompressSlotPoints = 16384;

int32_t cdl_g1_decompress(cdl_ctx* c, const uint8_t* in48, size_t n, cdl_g1_affine* out, uint8_t* status) {
  if (!c || (n && (!in48 || !out || !status))) return CDL_ERR_INVALID_ARG;
  if (n == 0) return CDL_OK;
  std::lock_guard<std::mutex> lk(c->mu);
  if (cdlh::slots_for(c, n, kDecompressSlotPoints) > 1) {
    // every block writes all of its points and statuses; the verdict is then taken over the whole call, so that
    // it names the call's first rejected point as the one-device call does
    const int32_t rc = cdlh::run_split_locked(c, n, [&](cdl_ctx* l, size_t lo, size_t hi) {
      const int32_t r = cdl_g1_decompress(l, in48 + 48 * lo, hi - lo, out + lo, status + lo);
      return r == CDL_ERR_DECODE ? CDL_OK : r;
    }, false, 1, kDecompressSlotPoints);
    return rc ? rc : decode_verdict(c, status, n);
  }
  CDL_CUDA(c, cudaSetDevice(c->device));
  if (!c->in.grow(n * 48, c->stream) || !c->out.grow(n * sizeof(G1Affine), c->stream) || !c->status.grow(n, c->stream))
    return c->fail(CDL_ERR_CUDA, "device allocation failed");
  uint8_t* d_in = (uint8_t*)c->in.d();
  G1Affine* d_out = (G1Affine*)c->out.d();
  uint8_t* d_st = (uint8_t*)c->status.d();
  CDL_CUDA(c, cudaMemcpyAsync(d_in, in48, n * 48, cudaMemcpyHostToDevice, c->stream));
  launch_decompress(d_in, d_out, d_st, (int)n, c->stream);
  CDL_CUDA(c, cudaGetLastError());
  CDL_CUDA(c, cudaMemcpyAsync(out, d_out, n * sizeof(G1Affine), cudaMemcpyDeviceToHost, c->stream));
  CDL_CUDA(c, cudaMemcpyAsync(status, d_st, n, cudaMemcpyDeviceToHost, c->stream));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  return decode_verdict(c, status, n);
}

// --------------------------------------------------------------------- diagnostics
int32_t cdl_fp_mul(cdl_ctx* c, const cdl_fp* a, const cdl_fp* b, size_t n, cdl_fp* out) {
  if (!c || (n && (!a || !b || !out))) return CDL_ERR_INVALID_ARG;
  if (n == 0) return CDL_OK;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  if (!c->in.grow(n * sizeof(Fp), c->stream) || !c->in2.grow(n * sizeof(Fp), c->stream) || !c->out.grow(n * sizeof(Fp), c->stream))
    return c->fail(CDL_ERR_CUDA, "device allocation failed");
  Fp* d_a = (Fp*)c->in.d();
  Fp* d_b = (Fp*)c->in2.d();
  Fp* d_o = (Fp*)c->out.d();
  CDL_CUDA(c, cudaMemcpyAsync(d_a, a, n * sizeof(Fp), cudaMemcpyHostToDevice, c->stream));
  CDL_CUDA(c, cudaMemcpyAsync(d_b, b, n * sizeof(Fp), cudaMemcpyHostToDevice, c->stream));
  launch_fp_mul(d_a, d_b, d_o, (int)n, c->stream);
  CDL_CUDA(c, cudaGetLastError());
  CDL_CUDA(c, cudaMemcpyAsync(out, d_o, n * sizeof(Fp), cudaMemcpyDeviceToHost, c->stream));
  CDL_CUDA(c, cudaStreamSynchronize(c->stream));
  return CDL_OK;
}

int32_t cdl_int_peak(cdl_ctx* c, int kind, int iters, double* ops_per_s, double* ms_out) {
  return cdl_int_peak_cfg(c, kind, iters, kind >= 2 ? 2 : 8, 256, ops_per_s, ms_out);
}

int32_t cdl_int_peak_cfg(cdl_ctx* c, int kind, int iters, int blocks_per_sm, int tpb, double* ops_per_s,
                         double* ms_out) {
  if (!c || iters <= 0 || kind < 0 || kind > 4 || blocks_per_sm < 1 || blocks_per_sm > 32 || tpb < 32 || tpb > 1024)
    return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  const int blocks = c->sm_count * blocks_per_sm;
  if (!c->out.grow((size_t)blocks * tpb * sizeof(Fp), c->stream)) return c->fail(CDL_ERR_CUDA, "device allocation failed");
  void* d = c->out.d();
  float best = 1e30f;
  for (int rep = 0; rep < 4; rep++) {  // rep 0 is the warm-up
    CDL_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    launch_peak(kind, d, blocks, tpb, iters, 12345u + rep, c->stream);
    CDL_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    CDL_CUDA(c, cudaStreamSynchronize(c->stream));
    CDL_CUDA(c, cudaGetLastError());
    float ms = 0;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    if (rep > 0 && ms < best) best = ms;
  }
  double ops = (double)blocks * tpb * (double)iters * (kind == 2 ? 2.0 : kind == 3 ? 4.0 : kind == 4 ? 6.0 : 64.0);
  if (ops_per_s) *ops_per_s = ops / (best * 1e-3);
  if (ms_out) *ms_out = best;
  return CDL_OK;
}

}  // extern "C"
