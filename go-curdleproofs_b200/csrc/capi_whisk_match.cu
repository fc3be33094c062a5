// Whisk tracker matching: cdl_whisk_match_trackers and the engine stage behind it (kernels in k_match.cu).
#include <cstring>
#include <mutex>
#include <vector>

#include "host/engine.hpp"

using cdlh::Engine;
using cdlh::engine_of;
using cdlh::Fr;

namespace {

// Keys from which the per-tracker tables beat the shared-scalar schedule (k_match.cu): the crossover measured
// on a B200 with T = 8 192 trackers by tools/match_trackers.py (profiles/r4_match_trackers.txt)
constexpr uint32_t kMatchTableMinKeys = 256;

static_assert(CDL_WHISK_MATCH_MAX == (1u << 24), "documented limit of cdl_whisk_match_trackers");

const uint8_t kInfEnc[48] = {0xc0};  // compressed point at infinity

}  // namespace

// Device scratch of the table path for one tile of trackers: the tables, then the window bases (Jacobian and
// affine).  Grow-only and kept by the engine, like the pool; false if it cannot be had.
bool Engine::match_scratch(uint32_t tile) {
  constexpr size_t W = cdl::fb_windows(cdl::kMatchC);
  return d_match_.grow(cdl::fixed_table_bytes<cdl::kMatchC>(tile) + tile * W * (sizeof(cdl::G1Jac) + sizeof(cdl::G1Affine)),
                       ctx_->stream);
}

int32_t Engine::match_trackers(uint32_t T, const Fr* ks, uint32_t V, int32_t* owner) {
  int32_t rc;
  if ((rc = reserve(s_sc_, (size_t)V * sizeof(Fr))) || (rc = reserve(s_out_, (size_t)T * 4))) return rc;
  const uint32_t tile = T < cdl::kMatchTile ? T : cdl::kMatchTile;
  // without room for the tables the shared-scalar path gives the same owners
  const bool tables = V >= kMatchTableMinKeys && match_scratch(tile);
  constexpr uint32_t W = cdl::fb_windows(cdl::kMatchC);
  cdl::G1Affine* tab = (cdl::G1Affine*)d_match_.d();
  cdl::G1Jac* wjac = (cdl::G1Jac*)((char*)d_match_.d() + cdl::fixed_table_bytes<cdl::kMatchC>(tile));
  cdl::G1Affine* wbase = (cdl::G1Affine*)(wjac + (size_t)tile * W);
  memcpy(s_sc_.h(), ks, (size_t)V * sizeof(Fr));
  cdl::Fr* d_ks = (cdl::Fr*)s_sc_.d();
  int32_t* d_owner = (int32_t*)s_out_.d();
  const cdl::G1Affine* rg = d_pool();
  const cdl::G1Affine* krg = d_pool() + T;
  CDL_CUDA(ctx_, cudaMemcpyAsync(d_ks, s_sc_.h(), (size_t)V * sizeof(Fr), cudaMemcpyHostToDevice, ctx_->stream));
  tick();
  cdl::launch_match_prep(d_ks, V, d_owner, T, ctx_->stream);
  uint64_t kernels = 1;
  if (tables) {
    for (uint32_t t0 = 0; t0 < T; t0 += cdl::kMatchTile) {
      const uint32_t nt = T - t0 < cdl::kMatchTile ? T - t0 : cdl::kMatchTile;
      cdl::launch_match_windows(rg + t0, nt, wjac, ctx_->stream);
      cdl::launch_jac_to_affine(wjac, wbase, (int)(nt * W), ctx_->stream);
      cdl::launch_fixed_build<cdl::kMatchC>(wbase, nt, tab, ctx_->stream);
      cdl::launch_match_table(tab, krg, t0, nt, d_ks, V, d_owner, ctx_->stream);
      kernels += 4;
    }
  } else {
    cdl::launch_match_shared(rg, krg, T, d_ks, V, d_owner, ctx_->stream);
    kernels += 1;
  }
  // §8d: 3193 modmul per scalar multiplication, one per (key, tracker) pair; both points of every tracker,
  // every key and every owner word cross the device once
  tock(1, 3193.0 * T * (double)V, 196.0 * T + 32.0 * V);
  launches += kernels - 1;  // tock counted one
  CDL_CUDA(ctx_, cudaGetLastError());
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_out_.h(), d_owner, (size_t)T * 4, cudaMemcpyDeviceToHost, ctx_->stream));
  CDL_CUDA(ctx_, ctx_->sync_stream());
  finish_timing();
  memcpy(owner, s_out_.h(), (size_t)T * 4);
  return CDL_OK;
}

extern "C" {

int32_t cdl_whisk_match_trackers(cdl_ctx* c, size_t T, const uint8_t* trackers, size_t V, const cdl_fr* ks,
                                 int32_t* owner, int32_t* status) {
  if (!c || !trackers || !ks || !owner || !status || T == 0 || V == 0) return CDL_ERR_INVALID_ARG;
  if (T > CDL_WHISK_MATCH_MAX || V > CDL_WHISK_MATCH_MAX) {
    std::lock_guard<std::mutex> lk(c->mu);
    return c->fail(CDL_ERR_TOO_LARGE, "whisk_match_trackers: %zu trackers x %zu keys exceed 2^24", T, V);
  }
  // every slot matches its own block of trackers against all keys; blocks start on table tiles
  if (cdlh::slots_for(c, T) > 1)
    return cdlh::run_split(c, T, [&](cdl_ctx* lane, size_t lo, size_t hi) {
      return cdl_whisk_match_trackers(lane, hi - lo, trackers + 96 * lo, V, ks, owner + lo, status + lo);
    }, false, cdl::kMatchTile);
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  Engine* E = engine_of(c);
  int32_t rc;
  if ((rc = E->ensure_pool(2 * T))) return rc;
  // tracker.getPoints() (curve + subgroup checks): rG_t to pool[t], krG_t to pool[T + t]
  std::vector<uint32_t> dst(2 * T);
  for (size_t t = 0; t < T; t++) { dst[2 * t] = (uint32_t)t; dst[2 * t + 1] = (uint32_t)(T + t); }
  std::vector<uint8_t> st;
  if ((rc = E->decompress(trackers, dst, st))) return rc;
  if ((rc = E->match_trackers((uint32_t)T, reinterpret_cast<const Fr*>(ks), (uint32_t)V, owner))) return rc;
  for (size_t t = 0; t < T; t++) {
    if (st[2 * t] || st[2 * t + 1]) status[t] = CDL_ERR_DECODE;
    else if (memcmp(trackers + 96 * t, kInfEnc, 48) == 0) status[t] = CDL_ERR_PROTOCOL;  // identifies nobody
    else status[t] = CDL_OK;
    if (status[t] != CDL_OK || owner[t] == INT32_MAX) owner[t] = -1;
  }
  return CDL_OK;
}

}  // extern "C"
