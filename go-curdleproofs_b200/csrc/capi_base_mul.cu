// Batched fixed-base scalar multiplication: cdl_g1_batch_scalar_mul_base and the engine stage behind it
// (kernels in k_base_mul.cu).
#include <algorithm>
#include <cstring>
#include <mutex>

#include "host/engine.hpp"

using cdlh::Engine;
using cdlh::engine_of;
using cdlh::Fr;

namespace {

// Scalars from which a base without a cached table gets one: below, the GLV path's n scalar multiplications
// take less time than building the table and running the table path (cold table path).  The crossover measured
// on a B200 by tools/base_mul.py (profiles/r8_base_mul.txt).
constexpr size_t kBaseTableMinScalars = 32768;
// Scalars per device slot from which a call is split over the slots of a multi-device context:
// max(1, min(D, n / kBaseSlotScalars)) slots, each running its block on its lane 0's engine.  Equal to
// kBaseTableMinScalars, so that a fresh base takes the table path on every slot exactly when the one-device
// call would.  Derived, not tuned: the split's cost and gain have not been measured.
constexpr size_t kBaseSlotScalars = 32768;
// Scalars per round trip through the pinned staging: 32 MB of scalars and up to 144 MB of results
constexpr size_t kBaseMulChunk = (size_t)1 << 20;

static_assert(CDL_BASE_MUL_MAX == (1u << 24), "documented limit of cdl_g1_batch_scalar_mul_base");
static_assert(kBaseTableMinScalars <= kBaseMulChunk, "the GLV path runs in one chunk");
static_assert(kBaseSlotScalars >= kBaseTableMinScalars, "a split call's blocks take the table path as the whole call would");

const uint8_t kInfEnc[48] = {0xc0};  // compressed point at infinity

// the layout of the device scratch s_base_: the base, the check status, the window bases (Jacobian, then
// affine), then the n copies of the base of the GLV path
constexpr size_t kOffStatus = sizeof(cdl::G1Affine);
constexpr size_t kOffWjac = 128;
constexpr size_t kOffWaff = kOffWjac + cdl::kFbW * sizeof(cdl::G1Jac);
constexpr size_t kOffCopies = kOffWaff + cdl::kFbW * sizeof(cdl::G1Affine);

}  // namespace

size_t cdlh::base_mul_min_block(size_t per_unit) { return (kBaseSlotScalars + per_unit - 1) / per_unit; }

int32_t Engine::base_mul(const cdl_g1_affine& base, const Fr* sc, size_t n, cdl_g1_affine* out, uint8_t* out48) {
  // the cached table of this base, if any
  BaseTable* hit = nullptr;
  for (BaseTable& b : base_tabs_)
    if (memcmp(&b.base, &base, sizeof base) == 0) hit = &b;
  const bool table = hit || n >= kBaseTableMinScalars;
  const bool build = table && !hit;
  const size_t m0 = std::min(n, kBaseMulChunk);
  int32_t rc;
  if ((rc = reserve(s_sc_, m0 * sizeof(Fr))) || ((out || !table) && (rc = reserve(s_out_, m0 * sizeof(cdl::G1Affine)))) ||
      (out48 && (rc = reserve(s_enc_, m0 * 48))) ||
      (rc = reserve(s_base_, kOffCopies + (table ? 0 : m0 * sizeof(cdl::G1Affine)))))
    return rc;
  cdl::G1Affine* tab = hit ? hit->tab : nullptr;
  if (build) {
    if (base_tabs_.size() == kBaseTables) {  // replace the least recently used table
      auto lru = std::min_element(base_tabs_.begin(), base_tabs_.end(),
                                  [](const BaseTable& a, const BaseTable& b) { return a.used < b.used; });
      cudaFree(lru->tab);
      base_tabs_.erase(lru);
    }
    if (cudaMalloc(&tab, cdl::fixed_table_bytes(1)) != cudaSuccess) {
      cudaGetLastError();
      return ctx_->fail(CDL_ERR_CUDA, "batch_scalar_mul_base: table allocation of %zu bytes failed",
                        cdl::fixed_table_bytes(1));
    }
  }
  char* d_scr = (char*)s_base_.d();
  const cdl::G1Affine* d_base = (const cdl::G1Affine*)d_scr;
  uint32_t* d_status = (uint32_t*)(d_scr + kOffStatus);
  cdl::G1Jac* wjac = (cdl::G1Jac*)(d_scr + kOffWjac);
  cdl::G1Affine* waff = (cdl::G1Affine*)(d_scr + kOffWaff);
  cdl::G1Affine* copies = (cdl::G1Affine*)(d_scr + kOffCopies);
  cdl::Fr* d_sc = (cdl::Fr*)s_sc_.d();
  cdl::G1Affine* d_out = (cdl::G1Affine*)s_out_.d();
  uint8_t* d_enc = (uint8_t*)s_enc_.d();
  const bool check = !hit;  // a cached table's base passed the check when its table was built
  memcpy(s_base_.h(), &base, sizeof base);
  uint32_t status = 0;
  for (size_t c0 = 0; c0 < n; c0 += kBaseMulChunk) {
    const size_t m = std::min(n - c0, kBaseMulChunk);
    const bool first = c0 == 0;
    memcpy(s_sc_.h(), sc + c0, m * sizeof(Fr));
    if (first) CDL_CUDA(ctx_, cudaMemcpyAsync(s_base_.d(), s_base_.h(), sizeof base, cudaMemcpyHostToDevice, ctx_->stream));
    CDL_CUDA(ctx_, cudaMemcpyAsync(d_sc, s_sc_.h(), m * sizeof(Fr), cudaMemcpyHostToDevice, ctx_->stream));
    tick();
    uint64_t kernels = 0;
    double bytes = 32.0 * m + (out ? 96.0 * m : 0.0) + (out48 ? 48.0 * m : 0.0);
    if (first && check) {
      cdl::launch_base_prep(d_base, d_status, build ? wjac : nullptr, ctx_->stream);
      kernels++;
    }
    if (first && build) {
      cdl::launch_jac_to_affine(wjac, waff, cdl::kFbW, ctx_->stream);
      cdl::launch_fixed_build<cdl::kFbC, true, cdl::kBaseSeg>(waff, 1, tab, ctx_->stream);
      kernels += 2;
      bytes += (double)cdl::fixed_table_bytes(1);
    }
    if (table) {
      cdl::launch_base_mul(tab, d_sc, (uint32_t)m, out ? d_out : nullptr, out48 ? d_enc : nullptr, ctx_->stream);
      kernels++;
    } else {
      cdl::launch_base_fill(d_base, copies, (uint32_t)m, ctx_->stream);
      cdl::launch_scalar_mul(copies, d_sc, 1, nullptr, d_out, (int)m, ctx_->stream);
      kernels += 2;
      if (out48) {
        cdl::launch_compress(d_out, d_enc, (int)m, ctx_->stream);
        kernels++;
      }
    }
    // §8d: 3193 modmul per scalar multiplication, whichever path runs
    tock(1, 3193.0 * (double)m, bytes);
    launches += kernels - 1;  // tock counted one
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && first && check)
      e = cudaMemcpyAsync((char*)s_base_.h() + kOffStatus, d_status, 4, cudaMemcpyDeviceToHost, ctx_->stream);
    if (e == cudaSuccess && out) e = cudaMemcpyAsync(s_out_.h(), d_out, m * sizeof(cdl::G1Affine), cudaMemcpyDeviceToHost, ctx_->stream);
    if (e == cudaSuccess && out48) e = cudaMemcpyAsync(s_enc_.h(), d_enc, m * 48, cudaMemcpyDeviceToHost, ctx_->stream);
    if (e == cudaSuccess) e = ctx_->sync_stream();
    finish_timing();
    if (e == cudaSuccess && first && check) memcpy(&status, (char*)s_base_.h() + kOffStatus, 4);
    if (e != cudaSuccess || status) {
      if (build) cudaFree(tab);
      if (e != cudaSuccess)
        return ctx_->fail(CDL_ERR_CUDA, "batch_scalar_mul_base: %s", cudaGetErrorString(e));
      static const char* const why[] = {"", "a coordinate is not a canonical field element", "it is not on the curve",
                                        "it is not in G1"};
      return ctx_->fail(CDL_ERR_INVALID_ARG, "batch_scalar_mul_base: base rejected: %s", why[status < 4 ? status : 0]);
    }
    if (first && build) {
      base_tabs_.push_back(BaseTable{base, tab, 0});
      hit = &base_tabs_.back();
    }
    if (out) memcpy(out + c0, s_out_.h(), m * sizeof(cdl::G1Affine));
    if (out48) memcpy(out48 + 48 * c0, s_enc_.h(), m * 48);
  }
  if (hit) hit->used = ++base_clock_;
  return CDL_OK;
}

extern "C" {

int32_t cdl_g1_batch_scalar_mul_base(cdl_ctx* c, const cdl_g1_affine* base, const cdl_fr* scalars, size_t n,
                                     cdl_g1_affine* out, uint8_t* out48) {
  if (!c || (n && (!base || !scalars || (!out && !out48)))) return CDL_ERR_INVALID_ARG;
  if (n > CDL_BASE_MUL_MAX) {
    std::lock_guard<std::mutex> lk(c->mu);
    return c->fail(CDL_ERR_TOO_LARGE, "batch_scalar_mul_base: %zu scalars exceed 2^24", n);
  }
  if (n == 0) return CDL_OK;
  const cdl_g1_affine zero = {};
  if (memcmp(base, &zero, sizeof zero) == 0) {  // the point at infinity: every product is infinity
    if (out) memset(out, 0, n * sizeof *out);
    if (out48)
      for (size_t i = 0; i < n; i++) memcpy(out48 + 48 * i, kInfEnc, 48);
    return CDL_OK;
  }
  // every slot in use multiplies its own block of scalars with its own engine's tables (disjoint outputs)
  if (cdlh::slots_for(c, n, kBaseSlotScalars) > 1)
    return cdlh::run_split(c, n, [&](cdl_ctx* lane, size_t lo, size_t hi) {
      return cdl_g1_batch_scalar_mul_base(lane, base, scalars + lo, hi - lo, out ? out + lo : nullptr,
                                          out48 ? out48 + 48 * lo : nullptr);
    }, false, 1, kBaseSlotScalars);
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  return engine_of(c)->base_mul(*base, reinterpret_cast<const Fr*>(scalars), n, out, out48);
}

}  // extern "C"
