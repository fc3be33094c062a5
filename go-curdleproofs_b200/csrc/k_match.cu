// Whisk tracker matching: which of V secrets k_v owns which of T trackers (rG_t, krG_t), i.e. for which
// pairs k_v * rG_t == krG_t.  Every pair is one scalar multiplication and one comparison; shuffles rescale
// trackers by fresh randomisers, so nothing can be indexed or cached across them.  Two schedules:
//   * shared scalar (k_match_shared): the lanes of a warp take 32 trackers under one key, so the GLV digit
//     schedule of jac_scalar_mul_glv is the same on every lane, as in the Whisk rescale (k_elem.cu);
//   * per-tracker tables (k_match_table): for a tile of kMatchTile trackers the width-kMatchC fixed-base
//     tables of rG (fixed_base.cuh, built by k_fixed_build<kMatchC>) turn k * rG into 32 mixed additions;
//     the lanes of a warp take 32 keys of one tracker.  Building a tracker's tables (k_match_windows, then
//     k_fixed_build<kMatchC>) costs about a hundred scalar multiplications' worth of work, so this pays off
//     only with many keys (kMatchTableMinKeys).
// The comparison needs no inversion: (X, Y, Z) equals the affine (x, y) iff X == x Z^2 and Y == y Z^3 (XYZZ:
// X == x ZZ and Y == y ZZZ); the point at infinity only equals itself.  A match stores the key index into
// owner[t] with atomicMin, so duplicate keys resolve to the smallest index whatever order pairs run in.
#define CDL_FP_MUL_CALL 1  // one shared product body, as in k_elem.cu
#include "fixed_base.cuh"
#include "launch.h"

namespace cdl {

CDL_FN bool jac_eq_affine(const G1Jac& r, const G1Affine& a) {
  const bool ri = jac_is_inf(r), ai = aff_is_inf(a);
  if (ri || ai) return ri && ai;
  Fp zz, t;
  FpM::sqr(zz, r.z);
  FpM::mul(t, a.x, zz);
  if (!FpM::eq(t, r.x)) return false;
  FpM::mul(zz, zz, r.z);
  FpM::mul(t, a.y, zz);
  return FpM::eq(t, r.y);
}

CDL_FN bool xyzz_eq_affine(const G1Xyzz& r, const G1Affine& a) {
  const bool ri = xyzz_is_inf(r), ai = aff_is_inf(a);
  if (ri || ai) return ri && ai;
  Fp t;
  FpM::mul(t, a.x, r.zz);
  if (!FpM::eq(t, r.x)) return false;
  FpM::mul(t, a.y, r.zzz);
  return FpM::eq(t, r.y);
}

// ks: Montgomery -> canonical in place; owner[0 .. T) = INT32_MAX (no match yet)
__global__ void __launch_bounds__(128) k_match_prep(Fr* __restrict__ ks, uint32_t V, int32_t* __restrict__ owner,
                                                    uint32_t T) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < V) {
    Fr k = ks[i];
    FrM::from_mont(k, k);
    ks[i] = k;
  }
  if (i < T) owner[i] = INT32_MAX;
}

// pair i of [0, V * Tp) is (key i / Tp, tracker i % Tp); Tp = T rounded up to 32, so a warp never spans two keys
__global__ void __launch_bounds__(64, 4)
k_match_shared(const G1Affine* __restrict__ rg, const G1Affine* __restrict__ krg, uint32_t T, uint32_t Tp,
               const Fr* __restrict__ ks, uint32_t V, int32_t* __restrict__ owner) {
  const uint64_t n = (uint64_t)V * Tp, stride = (uint64_t)gridDim.x * blockDim.x;
#pragma unroll 1
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint32_t v = (uint32_t)(i / Tp), t = (uint32_t)(i - (uint64_t)v * Tp);
    if (t >= T) continue;
    const Fr k = ks[v];
    G1Jac r;
    jac_scalar_mul_glv(r, rg[t], k.v);
    if (jac_eq_affine(r, krg[t])) atomicMin(owner + t, (int32_t)v);
  }
}

// thread b: the window bases 2^(8 w) rg[b] of its tracker's tables, by repeated doubling (Jacobian: the caller
// normalises all of them with one batched inversion per thread of launch_jac_to_affine)
__global__ void __launch_bounds__(64)
k_match_windows(const G1Affine* __restrict__ rg, uint32_t nt, G1Jac* __restrict__ out) {
  constexpr int W = fb_windows(kMatchC);
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nt) return;
  G1Jac j;
  jac_from_affine(j, rg[b]);
  G1Jac* o = out + (size_t)b * W;
  o[0] = j;
#pragma unroll 1
  for (int w = 1; w < W; w++) {
#pragma unroll 1
    for (int i = 0; i < kMatchC; i++) jac_dbl(j, j);
    o[w] = j;
  }
}

// trackers t0 .. t0 + nt against all keys; tab holds the tables of rG_t0 .. rG_(t0+nt-1).  Pair i of
// [0, nt * Vp) is (tracker t0 + i / Vp, key i % Vp); Vp = V rounded up to 32
__global__ void __launch_bounds__(128)
k_match_table(const G1Affine* __restrict__ tab, const G1Affine* __restrict__ krg, uint32_t t0, uint32_t nt,
              const Fr* __restrict__ ks, uint32_t V, uint32_t Vp, int32_t* __restrict__ owner) {
  const FixedTable ft{tab, nt};
  const uint64_t n = (uint64_t)nt * Vp, stride = (uint64_t)gridDim.x * blockDim.x;
#pragma unroll 1
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint32_t tl = (uint32_t)(i / Vp), v = (uint32_t)(i - (uint64_t)tl * Vp);
    if (v >= V) continue;
    const Fr k = ks[v];
    G1Xyzz acc;
    xyzz_set_inf(acc);
    fixed_base_accumulate<true, kMatchC>(acc, ft, tl, k.v, false);
    if (xyzz_eq_affine(acc, krg[t0 + tl])) atomicMin(owner + t0 + tl, (int32_t)v);
  }
}

// resident CTAs of a kernel on the current device (queried per launch: a host thread may drive several devices)
template <class K>
static int resident_ctas(K kernel, int tpb) {
  int dev = 0, sms = 0, per_sm = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, tpb, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
  return sms * per_sm;
}

// a grid of at most one wave of resident CTAs, no larger than n items need
static int match_blocks(uint64_t n, int tpb, int resident) {
  const uint64_t need = (n + tpb - 1) / tpb;
  return (int)(need < (uint64_t)resident ? need : (uint64_t)resident);
}

void launch_match_prep(Fr* ks, uint32_t V, int32_t* owner, uint32_t T, cudaStream_t st) {
  const uint32_t n = V > T ? V : T;
  k_match_prep<<<(n + 127) / 128, 128, 0, st>>>(ks, V, owner, T);
}

void launch_match_shared(const G1Affine* rg, const G1Affine* krg, uint32_t T, const Fr* ks, uint32_t V,
                         int32_t* owner, cudaStream_t st) {
  const uint32_t Tp = (T + 31) & ~31u;
  const int blocks = match_blocks((uint64_t)V * Tp, 64, resident_ctas(k_match_shared, 64));
  k_match_shared<<<blocks, 64, 0, st>>>(rg, krg, T, Tp, ks, V, owner);
}

void launch_match_windows(const G1Affine* rg, uint32_t nt, G1Jac* out, cudaStream_t st) {
  k_match_windows<<<(nt + 63) / 64, 64, 0, st>>>(rg, nt, out);
}

void launch_match_table(const G1Affine* tab, const G1Affine* krg, uint32_t t0, uint32_t nt, const Fr* ks,
                        uint32_t V, int32_t* owner, cudaStream_t st) {
  const uint32_t Vp = (V + 31) & ~31u;
  const int blocks = match_blocks((uint64_t)nt * Vp, 128, resident_ctas(k_match_table, 128));
  k_match_table<<<blocks, 128, 0, st>>>(tab, krg, t0, nt, ks, V, Vp, owner);
}

}  // namespace cdl
