// Batched fixed-base scalar multiplication: out[i] = k_i * P for many scalars and one caller-supplied base P
// (bls12381.BatchScalarMultiplicationG1).  Two paths, chosen by Engine::base_mul (capi_base_mul.cu):
//   * table path: the width-12 fixed-base table of P (fixed_base.cuh, 22 x 2 048 points, 4.3 MB) turns k * P
//     into 22 mixed additions (k_base_mul).  The table is built from P's 22 window bases 2^(12 w) P
//     (k_base_prep, one doubling chain) by k_fixed_build in row-base mode with 128 threads per row;
//   * GLV path: the generic per-element scalar multiplication (launch_scalar_mul) on n device copies of P
//     (k_base_fill), for a few scalars and a base without a table.
// k_base_prep also checks the base (canonical coordinates, on the curve, in G1 by the subgroup test of
// decompression): the GLV path assumes a base of prime order and the table path does not, so only for bases in
// G1 do the two agree.
#define CDL_FP_MUL_CALL 1  // one shared product body, as in k_elem.cu
#include "codec.cuh"
#include "fixed_base.cuh"
#include "launch.h"

namespace cdl {

// Warp 0 checks *base into *status (0 in G1, 1 non-canonical coordinate, 2 not on the curve, 3 not in G1); warp 1
// writes the window bases wjac[w] = 2^(12 w) base (Jacobian) when wjac is given.  Two warps, so that the two
// single-thread chains run side by side.
__global__ void __launch_bounds__(64) k_base_prep(const G1Affine* __restrict__ base, uint32_t* __restrict__ status,
                                                  G1Jac* __restrict__ wjac) {
  const G1Affine p = *base;
  if (threadIdx.x == 0) {
    uint32_t st = 0;
    if (!fp_is_canonical(p.x) || !fp_is_canonical(p.y)) st = 1;
    else if (!aff_on_curve(p)) st = 2;
    else if (!g1_in_subgroup_endo(p)) st = 3;
    *status = st;
  } else if (threadIdx.x == 32 && wjac) {
    G1Jac j;
    jac_from_affine(j, p);
    wjac[0] = j;
#pragma unroll 1
    for (int w = 1; w < kFbW; w++) {
#pragma unroll 1
      for (int i = 0; i < kFbC; i++) jac_dbl(j, j);
      wjac[w] = j;
    }
  }
}

// out[0 .. n) = *base
__global__ void __launch_bounds__(128) k_base_fill(const G1Affine* __restrict__ base, G1Affine* __restrict__ out,
                                                   uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = *base;
}

// Results of one thread normalised with one inversion (Montgomery's trick): 7 products and 1/16 inversion each.
constexpr int kBmNorm = 16;

// out[i] = sc[i] * P from P's width-12 table (sc Montgomery, as the caller gave them); affine to `out` and / or
// compressed to `out48` (either may be null).  A persistent grid of T threads: thread t takes items
// t, t + T, .. (a warp reads consecutive scalars), parks up to kBmNorm XYZZ sums in local memory and inverts the
// product of their ZZZ once.
__global__ void __launch_bounds__(128)
k_base_mul(const G1Affine* __restrict__ tab, const Fr* __restrict__ sc, uint32_t n, G1Affine* __restrict__ out,
           uint8_t* __restrict__ out48) {
  const FixedTable ft{tab, 1};
  const uint32_t T = gridDim.x * blockDim.x;
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  G1Xyzz pend[kBmNorm];
  Fp pre[kBmNorm];  // pre[e] = zzz_0 .. zzz_e over the finite sums of the chunk
#pragma unroll 1
  for (uint32_t first = t; first < n; first += kBmNorm * T) {
    Fp run;
    FpM::set_one(run);
    int cnt = 0;
#pragma unroll 1
    for (int e = 0; e < kBmNorm; e++) {
      const uint32_t i = first + (uint32_t)e * T;
      if (i >= n) break;
      Fr k = sc[i];
      FrM::from_mont(k, k);
      G1Xyzz acc;
      xyzz_set_inf(acc);
      fixed_base_accumulate<true, kFbC>(acc, ft, 0, k.v, false);
      if (!xyzz_is_inf(acc)) FpM::mul(run, run, acc.zzz);
      pend[e] = acc;
      pre[e] = run;
      cnt++;
    }
    Fp inv;
    fp_inv(inv, run);
#pragma unroll 1
    for (int e = cnt - 1; e >= 0; e--) {
      const G1Xyzz v = pend[e];
      G1Affine a;
      if (xyzz_is_inf(v)) {
        aff_set_inf(a);
      } else {
        Fp zi;  // 1 / ZZZ
        if (e > 0) FpM::mul(zi, inv, pre[e - 1]); else zi = inv;
        FpM::mul(inv, inv, v.zzz);
        // with ZZ^3 = ZZZ^2: 1 / ZZ = (ZZ / ZZZ)^2
        Fp u, izz;
        FpM::mul(u, v.zz, zi);
        FpM::sqr(izz, u);
        FpM::mul(a.x, v.x, izz);
        FpM::mul(a.y, v.y, zi);
      }
      const uint32_t i = first + (uint32_t)e * T;
      if (out) out[i] = a;
      if (out48) g1_compress_dev(out48 + 48 * (size_t)i, a);
    }
  }
}

void launch_base_prep(const G1Affine* base, uint32_t* status, G1Jac* wjac, cudaStream_t st) {
  k_base_prep<<<1, 64, 0, st>>>(base, status, wjac);
}

void launch_base_fill(const G1Affine* base, G1Affine* out, uint32_t n, cudaStream_t st) {
  if (n) k_base_fill<<<(n + 127) / 128, 128, 0, st>>>(base, out, n);
}

void launch_base_mul(const G1Affine* tab, const Fr* sc, uint32_t n, G1Affine* out, uint8_t* out48, cudaStream_t st) {
  if (!n) return;
  // at most one wave of resident CTAs (queried per launch: a host thread may drive several devices); with
  // k = ceil(n / resident threads) items per thread the grid shrinks to ceil(n / k) threads, so that no thread
  // does k while others idle through the last pass
  int dev = 0, sms = 0, per_sm = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_base_mul, 128, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
  const uint64_t resident = (uint64_t)sms * per_sm * 128;
  const uint64_t k = (n + resident - 1) / resident;
  const uint64_t threads = (n + k - 1) / k;
  k_base_mul<<<(unsigned)((threads + 127) / 128), 128, 0, st>>>(tab, sc, n, out, out48);
}

}  // namespace cdl
