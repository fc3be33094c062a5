// Builds fixed-base tables (fixed_base.cuh) on the device: those of a CRS (width 12), the per-tracker
// tables of Whisk tracker matching (width kMatchC, k_match.cu) and the table of a caller's base for batched
// fixed-base scalar multiplication (width 12, k_base_mul.cu).
#define CDL_FP_MUL_CALL 1
#include "fixed_base.cuh"
#include "launch.h"

namespace cdl {

constexpr int kFbNorm = 8;  // entries normalised with one inversion (CRS tables)

// thread (b, w, s) of a row cut into S segments of L = M / S entries: Q = 2^(C w) P_b, then the entries
// (L s + 1) Q .. (L s + L) Q by repeated addition of Q; consecutive entries share one inversion (Montgomery's
// trick).
// Point bases (CRS tables, built once per CRS): bases[b] = P_b, each thread doubles its way to Q; groups of 8.
// Row bases (tracker tables, built on every matching call, and the table of a caller's base):
// bases[b W + w] = 2^(C w) P_b is given (launch_match_windows, launch_base_windows), and a thread's L entries
// share one inversion.
template <int C, bool kRowBases, int kSeg>
__global__ void __launch_bounds__(64)
k_fixed_build(const G1Affine* __restrict__ bases, uint32_t nbase, G1Affine* __restrict__ tab) {
  constexpr int W = fb_windows(C), M = fb_entries(C), kFbSegLen = M / kSeg;
  constexpr int kNorm = kRowBases ? kFbSegLen : kFbNorm;
  static_assert(kFbSegLen % kNorm == 0, "segment length");
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nbase * (uint32_t)(W * kSeg)) return;
  const uint32_t b = t / (W * kSeg), r = t - b * (W * kSeg);
  const int w = (int)(r / kSeg), s = (int)(r - (uint32_t)w * kSeg);
  G1Affine* row = tab + ((size_t)b * W + w) * M + (size_t)s * kFbSegLen;
  G1Affine q;
  if constexpr (kRowBases) {
    q = bases[(size_t)b * W + w];
  } else {
    const G1Affine p = bases[b];
    G1Jac j;
    jac_from_affine(j, p);
#pragma unroll 1
    for (int i = 0; i < w * C; i++) jac_dbl(j, j);
    jac_to_affine(q, j);  // infinity stays infinity: the whole row is infinity then
  }
  // acc = (L s) Q
  G1Xyzz acc;
  xyzz_set_inf(acc);
  {
    const uint32_t e = (uint32_t)s * kFbSegLen;
    if (e) {
      const int top = 31 - __clz(e);
#pragma unroll 1
      for (int i = top; i >= 0; i--) {
        xyzz_dbl(acc, acc);
        if ((e >> i) & 1u) xyzz_add_mixed(acc, acc, q);
      }
    }
  }
  G1Xyzz pend[kNorm];
  Fp pre[kNorm];
#pragma unroll 1
  for (int base = 0; base < kFbSegLen; base += kNorm) {
    Fp run;
    FpM::set_one(run);
#pragma unroll 1
    for (int e = 0; e < kNorm; e++) {
      xyzz_add_mixed(acc, acc, q);
      if (!xyzz_is_inf(acc)) FpM::mul(run, run, acc.zzz);
      pend[e] = acc;
      pre[e] = run;
    }
    Fp inv;
    fp_inv(inv, run);
#pragma unroll 1
    for (int e = kNorm - 1; e >= 0; e--) {
      const G1Xyzz v = pend[e];
      G1Affine a;
      if (xyzz_is_inf(v)) {
        aff_set_inf(a);
      } else {
        Fp zi;  // 1 / zzz
        if (e > 0) FpM::mul(zi, inv, pre[e - 1]); else zi = inv;
        FpM::mul(inv, inv, v.zzz);
        // x = X / ZZ = X * ZZZ^-2 * ... : with ZZ^3 = ZZZ^2, 1/ZZ = (ZZ * (1/ZZZ))^2
        Fp u, izz;
        FpM::mul(u, v.zz, zi);  // ZZ / ZZZ = 1 / Z
        FpM::sqr(izz, u);       // 1 / ZZ
        FpM::mul(a.x, v.x, izz);
        FpM::mul(a.y, v.y, zi);
      }
      row[base + e] = a;
    }
  }
}

template <int C>
size_t fixed_table_bytes(uint32_t nbase) {
  return (size_t)nbase * fb_windows(C) * fb_entries(C) * sizeof(G1Affine);
}

template <int C, bool RowBases, int Seg>
void launch_fixed_build(const G1Affine* bases, uint32_t nbase, G1Affine* tab, cudaStream_t st) {
  const uint32_t threads = nbase * (uint32_t)(fb_windows(C) * Seg);
  if (threads) k_fixed_build<C, RowBases, Seg><<<(threads + 63) / 64, 64, 0, st>>>(bases, nbase, tab);
}

template size_t fixed_table_bytes<kFbC>(uint32_t);
template void launch_fixed_build<kFbC>(const G1Affine*, uint32_t, G1Affine*, cudaStream_t);
template size_t fixed_table_bytes<kMatchC>(uint32_t);
template void launch_fixed_build<kMatchC>(const G1Affine*, uint32_t, G1Affine*, cudaStream_t);
template void launch_fixed_build<kFbC, true, kBaseSeg>(const G1Affine*, uint32_t, G1Affine*, cudaStream_t);

}  // namespace cdl
