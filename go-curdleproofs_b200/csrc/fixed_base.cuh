// Fixed-base tables for the CRS points.
//
// The CRS (crs.go:20-59: Gs, Hs, H, Gt, Gu, Gsum, Hsum) is the same for every proof a context ever
// handles, and a sizeable share of the group work of a batch is multiples of exactly those points:
// the commitments A, C, B_c, B_a and M, the first round of both folding arguments (whose bases are
// still the unfolded Gs || Hs), the verifier's merged Gs / Hs terms, and Gs'[i] = beta^-(i+1) Gs[i]
// (grandproductargument.go:94-103).  For such a term the windowed sum needs no doublings and no
// buckets: with T[b][w][d] = d * 2^(12 w) * P_b tabulated for d = 1 .. 2048,
//     k * P_b = sum_w  sign(d_w) * T[b][w][|d_w|],   k = sum_w d_w 2^(12 w),  d_w in [-2047, 2048],
// is 22 mixed additions (220 field products) against ~ 700 for a term of the bucket kernel and
// ~ 1 500 for a scalar multiplication.  The table is 22 x 2 048 points = 4.3 MB per base, 580 MB for
// the 134 points of an ell = 124 CRS — HBM this path has to spare — and is built once per CRS on the
// device (k_fixed_build), the first time a large batch uses that CRS.  Results are the same group
// elements, hence the same bytes.
#pragma once
#include "g1.cuh"

namespace cdl {

constexpr int kFbC = 12;               // window width of the CRS tables
// Tables of window width C (2 <= C <= 16): fb_windows(C) windows of fb_entries(C) entries d = 1 .. 2^(C-1).
// The top window holds bits of k below 2^255 only, so it never carries out.
CDL_HD constexpr int fb_windows(int C) { return (255 + C) / C; }
CDL_HD constexpr int fb_entries(int C) { return 1 << (C - 1); }
constexpr int kFbW = fb_windows(kFbC);  // 22 * 12 = 264 >= 255 bits + carry
constexpr int kFbM = fb_entries(kFbC);  // d = 1 .. 2048
static_assert(kFbW == 22 && kFbM == 2048, "CRS table geometry");

struct FixedTable {
  const G1Affine* tab = nullptr;  // [nbase][W][M], entry (b, w, d - 1) = d * 2^(C w) * P_b (W, M of the width C)
  uint32_t nbase = 0;             // pool indices below this are tabulated
};

// signed C-bit digit of window w (carry in / out through `carry`): the table index |d| - 1 of a non-zero
// digit, its sign in bit 31; 0xffffffff for a zero digit
template <int C = kFbC>
CDL_FN uint32_t fixed_base_digit(const uint32_t* k, int w, uint32_t& carry) {
  static_assert(C >= 2 && C <= 16, "window width");
  const int bit = w * C;
  const int word = bit >> 5, sh = bit & 31;
  const uint32_t lo = k[word], hi = word + 1 < 8 ? k[word + 1] : 0u;
  uint32_t raw = sh ? ((lo >> sh) | (sh > 32 - C ? hi << (32 - sh) : 0u)) : lo;
  raw = (raw & ((1u << C) - 1u)) + carry;
  carry = raw > (uint32_t)fb_entries(C) ? 1u : 0u;
  if (raw == 0 || raw == (1u << C)) return 0xffffffffu;  // digit 0 (the second form carries into the next window)
  const uint32_t mag = carry ? (1u << C) - raw : raw;
  return (mag - 1) | (carry << 31);
}

// acc += (neg ? -k : k) * P_b, k canonical little-endian words (k < 2^255).  The look-ups do not depend
// on the running sum, so the next window's table entry is fetched while the current one is added.
// PREFETCH = false keeps one table entry live (24 registers less) for kernels that are short of registers.
template <bool PREFETCH = true, int C = kFbC>
CDL_FN void fixed_base_accumulate(G1Xyzz& acc, const FixedTable& ft, uint32_t b, const uint32_t* k, bool neg) {
  constexpr int W = fb_windows(C), M = fb_entries(C);
  const G1Affine* tb = ft.tab + (size_t)b * (W * M);
  uint32_t carry = 0;
  if (!PREFETCH) {
#pragma unroll 1
    for (int w = 0; w < W; w++) {
      const uint32_t d = fixed_base_digit<C>(k, w, carry);
      if (d == 0xffffffffu) continue;
      G1Affine q = tb[(size_t)w * M + (d & 0x7fffffffu)];
      if (((d >> 31) != 0) != neg) FpM::neg(q.y, q.y);
      xyzz_add_mixed(acc, acc, q);
    }
    return;
  }
  uint32_t d = fixed_base_digit<C>(k, 0, carry);
  G1Affine q;
  aff_set_inf(q);
  if (d != 0xffffffffu) q = tb[d & 0x7fffffffu];
#pragma unroll 1
  for (int w = 0; w < W; w++) {
    uint32_t dn = 0xffffffffu;
    G1Affine qn = q;
    if (w + 1 < W) {
      dn = fixed_base_digit<C>(k, w + 1, carry);
      if (dn != 0xffffffffu) qn = tb[(size_t)(w + 1) * M + (dn & 0x7fffffffu)];
    }
    if (d != 0xffffffffu) {
      if (((d >> 31) != 0) != neg) FpM::neg(q.y, q.y);
      xyzz_add_mixed(acc, acc, q);
    }
    d = dn;
    q = qn;
  }
}

}  // namespace cdl
