// BLS12-381 base field Fp (381 bit, 12 x 32-bit limbs) and scalar field Fr
// (255 bit, 8 x 32-bit limbs) parameters for the Montgomery core in mont.cuh.
// Replaces gnark-crypto's fp.Element / fr.Element arithmetic underneath every
// row of SURVEY.md §8a (the reference reaches it through go.mod:6).
#pragma once
#include "mont.cuh"

namespace cdl {

#define CDL_FP_MOD  {0xffffaaabu, 0xb9feffffu, 0xb153ffffu, 0x1eabfffeu, 0xf6b0f624u, 0x6730d2a0u, 0xf38512bfu, 0x64774b84u, 0x434bacd7u, 0x4b1ba7b6u, 0x397fe69au, 0x1a0111eau}
#define CDL_FP_ONE  {0x0002fffdu, 0x76090000u, 0xc40c0002u, 0xebf4000bu, 0x53c758bau, 0x5f489857u, 0x70525745u, 0x77ce5853u, 0xa256ec6du, 0x5c071a97u, 0xfa80e493u, 0x15f65ec3u}
#define CDL_FP_R2   {0x1c341746u, 0xf4df1f34u, 0x09d104f1u, 0x0a76e6a6u, 0x4c95b6d5u, 0x8de5476cu, 0x939d83c0u, 0x67eb88a9u, 0xb519952du, 0x9a793e85u, 0x92cae3aau, 0x11988fe5u}
#define CDL_FR_MOD  {0x00000001u, 0xffffffffu, 0xfffe5bfeu, 0x53bda402u, 0x09a1d805u, 0x3339d808u, 0x299d7d48u, 0x73eda753u}
#define CDL_FR_ONE  {0xfffffffeu, 0x00000001u, 0x00034802u, 0x5884b7fau, 0xecbc4ff5u, 0x998c4fefu, 0xacc5056fu, 0x1824b159u}
#define CDL_FR_R2   {0xf3f29c6du, 0xc999e990u, 0x87925c23u, 0x2b6cedcbu, 0x7254398fu, 0x05d31496u, 0x9f59ff11u, 0x0748d9d9u}

static const uint32_t FP_MOD_H[12] = CDL_FP_MOD;
static const uint32_t FP_ONE_H[12] = CDL_FP_ONE;
static const uint32_t FP_R2_H[12] = CDL_FP_R2;
static const uint32_t FR_MOD_H[8] = CDL_FR_MOD;
static const uint32_t FR_ONE_H[8] = CDL_FR_ONE;
static const uint32_t FR_R2_H[8] = CDL_FR_R2;
#if defined(__CUDACC__)
static __device__ __constant__ uint32_t FP_MOD_D[12] = CDL_FP_MOD;
static __device__ __constant__ uint32_t FP_ONE_D[12] = CDL_FP_ONE;
static __device__ __constant__ uint32_t FP_R2_D[12] = CDL_FP_R2;
static __device__ __constant__ uint32_t FR_MOD_D[8] = CDL_FR_MOD;
static __device__ __constant__ uint32_t FR_ONE_D[8] = CDL_FR_ONE;
static __device__ __constant__ uint32_t FR_R2_D[8] = CDL_FR_R2;
#endif

#if defined(__CUDA_ARCH__)
#define CDL_SEL(dev, host) dev
#else
#define CDL_SEL(dev, host) host
#endif

struct FpParams {
  static constexpr int N = 12;
  static constexpr uint32_t M0 = 0xfffcfffdu;  // -p^-1 mod 2^32
  static CDL_HD uint32_t mod(int i) { return CDL_SEL(FP_MOD_D, FP_MOD_H)[i]; }
  static CDL_HD uint32_t one(int i) { return CDL_SEL(FP_ONE_D, FP_ONE_H)[i]; }
  static CDL_HD uint32_t r2(int i) { return CDL_SEL(FP_R2_D, FP_R2_H)[i]; }
};

struct FrParams {
  static constexpr int N = 8;
  static constexpr uint32_t M0 = 0xffffffffu;  // -r^-1 mod 2^32
  static CDL_HD uint32_t mod(int i) { return CDL_SEL(FR_MOD_D, FR_MOD_H)[i]; }
  static CDL_HD uint32_t one(int i) { return CDL_SEL(FR_ONE_D, FR_ONE_H)[i]; }
  static CDL_HD uint32_t r2(int i) { return CDL_SEL(FR_R2_D, FR_R2_H)[i]; }
};

using FpM = Mont<FpParams>;
using FrM = Mont<FrParams>;
using Fp = FpM::El;  // 48 bytes == gnark fp.Element
using Fr = FrM::El;  // 32 bytes == gnark fr.Element

// public constants, little-endian 32-bit words
// (p-1)/2
#define CDL_FP_HALF  {0xffffd555u, 0xdcff7fffu, 0x58a9ffffu, 0x0f55ffffu, 0x7b587b12u, 0xb3986950u, 0x79c2895fu, 0xb23ba5c2u, 0x21a5d66bu, 0x258dd3dbu, 0x1cbff34du, 0x0d0088f5u}
// Montgomery form of curve constant b = 4 and of beta (cube root of unity with
// phi(x,y) = (beta*x, y) = lambda*(x,y), lambda = z^2 - 1)
#define CDL_FP_B     {0x000cfff3u, 0xaa270000u, 0xfc34000au, 0x53cc0032u, 0x6b0a807fu, 0x478fe97au, 0xe6ba24d7u, 0xb1d37ebeu, 0xbf78ab2fu, 0x8ec9733bu, 0x3d83de7eu, 0x09d64551u}
#define CDL_FP_BETA  {0x8671f071u, 0xcd03c9e4u, 0x1fcda5d2u, 0x5dab2246u, 0xd3851b95u, 0x587042afu, 0x01bacb9eu, 0x8eb60ebeu, 0x83d050d2u, 0x03f97d6eu, 0x54638741u, 0x18f02065u}

static const uint32_t FP_HALF_H[12] = CDL_FP_HALF;
static const uint32_t FP_B_H[12] = CDL_FP_B;
static const uint32_t FP_BETA_H[12] = CDL_FP_BETA;
#if defined(__CUDACC__)
static __device__ __constant__ uint32_t FP_HALF_D[12] = CDL_FP_HALF;
static __device__ __constant__ uint32_t FP_B_D[12] = CDL_FP_B;
static __device__ __constant__ uint32_t FP_BETA_D[12] = CDL_FP_BETA;
#endif

// Reference inversion (kept for the cross-check of fp_inv on the CPU tier): binary extended Euclid in a branch-free,
// fixed-length form: the invariants u = x1*A, v = x2*A (mod p) hold for the raw limbs A = a*R; a
// step makes u even (swapping so that u >= v and subtracting when it is odd) and halves it, so
// bitlen(u) + bitlen(v) drops by at least one per step and 768 steps always end with u = 0,
// v = 1, x2 = A^-1.  About 180 add/shift/select instructions per step instead of the ~480
// Montgomery products of Fermat's a^(p-2): a third of the latency of every normalisation
// (one per scalar multiplication, per MSM result, per Horner chain) and half its issue slots.
CDL_FN void fp_inv_eea(Fp& r, const Fp& a) {
  constexpr int N = 12;
  uint32_t u[N], v[N], x1[N], x2[N];
#pragma unroll
  for (int i = 0; i < N; i++) {
    u[i] = a.v[i];
    v[i] = FpParams::mod(i);
    x1[i] = i == 0 ? 1u : 0u;
    x2[i] = 0u;
  }
#pragma unroll 1
  for (int it = 0; it < 768; it++) {
    const uint32_t odd = 0u - (u[0] & 1u);
    uint32_t lt;
    {
      CC c;
      (void)sub_cc(c, u[0], v[0]);
#pragma unroll
      for (int i = 1; i < N; i++) (void)subc_cc(c, u[i], v[i]);
      lt = subc(c, 0, 0);  // all ones when u < v
    }
    const uint32_t sw = odd & lt;
#pragma unroll
    for (int i = 0; i < N; i++) {
      uint32_t t = (u[i] ^ v[i]) & sw;
      u[i] ^= t;
      v[i] ^= t;
      uint32_t s = (x1[i] ^ x2[i]) & sw;
      x1[i] ^= s;
      x2[i] ^= s;
    }
    {  // u -= v when u is odd (now u >= v)
      CC c;
      u[0] = sub_cc(c, u[0], v[0] & odd);
#pragma unroll
      for (int i = 1; i < N - 1; i++) u[i] = subc_cc(c, u[i], v[i] & odd);
      u[N - 1] = subc(c, u[N - 1], v[N - 1] & odd);
    }
    {  // x1 = x1 - x2 (mod p) when u was odd
      CC c;
      x1[0] = sub_cc(c, x1[0], x2[0] & odd);
#pragma unroll
      for (int i = 1; i < N; i++) x1[i] = subc_cc(c, x1[i], x2[i] & odd);
      const uint32_t borrow = subc(c, 0, 0);
      CC c2;
      x1[0] = add_cc(c2, x1[0], FpParams::mod(0) & borrow);
#pragma unroll
      for (int i = 1; i < N - 1; i++) x1[i] = addc_cc(c2, x1[i], FpParams::mod(i) & borrow);
      x1[N - 1] = addc(c2, x1[N - 1], FpParams::mod(N - 1) & borrow);
    }
#pragma unroll
    for (int i = 0; i < N - 1; i++) u[i] = (u[i] >> 1) | (u[i + 1] << 31);
    u[N - 1] >>= 1;
    {  // x1 = x1 / 2 (mod p): add p first when odd (x1 + p < 2^382, no carry out of the top limb)
      const uint32_t xo = 0u - (x1[0] & 1u);
      CC c;
      x1[0] = add_cc(c, x1[0], FpParams::mod(0) & xo);
#pragma unroll
      for (int i = 1; i < N - 1; i++) x1[i] = addc_cc(c, x1[i], FpParams::mod(i) & xo);
      x1[N - 1] = addc(c, x1[N - 1], FpParams::mod(N - 1) & xo);
#pragma unroll
      for (int i = 0; i < N - 1; i++) x1[i] = (x1[i] >> 1) | (x1[i + 1] << 31);
      x1[N - 1] >>= 1;
    }
  }
  // x2 = (a*R)^-1 = a^-1 * R^-1 as a plain residue; times R^3 in the Montgomery product gives a^-1 * R
  Fp raw, r2, r3;
#pragma unroll
  for (int i = 0; i < N; i++) {
    raw.v[i] = x2[i];
    r2.v[i] = FpParams::r2(i);
  }
  FpM::mul(r3, r2, r2);
  FpM::mul(r, raw, r3);
}

// ---------------------------------------------------------------------------------------------
// r = a^-1, inv(0) = 0 (Montgomery form in and out).
//
// Binary GCD with the inner steps run on 64-bit APPROXIMATIONS of the operands (Pornin, "Optimized
// binary GCD for modular inversion", 2020): per outer iteration the low 31 bits and the top 33 bits of
// (a, b) are packed into two 64-bit words, 31 divsteps run on those words only and record their effect
// as a 2x2 matrix (f0 g0 / f1 g1) of 33-bit signed factors, then the matrix is applied once to the full
// operands: (a, b) <- (a f0 + b g0, a f1 + b g1) / 2^31 (exact), and to the cofactors modulo p with a
// word-level Montgomery division by 2^31, which keeps the invariants a = x*u, b = x*v (mod p).  25 outer
// iterations (>= (2*381 - 1) / 31) end with a = 0, b = 1, v = x^-1.  About 30 k instructions, fixed
// length and branch-free, against 138 k for the limb-wide binary Euclid above it replaces: the
// normalisation at the end of every latency-bound stage drops from 0.2 ms to under 0.05 ms.
struct FpInvMat { uint32_t f0, g0, f1, g1; bool nf0, ng0, nf1, ng1; };  // magnitudes (<= 2^31) and signs

// 13-limb (two's complement, sign returned) t = (sx ? -x*fx : x*fx) + (sy ? -y*fy : y*fy), shifted
// right by 31 bits; the 31 dropped bits are zero by construction.  |result| < 2^383.
CDL_FN bool fp_inv_lincomb(uint32_t* out, const uint32_t* x, uint32_t fx, bool sx, const uint32_t* y, uint32_t fy, bool sy) {
  constexpr int N = 12;
  uint32_t X[N + 2], Y[N + 2];
  uint64_t cx = 0, cy = 0;
#pragma unroll
  for (int i = 0; i < N; i++) {
    cx += (uint64_t)x[i] * fx;
    X[i] = (uint32_t)cx;
    cx >>= 32;
    cy += (uint64_t)y[i] * fy;
    Y[i] = (uint32_t)cy;
    cy >>= 32;
  }
  X[N] = (uint32_t)cx; X[N + 1] = 0;
  Y[N] = (uint32_t)cy; Y[N + 1] = 0;
  // conditional negation folded into the addition: X ^ mx + (mx & 1) is -X in two's complement
  const uint32_t mx = sx ? 0xffffffffu : 0u, my = sy ? 0xffffffffu : 0u;
  uint64_t c = (uint64_t)(mx & 1u) + (my & 1u);
  uint32_t R[N + 2];
#pragma unroll
  for (int i = 0; i < N + 2; i++) {
    c += (uint64_t)(X[i] ^ mx) + (Y[i] ^ my);
    R[i] = (uint32_t)c;
    c >>= 32;
  }
  const bool neg = (R[N + 1] >> 31) != 0;
  // arithmetic shift right by 31, then absolute value
  const uint32_t mn = neg ? 0xffffffffu : 0u;
  uint64_t cn = mn & 1u;
#pragma unroll
  for (int i = 0; i < N + 1; i++) {
    uint32_t w = (R[i] >> 31) | (R[i + 1] << 1);
    cn += (uint64_t)(w ^ mn);
    out[i] = (uint32_t)cn;
    cn >>= 32;
  }
  return neg;
}

// w = (sx ? p - x : x) * fx + (sy ? p - y : y) * fy, Montgomery-divided by 2^31 and reduced below p
CDL_FN void fp_inv_cofactor(uint32_t* out, const uint32_t* x, uint32_t fx, bool sx, const uint32_t* y, uint32_t fy, bool sy) {
  constexpr int N = 12;
  uint32_t xs[N], ys[N];
  {
    uint64_t bx = 0, by = 0;
#pragma unroll
    for (int i = 0; i < N; i++) {
      uint64_t dx = (uint64_t)FpParams::mod(i) - x[i] - bx;
      uint64_t dy = (uint64_t)FpParams::mod(i) - y[i] - by;
      bx = (dx >> 63) & 1u;
      by = (dy >> 63) & 1u;
      xs[i] = sx ? (uint32_t)dx : x[i];
      ys[i] = sy ? (uint32_t)dy : y[i];
    }
  }
  uint32_t Z[N + 2];
  uint64_t c = 0;
#pragma unroll
  for (int i = 0; i < N; i++) {
    c += (uint64_t)xs[i] * fx;
    uint32_t lo = (uint32_t)c;
    c >>= 32;
    uint64_t t = (uint64_t)ys[i] * fy + lo;
    Z[i] = (uint32_t)t;
    c += t >> 32;
  }
  Z[N] = (uint32_t)c;
  Z[N + 1] = (uint32_t)(c >> 32);
  // Z += k * p with k = -Z * p^-1 mod 2^31: the low 31 bits cancel
  const uint32_t k = (Z[0] * FpParams::M0) & 0x7fffffffu;
  c = 0;
#pragma unroll
  for (int i = 0; i < N; i++) {
    c += (uint64_t)FpParams::mod(i) * k + Z[i];
    Z[i] = (uint32_t)c;
    c >>= 32;
  }
  c += Z[N];
  Z[N] = (uint32_t)c;
  Z[N + 1] += (uint32_t)(c >> 32);
  uint32_t w[N + 1];
#pragma unroll
  for (int i = 0; i < N + 1; i++) w[i] = (Z[i] >> 31) | (Z[i + 1] << 1);
  // w < 3p: two conditional subtractions
#pragma unroll 1
  for (int rep = 0; rep < 2; rep++) {
    uint32_t t[N + 1];
    uint64_t bw = 0;
#pragma unroll
    for (int i = 0; i < N + 1; i++) {
      uint64_t d = (uint64_t)w[i] - (i < N ? FpParams::mod(i) : 0u) - bw;
      t[i] = (uint32_t)d;
      bw = (d >> 63) & 1u;
    }
#pragma unroll
    for (int i = 0; i < N + 1; i++) w[i] = bw ? w[i] : t[i];
  }
#pragma unroll
  for (int i = 0; i < N; i++) out[i] = w[i];
}

CDL_FN void fp_inv(Fp& r, const Fp& x) {
  constexpr int N = 12;
  uint32_t a[N + 1], b[N + 1], u[N], v[N];
#pragma unroll
  for (int i = 0; i < N; i++) {
    a[i] = x.v[i];
    b[i] = FpParams::mod(i);
    u[i] = i == 0 ? 1u : 0u;
    v[i] = 0u;
  }
  a[N] = b[N] = 0;
#pragma unroll 1
  for (int it = 0; it < 25; it++) {
    // ---- 64-bit approximations: low 31 bits + the 33 bits below the top bit of max(a, b)
    uint32_t top = 0, ah = 0, am = 0, al = 0, bh = 0, bm = 0, bl = 0;
    bool found = false;
#pragma unroll
    for (int i = N - 1; i >= 2; i--) {
      const uint32_t o = a[i] | b[i];
      const bool take = !found && o != 0;
      top = take ? o : top;
      ah = take ? a[i] : ah; am = take ? a[i - 1] : am; al = take ? a[i - 2] : al;
      bh = take ? b[i] : bh; bm = take ? b[i - 1] : bm; bl = take ? b[i - 2] : bl;
      found = found || o != 0;
    }
    uint64_t abar, bbar;
    {
      int s = 0;  // clz(top); top != 0 when found
#if defined(__CUDA_ARCH__)
      s = found ? __clz((int)top) : 0;
#else
      for (uint32_t t = top; found && !(t & 0x80000000u); t <<= 1) s++;
#endif
      const uint64_t a96h = ((uint64_t)ah << 32) | am, b96h = ((uint64_t)bh << 32) | bm;
      const uint64_t a64 = s ? (a96h << s) | (al >> (32 - s)) : a96h;
      const uint64_t b64 = s ? (b96h << s) | (bl >> (32 - s)) : b96h;
      const uint64_t ax = ((a64 >> 31) << 31) | (a[0] & 0x7fffffffu);
      const uint64_t bx = ((b64 >> 31) << 31) | (b[0] & 0x7fffffffu);
      const uint64_t ae = ((uint64_t)a[1] << 32) | a[0], be = ((uint64_t)b[1] << 32) | b[0];  // exact below 2^64
      abar = found ? ax : ae;
      bbar = found ? bx : be;
    }
    // ---- 31 divsteps on the approximations
    int64_t f0 = 1, g0 = 0, f1 = 0, g1 = 1;
#pragma unroll 1
    for (int j = 0; j < 31; j++) {
      const uint64_t odd = 0ull - (abar & 1ull);
      const uint64_t sw = odd & (abar < bbar ? ~0ull : 0ull);
      uint64_t t = (abar ^ bbar) & sw;
      abar ^= t; bbar ^= t;
      t = (uint64_t)(f0 ^ f1) & sw;
      f0 ^= (int64_t)t; f1 ^= (int64_t)t;
      t = (uint64_t)(g0 ^ g1) & sw;
      g0 ^= (int64_t)t; g1 ^= (int64_t)t;
      abar -= bbar & odd;
      f0 -= f1 & (int64_t)odd;
      g0 -= g1 & (int64_t)odd;
      abar >>= 1;
      f1 = (int64_t)((uint64_t)f1 << 1);
      g1 = (int64_t)((uint64_t)g1 << 1);
    }
    bool nf0 = f0 < 0, ng0 = g0 < 0, nf1 = f1 < 0, ng1 = g1 < 0;
    const uint32_t mf0 = (uint32_t)(nf0 ? -f0 : f0), mg0 = (uint32_t)(ng0 ? -g0 : g0);
    const uint32_t mf1 = (uint32_t)(nf1 ? -f1 : f1), mg1 = (uint32_t)(ng1 ? -g1 : g1);
    // ---- apply to the operands; a negative result is negated together with its matrix row
    uint32_t na[N + 1], nb[N + 1];
    const bool sa = fp_inv_lincomb(na, a, mf0, nf0, b, mg0, ng0);
    const bool sb = fp_inv_lincomb(nb, a, mf1, nf1, b, mg1, ng1);
    nf0 = nf0 != sa; ng0 = ng0 != sa;
    nf1 = nf1 != sb; ng1 = ng1 != sb;
    // ---- and to the cofactors, modulo p
    uint32_t nu[N], nv[N];
    fp_inv_cofactor(nu, u, mf0, nf0, v, mg0, ng0);
    fp_inv_cofactor(nv, u, mf1, nf1, v, mg1, ng1);
#pragma unroll
    for (int i = 0; i < N; i++) { a[i] = na[i]; b[i] = nb[i]; u[i] = nu[i]; v[i] = nv[i]; }
  }
  // v = (x*R)^-1 = x^-1 * R^-1 as a plain residue; times R^3 in the Montgomery product gives x^-1 * R.
  // (x = 0 leaves a = 0, b = p, v = 0 throughout: inv(0) = 0.)
  Fp raw, r2, r3;
#pragma unroll
  for (int i = 0; i < N; i++) {
    raw.v[i] = v[i];
    r2.v[i] = FpParams::r2(i);
  }
  FpM::mul(r3, r2, r2);
  FpM::mul(r, raw, r3);
}

// r = r^(2^n): a loop, so that a squaring run costs one squaring's code (inlined or the shared body)
CDL_FN void fp_sqr_n(Fp& r, int n) {
#pragma unroll 1
  for (int i = 0; i < n; i++) FpM::sqr(r, r);
}

#include "fp_sqrt_chain.cuh"  // fp_pow_sqrt_exp(r, a): r = a^((p+1)/4) by a fixed addition chain

// candidate square root a^((p+1)/4) (p = 3 mod 4); returns whether it squares to a
CDL_FN bool fp_sqrt(Fp& r, const Fp& a) {
  Fp s, t;
  fp_pow_sqrt_exp(s, a);
  FpM::sqr(t, s);
  r = s;
  return FpM::eq(t, a);
}

CDL_HD void fp_set_b(Fp& r) {
#pragma unroll
  for (int i = 0; i < 12; i++) r.v[i] = CDL_SEL(FP_B_D, FP_B_H)[i];
}

CDL_HD void fp_set_beta(Fp& r) {
#pragma unroll
  for (int i = 0; i < 12; i++) r.v[i] = CDL_SEL(FP_BETA_D, FP_BETA_H)[i];
}

// gnark fp.Element.LexicographicallyLargest: canonical(a) > (p-1)/2
CDL_FN bool fp_lex_largest(const Fp& a_mont) {
  Fp c;
  FpM::from_mont(c, a_mont);
  CC cc;  // (p-1)/2 - c borrows  <=>  c > (p-1)/2
  (void)sub_cc(cc, CDL_SEL(FP_HALF_D, FP_HALF_H)[0], c.v[0]);
#pragma unroll
  for (int i = 1; i < 12; i++) (void)subc_cc(cc, CDL_SEL(FP_HALF_D, FP_HALF_H)[i], c.v[i]);
  return subc(cc, 0, 0) != 0;
}

// canonical limbs < p ?
CDL_HD bool fp_is_canonical(const Fp& c) {
  CC cc;
  (void)sub_cc(cc, c.v[0], FpParams::mod(0));
#pragma unroll
  for (int i = 1; i < 12; i++) (void)subc_cc(cc, c.v[i], FpParams::mod(i));
  return subc(cc, 0, 0) != 0;
}

}  // namespace cdl
