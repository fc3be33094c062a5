// Montgomery arithmetic on N 32-bit limbs (N even), generic over the modulus.
//
// Elements are plain little-endian limb arrays in Montgomery form, always fully
// reduced to [0, p).  This is byte-for-byte gnark-crypto's fp.Element /
// fr.Element memory layout ([6]uint64 / [4]uint64 little-endian, Montgomery,
// R = 2^(32N)), so host buffers cross the C ABI without conversion
// (SURVEY.md §8 header).
//
// Multiplication is a CIOS product with the partial products split into an
// "even" and an "odd" accumulator so that every a[j]*b_i lands on an aligned
// 64-bit column pair: each row is N/2 + N/2 IMAD.WIDE for the product, the same
// again for the reduction, plus one low multiply for the quotient digit —
// 2N^2 + N wide multiply-adds per product (300 for the 381-bit field), which is
// the unit the integer-pipe roofline is stated in (SURVEY.md §8d).
#pragma once
#include "carry.cuh"

namespace cdl {

template <class F>
struct Mont {
  static constexpr int N = F::N;
  // 16-byte aligned in device code so that loads/stores vectorise to 128 bit
  // (cudaMalloc'ed arrays of 32/48/96/144/192-byte elements keep that alignment).
#if defined(__CUDACC__)
  struct alignas(16) El { uint32_t v[N]; };
#else
  struct El { uint32_t v[N]; };
#endif

  // acc[0..N) = a[j]*bi for j = 0,2,4,.. (64-bit products on aligned pairs)
  static CDL_HD void mul_n(uint32_t* acc, const uint32_t* a, uint32_t bi) {
#pragma unroll
    for (int j = 0; j < N; j += 2) {
      acc[j] = mul_lo(a[j], bi);
      acc[j + 1] = mul_hi(a[j], bi);
    }
  }

  // acc[0..N) += a[j]*bi for j = 0,2,4,.. ; returns with the carry-out in cc.
  static CDL_HD void cmad_n(CC& cc, uint32_t* acc, const uint32_t* a, uint32_t bi) {
    acc[0] = mad_lo_cc(cc, a[0], bi, acc[0]);
    acc[1] = madc_hi_cc(cc, a[0], bi, acc[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      acc[j] = madc_lo_cc(cc, a[j], bi, acc[j]);
      acc[j + 1] = madc_hi_cc(cc, a[j], bi, acc[j + 1]);
    }
  }

  // Same with the modulus as multiplicand (limbs start .. start+N step 2).
  template <int START>
  static CDL_HD void cmad_mod(CC& cc, uint32_t* acc, uint32_t mi) {
    acc[0] = mad_lo_cc(cc, F::mod(START), mi, acc[0]);
    acc[1] = madc_hi_cc(cc, F::mod(START), mi, acc[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      acc[j] = madc_lo_cc(cc, F::mod(START + j), mi, acc[j]);
      acc[j + 1] = madc_hi_cc(cc, F::mod(START + j), mi, acc[j + 1]);
    }
  }

  // odd[] >>= 64 bits while accumulating a[j]*bi (j = 0,2,..) with carry-in.
  static CDL_HD void madc_n_rshift(CC& cc, uint32_t* odd, const uint32_t* a, uint32_t bi) {
#pragma unroll
    for (int j = 0; j < N - 2; j += 2) {
      odd[j] = madc_lo_cc(cc, a[j], bi, odd[j + 2]);
      odd[j + 1] = madc_hi_cc(cc, a[j], bi, odd[j + 3]);
    }
    odd[N - 2] = madc_lo_cc(cc, a[N - 2], bi, 0);
    odd[N - 1] = madc_hi(cc, a[N - 2], bi, 0);
  }

  // One CIOS row: T = (T >> 32) + a*bi, then T += m*p with m chosen so that the
  // low word cancels.  T = even + (odd << 32).
  static CDL_HD void row(uint32_t* even, uint32_t* odd, const uint32_t* a, uint32_t bi, bool first) {
    CC cc;
    if (first) {
      mul_n(odd, a + 1, bi);
      mul_n(even, a, bi);
    } else {
      even[0] = add_cc(cc, even[0], odd[1]);
      madc_n_rshift(cc, odd, a + 1, bi);
      cmad_n(cc, even, a, bi);
      odd[N - 1] = addc(cc, odd[N - 1], 0);
    }
    uint32_t mi = even[0] * F::M0;
    cmad_mod<1>(cc, odd, mi);
    cmad_mod<0>(cc, even, mi);
    odd[N - 1] = addc(cc, odd[N - 1], 0);
  }

  // r = r - p if r >= p
  static CDL_HD void final_sub(uint32_t* r) {
    uint32_t t[N];
    CC cc;
    t[0] = sub_cc(cc, r[0], F::mod(0));
#pragma unroll
    for (int i = 1; i < N; i++) t[i] = subc_cc(cc, r[i], F::mod(i));
    uint32_t borrow = subc(cc, 0, 0);  // 0 - 0 - CF : 0 or 0xffffffff
#pragma unroll
    for (int i = 0; i < N; i++) r[i] = borrow ? r[i] : t[i];
  }

  // Translation units that define CDL_FP_MUL_CALL route every product through one shared,
  // non-inlined body (operands and result by value, in registers): a kernel whose hot loop
  // would otherwise hold ten inlined copies of the 420-instruction product (~70 KB of
  // SASS) then fits the instruction caches.
#if defined(__CUDA_ARCH__) && defined(CDL_FP_MUL_CALL)
  static __device__ __noinline__ El mul_call(El a, El b) {
    El r;
    mul_inline(r, a, b);
    return r;
  }
  static CDL_HD void mul(El& r, const El& a, const El& b) { r = mul_call(a, b); }
#else
  static CDL_HD void mul(El& r, const El& a, const El& b) { mul_inline(r, a, b); }
#endif

  static CDL_HD void mul_inline(El& r, const El& a, const El& b) {
    uint32_t even[N], odd[N];
#pragma unroll
    for (int i = 0; i < N; i += 2) {
      row(even, odd, a.v, b.v[i], i == 0);
      row(odd, even, a.v, b.v[i + 1], false);
    }
    CC cc;
    even[0] = add_cc(cc, even[0], odd[1]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) even[i] = addc_cc(cc, even[i], odd[i + 1]);
    even[N - 1] = addc(cc, even[N - 1], 0);
    final_sub(even);
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = even[i];
  }

  // ---- dedicated squaring: N(N-1)/2 off-diagonal + N diagonal products for the 2N-limb square, then
  // a pure reduction of its low half (N^2 + N multiply-adds): 78 + 144 + 12 = 234 wide multiply-adds
  // for the 381-bit field against 300 for a general product.
  //
  // The off-diagonal products a_i*a_j (i < j) land at limb i+j: even sums accumulate in E, odd sums
  // in O (a value shifted by 32 bits), so every product is an aligned 64-bit column of one of the two
  // arrays, exactly as in row().  Row i is two carry chains (j = i+1, i+3, .. into O from limb 2i;
  // j = i+2, i+4, .. into E from limb 2i+2); rows are taken in increasing i, so the top of a chain is
  // either a fresh column (absorbs the carry) or spills one bit into a limb nobody has written yet.

  // acc[0..2*cnt) += a[0], a[2], .. (cnt limbs, stride 2) * bi; `fresh` = number of trailing limbs of
  // the chain that have never been written (0, 1 or 2); with fresh == 0 the carry goes to acc[2*cnt].
  template <int CNT, int FRESH>
  static CDL_HD void sq_chain(uint32_t* acc, const uint32_t* a, uint32_t bi) {
    CC cc;
    if (CNT == 1 && FRESH == 2) {
      acc[0] = mul_lo(a[0], bi);
      acc[1] = mul_hi(a[0], bi);
      return;
    }
#pragma unroll
    for (int k = 0; k < CNT; k++) {
      const bool last = k == CNT - 1;
      const uint32_t lo_in = (last && FRESH == 2) ? 0u : acc[2 * k];
      const uint32_t hi_in = (last && FRESH >= 1) ? 0u : acc[2 * k + 1];
      acc[2 * k] = k == 0 ? mad_lo_cc(cc, a[2 * k], bi, lo_in) : madc_lo_cc(cc, a[2 * k], bi, lo_in);
      if (last && FRESH >= 1) acc[2 * k + 1] = madc_hi(cc, a[2 * k], bi, hi_in);
      else acc[2 * k + 1] = madc_hi_cc(cc, a[2 * k], bi, hi_in);
    }
    if (FRESH == 0) acc[2 * CNT] = addc(cc, 0, 0);
  }

  // Number of limbs of E (PAR = 0) / O (PAR = 1) written before row I starts: E rows start at limb
  // 2i+2 and row i's top limb is i + jmax + 1 with jmax the largest j <= N-1 of the right parity.
  template <int PAR>
#if defined(__CUDACC__)
  __host__ __device__
#endif
  static constexpr int sq_written(int I) {
    int top = PAR == 0 ? 2 : 0;  // E[0], E[1] are never written (kept zero); O starts empty
    for (int i = 0; i < I; i++) {
      const int j0 = i + (PAR == 0 ? 2 : 1);
      if (j0 > N - 1) continue;
      const int cnt = (N - 1 - j0) / 2 + 1;
      const int base = PAR == 0 ? 2 * i + 2 : 2 * i;
      int end = base + 2 * cnt;                 // one past the chain's last limb
      if (end <= top) end = base + 2 * cnt + 1; // the chain ended inside written limbs: carry limb
      if (end > top) top = end;
    }
    return top;
  }

  template <int I, int PAR>
  static CDL_HD void sq_row_half(uint32_t* acc, const uint32_t* a) {
    constexpr int j0 = I + (PAR == 0 ? 2 : 1);
    if constexpr (j0 <= N - 1) {
      constexpr int cnt = (N - 1 - j0) / 2 + 1;
      constexpr int base = PAR == 0 ? 2 * I + 2 : 2 * I;
      constexpr int written = sq_written<PAR>(I);
      constexpr int end = base + 2 * cnt;
      static_assert(end >= written, "a chain must end at or above every limb written so far");
      constexpr int fresh = end - written >= 2 ? 2 : (end - written == 1 ? 1 : 0);
      // limbs of the chain below `written` that were skipped by earlier rows cannot exist: every row
      // starts at or above the previous row's start and chains are contiguous
      sq_chain<cnt, fresh>(acc + base, a + j0, a[I]);
    }
  }

  template <int I>
  static CDL_HD void sq_rows(uint32_t* E, uint32_t* O, const uint32_t* a) {
    if constexpr (I < N - 1) {
      sq_row_half<I, 1>(O, a);
      sq_row_half<I, 0>(E, a);
      sq_rows<I + 1>(E, O, a);
    }
  }

  // pure reduction row (row() without the a*b_i part): T = (T + m*p) >> 32
  static CDL_HD void redc_row(uint32_t* even, uint32_t* odd, bool first) {
    CC cc;
    if (first) {
      uint32_t mi = even[0] * F::M0;
      // odd = p_odd * mi (fresh), even += p_even * mi
#pragma unroll
      for (int j = 0; j < N; j += 2) {
        odd[j] = mul_lo(F::mod(1 + j), mi);
        odd[j + 1] = mul_hi(F::mod(1 + j), mi);
      }
      cmad_mod<0>(cc, even, mi);
      odd[N - 1] = addc(cc, odd[N - 1], 0);
      return;
    }
    even[0] = add_cc(cc, even[0], odd[1]);
    uint32_t mi = even[0] * F::M0;
    // odd = (odd >> 64) + p_odd * mi, carry-in from the fold above
#pragma unroll
    for (int j = 0; j < N - 2; j += 2) {
      odd[j] = madc_lo_cc(cc, F::mod(1 + j), mi, odd[j + 2]);
      odd[j + 1] = madc_hi_cc(cc, F::mod(1 + j), mi, odd[j + 3]);
    }
    odd[N - 2] = madc_lo_cc(cc, F::mod(N - 1), mi, 0);
    odd[N - 1] = madc_hi(cc, F::mod(N - 1), mi, 0);
    cmad_mod<0>(cc, even, mi);
    odd[N - 1] = addc(cc, odd[N - 1], 0);
  }

  static CDL_HD void sqr_inline(El& r, const El& a) {
    uint32_t E[2 * N], O[2 * N];
#pragma unroll
    for (int i = 0; i < 2 * N; i++) E[i] = O[i] = 0;
    sq_rows<0>(E, O, a.v);
    // X = E + (O << 32): the off-diagonal half-sum, 2N limbs (X[0] = E[0] = 0)
    uint32_t X[2 * N];
    {
      CC cc;
      X[0] = 0;
      X[1] = add_cc(cc, E[1], O[0]);
#pragma unroll
      for (int i = 2; i < 2 * N - 1; i++) X[i] = addc_cc(cc, E[i], O[i - 1]);
      X[2 * N - 1] = addc(cc, E[2 * N - 1], O[2 * N - 2]);
    }
    // T = 2X + diag: the doubling is a funnel shift, the diagonal squares ride the carry chain
    uint32_t T[2 * N];
    {
      CC cc;
#pragma unroll
      for (int i = 0; i < N; i++) {
        const uint32_t d0 = i == 0 ? 0u : ((X[2 * i] << 1) | (X[2 * i - 1] >> 31));
        const uint32_t d1 = (X[2 * i + 1] << 1) | (X[2 * i] >> 31);
        T[2 * i] = i == 0 ? mad_lo_cc(cc, a.v[i], a.v[i], d0) : madc_lo_cc(cc, a.v[i], a.v[i], d0);
        if (i == N - 1) T[2 * i + 1] = madc_hi(cc, a.v[i], a.v[i], d1);
        else T[2 * i + 1] = madc_hi_cc(cc, a.v[i], a.v[i], d1);
      }
    }
    // reduce the low half (the Montgomery product of T_lo with 1), then add the high half
    uint32_t even[N], odd[N];
#pragma unroll
    for (int i = 0; i < N; i++) even[i] = T[i];
#pragma unroll
    for (int i = 0; i < N; i += 2) {
      redc_row(even, odd, i == 0);
      redc_row(odd, even, false);
    }
    CC cc;
    even[0] = add_cc(cc, even[0], odd[1]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) even[i] = addc_cc(cc, even[i], odd[i + 1]);
    even[N - 1] = addc(cc, even[N - 1], 0);
    CC c2;
    even[0] = add_cc(c2, even[0], T[N]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) even[i] = addc_cc(c2, even[i], T[N + i]);
    even[N - 1] = addc(c2, even[N - 1], T[2 * N - 1]);
    final_sub(even);
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = even[i];
  }

#if defined(CDL_NO_DEDICATED_SQR)  // A/B switch for tools/kbench.cu
  static CDL_HD void sqr(El& r, const El& a) { mul(r, a, a); }
#elif defined(__CUDA_ARCH__) && defined(CDL_FP_MUL_CALL)
  static __device__ __noinline__ El sqr_call(El a) {
    El r;
    sqr_inline(r, a);
    return r;
  }
  static CDL_HD void sqr(El& r, const El& a) { r = sqr_call(a); }
#else
  static CDL_HD void sqr(El& r, const El& a) { sqr_inline(r, a); }
#endif

  static CDL_HD void add(El& r, const El& a, const El& b) {
    uint32_t t[N];
    CC cc;
    t[0] = add_cc(cc, a.v[0], b.v[0]);
#pragma unroll
    for (int i = 1; i < N; i++) t[i] = addc_cc(cc, a.v[i], b.v[i]);
    final_sub(t);  // moduli here leave >= 1 spare top bit: no carry out of limb N-1
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = t[i];
  }

  static CDL_HD void sub(El& r, const El& a, const El& b) {
    uint32_t t[N];
    CC cc;
    t[0] = sub_cc(cc, a.v[0], b.v[0]);
#pragma unroll
    for (int i = 1; i < N; i++) t[i] = subc_cc(cc, a.v[i], b.v[i]);
    uint32_t borrow = subc(cc, 0, 0);
    CC c2;
    t[0] = add_cc(c2, t[0], borrow & F::mod(0));
#pragma unroll
    for (int i = 1; i < N - 1; i++) t[i] = addc_cc(c2, t[i], borrow & F::mod(i));
    t[N - 1] = addc(c2, t[N - 1], borrow & F::mod(N - 1));
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = t[i];
  }

  static CDL_HD void dbl(El& r, const El& a) { add(r, a, a); }

  static CDL_HD bool is_zero(const El& a) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < N; i++) o |= a.v[i];
    return o == 0;
  }

  static CDL_HD void neg(El& r, const El& a) {
    uint32_t t[N];
    CC cc;
    t[0] = sub_cc(cc, F::mod(0), a.v[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) t[i] = subc_cc(cc, F::mod(i), a.v[i]);
    t[N - 1] = subc(cc, F::mod(N - 1), a.v[N - 1]);
    bool z = is_zero(a);
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = z ? 0u : t[i];
  }

  static CDL_HD bool eq(const El& a, const El& b) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < N; i++) o |= a.v[i] ^ b.v[i];
    return o == 0;
  }

  static CDL_HD void set_zero(El& r) {
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = 0;
  }

  static CDL_HD void set_one(El& r) {
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = F::one(i);
  }

  static CDL_HD void cmov(El& r, const El& a, bool c) {
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = c ? a.v[i] : r.v[i];
  }

  // Montgomery form -> canonical integer limbs (one reduction pass: a * 1).
  static CDL_HD void from_mont(El& r, const El& a) {
    El one_raw;
    set_zero(one_raw);
    one_raw.v[0] = 1;
    mul(r, a, one_raw);
  }

  static CDL_HD void to_mont(El& r, const El& a) {
    El r2;
#pragma unroll
    for (int i = 0; i < N; i++) r2.v[i] = F::r2(i);
    mul(r, a, r2);
  }
};

}  // namespace cdl
