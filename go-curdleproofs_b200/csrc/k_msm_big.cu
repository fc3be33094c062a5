// Large single MSM: signed-digit Pippenger with an on-GPU counting sort of bucket
// indices.  Replaces (*G1Jac).MultiExp when one call carries thousands to
// millions of terms (BASELINE.json config 5, the standalone sweep 2^10..2^22;
// gnark's MultiExp is reached from msmaccumulator/msmaccumulator.go:59 and
// common/util.go:75 with the same signature).
//
//   k_big_tables     gather table of the bases: P and phi(P) = (beta*x, y) (the GLV endomorphism),
//                    one 128-byte line each
//   k_big_digits<0>  thread per scalar: Montgomery -> canonical -> GLV halves (< 2^127),
//                    signed c-bit digits d_w in [-2^(c-1), 2^(c-1)] of both halves,
//                    histogram of (window, |d|) keys
//   k_scan_*         exclusive prefix sum of the histogram (bucket offsets)
//   k_big_digits<1>  same digits again, scatter (point index | sign) to the bucket's
//                    slot — a counting sort; order inside a bucket is irrelevant
//   k_big_size_sort  buckets ordered by decreasing length (counting sort), so that the
//                    32 buckets of a warp have nearly equal trip counts
//   k_ba_fwd / k_ba_inv / k_ba_bwd
//                    batch-affine rounds (batch_affine.cuh): every bucket's region of the sorted
//                    entries is padded to a multiple of 2^R slots, so that for R rounds the
//                    neighbouring slots (2k, 2k+1) of the whole array are summed pairwise as
//                    AFFINE additions — 6 field products each, the inversions shared by
//                    Montgomery's trick across the pairs of a thread and then across threads —
//                    and a bucket's region simply halves.  What is left (count / 2^R points
//                    per bucket) goes to k_big_accum.
//   k_big_accum      thread per bucket: XYZZ mixed additions of the bucket's points
//   k_big_slice / k_big_large_finish
//                    buckets above kBigLargeBucket entries (degenerate inputs: all
//                    equal scalars, tiny scalars) are cut into slices summed by a
//                    whole CTA each, so no thread ever walks a long list alone
//   k_big_reduce1    thread per chunk of L buckets: running-sum trick inside the
//                    chunk plus (chunk base)*sum by a short double-and-add
//   k_big_sum        tree of plain sums down to one point per window
//   k_big_horner     windows top-down (c doublings each), optional normalisation
//
// A rank of a multi-GPU job owns windows wfirst, wfirst + wstep, ... and returns
// its partial sum already shifted, so the exchange is one all-gather of one point
// per rank (k_big_combine adds them).
#define CDL_FP_MUL_CALL 1  // one shared product body: the hot loops fit the instruction caches (mont.cuh)
#include <cstdlib>
#include "quad.cuh"
#include "batch_affine.cuh"
#include "launch.h"

namespace cdl {

constexpr uint32_t kBigLargeBucket = 2048;  // upper bound of BigMsmDims::large (entries); longer buckets take the slice path
constexpr uint32_t kBigSliceLen = 2048;     // entries per slice (16 per thread of a 128-thread CTA)
constexpr int kBigCtaThreads = 128;

struct BigSliceRec {
  uint32_t first, count;
};
struct BigLargeRec {
  uint32_t bucket, slice_first, slice_count, pad;
};

// The bucket sums gather their operands at random, and a random read costs a whole 128-byte L2 line
// of DRAM traffic whatever its size (measured: 117 B per 48-byte coordinate in a 64-byte slot, 257 B per
// point as two such slots, 203 B per 96-byte point straddling lines).  So the bases are re-laid once
// per MSM as one table of 2n points, tab[0 .. n) = P and tab[n .. 2n) = phi(P) = (beta * x, y) (the GLV
// endomorphism), each in its own 128-byte line: a gathered point, or its x alone, is exactly one line.
struct alignas(128) BigPoint {
  Fp x, y;
  uint32_t pad[8];
};

// Where the summands of a bucket come from: the sorted entries (a gather from the coordinate tables,
// bit 31 = negate, an index beyond the tables = padding = infinity), or — after batch-affine
// rounds — the affine pair sums of the last round, in place.
struct BigSrc {
  const BigPoint* tab;  // 2n slots: [P | phi(P)]
  uint32_t n;
  const uint32_t* entries;
  const G1Affine* direct;  // non-null: slot t holds its point
};
template <bool DIRECT>
__device__ __forceinline__ G1Affine big_src_load(const BigSrc& s, uint32_t t) {
  if (DIRECT) return s.direct[t];
  G1Affine q;
  const uint32_t en = s.entries[t];
  const uint32_t pi = en & 0x7fffffffu;
  if (pi >= 2u * s.n) {
    aff_set_inf(q);
    return q;
  }
  q.x = s.tab[pi].x;
  q.y = s.tab[pi].y;
  if (en >> 31) FpM::neg(q.y, q.y);
  return q;
}
// x coordinate only (the forward pass of a batch-affine round needs nothing else for almost every pair)
template <bool DIRECT>
__device__ __forceinline__ Fp big_src_load_x(const BigSrc& s, uint32_t t) {
  if (DIRECT) return s.direct[t].x;
  const uint32_t pi = s.entries[t] & 0x7fffffffu;
  if (pi >= 2u * s.n) {
    Fp x;
    FpM::set_zero(x);
    return x;
  }
  return s.tab[pi].x;
}

// ---------------------------------------------------------------- digits
// Every scalar is split with the GLV endomorphism, k = +-|k1| +- k2*lambda with |k1|, k2 <
// 2^127 (glv.cuh), so a term contributes to W = ceil(128/c) windows twice — once with P,
// once with phi(P) = (beta*x, y), which k_big_phi tabulates — instead of to ceil(256/c)
// windows once: the same number of bucket additions, but half the windows to reduce and
// half the doublings in the final Horner chain.
// window w digit of a 128-bit magnitude (6 words, top two zero)
__device__ __forceinline__ uint32_t big_raw_digit(const uint32_t* k6, int w, int c) {
  int bit = w * c;
  int word = bit >> 5, sh = bit & 31;
  uint32_t lo = k6[word], hi = k6[word + 1];
  uint32_t v = __funnelshift_r(lo, hi, sh);
  return v & ((1u << c) - 1u);
}

__global__ void __launch_bounds__(256)
k_big_tables(const G1Affine* __restrict__ points, const uint32_t* __restrict__ idx, int n, BigPoint* __restrict__ tab) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const G1Affine p = points[idx ? idx[i] : (uint32_t)i];
  Fp beta, bx;
  fp_set_beta(beta);
  FpM::mul(bx, p.x, beta);  // infinity (0, 0) stays (0, 0)
  tab[i].x = p.x;
  tab[i].y = p.y;
  tab[i + n].x = bx;
  tab[i + n].y = p.y;
}

// entry = index into tab[] = [P | phi(P)] (bit 31: negate)
template <int PASS>
__global__ void __launch_bounds__(256)
k_big_digits(const Fr* __restrict__ scalars, int n, BigMsmDims dm, uint32_t* __restrict__ counters,
             const uint32_t* __restrict__ offsets, uint32_t* __restrict__ entries) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = i < n;
  uint32_t k6[2][6];
  bool neg[2] = {false, false};
#pragma unroll
  for (int h = 0; h < 2; h++)
#pragma unroll
    for (int j = 0; j < 6; j++) k6[h][j] = 0;
  if (live) {
    Fr km = scalars[i], k;
    FrM::from_mont(k, km);
    Glv g;
    glv_decompose(g, k.v);
#pragma unroll
    for (int j = 0; j < 4; j++) { k6[0][j] = g.k1[j]; k6[1][j] = g.k2[j]; }
    neg[0] = g.neg1;
    neg[1] = g.neg2;
  }
  const uint32_t lane = threadIdx.x & 31;
#pragma unroll 1
  for (int h = 0; h < 2; h++) {
    uint32_t carry = 0;
    int next_local = dm.wfirst, j = 0;
#pragma unroll 1
    for (int w = 0; w < dm.W; w++) {
      uint32_t t = (w * dm.c < 128 ? big_raw_digit(k6[h], w, dm.c) : 0u) + carry;
      carry = t > (uint32_t)dm.M ? 1u : 0u;
      if (w != next_local) continue;  // uniform: every lane walks the same windows
      int32_t d = carry ? (int32_t)t - (int32_t)(2 * dm.M) : (int32_t)t;
      uint32_t key = 0xffffffffu;
      if (live && d != 0) key = (uint32_t)j * (uint32_t)dm.M + (uint32_t)(d < 0 ? -d : d) - 1u;
      // warp-aggregated atomic: one add per distinct key in the warp (degenerate inputs put
      // all 32 lanes on one counter)
      uint32_t peers = __match_any_sync(0xffffffffu, key);
      uint32_t leader = __ffs(peers) - 1;
      uint32_t rank = __popc(peers & ((1u << lane) - 1u));
      uint32_t base = 0;
      if (key != 0xffffffffu && lane == leader) base = atomicAdd(&counters[key], (uint32_t)__popc(peers));
      base = __shfl_sync(0xffffffffu, base, leader);
      if (PASS == 1 && key != 0xffffffffu)
        entries[offsets[key] + base + rank] =
            ((uint32_t)i + (h ? (uint32_t)n : 0u)) | (((d < 0) != neg[h]) ? 0x80000000u : 0u);
      next_local += dm.wstep;
      j++;
    }
  }
}

// ---------------------------------------------------------------- scan (exclusive, n + 1 outputs)
// Three launches: per-block sums, one block scanning the block sums, per-block rescan.
// A block covers 256 * ipt counters (ipt <= 16), so n <= 4096 * 4096.
constexpr int kScanMaxIpt = 16;

__global__ void __launch_bounds__(256)
k_scan_block_sums(const uint32_t* __restrict__ in, uint32_t n, int ipt, uint32_t pad, uint32_t* __restrict__ bsum) {
  __shared__ uint32_t sh[256];
  uint32_t base = (blockIdx.x * 256u + threadIdx.x) * (uint32_t)ipt;
  uint32_t s = 0;
  for (int k = 0; k < ipt; k++) s += (base + k < n) ? ((in[base + k] + pad) & ~pad) : 0u;
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int st = 128; st >= 1; st >>= 1) {
    if ((int)threadIdx.x < st) sh[threadIdx.x] += sh[threadIdx.x + st];
    __syncthreads();
  }
  if (threadIdx.x == 0) bsum[blockIdx.x] = sh[0];
}

// single block: exclusive scan of nblk block sums in place (nblk <= 4096)
__global__ void __launch_bounds__(1024)
k_scan_top(uint32_t* __restrict__ bsum, uint32_t nblk) {
  __shared__ uint32_t sh[1024];
  uint32_t v[4];
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    uint32_t idx = threadIdx.x * 4 + k;
    v[k] = idx < nblk ? bsum[idx] : 0u;
    s += v[k];
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {  // Hillis-Steele inclusive scan
    uint32_t t = (int)threadIdx.x >= off ? sh[threadIdx.x - off] : 0u;
    __syncthreads();
    sh[threadIdx.x] += t;
    __syncthreads();
  }
  uint32_t run = sh[threadIdx.x] - s;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    uint32_t idx = threadIdx.x * 4 + k;
    if (idx < nblk) bsum[idx] = run;
    run += v[k];
  }
}

// offsets[i] = exclusive prefix of counts (each rounded up to a multiple of pad + 1); offsets[n] =
// total; counts are zeroed (they become the scatter cursors)
__global__ void __launch_bounds__(256)
k_scan_apply(uint32_t* __restrict__ counts, uint32_t n, int ipt, uint32_t pad, const uint32_t* __restrict__ bsum,
             uint32_t* __restrict__ offsets) {
  __shared__ uint32_t sh[256];
  uint32_t base = (blockIdx.x * 256u + threadIdx.x) * (uint32_t)ipt;
  uint32_t v[kScanMaxIpt];
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < kScanMaxIpt; k++) {
    v[k] = (k < ipt && base + k < n) ? ((counts[base + k] + pad) & ~pad) : 0u;
    s += v[k];
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int off = 1; off < 256; off <<= 1) {
    uint32_t t = (int)threadIdx.x >= off ? sh[threadIdx.x - off] : 0u;
    __syncthreads();
    sh[threadIdx.x] += t;
    __syncthreads();
  }
  uint32_t run = bsum[blockIdx.x] + sh[threadIdx.x] - s;
#pragma unroll
  for (int k = 0; k < kScanMaxIpt; k++) {
    if (k < ipt && base + k < n) {
      offsets[base + k] = run;
      counts[base + k] = 0;
      if (base + k + 1 == n) offsets[n] = run + v[k];
    }
    run += v[k];
  }
}

// counts[0..n) -> offsets[0..n] (exclusive prefix, total in offsets[n]); counts zeroed; bsum: 4096 words.
// pad = 2^R - 1 rounds every count up to a multiple of 2^R first (batch-affine layout).
cudaError_t launch_exclusive_scan(uint32_t* counts, uint32_t n, uint32_t* bsum, uint32_t* offsets, cudaStream_t st,
                                  uint32_t pad) {
  if (n == 0) return cudaMemsetAsync(offsets, 0, 4, st);
  int ipt = 4;
  while ((uint64_t)4096 * 256 * ipt < n && ipt < kScanMaxIpt) ipt *= 2;
  uint32_t per = 256u * (uint32_t)ipt;
  uint32_t nblk = (n + per - 1) / per;
  if (nblk > 4096) return cudaErrorInvalidValue;
  k_scan_block_sums<<<nblk, 256, 0, st>>>(counts, n, ipt, pad, bsum);
  k_scan_top<<<1, 1024, 0, st>>>(bsum, nblk);
  k_scan_apply<<<nblk, 256, 0, st>>>(counts, n, ipt, pad, bsum, offsets);
  return cudaGetLastError();
}

// ---------------------------------------------------------------- large buckets
// meta[0] = number of large buckets, meta[1] = number of slices
__global__ void __launch_bounds__(256)
k_big_mark_large(const uint32_t* __restrict__ offsets, int shift, uint32_t nb, uint32_t large_thresh,
                 uint32_t* __restrict__ meta, BigLargeRec* __restrict__ large, BigSliceRec* __restrict__ slices) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  uint32_t s = offsets[b] >> shift, cnt = (offsets[b + 1] >> shift) - s;
  if (cnt <= large_thresh) return;
  uint32_t ns = (cnt + kBigSliceLen - 1) / kBigSliceLen;
  uint32_t li = atomicAdd(&meta[0], 1u);
  uint32_t sf = atomicAdd(&meta[1], ns);
  large[li] = BigLargeRec{b, sf, ns, 0};
  for (uint32_t k = 0; k < ns; k++) {
    uint32_t first = s + k * kBigSliceLen;
    uint32_t c = cnt - k * kBigSliceLen;
    slices[sf + k] = BigSliceRec{first, c < kBigSliceLen ? c : kBigSliceLen};
  }
}

// CTA-wide sum of one XYZZ value per thread; result in sh[0]
__device__ __forceinline__ void big_cta_tree(G1Xyzz* sh, const G1Xyzz& mine) {
  const int t = threadIdx.x;
  sh[t] = mine;
  __syncthreads();
#pragma unroll 1
  for (int s = kBigCtaThreads / 2; s >= 1; s >>= 1) {
    if (t < s) {
      G1Xyzz a = sh[t], b = sh[t + s];
      xyzz_add(a, a, b);
      sh[t] = a;
    }
    __syncthreads();
  }
}

template <bool DIRECT>
__global__ void __launch_bounds__(kBigCtaThreads)
k_big_slice(const BigSrc src, const uint32_t* __restrict__ meta,
            const BigSliceRec* __restrict__ slices, G1Xyzz* __restrict__ slice_out) {
  __shared__ G1Xyzz sh[kBigCtaThreads];
  const uint32_t nslices = meta[1];
#pragma unroll 1
  for (uint32_t s = blockIdx.x; s < nslices; s += gridDim.x) {
    BigSliceRec r = slices[s];
    G1Xyzz acc;
    xyzz_set_inf(acc);
#pragma unroll 1
    for (uint32_t t = threadIdx.x; t < r.count; t += kBigCtaThreads) {
      const G1Affine q = big_src_load<DIRECT>(src, r.first + t);
      xyzz_add_mixed(acc, acc, q);
    }
    big_cta_tree(sh, acc);
    if (threadIdx.x == 0) slice_out[s] = sh[0];
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kBigCtaThreads)
k_big_large_finish(const uint32_t* __restrict__ meta, const BigLargeRec* __restrict__ large,
                   const G1Xyzz* __restrict__ slice_out, G1Xyzz* __restrict__ buckets) {
  __shared__ G1Xyzz sh[kBigCtaThreads];
  const uint32_t nlarge = meta[0];
#pragma unroll 1
  for (uint32_t l = blockIdx.x; l < nlarge; l += gridDim.x) {
    BigLargeRec r = large[l];
    G1Xyzz acc;
    xyzz_set_inf(acc);
#pragma unroll 1
    for (uint32_t t = threadIdx.x; t < r.slice_count; t += kBigCtaThreads) {
      G1Xyzz p = slice_out[r.slice_first + t];
      xyzz_add(acc, acc, p);
    }
    big_cta_tree(sh, acc);
    if (threadIdx.x == 0) buckets[r.bucket] = sh[0];
    __syncthreads();
  }
}

// ---------------------------------------------------------------- size-ordered schedule
// Buckets are handed to threads in order of decreasing length (a counting sort on the
// length), so the 32 buckets of a warp have (almost) the same trip count and no lane waits
// for a longer neighbour.  Lengths above kBigLargeBucket count as 0 (slice path).
__device__ __forceinline__ uint32_t big_size_bin(const uint32_t* __restrict__ offsets, int shift, uint32_t b, uint32_t large_thresh) {
  uint32_t cnt = (offsets[b + 1] >> shift) - (offsets[b] >> shift);
  if (cnt > large_thresh) cnt = 0;
  return large_thresh - cnt;  // bin 0 = longest
}

template <int PASS>
__global__ void __launch_bounds__(256)
k_big_size_sort(const uint32_t* __restrict__ offsets, int shift, uint32_t nb, uint32_t large_thresh,
                uint32_t* __restrict__ bin_counters, const uint32_t* __restrict__ bin_offsets,
                uint32_t* __restrict__ order) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t lane = threadIdx.x & 31;
  uint32_t bin = b < nb ? big_size_bin(offsets, shift, b, large_thresh) : 0xffffffffu;
  uint32_t peers = __match_any_sync(0xffffffffu, bin);
  uint32_t leader = __ffs(peers) - 1;
  uint32_t rank = __popc(peers & ((1u << lane) - 1u));
  uint32_t base = 0;
  if (bin != 0xffffffffu && lane == leader) base = atomicAdd(&bin_counters[bin], (uint32_t)__popc(peers));
  base = __shfl_sync(0xffffffffu, base, leader);
  if (PASS == 1 && bin != 0xffffffffu) order[bin_offsets[bin] + base + rank] = b;
}

// ---------------------------------------------------------------- batch-affine rounds
// Round r sums the slots (2k, 2k + 1) of its input (the sorted entries in round 1, the previous
// round's sums afterwards) into slot k of its output.  Every bucket's region starts at a multiple of
// 2^R slots and spans a multiple of 2^R, so pairs never straddle two buckets and the regions are
// offsets >> r after round r; padding slots hold infinity.  total_ptr -> offsets[nb] (the padded
// number of entries, known only on the device); the grid is sized by its host-side upper bound.
//
// The grid is a whole number of waves of resident CTAs and every CTA owns the same number of
// consecutive pairs, kBaThreads * bpt with bpt = ceil(pairs / threads) — no half-empty last wave.
// Thread t of a CTA takes the pairs base + t + j * kBaThreads (so a warp's loads and stores are
// contiguous), and the pairs of a thread share one inversion
// (batch_affine.cuh): k_ba_fwd leaves the running products of the denominators in pre[] and the
// thread's total in totals[]; k_ba_inv inverts all totals (the same trick one level up, one real
// inversion per thread); k_ba_bwd peels the factors off and writes the sums.
constexpr int kBaThreads = 128;
__host__ __device__ __forceinline__ uint32_t ba_pairs_per_thread(uint32_t npairs, uint32_t nblk) {
  const uint32_t threads = nblk * (uint32_t)kBaThreads;
  return (npairs + threads - 1) / threads;
}

template <bool DIRECT>
__global__ void __launch_bounds__(kBaThreads)
k_ba_fwd(const BigSrc src, const uint32_t* __restrict__ total_ptr, int shift, Fp* __restrict__ pre,
         Fp* __restrict__ totals) {
  const uint32_t npairs = (total_ptr[0] >> shift) >> 1;
  const int bpt = (int)ba_pairs_per_thread(npairs, gridDim.x);
  uint32_t k = blockIdx.x * (uint32_t)(kBaThreads * bpt) + threadIdx.x;
  Fp run;
  FpM::set_one(run);
#pragma unroll 1
  for (int j = 0; j < bpt && k < npairs; j++, k += kBaThreads) {
    const Fp x1 = big_src_load_x<DIRECT>(src, 2 * k), x2 = big_src_load_x<DIRECT>(src, 2 * k + 1);
    Fp d;
    FpM::sub(d, x2, x1);
    if (FpM::is_zero(d)) {  // rare: equal points, opposite points, padding
      const G1Affine p1 = big_src_load<DIRECT>(src, 2 * k), p2 = big_src_load<DIRECT>(src, 2 * k + 1);
      ba_denominator_equal_x(d, p1.y, p2.y);
    }
    if (j == 0) run = d;
    else FpM::mul(run, run, d);
    pre[k] = run;
  }
  totals[blockIdx.x * kBaThreads + threadIdx.x] = run;
}

// totals[i] <- 1 / totals[i]; thread t of a CTA owns the G totals base + t + j * blockDim
__global__ void __launch_bounds__(kBaThreads)
k_ba_inv(Fp* __restrict__ totals, Fp* __restrict__ tpre, uint32_t ntot, int G) {
  const uint32_t first = blockIdx.x * (uint32_t)(kBaThreads * G) + threadIdx.x;
  if (first >= ntot) return;
  Fp run = totals[first];
  int cnt = 1;
#pragma unroll 1
  for (uint32_t i = first + kBaThreads; cnt < G && i < ntot; i += kBaThreads, cnt++) {
    tpre[i - kBaThreads] = run;
    const Fp t = totals[i];
    FpM::mul(run, run, t);
  }
  Fp inv;
  fp_inv(inv, run);
#pragma unroll 1
  for (int j = cnt - 1; j >= 1; j--) {
    const uint32_t i = first + (uint32_t)j * kBaThreads;
    const Fp t = totals[i], p = tpre[i - kBaThreads];
    Fp o;
    FpM::mul(o, inv, p);
    totals[i] = o;
    FpM::mul(inv, inv, t);
  }
  totals[first] = inv;
}

template <bool DIRECT>
__global__ void __launch_bounds__(kBaThreads, 4)
k_ba_bwd(const BigSrc src, const uint32_t* __restrict__ total_ptr, int shift, const Fp* __restrict__ pre,
         const Fp* __restrict__ totals, G1Affine* __restrict__ dst) {
  const uint32_t npairs = (total_ptr[0] >> shift) >> 1;
  const int bpt = (int)ba_pairs_per_thread(npairs, gridDim.x);
  const uint32_t k0 = blockIdx.x * (uint32_t)(kBaThreads * bpt) + threadIdx.x;
  if (k0 >= npairs) return;
  uint32_t cnt = (npairs - k0 + kBaThreads - 1) / kBaThreads;
  if (cnt > (uint32_t)bpt) cnt = (uint32_t)bpt;
  Fp inv = totals[blockIdx.x * kBaThreads + threadIdx.x];
#pragma unroll 1
  for (int j = (int)cnt - 1; j >= 0; j--) {
    const uint32_t k = k0 + (uint32_t)j * kBaThreads;
    const G1Affine p1 = big_src_load<DIRECT>(src, 2 * k), p2 = big_src_load<DIRECT>(src, 2 * k + 1);
    Fp invj = inv;
    if (j > 0) {
      Fp d;
      ba_denominator(d, p1, p2);
      const Fp pj = pre[k - kBaThreads];
      FpM::mul(invj, inv, pj);
      FpM::mul(inv, inv, d);
    }
    G1Affine r;
    ba_pair_sum(r, p1, p2, invj);
    dst[k] = r;
  }
}

// ---------------------------------------------------------------- bucket accumulation
template <bool DIRECT>
__global__ void __launch_bounds__(128, 3)
k_big_accum(const BigSrc src, const uint32_t* __restrict__ offsets, int shift,
            const uint32_t* __restrict__ order, uint32_t nb, uint32_t large_thresh,
            G1Xyzz* __restrict__ buckets) {
  uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= nb) return;
  const uint32_t b = order[tid];
  uint32_t s = offsets[b] >> shift, e = offsets[b + 1] >> shift;
  G1Xyzz acc;
  xyzz_set_inf(acc);
  if (e - s <= large_thresh) {
#pragma unroll 1
    for (uint32_t t = s; t < e; t++) {
      const G1Affine q = big_src_load<DIRECT>(src, t);
      xyzz_add_mixed(acc, acc, q);
    }
  }
  buckets[b] = acc;  // large buckets are filled in by k_big_large_finish
}

// ---------------------------------------------------------------- bucket reduction
// r = e * p, small public-size e (MSB-first double-and-add)
__device__ __forceinline__ void xyzz_mul_small(G1Xyzz& r, const G1Xyzz& p, uint32_t e) {
  xyzz_set_inf(r);
  if (e == 0) return;
  int top = 31 - __clz(e);
  r = p;
#pragma unroll 1
  for (int i = top - 1; i >= 0; i--) {
    xyzz_dbl(r, r);
    if ((e >> i) & 1u) xyzz_add(r, r, p);
  }
}

// thread (j, ch): P = sum_{i < L} (ch*L + i + 1) * B[j*M + ch*L + i]
__global__ void __launch_bounds__(128, 3)
k_big_reduce1(const G1Xyzz* __restrict__ buckets, int M, int L, int nchunks_total, G1Xyzz* __restrict__ out) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nchunks_total) return;
  const int per = M / L;
  const int j = t / per, ch = t - j * per;
  const G1Xyzz* B = buckets + (size_t)j * M + (size_t)ch * L;
  G1Xyzz run, acc;
  xyzz_set_inf(run);
  xyzz_set_inf(acc);
#pragma unroll 1
  for (int i = L - 1; i >= 0; i--) {
    G1Xyzz b = B[i];
    xyzz_add(run, run, b);
    xyzz_add(acc, acc, run);
  }
  if (ch > 0) {
    G1Xyzz s;
    xyzz_mul_small(s, run, (uint32_t)ch * (uint32_t)L);
    xyzz_add(acc, acc, s);
  }
  out[t] = acc;
}

// The same two reductions with a QUAD of lanes per output (quad.cuh), for small MSMs: with a few hundred
// outputs the serial chains above (30 and 16 group operations) are pure latency; a quad runs each
// addition in four product latencies instead of fourteen.
__device__ __forceinline__ void qxyzz_mul_small(const Quad& q, G1Xyzz& r, const G1Xyzz& p, uint32_t e) {
  xyzz_set_inf(r);
  if (e == 0) return;
  int top = 31 - __clz(e);
  r = p;
#pragma unroll 1
  for (int i = top - 1; i >= 0; i--) {
    qxyzz_dbl(q, r, r);
    if ((e >> i) & 1u) qxyzz_add(q, r, r, p);
  }
}

__global__ void __launch_bounds__(128)
k_big_reduce1_quad(const G1Xyzz* __restrict__ buckets, int M, int L, int nchunks_total, G1Xyzz* __restrict__ out) {
  const Quad q;
  int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;
  if (t >= nchunks_total) return;  // the whole quad
  const int per = M / L;
  const int j = t / per, ch = t - j * per;
  const G1Xyzz* B = buckets + (size_t)j * M + (size_t)ch * L;
  G1Xyzz run, acc;
  xyzz_set_inf(run);
  xyzz_set_inf(acc);
#pragma unroll 1
  for (int i = L - 1; i >= 0; i--) {
    const G1Xyzz b = B[i];
    qxyzz_add(q, run, run, b);
    qxyzz_add(q, acc, acc, run);
  }
  if (ch > 0) {
    G1Xyzz s;
    qxyzz_mul_small(q, s, run, (uint32_t)ch * (uint32_t)L);
    qxyzz_add(q, acc, acc, s);
  }
  if (q.lane == 0) out[t] = acc;
}

__global__ void __launch_bounds__(128)
k_big_sum_quad(const G1Xyzz* __restrict__ in, int pin, int G, int pout, int total_out, G1Xyzz* __restrict__ out) {
  const Quad q;
  int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;
  if (t >= total_out) return;
  const int j = t / pout, g = t - j * pout;
  int lo = g * G, hi = lo + G < pin ? lo + G : pin;
  G1Xyzz acc;
  xyzz_set_inf(acc);
#pragma unroll 1
  for (int i = lo; i < hi; i++) {
    const G1Xyzz p = in[(size_t)j * pin + i];
    qxyzz_add(q, acc, acc, p);
  }
  if (q.lane == 0) out[t] = acc;
}
constexpr int kBigQuadMaxOutputs = 8192;  // below this many outputs the reductions run a quad per output

// out[j*pout + g] = sum of in[j*pin + g*G .. +G)
__global__ void __launch_bounds__(128, 3)
k_big_sum(const G1Xyzz* __restrict__ in, int pin, int G, int pout, int total_out, G1Xyzz* __restrict__ out) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total_out) return;
  const int j = t / pout, g = t - j * pout;
  int lo = g * G, hi = lo + G < pin ? lo + G : pin;
  G1Xyzz acc;
  xyzz_set_inf(acc);
#pragma unroll 1
  for (int i = lo; i < hi; i++) {
    G1Xyzz p = in[(size_t)j * pin + i];
    xyzz_add(acc, acc, p);
  }
  out[t] = acc;
}

// acc = sum_j 2^(c*(wfirst + j*wstep)) * S_j ; optional normalisation to (x, y, 1) / (1, 1, 0).
// The chain is serial by nature (c * W doublings), so it runs on one QUAD of lanes (quad.cuh): three
// product latencies per doubling instead of nine.
__global__ void k_big_horner(const G1Xyzz* __restrict__ S, BigMsmDims dm, int normalize, G1Jac* __restrict__ out) {
  if (threadIdx.x >= 4 || blockIdx.x != 0) return;
  const Quad q;
  G1Xyzz acc;
  xyzz_set_inf(acc);
#pragma unroll 1
  for (int j = dm.nlocal - 1; j >= 0; j--) {
    if (j != dm.nlocal - 1) {
#pragma unroll 1
      for (int k = 0; k < dm.c * dm.wstep; k++) qxyzz_dbl(q, acc, acc);
    }
    const G1Xyzz s = S[j];
    qxyzz_add(q, acc, acc, s);
  }
#pragma unroll 1
  for (int k = 0; k < dm.c * dm.wfirst; k++) qxyzz_dbl(q, acc, acc);
  G1Jac r;
  if (normalize) {
    G1Affine a;
    qxyzz_to_affine(q, a, acc);
    jac_from_affine(r, a);
  } else {
    xyzz_to_jac(r, acc);
  }
  if (q.lane == 0) out[0] = r;
}

// out = sum of n Jacobian points (the per-rank partial sums), normalised
__global__ void k_big_combine(const G1Jac* __restrict__ in, int n, G1Jac* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  G1Jac acc;
  jac_set_inf(acc);
#pragma unroll 1
  for (int i = 0; i < n; i++) {
    G1Jac p = in[i];
    jac_add(acc, acc, p);
  }
  G1Affine a;
  jac_to_affine(a, acc);
  jac_from_affine(acc, a);
  out[0] = acc;
}

// ---------------------------------------------------------------- host side
// window width by size, measured on B200 (tools/msm_sweep.py --scan-c, profiles/r2_msm_window_scan.txt)
int big_msm_pick_c(size_t n) {
  int lg = 0;
  while (((size_t)1 << (lg + 1)) <= n) lg++;
  static const int table[] = {8, 8, 8, 8, 8, 8, 8, 8, 8, 8, 8, 9, 11, 12, 12, 15, 16, 16, 16, 16, 16};
  return lg <= 20 ? table[lg] : 16;
}

// Batch-affine rounds by the mean number of entries per bucket: a round halves every bucket at 6.3
// instead of 10 products per addition, but pads every bucket to a multiple of 2^R slots (2^R / 2 wasted
// pair slots on average) and costs three more launches, one of them a field inversion's latency long;
// below ~ 16 entries per bucket it does not pay (measured with c = 16, profiles/r3_msm_ba_scan.txt:
// 2^17 -> 0 rounds, 2^18 -> 1, 2^19 / 2^20 -> 2, 2^21 -> 3, 2^22 -> 4).
static int big_msm_pick_rounds(size_t mean) {
  static const int forced = [] {
    const char* e = getenv("CDL_MSM_BATCH_AFFINE");
    return e ? atoi(e) : -1;
  }();
  if (forced >= 0) return forced > kBigMaxBaRounds ? kBigMaxBaRounds : forced;
  int lg = 0;
  while (((size_t)2 << lg) <= mean) lg++;
  int r = lg <= 5 ? lg - 3 : lg - 4;  // leaves 8 .. 31 points per bucket to the XYZZ pass
  return r < 0 ? 0 : r > kBigMaxBaRounds ? kBigMaxBaRounds : r;
}

BigMsmDims big_msm_dims(size_t n, int c, int wfirst, int wstep, int ba_rounds) {
  BigMsmDims d;
  d.n = (int)n;
  d.c = c;
  d.W = (128 + c - 1) / c;  // windows over the 128-bit GLV halves
  d.M = 1 << (c - 1);
  d.wfirst = wfirst;
  d.wstep = wstep;
  d.nlocal = wfirst < d.W ? (d.W - wfirst + wstep - 1) / wstep : 0;
  d.nb = (uint32_t)d.nlocal * (uint32_t)d.M;
  size_t mean = 2 * n / (size_t)d.M + 1;
  d.R = ba_rounds >= 0 ? (ba_rounds > kBigMaxBaRounds ? kBigMaxBaRounds : ba_rounds) : big_msm_pick_rounds(mean);
  if (d.nlocal == 0 || n == 0) d.R = 0;
  // a bucket longer than 8x the mean goes to the CTA-per-slice path instead of one thread
  // (degenerate scalars, and the top window, which holds only 256 - c*(W-1) scalar bits);
  // lengths are those the XYZZ pass sees, i.e. after the batch-affine rounds
  size_t lt = 8 * ((mean >> d.R) + 1);
  d.large = (uint32_t)(lt < 64 ? 64 : lt > kBigLargeBucket ? kBigLargeBucket : lt);
  return d;
}

static inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

// CTAs of a batch-affine round.  The forward and the backward kernel must cut the pairs into the same
// per-thread runs, so they share the grid: a multiple of the number of CTAs that are resident at once
// for EITHER kernel (they differ in registers), as many waves as bring a thread's run down to about
// kBaTargetPairs pairs; a round too small for one such wave gets two pairs per thread.
constexpr uint32_t kBaTargetPairs = 24;
static uint32_t ba_grid(uint64_t npairs, int sm_count) {
  static const uint32_t per_sm = [] {
    int of = 0, ob = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&of, k_ba_fwd<false>, kBaThreads, 0);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ob, k_ba_bwd<false>, kBaThreads, 0);
    if (of < 1) of = 1;
    if (ob < 1) ob = 1;
    uint32_t a = (uint32_t)of, b = (uint32_t)ob, g = a, h = b;
    while (h) { uint32_t t = g % h; g = h; h = t; }
    return a / g * b;  // lcm
  }();
  const uint64_t wave = (uint64_t)per_sm * (uint64_t)sm_count;
  if (npairs < wave * kBaThreads * 2) return (uint32_t)((npairs + 2 * kBaThreads - 1) / (2 * kBaThreads));
  uint64_t m = (npairs + wave * kBaThreads * kBaTargetPairs / 2) / (wave * kBaThreads * kBaTargetPairs);
  if (m < 1) m = 1;
  return (uint32_t)(m * wave);
}

struct BigLayout {
  size_t counts, offsets, bsum, meta, entries, buckets, large, slices, slice_out, red0, red1, bins, bin_off, order, tab;
  size_t work0, work1, pre, totals, tpre, total;
  uint32_t max_slices, max_large;
};

static BigLayout big_layout(const BigMsmDims& d) {
  BigLayout L;
  size_t nent = (size_t)big_msm_entries(d);  // padded upper bound
  size_t nfinal = nent >> d.R;               // summands left for the XYZZ pass
  L.max_large = (uint32_t)(nfinal / d.large + 1);
  L.max_slices = (uint32_t)(nfinal / kBigSliceLen + L.max_large + 1);
  size_t o = 0;
  L.counts = o; o += al256(((size_t)d.nb + 1) * 4);
  L.offsets = o; o += al256(((size_t)d.nb + 2) * 4);
  L.bsum = o; o += al256(4096 * 4);
  L.meta = o; o += 256;
  L.entries = o; o += al256((nent + 2) * 4);
  L.buckets = o; o += al256(((size_t)d.nb + 1) * sizeof(G1Xyzz));
  L.large = o; o += al256((size_t)L.max_large * sizeof(BigLargeRec));
  L.slices = o; o += al256((size_t)L.max_slices * sizeof(BigSliceRec));
  L.slice_out = o; o += al256((size_t)L.max_slices * sizeof(G1Xyzz));
  size_t red = ((size_t)d.nb / 2 + (size_t)d.nlocal + 1) * sizeof(G1Xyzz);
  L.red0 = o; o += al256(red);
  L.red1 = o; o += al256(red);
  L.bins = o; o += al256(((size_t)kBigLargeBucket + 2) * 4);
  L.bin_off = o; o += al256(((size_t)kBigLargeBucket + 3) * 4);
  L.order = o; o += al256(((size_t)d.nb + 1) * 4);
  L.tab = o; o += al256((2 * (size_t)d.n + 1) * sizeof(BigPoint));
  L.work0 = L.work1 = L.pre = L.totals = L.tpre = o;
  if (d.R > 0) {
    size_t p1 = nent / 2 + 1;  // pairs of round 1
    // a thread owns at least 2 pairs; every CTA writes kBaThreads totals
    size_t ntot = (p1 / 2 / kBaThreads + 2) * kBaThreads;
    L.work0 = o; o += al256(p1 * sizeof(G1Affine));
    L.work1 = o; o += al256((p1 / 2 + 1) * sizeof(G1Affine));
    L.pre = o; o += al256(p1 * sizeof(Fp));
    L.totals = o; o += al256(ntot * sizeof(Fp));
    L.tpre = o; o += al256(ntot * sizeof(Fp));
  }
  L.total = o;
  return L;
}

size_t big_msm_scratch_bytes(const BigMsmDims& d) { return big_layout(d).total; }

// All launches go to `st`; nothing synchronises.  d_out receives one G1Jac.
cudaError_t launch_big_msm(const G1Affine* points, const Fr* scalars, const BigMsmDims& d, int normalize,
                           void* scratch, int sm_count, G1Jac* d_out, cudaStream_t st, const uint32_t* idx,
                           bool release_l2, int* nkernels) {
  if (release_l2) msm_l2_carveout(false);  // the point gathers want the whole L2
  uint8_t* base = (uint8_t*)scratch;
  BigLayout L = big_layout(d);
  uint32_t* counts = (uint32_t*)(base + L.counts);
  uint32_t* offsets = (uint32_t*)(base + L.offsets);
  uint32_t* bsum = (uint32_t*)(base + L.bsum);
  uint32_t* meta = (uint32_t*)(base + L.meta);
  uint32_t* entries = (uint32_t*)(base + L.entries);
  G1Xyzz* buckets = (G1Xyzz*)(base + L.buckets);
  BigLargeRec* large = (BigLargeRec*)(base + L.large);
  BigSliceRec* slices = (BigSliceRec*)(base + L.slices);
  G1Xyzz* slice_out = (G1Xyzz*)(base + L.slice_out);
  G1Xyzz* red[2] = {(G1Xyzz*)(base + L.red0), (G1Xyzz*)(base + L.red1)};
  uint32_t* bins = (uint32_t*)(base + L.bins);
  uint32_t* bin_off = (uint32_t*)(base + L.bin_off);
  uint32_t* order = (uint32_t*)(base + L.order);
  BigPoint* tab = (BigPoint*)(base + L.tab);

  if (d.nlocal == 0 || d.n == 0) {  // this rank owns no window: partial sum = infinity
    G1Xyzz* one = red[0];
    cudaMemsetAsync(one, 0, sizeof(G1Xyzz), st);  // zz = 0 => infinity
    BigMsmDims e = d;
    e.nlocal = 1; e.wfirst = 0; e.wstep = 1; e.c = 0;
    k_big_horner<<<1, 32, 0, st>>>(one, e, normalize, d_out);
    if (nkernels) *nkernels = 1;
    return cudaGetLastError();
  }
  const uint32_t nb = d.nb;
  const int R = d.R;
  const uint64_t nent = big_msm_entries(d);
  cudaMemsetAsync(counts, 0, ((size_t)nb + 1) * 4, st);
  cudaMemsetAsync(meta, 0, 256, st);
  const int gd = (d.n + 255) / 256;
  k_big_tables<<<gd, 256, 0, st>>>(points, idx, d.n, tab);
  k_big_digits<0><<<gd, 256, 0, st>>>(scalars, d.n, d, counts, nullptr, nullptr);
  cudaError_t se = launch_exclusive_scan(counts, nb, bsum, offsets, st, (1u << R) - 1u);
  if (se != cudaSuccess) return se;
  if (R > 0) cudaMemsetAsync(entries, 0xff, (size_t)(nent + 2) * 4, st);  // padding slots = infinity
  k_big_digits<1><<<gd, 256, 0, st>>>(scalars, d.n, d, counts, offsets, entries);

  BigSrc src{tab, (uint32_t)d.n, entries, nullptr};
  if (R > 0) {
    G1Affine* work[2] = {(G1Affine*)(base + L.work0), (G1Affine*)(base + L.work1)};
    Fp* pre = (Fp*)(base + L.pre);
    Fp* totals = (Fp*)(base + L.totals);
    Fp* tpre = (Fp*)(base + L.tpre);
    for (int r = 1; r <= R; r++) {
      const uint64_t npairs = nent >> r;  // upper bound; the kernels read the exact count
      if (npairs == 0) break;
      const uint32_t nblk = ba_grid(npairs, sm_count);
      const uint32_t ntot = nblk * (uint32_t)kBaThreads;
      // totals per inverting thread: one field inversion costs ~ 85 products, so as few threads as keep
      // every scheduler busy (kBaInvThreadsPerSm per SM) share the totals among them
      constexpr uint32_t kBaInvThreadsPerSm = 256;
      int G = (int)(ntot / ((uint32_t)sm_count * kBaInvThreadsPerSm));
      G = G < 1 ? 1 : G > 256 ? 256 : G;
      G1Affine* dst = work[(r - 1) & 1];
      if (r == 1) k_ba_fwd<false><<<nblk, kBaThreads, 0, st>>>(src, offsets + nb, r - 1, pre, totals);
      else k_ba_fwd<true><<<nblk, kBaThreads, 0, st>>>(src, offsets + nb, r - 1, pre, totals);
      k_ba_inv<<<(ntot + kBaThreads * G - 1) / (kBaThreads * G), kBaThreads, 0, st>>>(totals, tpre, ntot, G);
      if (r == 1) k_ba_bwd<false><<<nblk, kBaThreads, 0, st>>>(src, offsets + nb, r - 1, pre, totals, dst);
      else k_ba_bwd<true><<<nblk, kBaThreads, 0, st>>>(src, offsets + nb, r - 1, pre, totals, dst);
      src.direct = dst;
    }
  }

  k_big_mark_large<<<(nb + 255) / 256, 256, 0, st>>>(offsets, R, nb, d.large, meta, large, slices);
  const uint32_t nbins = d.large + 1;
  cudaMemsetAsync(bins, 0, ((size_t)nbins + 1) * 4, st);
  k_big_size_sort<0><<<(nb + 255) / 256, 256, 0, st>>>(offsets, R, nb, d.large, bins, nullptr, nullptr);
  se = launch_exclusive_scan(bins, nbins, bsum, bin_off, st);
  if (se != cudaSuccess) return se;
  k_big_size_sort<1><<<(nb + 255) / 256, 256, 0, st>>>(offsets, R, nb, d.large, bins, bin_off, order);
  if (src.direct) {
    k_big_accum<true><<<(nb + 127) / 128, 128, 0, st>>>(src, offsets, R, order, nb, d.large, buckets);
    k_big_slice<true><<<sm_count * 4, kBigCtaThreads, 0, st>>>(src, meta, slices, slice_out);
  } else {
    k_big_accum<false><<<(nb + 127) / 128, 128, 0, st>>>(src, offsets, R, order, nb, d.large, buckets);
    k_big_slice<false><<<sm_count * 4, kBigCtaThreads, 0, st>>>(src, meta, slices, slice_out);
  }
  k_big_large_finish<<<sm_count, kBigCtaThreads, 0, st>>>(meta, large, slice_out, buckets);
  // bucket reduction
  int Lc = d.M < 8 ? d.M : 8;  // buckets per reduce1 thread: shorter serial chain, more threads
  int per = d.M / Lc;
  int total = d.nlocal * per;
  if (total <= kBigQuadMaxOutputs) k_big_reduce1_quad<<<(4 * total + 127) / 128, 128, 0, st>>>(buckets, d.M, Lc, total, red[0]);
  else k_big_reduce1<<<(total + 127) / 128, 128, 0, st>>>(buckets, d.M, Lc, total, red[0]);
  int cur = 0, nsum = 0;
  while (per > 1) {
    nsum++;
    int G = per > 256 ? 16 : (per > 16 ? 8 : per);
    int pout = (per + G - 1) / G;
    int tot = d.nlocal * pout;
    if (tot <= kBigQuadMaxOutputs) k_big_sum_quad<<<(4 * tot + 127) / 128, 128, 0, st>>>(red[cur], per, G, pout, tot, red[cur ^ 1]);
    else k_big_sum<<<(tot + 127) / 128, 128, 0, st>>>(red[cur], per, G, pout, tot, red[cur ^ 1]);
    cur ^= 1;
    per = pout;
  }
  k_big_horner<<<1, 32, 0, st>>>(red[cur], d, normalize, d_out);
  // tables, 2 digits, 2 x 3 scan, 2 size sort, mark, accum, slice, finish, reduce1, horner: 17; 3 per round
  if (nkernels) *nkernels = 17 + 3 * R + nsum;
  return cudaGetLastError();
}

void launch_big_combine(const G1Jac* in, int n, G1Jac* out, cudaStream_t st) {
  k_big_combine<<<1, 32, 0, st>>>(in, n, out);
}

}  // namespace cdl
