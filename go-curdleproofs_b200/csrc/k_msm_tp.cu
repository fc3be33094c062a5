// Throughput path for many small MSMs per launch (batched proving / verification), and for a
// few long ones (the verifier's 5*ell + 8 terms for a single proof).
//
//   k_msm_recode    thread per term: fr.Element (Montgomery) -> canonical -> GLV split
//                   k = s0*(s1*|k1| + k2*lambda), both < 2^127, stored biased so that a window
//                   digit is one nibble - 8; beta*x of the base (the x of phi(P)) once per term
//   k_msm_warp_gmem warp per chunk (<= 128 terms, msm_tp_pick_chunk) of a task, lane = one of the
//                   32 signed 4-bit windows: every lane walks the chunk's terms serially and adds
//                   +-P / +-phi(P) into its 8 XYZZ buckets, then reduces them with the running-sum
//                   trick from the highest non-empty bucket.  All 32 lanes do the same amount of
//                   work on every term (the term's point is one broadcast load), so lane
//                   efficiency is ~15/16 whatever the MSM size — unlike thread-per-bucket, whose
//                   lanes idle on load imbalance when a window has few points per bucket.
//                   The buckets (49 KB per warp) live in a per-launch global scratch that a persistent
//                   grid reuses chunk after chunk and that stays in L2 (see k_msm_warp_gmem).
//   k_msm_chunk_sum thread per (task, window): sums the chunk partials
//   k_msm_combine_tp thread per task: walks the windows top-down (4 doublings + 1 addition),
//                   normalises, stores the affine point and its 48-byte encoding.  The 124-doubling
//                   chain is serial per MSM but runs at full lane efficiency across thousands of
//                   MSMs, and overlaps the other lanes' kernels in a batched call.
#include <algorithm>
#include <mutex>

#define CDL_FP_MUL_CALL 1
#include "codec.cuh"
#include "quad.cuh"
#include "launch.h"

namespace cdl {

constexpr int kTpWindows = 32;
constexpr int kTpRows = kTpWindows + 1;  // rows of the window-sum arrays: 32 windows + the chunk's fixed-base sum (weight 1)
constexpr uint32_t kIdxFixed = kMsmIdxFixed;  // term index flag set by the host: sum this term from the fixed-base tables

// Streaming (evict-first) loads for data a warp reads once — the recoded terms and the base
// points — so that they do not push the warps' bucket arrays (local memory, re-read on every
// addition) out of L2.
template <class T>
__device__ __forceinline__ T ld_stream8(const T* p) {
  static_assert(sizeof(T) % 8 == 0, "8-byte granules");
  T v;
  const uint2* s = reinterpret_cast<const uint2*>(p);
  uint2* d = reinterpret_cast<uint2*>(&v);
#pragma unroll
  for (int i = 0; i < (int)(sizeof(T) / 8); i++) d[i] = __ldcs(s + i);
  return v;
}
template <class T>
__device__ __forceinline__ T ld_stream16(const T* p) {
  static_assert(sizeof(T) % 16 == 0, "16-byte granules");
  T v;
  const uint4* s = reinterpret_cast<const uint4*>(p);
  uint4* d = reinterpret_cast<uint4*>(&v);
#pragma unroll
  for (int i = 0; i < (int)(sizeof(T) / 16); i++) d[i] = __ldcs(s + i);
  return v;
}

struct alignas(16) MsmRec {
  uint32_t k1p[4];
  uint32_t k2p[4];
  uint32_t pidx;   // pool index of the base
  uint32_t flags;  // bit 0: negate the P part, bit 1: negate the phi(P) part, bit 2: the base is the point at infinity,
                   // bit 3: fixed-base term (summed from the tables by k_msm_fixed; bucket warps skip it), bit 4: negate it
  uint32_t pad[2];
  Fp bx;           // beta * x of the base: the x coordinate of phi(P), computed once per term here
                   // instead of once per term by all 32 lanes of the bucket warp
};

__global__ void k_msm_recode(const G1Affine* __restrict__ points, const uint32_t* __restrict__ idx,
                             const Fr* __restrict__ scalars, MsmRec* __restrict__ rec, int nterm, uint32_t nfixed) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nterm) return;
  Fr km = scalars[t], k;
  FrM::from_mont(k, km);
  Glv g;
  glv_decompose(g, k.v);
  MsmRec r;
  glv_bias(r.k1p, g.k1);
  glv_bias(r.k2p, g.k2);
  r.pidx = idx[t] & 0x3fffffffu;
  bool flip = (idx[t] >> 31) != 0;
  const bool fixed_term = (idx[t] & kIdxFixed) != 0 && r.pidx < nfixed;
  const G1Affine base = points[r.pidx];
  r.flags = ((g.neg1 != flip) ? 1u : 0u) | ((g.neg2 != flip) ? 2u : 0u) | (aff_is_inf(base) ? 4u : 0u) |
            (fixed_term ? 8u : 0u) | (flip ? 16u : 0u);
  r.pad[0] = r.pad[1] = 0;
  Fp beta;
  fp_set_beta(beta);
  FpM::mul(r.bx, base.x, beta);
  rec[t] = r;
}

// Bucket warps.  The 8 XYZZ buckets of every lane (49 KB per warp) live in an explicitly managed
// GLOBAL scratch that is part of the launch's own scratch allocation: the grid is persistent (two
// 128-thread CTAs per SM), warp (blockIdx, warp) owns region blockIdx*4 + warp for the whole launch
// and fetches chunks from a per-launch work counter until none are left.  Every chunk a warp ever
// processes therefore reuses the same addresses, the working set is resident warps x 49 KB = 58 MB and
// stays in L2 (persisting access-policy window on the launching stream), and nothing survives the
// launch: no device-global allocator state, no spinning, nothing a faulted kernel could leave behind.
// uint4 granules, layout [bucket][granule][lane]: a warp access is 512 contiguous bytes.
constexpr size_t kWarpBucketBytes = 8 * sizeof(G1Xyzz) * 32;
constexpr int kWarpsPerCta = 4;
#ifndef CDL_TP_CTAS_PER_SM
#define CDL_TP_CTAS_PER_SM 2
#endif
constexpr int kCtasPerSm = CDL_TP_CTAS_PER_SM;

__global__ void __launch_bounds__(32 * kWarpsPerCta, kCtasPerSm)
k_msm_warp_gmem(const G1Affine* __restrict__ points, const MsmRec* __restrict__ rec, const MsmSub* __restrict__ subs,
                int nsub, G1Jac* __restrict__ win, uint4* __restrict__ scratch, uint32_t* __restrict__ next) {
  const int w = threadIdx.x & 31;
  uint4* bk = scratch + ((size_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5)) * (kWarpBucketBytes / 16) + w;
#pragma unroll 1
  for (;;) {
    uint32_t sub = 0;
    if (w == 0) sub = atomicAdd(next, 1u);
    sub = __shfl_sync(0xffffffffu, sub, 0);
    if (sub >= (uint32_t)nsub) break;
    const MsmSub s = subs[sub];
    uint32_t nonempty = 0;
#pragma unroll 1
    for (uint32_t t = 0; t < s.term_cnt; t++) {
      // only the digits stay in registers across the two halves; the coordinates of the half's point
      // (x or beta*x, y: warp-uniform broadcast loads) are fetched when that half is added
      const MsmRec* rp = rec + s.term_off + t;
      const uint4 k1 = __ldcs(reinterpret_cast<const uint4*>(rp->k1p));
      const uint4 k2 = __ldcs(reinterpret_cast<const uint4*>(rp->k2p));
      const uint2 pf = __ldcs(reinterpret_cast<const uint2*>(&rp->pidx));  // pidx, flags
      if (pf.y & 12u) continue;  // base at infinity, or a fixed-base term (uniform across the warp)
#pragma unroll 1
      for (int h = 0; h < 2; h++) {
        const uint4 kk = h == 0 ? k1 : k2;
        const int wi = w >> 3;  // the lane's window sits in word wi (register selects, no local array)
        const uint32_t word = wi == 0 ? kk.x : wi == 1 ? kk.y : wi == 2 ? kk.z : kk.w;
        const int nib = (int)((word >> ((w & 7) * 4)) & 15u);
        const int d = w == 31 ? nib : nib - 8;  // glv_digit()
        if (d == 0) continue;
        bool neg = (d < 0) != (((pf.y >> h) & 1u) != 0);
        int a = (d < 0 ? -d : d) - 1;
        G1Affine q;
        q.x = h == 0 ? ld_stream16(&points[pf.x].x) : ld_stream16(&rp->bx);
        q.y = ld_stream16(&points[pf.x].y);
        if (neg) FpM::neg(q.y, q.y);
        uint4* slotp = bk + (size_t)a * 12 * 32;
        G1Xyzz b;
        uint4* bw = reinterpret_cast<uint4*>(&b);
        if (!((nonempty >> a) & 1u)) {
          xyzz_from_affine(b, q);
          nonempty |= 1u << a;
        } else {
#pragma unroll
          for (int i = 0; i < 12; i++) bw[i] = slotp[i * 32];
          xyzz_add_mixed(b, b, q);
        }
#pragma unroll
        for (int i = 0; i < 12; i++) slotp[i * 32] = bw[i];
      }
    }
    // sum_d d * B_d by the running-sum trick, from the highest non-empty bucket down (short chunks in
    // the late folding rounds touch one or two buckets per window)
    G1Xyzz run, acc;
    xyzz_set_inf(run);
    xyzz_set_inf(acc);
#pragma unroll 1
    for (int a = nonempty ? 31 - __clz(nonempty) : -1; a >= 0; a--) {
      if ((nonempty >> a) & 1u) {
        G1Xyzz b;
        uint4* bw = reinterpret_cast<uint4*>(&b);
        const uint4* slotp = bk + (size_t)a * 12 * 32;
#pragma unroll
        for (int i = 0; i < 12; i++) bw[i] = slotp[i * 32];
        xyzz_add(run, run, b);
      }
      xyzz_add(acc, acc, run);
    }
    G1Jac j;
    xyzz_to_jac(j, acc);
    win[(size_t)w * nsub + sub] = j;
  }
}

// The persisting L2 carve-out takes L2 away from everything else on the device, so it is only held
// while batched-MSM launches are being issued: the large-MSM path (whose point gathers want the
// whole L2) releases it, the next batched launch takes it back.
struct L2Persist {
  int sms = 0;
  size_t bytes = 0;       // carve-out this path asks for (0: unsupported)
  int max_window = 0;
  bool queried = false, on = false;
};
static std::mutex g_l2_mu;
static L2Persist g_l2[64];

static L2Persist& l2_state(int dev) {  // g_l2_mu held
  L2Persist& g = g_l2[dev & 63];
  if (!g.queried) {
    g.queried = true;
    cudaDeviceGetAttribute(&g.sms, cudaDevAttrMultiProcessorCount, dev);
    if (g.sms < 1) g.sms = 1;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) {
      const size_t hot = (size_t)g.sms * kCtasPerSm * kWarpsPerCta * kWarpBucketBytes;
      if (prop.persistingL2CacheMaxSize > 0)
        g.bytes = std::min<size_t>((size_t)prop.persistingL2CacheMaxSize, hot);
      cudaDeviceGetAttribute(&g.max_window, cudaDevAttrMaxAccessPolicyWindowSize, dev);
    }
    cudaGetLastError();
  }
  return g;
}

void msm_l2_carveout(bool on) {
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lk(g_l2_mu);
  L2Persist& g = l2_state(dev);
  if (!g.bytes || g.on == on) return;
  if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, on ? g.bytes : 0) == cudaSuccess) g.on = on;
  cudaGetLastError();
}

static size_t bucket_scratch_bytes(int sms) { return (size_t)sms * kCtasPerSm * kWarpsPerCta * kWarpBucketBytes; }

// Fixed-base terms (fixed_base.cuh): one warp per chunk, lane l takes the chunk's terms l, l + 32, ..; a
// term flagged by the host (kIdxFixed: its task holds enough terms on tabulated points to pay for the
// pass) is 22 table look-ups and mixed additions, no doublings, no buckets.  The lanes' sums are added
// up with a shuffle tree into row 32 of the chunk's window sums, which k_msm_chunk_sum and
// k_msm_combine_* carry along with weight 1.
// One warp per CTA, launched for the listed chunks only (row 32 of every other chunk is zeroed = infinity).
__global__ void __launch_bounds__(32)
k_msm_fixed(const MsmRec* __restrict__ rec, const Fr* __restrict__ scalars, const MsmSub* __restrict__ subs, int nsub,
            const uint32_t* __restrict__ fsubs, FixedTable ft, G1Jac* __restrict__ win) {
  const int sub = (int)fsubs[blockIdx.x];  // the host lists the chunks of the tasks it flagged
  const int lane = threadIdx.x;
  const MsmSub s = subs[sub];
  G1Xyzz acc;
  xyzz_set_inf(acc);
#pragma unroll 1
  for (uint32_t t = s.term_off + (uint32_t)lane; t < s.term_off + s.term_cnt; t += 32) {
    const uint2 pf = *reinterpret_cast<const uint2*>(&rec[t].pidx);
    if ((pf.y & 12u) != 8u) continue;
    Fr k;
    FrM::from_mont(k, scalars[t]);
    fixed_base_accumulate(acc, ft, pf.x, k.v, (pf.y & 16u) != 0);
  }
  G1Jac* out = win + (size_t)kTpWindows * nsub + sub;
  // sum over the lanes (any lane may hold infinity)
  if (!__any_sync(0xffffffffu, !xyzz_is_inf(acc))) {
    if (lane == 0) { G1Jac z; jac_set_inf(z); *out = z; }
    return;
  }
#pragma unroll 1
  for (int off = 16; off >= 1; off >>= 1) {
    G1Xyzz o;
    uint32_t* ow = reinterpret_cast<uint32_t*>(&o);
    const uint32_t* aw = reinterpret_cast<const uint32_t*>(&acc);
#pragma unroll
    for (int i = 0; i < 48; i++) ow[i] = __shfl_down_sync(0xffffffffu, aw[i], off);
    if (lane < off) xyzz_add(acc, acc, o);
  }
  if (lane == 0) {
    G1Jac r;
    xyzz_to_jac(r, acc);
    *out = r;
  }
}

// thread per (task, window): sum of the task's chunk partials, so that the serial Horner
// chain of k_msm_combine_tp sees one point per window however finely a task was cut
__global__ void __launch_bounds__(128)
k_msm_chunk_sum(const G1Jac* __restrict__ win, const MsmTask2* __restrict__ tasks, int ntasks, int nsub, int nrows,
                G1Jac* __restrict__ wsum) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ntasks * nrows) return;
  const int w = t / ntasks, j = t - w * ntasks;
  const MsmTask2 task = tasks[j];
  G1Jac acc;
  jac_set_inf(acc);
#pragma unroll 1
  for (uint32_t c = 0; c < task.sub_cnt; c++) {
    G1Jac s = win[(size_t)w * nsub + task.sub_off + c];
    jac_add(acc, acc, s);
  }
  wsum[(size_t)w * ntasks + j] = acc;
}

__global__ void __launch_bounds__(64)
k_msm_combine_tp(const G1Jac* __restrict__ wsum, const MsmTask2* __restrict__ tasks, int ntasks,
                 int has_fixed, G1Affine* __restrict__ out_aff, uint8_t* __restrict__ out_c48) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= ntasks) return;
  const MsmTask2 task = tasks[j];
  G1Jac acc;
  jac_set_inf(acc);
#pragma unroll 1
  for (int w = kTpWindows - 1; w >= 0; w--) {
    if (w != kTpWindows - 1) {
#pragma unroll 1
      for (int i = 0; i < 4; i++) jac_dbl(acc, acc);
    }
    G1Jac s = wsum[(size_t)w * ntasks + j];
    jac_add(acc, acc, s);
  }
  if (has_fixed) {  // the task's fixed-base terms (k_msm_fixed), row 32
    G1Jac f = wsum[(size_t)kTpWindows * ntasks + j];
    jac_add(acc, acc, f);
  }
  G1Affine a;
  jac_to_affine(a, acc);
  if (out_aff) out_aff[task.out_idx] = a;
  if (out_c48) g1_compress_dev(out_c48 + 48 * (size_t)j, a);
}

// acc += s for a Jacobian s (Jacobian -> XYZZ: ZZ = Z^2, ZZZ = Z^3), one quad per point
__device__ __forceinline__ void quad_add_jac(const Quad& q, G1Xyzz& acc, const G1Jac& s) {
  if (jac_is_inf(s)) return;
  G1Xyzz sx;
  Fp a[4], b[4], o[4];
  a[0] = s.z; b[0] = s.z;
  qmul<1>(q, o, a, b);
  sx.zz = o[0];
  a[0] = o[0]; b[0] = s.z;
  qmul<1>(q, o, a, b);
  sx.zzz = o[0];
  sx.x = s.x;
  sx.y = s.y;
  qxyzz_add(q, acc, acc, sx);
}

// The same Horner walk with a QUAD of lanes per task (quad.cuh) for launches with few tasks (one proof
// at a time): 124 x 3 + 32 x 4 product latencies instead of 124 x 7 + 32 x 16.
__global__ void __launch_bounds__(32)
k_msm_combine_quad(const G1Jac* __restrict__ wsum, const MsmTask2* __restrict__ tasks, int ntasks,
                   int has_fixed, G1Affine* __restrict__ out_aff, uint8_t* __restrict__ out_c48) {
  const Quad q;
  const int j = blockIdx.x * 8 + (threadIdx.x >> 2);
  if (j >= ntasks) return;  // the whole quad
  const MsmTask2 task = tasks[j];
  G1Xyzz acc;
  xyzz_set_inf(acc);
#pragma unroll 1
  for (int w = kTpWindows - 1; w >= 0; w--) {
    if (w != kTpWindows - 1) {
#pragma unroll 1
      for (int i = 0; i < 4; i++) qxyzz_dbl(q, acc, acc);
    }
    const G1Jac s = wsum[(size_t)w * ntasks + j];
    quad_add_jac(q, acc, s);
  }
  if (has_fixed) {  // the task's fixed-base terms (k_msm_fixed), row 32
    const G1Jac f = wsum[(size_t)kTpWindows * ntasks + j];
    quad_add_jac(q, acc, f);
  }
  G1Affine a;
  qxyzz_to_affine(q, a, acc);
  if (q.lane == 0) {
    if (out_aff) out_aff[task.out_idx] = a;
    if (out_c48) g1_compress_dev(out_c48 + 48 * (size_t)j, a);
  }
}
constexpr int kCombineQuadMaxTasks = 4096;  // above this the thread-per-task kernel has enough warps (measured: no difference from 4 096 up)

// [work counter | recoded terms | chunk window sums | task window sums | bucket scratch]; the sums have 33 rows
size_t msm_tp_scratch_bytes(size_t nterm, size_t nsub, size_t ntasks) {
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  size_t rec = (nterm * sizeof(MsmRec) + 255) & ~(size_t)255;
  size_t win = (nsub * kTpRows * sizeof(G1Jac) + 255) & ~(size_t)255;
  size_t ws = (ntasks * kTpRows * sizeof(G1Jac) + 255) & ~(size_t)255;
  return 256 + rec + win + ws + bucket_scratch_bytes(sms);
}

// Chunk length for a launch.  Long chunks amortise the per-chunk bucket reduction (up to 16 full
// additions against 2 mixed additions per term); shorter ones give more warps and a shorter tail.
// Measured on B200 with batches of 2 048 Whisk round trips (MSM class per step): 64 terms 377 ms,
// 128: 378, 160: 374, 256: 384, 512: 404, 1 024: 427; batched verification alone (one 712-term MSM
// per proof) gains 5-12 % from 64-128 over 256.
uint32_t msm_tp_pick_chunk(size_t nterm, int sm_count) {
  // latency regime (a handful of large MSMs, e.g. the verifier's 5*ell + 8 terms for one proof):
  // too few 128-term chunks to occupy the machine, so cut finer and shorten each warp's serial walk
  if (nterm / kMsmChunk < (size_t)2 * sm_count) return 32;
  return kMsmChunk;
}

void launch_msm_tp(const G1Affine* points, const uint32_t* idx, const Fr* scalars, int nterm, const MsmSub* subs,
                   int nsub, const MsmTask2* tasks, int ntasks, G1Affine* out_aff, uint8_t* out_c48, void* scratch,
                   cudaStream_t st, FixedTable ft, const uint32_t* fixed_subs, int nfixed_subs) {
  int dev = 0;
  cudaGetDevice(&dev);
  L2Persist g;
  {
    std::lock_guard<std::mutex> lk(g_l2_mu);
    g = l2_state(dev);
  }
  uint32_t* next = (uint32_t*)scratch;
  MsmRec* rec = (MsmRec*)((uint8_t*)scratch + 256);
  size_t rec_bytes = ((size_t)nterm * sizeof(MsmRec) + 255) & ~(size_t)255;
  size_t win_bytes = ((size_t)nsub * kTpRows * sizeof(G1Jac) + 255) & ~(size_t)255;
  size_t ws_bytes = ((size_t)ntasks * kTpRows * sizeof(G1Jac) + 255) & ~(size_t)255;
  G1Jac* win = (G1Jac*)((uint8_t*)rec + rec_bytes);
  G1Jac* wsum = (G1Jac*)((uint8_t*)win + win_bytes);
  uint4* buckets = (uint4*)((uint8_t*)wsum + ws_bytes);
  const bool fixed = ft.tab != nullptr && ft.nbase > 0 && fixed_subs != nullptr && nfixed_subs > 0;
  if (nterm > 0)
    k_msm_recode<<<(nterm + 127) / 128, 128, 0, st>>>(points, idx, scalars, rec, nterm, fixed ? ft.nbase : 0u);
  if (fixed) {
    cudaMemsetAsync(win + (size_t)kTpWindows * nsub, 0, (size_t)nsub * sizeof(G1Jac), st);  // Z = 0: infinity
    k_msm_fixed<<<nfixed_subs, 32, 0, st>>>(rec, scalars, subs, nsub, fixed_subs, ft, win);
  }
  const int nrows = fixed ? kTpRows : kTpWindows;
  if (nsub > 0) {
    cudaMemsetAsync(next, 0, 4, st);
    if (g.bytes) {  // keep the bucket scratch resident in L2: persisting carve-out + access-policy window
      msm_l2_carveout(true);
      cudaStreamAttrValue av = {};
      av.accessPolicyWindow.base_ptr = buckets;
      av.accessPolicyWindow.num_bytes = std::min<size_t>(bucket_scratch_bytes(g.sms), (size_t)g.max_window);
      av.accessPolicyWindow.hitRatio = 1.0f;
      av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
      av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
      cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &av);
    }
    const int ctas = std::min((nsub + kWarpsPerCta - 1) / kWarpsPerCta, g.sms * kCtasPerSm);
    k_msm_warp_gmem<<<ctas, 32 * kWarpsPerCta, 0, st>>>(points, rec, subs, nsub, win, buckets, next);
  }
  k_msm_chunk_sum<<<(ntasks * nrows + 127) / 128, 128, 0, st>>>(win, tasks, ntasks, nsub, nrows, wsum);
  const int fs = fixed ? 1 : 0;
  if (ntasks <= kCombineQuadMaxTasks) k_msm_combine_quad<<<(ntasks + 7) / 8, 32, 0, st>>>(wsum, tasks, ntasks, fs, out_aff, out_c48);
  else k_msm_combine_tp<<<(ntasks + 63) / 64, 64, 0, st>>>(wsum, tasks, ntasks, fs, out_aff, out_c48);
}

}  // namespace cdl
