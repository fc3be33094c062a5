// Host-callable kernel launchers; each is defined next to its kernel so that the
// kernels live in separate translation units (compiled in parallel).
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>
#include "g1.cuh"
#include "fixed_base.cuh"

namespace cdl {

struct MsmTask {
  uint32_t term_off;  // first term in idx[] / scalars[]
  uint32_t term_cnt;
  uint32_t out_idx;   // result slot: out_aff[out_idx]
  uint32_t pad;
};
// elementwise op on a pool of affine points:
//   pool[dst] = scalars[sc] * pool[src]  (+ pool[add] unless add == kNoPoint)
struct ElemOp {
  uint32_t src, add, dst, sc;
};
constexpr uint32_t kNoPoint = 0xffffffffu;
// pool[dst .. dst+count) = pool[src .. src+count); src == kNoPoint fills with the point at infinity.
// Ranges of one launch must not overlap each other's destinations.
struct CopyRange {
  uint32_t src, dst, count, pad;
};
constexpr size_t kMsmMaxSmem = 220 * 1024;         // dynamic shared memory opt-in for the small-MSM kernel
constexpr size_t kMsmMaxTerms = kMsmMaxSmem / 36;  // 36 B of staging per term

void launch_compress(const G1Affine* in, uint8_t* out, int n, cudaStream_t s);
void launch_decompress(const uint8_t* in, G1Affine* out, uint8_t* status, int n, cudaStream_t s);
void launch_fp_mul(const Fp* a, const Fp* b, Fp* out, int n, cudaStream_t s);
void launch_peak(int kind, void* out, int blocks, int tpb, int iters, uint32_t seed, cudaStream_t s);
void launch_scalar_mul(const G1Affine* P, const Fr* s, int stride, const G1Affine* L, G1Affine* out, int n,
                       cudaStream_t st);
void launch_jac_to_affine(const G1Jac* in, G1Affine* out, int n, cudaStream_t st);
// ft: fixed-base tables of the pool's first ft.nbase points (fixed_base.cuh); ops on those sources skip the
// double-and-add (the thread-per-op kernel only; small launches take the quad kernel)
void launch_elem_ops(G1Affine* pool, const ElemOp* ops, const Fr* scalars, int n, cudaStream_t st,
                     FixedTable ft = FixedTable());
// --- Whisk tracker matching (k_match.cu): owner[t] = min { v : ks[v] * rg[t] == krg[t] }, INT32_MAX if none.
// launch_match_prep converts ks (device, Montgomery) to canonical form in place and resets owner[0 .. T).
constexpr int kMatchC = 8;              // window width of the per-tracker tables: 32 windows x 128 entries, 384 KiB
// Trackers whose tables are built, then used, together: bounds the table memory (96 MiB).  The resident warps of
// k_match_table walk the keys of a few trackers at a time, so the tile's tables need not stay in the L2.
constexpr uint32_t kMatchTile = 256;
void launch_match_prep(Fr* ks, uint32_t V, int32_t* owner, uint32_t T, cudaStream_t st);
void launch_match_shared(const G1Affine* rg, const G1Affine* krg, uint32_t T, const Fr* ks, uint32_t V,
                         int32_t* owner, cudaStream_t st);
// out[b W + w] = 2^(kMatchC w) rg[b], w < W = fb_windows(kMatchC), Jacobian (normalise with launch_jac_to_affine)
void launch_match_windows(const G1Affine* rg, uint32_t nt, G1Jac* out, cudaStream_t st);
// trackers t0 .. t0 + nt - 1 against every key; tab = launch_fixed_build<kMatchC>(window bases of rg + t0, nt, ..)
void launch_match_table(const G1Affine* tab, const G1Affine* krg, uint32_t t0, uint32_t nt, const Fr* ks,
                        uint32_t V, int32_t* owner, cudaStream_t st);
// fixed-base tables of window width C for nbase points, every (point, window) row built by Seg threads.
// Point bases (C = 12 the CRS tables): bases = the points.  Row bases (C = kMatchC the tracker tables, C = 12
// with kBaseSeg the table of a caller's base): bases = their fb_windows(C) window bases each
// (launch_match_windows, launch_base_windows)
constexpr int kFbSeg = 8;      // threads per row of the CRS and tracker tables
constexpr int kBaseSeg = 128;  // threads per row of a caller's base table: 22 x 128 threads, 16 entries each
template <int C = kFbC>
size_t fixed_table_bytes(uint32_t nbase);
template <int C = kFbC, bool RowBases = (C != kFbC), int Seg = kFbSeg>
void launch_fixed_build(const G1Affine* bases, uint32_t nbase, G1Affine* tab, cudaStream_t st);
// --- batched fixed-base scalar multiplication (k_base_mul.cu): out[i] = sc[i] * P for one base P.
// *status = 0 when *base is in G1 (1 non-canonical coordinate, 2 off the curve, 3 outside G1); with wjac, also
// wjac[w] = 2^(12 w) P for w < kFbW (Jacobian: normalise with launch_jac_to_affine, then
// launch_fixed_build<kFbC, true, kBaseSeg>(affine window bases, 1, tab, ..))
void launch_base_prep(const G1Affine* base, uint32_t* status, G1Jac* wjac, cudaStream_t st);
void launch_base_fill(const G1Affine* base, G1Affine* out, uint32_t n, cudaStream_t st);  // out[0 .. n) = *base
// from P's table (fixed_table_bytes(1) bytes); sc Montgomery; out (affine) and / or out48 (compressed), either null
void launch_base_mul(const G1Affine* tab, const Fr* sc, uint32_t n, G1Affine* out, uint8_t* out48, cudaStream_t st);
void launch_copy_ranges(G1Affine* pool, const CopyRange* ranges, int n, cudaStream_t st);
// verifier scalar pipeline on the device (k_verify_scalars.cu): per-proof inputs, all Montgomery fr.Element
constexpr int kVsMaxM = 16;  // rounds (n <= 2^16)
struct VsParams {
  Fr a1b, a2c0, a3d0, a4xf, a5xf, a6xf, a7, a8, beta_inv, sH_host;
  Fr gamma[kVsMaxM], gamma_inv[kVsMaxM], ch[kVsMaxM];
  uint32_t sc_base;  // first merged-base scalar of this proof in the stage's scalar array
  uint32_t as_base;  // first vector challenge of this proof in the `as` array
  uint32_t pad[2];
};
void launch_verify_scalars(const VsParams* params, const Fr* as, Fr* sc, uint32_t nproofs, uint32_t ell, uint32_t n,
                           uint32_t m, cudaStream_t st);
// combined verifier check (k_batch_verify.cu), all scalars Montgomery: term j < nterm of the stage becomes
// (idx[j] without flags, sc[j] * rho[task of j]); then for each CRS base b < ncrs the weighted scalars of its
// terms (stage positions crs_pos[crs_off[b] .. crs_off[b + 1])) are summed into term nterm + b and zeroed in place
void launch_bv_assemble(const uint32_t* idx, const Fr* sc, const MsmTask* tasks, uint32_t ntask, const Fr* rho,
                        uint32_t nterm, const uint32_t* crs_off, const uint32_t* crs_pos, uint32_t ncrs, uint32_t* cidx,
                        Fr* csc, cudaStream_t st);
// flag[0] = 1 if r[0] is the point at infinity, else 0
void launch_bv_is_inf(const G1Jac* r, uint32_t* flag, cudaStream_t st);
// indexed codecs on a pool: enc[i] <- pool[src[i]] ; pool[dst[i]] <- enc[i]
void launch_compress_idx(const G1Affine* pool, const uint32_t* src, uint8_t* out48, int n, cudaStream_t s);
void launch_decompress_idx(const uint8_t* in48, G1Affine* pool, const uint32_t* dst, uint8_t* status, int n,
                           cudaStream_t s);
// one CTA per task; out_aff / out_c48 may be null
cudaError_t msm_small_init();
// --- throughput path (k_msm_tp.cu): tasks are cut into chunks ("subs") of at most
// kMsmChunk terms; one warp per sub, one combine thread per task.
struct MsmSub {
  uint32_t term_off, term_cnt;
};
struct MsmTask2 {
  uint32_t sub_off, sub_cnt, out_idx, pad;
};
constexpr uint32_t kMsmIdxFixed = 1u << 30;  // idx[] flag (throughput path only): sum this term from the fixed-base tables
constexpr uint32_t kMsmChunk = 128;  // terms per bucket warp (msm_tp_pick_chunk)
size_t msm_tp_scratch_bytes(size_t nterm, size_t nsub, size_t ntasks);
uint32_t msm_tp_pick_chunk(size_t nterm, int sm_count);
void msm_l2_carveout(bool on);  // persisting-L2 window of the bucket scratch: held by the batched path only
// ft + fixed_subs: terms flagged kMsmIdxFixed (on the pool's first ft.nbase points) are summed from the fixed-base
// tables by one warp per listed chunk (k_msm_fixed; fixed_subs = device list of the chunks holding such terms)
// and skipped by the bucket warps
void launch_msm_tp(const G1Affine* points, const uint32_t* idx, const Fr* scalars, int nterm, const MsmSub* subs,
                   int nsub, const MsmTask2* tasks, int ntasks, G1Affine* out_aff, uint8_t* out_c48, void* scratch,
                   cudaStream_t st, FixedTable ft = FixedTable(), const uint32_t* fixed_subs = nullptr,
                   int nfixed_subs = 0);
// host helper: cut tasks into subs
template <class VecSub, class VecTask2>
inline void msm_build_subs(const MsmTask* tasks, size_t ntasks, uint32_t chunk, VecSub& subs, VecTask2& tasks2) {
  subs.clear();
  tasks2.clear();
  for (size_t j = 0; j < ntasks; j++) {
    MsmTask2 t2{(uint32_t)subs.size(), 0, tasks[j].out_idx, 0};
    for (uint32_t o = 0; o < tasks[j].term_cnt; o += chunk) {
      uint32_t c = tasks[j].term_cnt - o < chunk ? tasks[j].term_cnt - o : chunk;
      subs.push_back(MsmSub{tasks[j].term_off + o, c});
      t2.sub_cnt++;
    }
    tasks2.push_back(t2);
  }
}

// counts[0..n) -> offsets[0..n] exclusive prefix (total in offsets[n]); counts are zeroed; bsum: 4096 words
cudaError_t launch_exclusive_scan(uint32_t* counts, uint32_t n, uint32_t* bsum, uint32_t* offsets, cudaStream_t st,
                                  uint32_t pad = 0);

// Latency path (k_msm.cu): one CTA per task.  Engine::run_msm switches to the throughput path at
// kMsmSplitThreshold tasks per launch.
constexpr int kMsmSplitThreshold = 96;
// ... or when one task is long enough that a single CTA's thread-per-bucket walk is the slower choice
constexpr size_t kMsmSplitTerms = 384;
void launch_msm_small(const G1Affine* points, const uint32_t* idx, const Fr* scalars, const MsmTask* tasks,
                      int ntasks, size_t max_terms, G1Affine* out_aff, uint8_t* out_c48, cudaStream_t st);


// --- single large MSM (k_msm_big.cu): signed-digit Pippenger, counting sort of bucket
// indices, thread-per-bucket accumulation.  A caller may own only the windows
// wfirst, wfirst + wstep, ... (multi-GPU window partition).
struct BigMsmDims {
  int n, c, W, M, wfirst, wstep, nlocal;
  uint32_t nb;     // nlocal * M buckets
  uint32_t large;  // buckets with more entries than this (after the batch-affine rounds) are summed by whole CTAs (slices)
  int R;           // batch-affine rounds: bucket regions padded to 2^R slots and halved R times (0 = XYZZ only)
};
constexpr size_t kBigMsmThreshold = 1024;  // cdl_g1_msm switches to the Pippenger path above this size
int big_msm_pick_c(size_t n);
// ba_rounds < 0: pick the number of batch-affine rounds by the mean bucket load
BigMsmDims big_msm_dims(size_t n, int c, int wfirst, int wstep, int ba_rounds = -1);
constexpr int kBigMaxBaRounds = 8;
size_t big_msm_scratch_bytes(const BigMsmDims& d);
// sorted (point, sign) entries of a launch: both GLV halves of every term in every owned window, plus
// the padding of every bucket's region to a multiple of 2^R slots (upper bound)
inline uint64_t big_msm_entries(const BigMsmDims& d) {
  return 2ull * (uint64_t)d.n * (uint64_t)d.nlocal + (uint64_t)d.nb * (((uint64_t)1 << d.R) - 1);
}
// idx (optional): term i's base is points[idx[i]].  release_l2: drop the persisting-L2 window of the batched
// small-MSM path first (a process-wide limit; a caller whose other streams run that path keeps it).
// nkernels (optional) receives the number of kernels launched.
cudaError_t launch_big_msm(const G1Affine* points, const Fr* scalars, const BigMsmDims& d, int normalize,
                           void* scratch, int sm_count, G1Jac* d_out, cudaStream_t st, const uint32_t* idx = nullptr,
                           bool release_l2 = true, int* nkernels = nullptr);
void launch_big_combine(const G1Jac* in, int n, G1Jac* out, cudaStream_t st);

}  // namespace cdl
