// Batched protocol engine: drives curdleproofs Prove / Verify / ShufflePermuteCommit
// and the Whisk wrappers for B independent instances in lock step.  The host
// keeps what the reference keeps on the host (Merlin transcript, Fiat-Shamir
// challenges, Fr vector arithmetic, RNG, wire format); every group operation is
// a GPU stage over a device-resident pool of affine points:
//   * an MSM stage   — many independent small MSMs in one launch (k_msm_small),
//   * an elementwise stage — pool[dst] = s * pool[src] (+ pool[add]) (k_elem_ops),
//   * (de)compression to/from 48-byte encodings.
// Group elements reach the host only as canonical 48-byte encodings, which is
// all the reference ever observes (SURVEY.md §8c), so no Fp arithmetic exists on
// the host.
#pragma once
#include <cstdint>
#include <functional>
#include <memory>
#include <string>
#include <vector>

#include "../context.cuh"
#include "../launch.h"
#include "fr.hpp"
#include "pool.hpp"
#include "transcript.hpp"

struct cdl_rand {
  cdlh::Rand r;
  explicit cdl_rand(uint64_t seed) : r(seed) {}
};

// crs.go:10-18.  Points are kept on the host (image), on the device of every slot of the owning context
// (pool image) and as compressed encodings on the host (for transcript appends of H).
struct cdl_crs {
  cdl_ctx* ctx = nullptr;
  uint32_t ell = 0;
  std::vector<cdl_g1_affine> host;    // Gs[ell] Hs[4] H Gt Gu Gsum Hsum INF  (ell + 10 points)
  std::vector<uint8_t> enc;           // same order, 48 B each
  // One replica per device slot of ctx: the image (slot 0's made with the CRS, the others uploaded from `host`
  // by their first call) and its fixed-base tables (csrc/fixed_base.cuh), built by the first large batch of
  // that slot that uses this CRS.  Guarded by fixed_mu.
  struct Replica {
    cdl::G1Affine* d_points = nullptr;
    cdl::G1Affine* d_fixed = nullptr;
    bool fixed_failed = false;
  };
  mutable std::mutex fixed_mu;
  mutable std::vector<Replica> rep;
  // slot `s`'s image, uploaded on first use (fixed_mu held, the slot's device current); null if that fails
  const cdl::G1Affine* points_on(size_t s) const;
};

namespace cdlh {

constexpr uint32_t kBlinders = 4;  // common/constants.go:3

struct Layout {
  uint32_t ell, n, m;
  // shared CRS image at the start of the pool
  uint32_t Gs, Hs, H, Gt, Gu, Gsum, Hsum, INF, crs_size;
  // per-instance region (offsets relative to base(b))
  uint32_t Rs, Ss, Ts, Us, M, A, B, scratch, G, Gp, Gm, Tp, Up, PP, inst_size;
  static constexpr uint32_t kScratch = 24;
  explicit Layout(uint32_t ell_);
  uint32_t base(uint32_t b) const { return crs_size + b * inst_size; }
  uint32_t npp() const { return 19 + 10 * m; }  // points in a Whisk shuffle proof (M + 18 + 10m)
};

struct MsmStage {
  std::vector<uint32_t> idx;
  std::vector<Fr> sc;
  std::vector<cdl::MsmTask> tasks;
  std::vector<uint8_t> out48;  // filled by run: tasks.size() * 48
  // host-side accounting only (empty, or one entry per task): terms of the task that exist because one base of
  // the reference's MSM was written as several CRS points (lazy folding); not counted as algorithmic work
  std::vector<uint32_t> extra;
  void clear() { idx.clear(); sc.clear(); tasks.clear(); extra.clear(); }
};

// per-instance builder writing into a pre-sized slice of a stage
struct MsmSlice {
  uint32_t* idx;
  Fr* sc;
  cdl::MsmTask* tasks;
  uint32_t* extra = nullptr;  // MsmStage::extra of this slice's tasks
  uint32_t term_base;  // global index of idx[0]
  uint32_t nterm = 0, ntask = 0;
  void begin(uint32_t out_idx) {
    tasks[ntask].term_off = term_base + nterm;
    tasks[ntask].term_cnt = 0;
    tasks[ntask].out_idx = out_idx;
    tasks[ntask].pad = 0;
  }
  void term(uint32_t point, const Fr& s) {
    idx[nterm] = point;
    sc[nterm] = s;
    nterm++;
    tasks[ntask].term_cnt++;
  }
  // a further term of the base the previous term() call started (see MsmStage::extra)
  void term_more(uint32_t point, const Fr& s) {
    term(point, s);
    if (extra) extra[ntask]++;
  }
  void end() { ntask++; }
};

class Engine {
 public:
  explicit Engine(cdl_ctx* ctx);
  ~Engine();

  // --- API-level operations (all batched over B instances) -----------------
  // common.ShufflePermuteCommit (common/util.go:45-88) on instance points that
  // are already in the pool (Rs, Ss); writes Ts, Us, M into the pool.
  int32_t shuffle_permute_commit(const Layout& L, uint32_t B, const std::vector<std::vector<uint32_t>>& perms,
                                 const std::vector<Fr>& ks, std::vector<cdl_rand*>& rands,
                                 std::vector<std::vector<Fr>>& rs_m);
  // curdleproof.Prove (curdleproof.go:38-197); proofs[b] receives the serialized
  // proof (curdleproof.go:358-387).  status[b] = CDL_OK or the error.
  // inst_enc receives, per instance, the encodings of Rs | Ss | Ts | Us | M.
  // witness_is_ours: M and rs_m were produced by shuffle_permute_commit in the same call (the Whisk
  // wrapper), so the reference's msm(G', d) == D self-check (grandproductargument.go:171-177) cannot fail.
  int32_t prove(const Layout& L, uint32_t B, const cdl_crs* crs, const std::vector<std::vector<uint32_t>>& perms,
                const std::vector<Fr>& ks, const std::vector<std::vector<Fr>>& rs_m, std::vector<cdl_rand*>& rands,
                std::vector<std::vector<uint8_t>>& proofs, std::vector<int32_t>& status,
                std::vector<std::string>& errs, std::vector<uint8_t>& inst_enc, bool witness_is_ours);
  // curdleproof.Verify (curdleproof.go:199-318) for proofs whose points have
  // been decompressed into PP (see parse_and_load_proofs).
  struct ParsedProof {
    bool ok = false;          // decoded without error
    std::string err;
    uint32_t lens[10] = {};   // the ten slice lengths in wire order
    std::vector<uint32_t> pt; // pool index of each decoded point, wire order, M first
    std::vector<const uint8_t*> enc;  // 48-byte encoding of each of those points
    std::vector<Fr> sc;       // the 7 scalars in wire order: Rp c0 d0 Z_k Z_t Z_u x
    const uint8_t* inst_enc = nullptr;  // Rs | Ss | Ts | Us encodings, 4*ell*48 bytes
  };
  int32_t verify(const Layout& L, uint32_t B, const cdl_crs* crs, std::vector<ParsedProof>& pp,
                 std::vector<cdl_rand*>& rands, std::vector<int32_t>& verdict, std::vector<int32_t>& status,
                 std::vector<std::string>& errs);

  // --- pool plumbing ----------------------------------------------------------
  int32_t ensure_pool(size_t npoints);
  int32_t load_crs(const Layout& L, const cdl_crs* crs);
  // fixed-base tables for this call's CRS image (pool indices below crs_size); B = instances of the call
  void select_fixed(const Layout& L, const cdl_crs* crs, size_t B);
  void clear_fixed() { fixed_ = cdl::FixedTable(); }  // calls whose pool does not start with a CRS image
  int32_t upload_points(uint32_t dst, const void* host_affine, size_t count);
  int32_t download_points(uint32_t src, void* host_affine, size_t count);
  int32_t copy_points(uint32_t dst, uint32_t src, size_t count);
  int32_t set_infinity(uint32_t dst, size_t count);
  int32_t copy_ranges(const std::vector<cdl::CopyRange>& ranges);  // many pool-to-pool copies in one launch
  // Instance intake of the batched C ABI calls: instance j of the engine call is the caller's instance sel[j].
  // pts[a] + sel[j] * ell (a < npts: Rs, Ss[, Ts, Us]) go to pool[base(j) + a * ell ..) and, when M is given,
  // M[sel[j]] (gnark G1Jac) to pool[base(j) + M].  One pinned host-to-device copy into the pool behind the
  // instance regions, one normalisation of every M and one copy_ranges launch, so the pool must hold
  // base(sel.size()) + intake_points(L, sel.size()) points.
  int32_t load_instances(const Layout& L, const std::vector<uint32_t>& sel, const cdl_g1_affine* const* pts,
                         uint32_t npts, const cdl_g1_jac* M);
  static size_t intake_points(const Layout& L, size_t B) { return B * ((size_t)4 * L.ell + 1); }
  int32_t compress(const std::vector<uint32_t>& src, std::vector<uint8_t>& out48);
  int32_t decompress(const uint8_t* enc48, const std::vector<uint32_t>& dst, std::vector<uint8_t>& status);
  // `before` (optional) runs on the stream after the stage's indices / scalars reached the device and before
  // the MSM kernels: the verifier's scalar pipeline fills part of the scalar array there (d_scalars), and its
  // combined check reads the stage (d_idx: host indices plus kMsmIdxFixed flags; d_tasks).  Setting `done`
  // skips the MSM kernels: out48 is then left zero.
  // `points` (optional) is a device array the stage's indices refer to instead of the pool; results always
  // go to pool[task.out_idx].
  using MsmBefore = std::function<int32_t(const uint32_t* d_idx, cdl::Fr* d_scalars, const cdl::MsmTask* d_tasks, bool& done)>;
  int32_t run_msm(MsmStage& st, const MsmBefore& before = nullptr, const cdl::G1Affine* points = nullptr);
  int32_t run_elem(const std::vector<cdl::ElemOp>& ops, const std::vector<Fr>& sc);
  // Whisk tracker matching (capi_whisk_match.cu) on decoded trackers pool[t] = rG_t, pool[T + t] = krG_t:
  // owner[t] = the smallest v with ks[v] * rG_t == krG_t, else INT32_MAX.  ks: V gnark fr.Element (Montgomery)
  int32_t match_trackers(uint32_t T, const Fr* ks, uint32_t V, int32_t* owner);
  // Batched fixed-base scalar multiplication (capi_base_mul.cu): out[i] = sc[i] * base, i < n (sc: gnark
  // fr.Element, Montgomery), affine to out and / or compressed to out48 (either may be null).  CDL_ERR_INVALID_ARG
  // for a base outside G1.  The base is not the point at infinity.
  int32_t base_mul(const cdl_g1_affine& base, const Fr* sc, size_t n, cdl_g1_affine* out, uint8_t* out48);

  cdl_ctx* ctx() { return ctx_; }
  cdl::G1Affine* d_pool() { return (cdl::G1Affine*)pool_mem_.d(); }
  ThreadPool& threads() { return pool_; }
  // instrumentation for bench.py: per kernel class (0 msm, 1 elementwise, 2 decompress,
  // 3 compress / normalise): launches, CUDA-event time on the launching stream,
  // algorithmic modmul (SURVEY.md §8d conventions) and algorithmic bytes
  uint64_t launches = 0;
  // [start, end) of every timed kernel chain on its slot's timeline (ms since the slot's base_ev);
  // the union over the slot's engines is that device slot's busy time
  std::vector<std::pair<float, float>> intervals;
  struct Stats {
    uint64_t n[4] = {};
    double ms[4] = {};
    double modmul[4] = {};
    double bytes[4] = {};
  } stats;
  static double msm_algorithmic_modmul(uint64_t terms);
  // CDL_PROFILE=1: wall-clock split of the protocol calls, printed when the engine is destroyed
  struct HostProf {
    double par = 0;    // inside parallel_for sections (per-proof host work)
    double gpu = 0;    // inside GPU stage calls (staging copies + launch + wait)
    double copy = 0;   // of which: filling the pinned staging buffers
    double total = 0;  // prove + verify + shuffle_permute_commit calls
  } prof;
  // Per-proof host work of a stage.  Eight proofs at a time share a pool thread as cooperating
  // fibers so that their Keccak permutations run as one eight-way call (host/fiber.hpp).
  template <class F>
  void par(size_t n, F&& f) {
    double t0 = now();
    std::function<void(size_t)> fn(std::forward<F>(f));
    if (n >= 4 && fibers_available()) {
      const size_t groups = (n + 7) / 8;
      pool_.parallel_for(groups, std::function<void(size_t)>([&](size_t g) {
        run_fiber_group(fn, 8 * g, n - 8 * g < 8 ? n - 8 * g : 8);
      }));
    } else {
      pool_.parallel_for(n, fn);
    }
    prof.par += now() - t0;
  }
  static double now();
  static unsigned host_threads(bool lane, size_t slots);

 private:
  cdl_ctx* ctx_;
  ThreadPool pool_;
  DeviceScratch pool_mem_;  // the point pool (d_pool())
  cdl::FixedTable fixed_;  // tables of the current call's CRS, or empty
  DeviceScratch d_win_;  // window sums of the two-kernel MSM path
  DeviceScratch d_match_;  // tables and window bases of one tile of trackers (match_scratch)
  bool match_scratch(uint32_t tile);
  // Width-12 fixed-base tables of callers' bases (base_mul), keyed by the 96 base bytes: at most kBaseTables,
  // the least recently used replaced.  Separate allocations, so the pool and the match scratch stay as they are.
  struct BaseTable {
    cdl_g1_affine base;
    cdl::G1Affine* tab = nullptr;
    uint64_t used = 0;  // base_clock_ at the last call that used it
  };
  static constexpr size_t kBaseTables = 4;
  std::vector<BaseTable> base_tabs_;
  uint64_t base_clock_ = 0;
  DeviceScratch d_bv_;  // combined verifier check: term list, large-MSM scratch, result (batch_check)
  // The verifier's second MSM stage `st`, uploaded (d_idx, d_sc, d_tasks), as one large MSM with the weight
  // rho[t] (Montgomery) on task t and the CRS bases (pool indices < crs_size) merged: *all_inf = whether it
  // is the point at infinity.
  int32_t batch_check(const MsmStage& st, const std::vector<Fr>& rho, uint32_t crs_size, const uint32_t* d_idx,
                      const cdl::Fr* d_sc, const cdl::MsmTask* d_tasks, bool* all_inf);
  // pinned host staging + device scratch
  Staging s_idx_, s_sc_, s_task_, s_out_, s_ops_, s_enc_, s_st_, s_jac_, s_sub_, s_t2_, s_cr_, s_fsub_, s_vs_, s_as_, s_bv_,
      s_in_, s_base_;
  // s.grow on the engine's stream, with the error recorded when it fails
  int32_t reserve(Staging& s, size_t bytes);
  void tick();                                   // event before a kernel
  void tock(int cls, double modmul, double bytes);  // event after; call finish_timing() after the sync
  int pending_cls_ = -1;
  void finish_timing();
};

// Whisk proof wire walker (whisk/types.go:39-72, curdleproof.go:320-387):
// splits a serialized proof into point encodings, slice lengths and scalars.
struct WireProof {
  std::vector<const uint8_t*> points;  // 48-byte compressed encodings, wire order
  uint32_t lens[10];
  const uint8_t* scalars[7];
};
// returns empty string on success, else the decode error
std::string parse_wire_proof(const uint8_t* buf, size_t len, bool with_m, WireProof& out, size_t* used);

// C ABI helpers (capi_protocol.cu).  The context's engine, created on first use; its fixed-base tables are
// cleared (only a protocol call selects those of its CRS).
Engine* engine_of(cdl_ctx* c);
// gnark's G1Jac of an affine point: (x, y, 1), or (1, 1, 0) for infinity
void affine_to_jac(cdl_g1_jac* out, const cdl_g1_affine& a);
constexpr size_t kMinLaneBatch = 32;  // below this a sub-batch no longer fills its launches
// Device slots a call of B units on c uses: max(1, min(slots, B / min_block)), with min_block = 32 for the
// batched protocol calls and matching; 1 on a lane context.
size_t slots_for(cdl_ctx* c, size_t B, size_t min_block = kMinLaneBatch);
// Runs fn(lane ctx, lo, hi) for contiguous pieces [lo, hi) of a call of B units on a root context concurrently,
// one host thread per piece (DESIGN §4): slot s of the D = slots_for(c, B, min_block) slots in use takes the
// block that sharding.shard_bounds(B, D, s) gives, its bounds rounded to multiples of `align` (empty blocks are
// skipped); with `lanes` it cuts its block into up to n_lanes lanes of at least 32 units, else the block is one
// piece on the slot's lane 0.  Holds c's mutex while the pieces run.
int32_t run_split(cdl_ctx* c, size_t B, const std::function<int32_t(cdl_ctx*, size_t, size_t)>& fn, bool lanes = true,
                  size_t align = 1, size_t min_block = kMinLaneBatch);
// Minimum block of a split call whose units are `per_unit` scalars each of one Engine::base_mul (capi_base_mul.cu):
// ceil(kBaseSlotScalars / per_unit) units, so that every slot's base_mul takes the table path exactly when the
// one-device call would.
size_t base_mul_min_block(size_t per_unit);
// run_split for a caller that already holds c's mutex (and keeps it for work after the pieces)
int32_t run_split_locked(cdl_ctx* c, size_t B, const std::function<int32_t(cdl_ctx*, size_t, size_t)>& fn,
                         bool lanes, size_t align, size_t min_block);

}  // namespace cdlh
