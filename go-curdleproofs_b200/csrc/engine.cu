// Batched curdleproofs engine — see host/engine.hpp.
#include "host/engine.hpp"

#include <algorithm>
#include <array>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>

using cdl::ElemOp;
using cdl::G1Affine;
using cdl::MsmTask;

namespace cdlh {

static const uint8_t kInfEnc[48] = {0xc0};

Layout::Layout(uint32_t ell_) {
  ell = ell_;
  n = ell + kBlinders;
  m = 0;
  while ((1u << m) < n) m++;
  Gs = 0; Hs = ell; H = ell + 4; Gt = ell + 5; Gu = ell + 6; Gsum = ell + 7; Hsum = ell + 8; INF = ell + 9;
  crs_size = ell + 10;
  uint32_t o = 0;
  Rs = o; o += ell;
  Ss = o; o += ell;
  Ts = o; o += ell;
  Us = o; o += ell;
  M = o++; A = o++; B = o++;
  scratch = o; o += kScratch;
  G = o; o += n;
  Gp = o; o += n;
  Gm = o; o += n;
  Tp = o; o += n;
  Up = o; o += n;
  PP = o; o += 19 + 10 * 32;  // room for the largest accepted proof (lg n < 32)
  inst_size = o;
}

// ------------------------------------------------------------------ plumbing
// a lane engine shares the host cores with its sibling lanes, and the device slots of a context share them
Engine::Engine(cdl_ctx* ctx)
    : ctx_(ctx),
      pool_(host_threads(ctx->parent != nullptr, ctx->root()->slots.size())) {}

// CDL_HOST_THREADS caps the host cores one context may use (several ranks on one box share them); each of
// the context's device slots gets an equal share
unsigned Engine::host_threads(bool lane, size_t slots) {
  unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  if (const char* e = getenv("CDL_HOST_THREADS")) {
    int v = atoi(e);
    if (v >= 1) hw = std::min(hw, (unsigned)v);
  }
  hw = std::max(1u, hw / (unsigned)std::max<size_t>(1, slots));
  return lane ? std::max(2u, std::min(32u, hw / 2)) : std::max(1u, std::min(64u, hw));
}

double Engine::now() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

Engine::~Engine() {
  if (getenv("CDL_PROFILE"))
    fprintf(stderr, "[cdl profile] engine %p (lane %d): total %.1f ms = parallel host %.1f + gpu stages %.1f (staging copies %.1f) + serial host %.1f\n",
            (void*)this, ctx_->parent ? 1 : 0, prof.total * 1e3, prof.par * 1e3, prof.gpu * 1e3, prof.copy * 1e3,
            (prof.total - prof.par - prof.gpu) * 1e3);
  cudaSetDevice(ctx_->device);  // before the members free their memory
  for (BaseTable& b : base_tabs_) cudaFree(b.tab);
}

// SURVEY.md §8d: modmul(N) = min_c [6 N W + 28 2^(c-1) W + 9 c (W-1) + 14 W], W = ceil(256/c)
double Engine::msm_algorithmic_modmul(uint64_t N) {
  if (N == 0) return 0;
  double best = 1e300;
  for (int c = 1; c <= 24; c++) {
    double W = (double)((256 + c - 1) / c);
    double v = 6.0 * N * W + 28.0 * (double)(1ull << (c - 1)) * W + 9.0 * c * (W - 1) + 14.0 * W;
    if (v < best) best = v;
  }
  return best;
}

void Engine::tick() { cudaEventRecord(ctx_->ev0, ctx_->stream); }
void Engine::tock(int cls, double modmul, double bytes) {
  cudaEventRecord(ctx_->ev1, ctx_->stream);
  pending_cls_ = cls;
  stats.n[cls]++;
  stats.modmul[cls] += modmul;
  stats.bytes[cls] += bytes;
  launches++;
}
void Engine::finish_timing() {
  if (pending_cls_ < 0) return;
  float ms = 0;
  if (cudaEventElapsedTime(&ms, ctx_->ev0, ctx_->ev1) == cudaSuccess) stats.ms[pending_cls_] += ms;
  float t0 = 0;
  if (cudaEventElapsedTime(&t0, ctx_->root()->slots[ctx_->dev_slot].base_ev, ctx_->ev0) == cudaSuccess && intervals.size() < (1u << 22))
    intervals.emplace_back(t0, t0 + ms);
  pending_cls_ = -1;
}

int32_t Engine::reserve(Staging& s, size_t bytes) {
  if (s.grow(bytes, ctx_->stream)) return CDL_OK;
  return ctx_->fail(CDL_ERR_CUDA, "engine staging allocation of %zu bytes failed", bytes);
}

int32_t Engine::ensure_pool(size_t npoints) {
  if (pool_mem_.grow(npoints * sizeof(G1Affine), ctx_->stream)) return CDL_OK;
  return ctx_->fail(CDL_ERR_CUDA, "point pool allocation of %zu points failed", npoints);
}

int32_t Engine::load_crs(const Layout& L, const cdl_crs* crs) {
  const G1Affine* pts;
  {
    std::lock_guard<std::mutex> lk(crs->fixed_mu);
    pts = crs->points_on(ctx_->dev_slot);
  }
  if (!pts) return ctx_->fail(CDL_ERR_CUDA, "crs replica for device slot %zu could not be made", ctx_->dev_slot);
  CDL_CUDA(ctx_, cudaMemcpyAsync(d_pool(), pts, (size_t)L.crs_size * sizeof(G1Affine), cudaMemcpyDeviceToDevice,
                                 ctx_->stream));
  return CDL_OK;
}

// Batches of at least CDL_FIXED_BASE_MINB instances (default 64 per lane; 0 = never) use fixed-base tables
// for the CRS points.  The tables belong to the CRS object, one copy per device slot, and are built on
// that slot's first use (~ 10 ms and 4.3 MB per point); a failed allocation simply leaves the generic
// kernels in charge.
void Engine::select_fixed(const Layout& L, const cdl_crs* crs, size_t B) {
  fixed_ = cdl::FixedTable();
  static const long min_b = [] {
    const char* e = getenv("CDL_FIXED_BASE_MINB");
    return e ? atol(e) : 64L;
  }();
  const long over = ctx_->root()->fixed_min_batch;
  const long lim = over >= 0 ? over : min_b;
  if (lim <= 0 || (long)B < lim) return;
  std::lock_guard<std::mutex> lk(crs->fixed_mu);
  cdl_crs::Replica& r = crs->rep[ctx_->dev_slot];
  if (!r.d_fixed && !r.fixed_failed) {
    const G1Affine* pts = crs->points_on(ctx_->dev_slot);
    cdl::G1Affine* tab = nullptr;
    if (!pts || cudaMalloc(&tab, cdl::fixed_table_bytes(L.crs_size)) != cudaSuccess) {
      cudaGetLastError();
      r.fixed_failed = true;
      return;
    }
    cdl::launch_fixed_build(pts, L.crs_size, tab, ctx_->stream);
    if (cudaStreamSynchronize(ctx_->stream) != cudaSuccess) {
      cudaFree(tab);
      r.fixed_failed = true;
      return;
    }
    r.d_fixed = tab;
  }
  if (r.d_fixed) {
    fixed_.tab = r.d_fixed;
    fixed_.nbase = L.crs_size;
  }
}

int32_t Engine::upload_points(uint32_t dst, const void* host_affine, size_t count) {
  if (!count) return CDL_OK;
  CDL_CUDA(ctx_, cudaMemcpyAsync(d_pool() + dst, host_affine, count * sizeof(G1Affine), cudaMemcpyHostToDevice, ctx_->stream));
  CDL_CUDA(ctx_, ctx_->sync_stream());  // caller memory is pageable and may go away
  return CDL_OK;
}

int32_t Engine::download_points(uint32_t src, void* host_affine, size_t count) {
  if (!count) return CDL_OK;
  CDL_CUDA(ctx_, cudaMemcpyAsync(host_affine, d_pool() + src, count * sizeof(G1Affine), cudaMemcpyDeviceToHost, ctx_->stream));
  CDL_CUDA(ctx_, ctx_->sync_stream());
  return CDL_OK;
}

int32_t Engine::copy_points(uint32_t dst, uint32_t src, size_t count) {
  if (!count) return CDL_OK;
  CDL_CUDA(ctx_, cudaMemcpyAsync(d_pool() + dst, d_pool() + src, count * sizeof(G1Affine), cudaMemcpyDeviceToDevice, ctx_->stream));
  return CDL_OK;
}

int32_t Engine::set_infinity(uint32_t dst, size_t count) {
  if (!count) return CDL_OK;
  CDL_CUDA(ctx_, cudaMemsetAsync(d_pool() + dst, 0, count * sizeof(G1Affine), ctx_->stream));
  return CDL_OK;
}

int32_t Engine::copy_ranges(const std::vector<cdl::CopyRange>& ranges) {
  const size_t n = ranges.size();
  if (!n) return CDL_OK;
  // own staging buffer: the copy is left in flight (the next stage's launch syncs), so the pinned
  // descriptors must not be shared with a stage that refills its staging before that sync
  CDL_CUDA(ctx_, ctx_->sync_stream());  // a previous copy_ranges may still be reading s_cr_
  int32_t rc = reserve(s_cr_, n * sizeof(cdl::CopyRange));
  if (rc) return rc;
  memcpy(s_cr_.h(), ranges.data(), n * sizeof(cdl::CopyRange));
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_cr_.d(), s_cr_.h(), n * sizeof(cdl::CopyRange), cudaMemcpyHostToDevice, ctx_->stream));
  cdl::launch_copy_ranges(d_pool(), (const cdl::CopyRange*)s_cr_.d(), (int)n, ctx_->stream);
  CDL_CUDA(ctx_, cudaGetLastError());
  launches++;
  return CDL_OK;
}

namespace {
struct ProfScope {
  double& acc;
  double t0;
  explicit ProfScope(double& a) : acc(a), t0(Engine::now()) {}
  ~ProfScope() { acc += Engine::now() - t0; }
};
}  // namespace

int32_t Engine::load_instances(const Layout& L, const std::vector<uint32_t>& sel, const cdl_g1_affine* const* pts,
                               uint32_t npts, const cdl_g1_jac* M) {
  ProfScope ps(prof.gpu);
  const size_t B = sel.size(), per = (size_t)npts * L.ell;
  if (!B) return CDL_OK;
  const uint32_t tail = L.base((uint32_t)B), tail_m = tail + (uint32_t)(B * per);
  int32_t rc;
  if ((rc = reserve(s_in_, B * per * sizeof(G1Affine))) || (M && (rc = reserve(s_jac_, B * sizeof(cdl::G1Jac)))))
    return rc;
  {
    ProfScope pc(prof.copy);
    G1Affine* h = (G1Affine*)s_in_.h();
    pool_.parallel_for(B, std::function<void(size_t)>([&](size_t j) {
      for (uint32_t a = 0; a < npts; a++)
        memcpy(h + j * per + (size_t)a * L.ell, pts[a] + (size_t)sel[j] * L.ell, (size_t)L.ell * sizeof(G1Affine));
    }));
    if (M)
      for (size_t j = 0; j < B; j++) memcpy((cdl::G1Jac*)s_jac_.h() + j, M + sel[j], sizeof(cdl::G1Jac));
  }
  CDL_CUDA(ctx_, cudaMemcpyAsync(d_pool() + tail, s_in_.h(), B * per * sizeof(G1Affine), cudaMemcpyHostToDevice, ctx_->stream));
  if (M) {
    CDL_CUDA(ctx_, cudaMemcpyAsync(s_jac_.d(), s_jac_.h(), B * sizeof(cdl::G1Jac), cudaMemcpyHostToDevice, ctx_->stream));
    tick();
    cdl::launch_jac_to_affine((const cdl::G1Jac*)s_jac_.d(), d_pool() + tail_m, (int)B, ctx_->stream);
    tock(3, 0, 240.0 * B);
    CDL_CUDA(ctx_, cudaGetLastError());
  }
  std::vector<cdl::CopyRange> ranges;
  ranges.reserve(M ? 2 * B : B);
  for (size_t j = 0; j < B; j++) {
    const uint32_t base = L.base((uint32_t)j);
    ranges.push_back(cdl::CopyRange{tail + (uint32_t)(j * per), base + L.Rs, (uint32_t)per, 0});
    if (M) ranges.push_back(cdl::CopyRange{tail_m + (uint32_t)j, base + L.M, 1, 0});
  }
  // copy_ranges waits for the stream before it refills its descriptors, so the staging buffers are free and
  // the normalisation's events complete when it returns; the copy itself is ordered before the next stage
  if ((rc = copy_ranges(ranges))) return rc;
  finish_timing();
  return CDL_OK;
}

int32_t Engine::compress(const std::vector<uint32_t>& src, std::vector<uint8_t>& out48) {
  ProfScope ps(prof.gpu);
  size_t n = src.size();
  out48.resize(n * 48);
  if (!n) return CDL_OK;
  int32_t rc;
  if ((rc = reserve(s_idx_, n * 4)) || (rc = reserve(s_out_, n * 48))) return rc;
  memcpy(s_idx_.h(), src.data(), n * 4);
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_idx_.d(), s_idx_.h(), n * 4, cudaMemcpyHostToDevice, ctx_->stream));
  tick();
  cdl::launch_compress_idx(d_pool(), (const uint32_t*)s_idx_.d(), (uint8_t*)s_out_.d(), (int)n, ctx_->stream);
  tock(3, 3.0 * n, 148.0 * n);
  CDL_CUDA(ctx_, cudaGetLastError());
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_out_.h(), s_out_.d(), n * 48, cudaMemcpyDeviceToHost, ctx_->stream));
  CDL_CUDA(ctx_, ctx_->sync_stream());
  finish_timing();
  memcpy(out48.data(), s_out_.h(), n * 48);
  return CDL_OK;
}

int32_t Engine::decompress(const uint8_t* enc48, const std::vector<uint32_t>& dst, std::vector<uint8_t>& status) {
  ProfScope ps(prof.gpu);
  size_t n = dst.size();
  status.assign(n, 0);
  if (!n) return CDL_OK;
  int32_t rc;
  if ((rc = reserve(s_idx_, n * 4)) || (rc = reserve(s_enc_, n * 48)) || (rc = reserve(s_st_, n))) return rc;
  memcpy(s_idx_.h(), dst.data(), n * 4);
  memcpy(s_enc_.h(), enc48, n * 48);
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_idx_.d(), s_idx_.h(), n * 4, cudaMemcpyHostToDevice, ctx_->stream));
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_enc_.d(), s_enc_.h(), n * 48, cudaMemcpyHostToDevice, ctx_->stream));
  tick();
  cdl::launch_decompress_idx((const uint8_t*)s_enc_.d(), d_pool(), (const uint32_t*)s_idx_.d(), (uint8_t*)s_st_.d(), (int)n, ctx_->stream);
  // sqrt = one fixed 381-bit exponentiation (~480 modmul) + subgroup check [r]P (3193 by the §8d convention)
  tock(2, (480.0 + 3193.0) * n, 148.0 * n);
  CDL_CUDA(ctx_, cudaGetLastError());
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_st_.h(), s_st_.d(), n, cudaMemcpyDeviceToHost, ctx_->stream));
  CDL_CUDA(ctx_, ctx_->sync_stream());
  finish_timing();
  memcpy(status.data(), s_st_.h(), n);
  return CDL_OK;
}

static constexpr uint32_t kFixedMinTerms = 16;

int32_t Engine::run_msm(MsmStage& st, const MsmBefore& before, const G1Affine* points) {
  ProfScope ps(prof.gpu);
  size_t nt = st.tasks.size(), nterm = st.idx.size();
  st.out48.resize(nt * 48);
  if (!nt) return CDL_OK;
  if (!points) points = d_pool();
  size_t max_terms = 0;
  for (auto& t : st.tasks) max_terms = std::max<size_t>(max_terms, t.term_cnt);
  int32_t rc;
  if ((rc = reserve(s_idx_, (nterm + 1) * 4)) || (rc = reserve(s_sc_, (nterm + 1) * 32)) ||
      (rc = reserve(s_task_, nt * sizeof(MsmTask))) || (rc = reserve(s_out_, nt * 48)))
    return rc;
  // the latency kernel stages a task's terms in shared memory: every task it gets must fit
  static_assert(cdl::kMsmSplitTerms <= cdl::kMsmMaxTerms, "small-MSM tasks must fit the kernel's staging");
  const bool throughput = (int)nt >= cdl::kMsmSplitThreshold || max_terms > cdl::kMsmSplitTerms;
  std::vector<uint32_t> fixed_tasks;  // tasks whose CRS terms go through the fixed-base tables
  {
    ProfScope pc(prof.copy);
    memcpy(s_idx_.h(), st.idx.data(), nterm * 4);
    memcpy(s_sc_.h(), st.sc.data(), nterm * 32);
    memcpy(s_task_.h(), st.tasks.data(), nt * sizeof(MsmTask));
    if (throughput && fixed_.tab) {
      // terms on CRS points go through the fixed-base tables when their task holds enough of them to pay
      // for the extra pass (a chunk's lanes share 22 look-ups per 32 such terms; a lone term costs as much)
      uint32_t* idx = (uint32_t*)s_idx_.h();
      for (size_t j = 0; j < nt; j++) {
        const MsmTask& t = st.tasks[j];
        uint32_t cnt = 0;
        for (uint32_t k = 0; k < t.term_cnt; k++) cnt += (idx[t.term_off + k] & 0x7fffffffu) < fixed_.nbase;
        if (cnt < kFixedMinTerms) continue;
        for (uint32_t k = 0; k < t.term_cnt; k++)
          if ((idx[t.term_off + k] & 0x7fffffffu) < fixed_.nbase) idx[t.term_off + k] |= cdl::kMsmIdxFixed;
        fixed_tasks.push_back((uint32_t)j);
      }
    }
  }
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_idx_.d(), s_idx_.h(), nterm * 4, cudaMemcpyHostToDevice, ctx_->stream));
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_sc_.d(), s_sc_.h(), nterm * 32, cudaMemcpyHostToDevice, ctx_->stream));
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_task_.d(), s_task_.h(), nt * sizeof(MsmTask), cudaMemcpyHostToDevice, ctx_->stream));
  if (before) {
    bool done = false;
    int32_t brc = before((const uint32_t*)s_idx_.d(), (cdl::Fr*)s_sc_.d(), (const MsmTask*)s_task_.d(), done);
    if (brc) return brc;
    if (done) {
      std::fill(st.out48.begin(), st.out48.end(), 0);
      return CDL_OK;
    }
  }
  double alg = 0;
  // credited per task at the reference's term count (a base expanded into several CRS terms counts once)
  for (size_t j = 0; j < st.tasks.size(); j++)
    alg += msm_algorithmic_modmul(st.tasks[j].term_cnt - (st.extra.size() == st.tasks.size() ? st.extra[j] : 0));
  if (throughput) {
    // throughput path: recode + warp-per-chunk + per-task combine
    std::vector<cdl::MsmSub> subs;
    std::vector<cdl::MsmTask2> tasks2;
    cdl::msm_build_subs(st.tasks.data(), nt, cdl::msm_tp_pick_chunk(nterm, ctx_->sm_count), subs, tasks2);
    if ((rc = reserve(s_sub_, subs.size() * sizeof(cdl::MsmSub))) || (rc = reserve(s_t2_, tasks2.size() * sizeof(cdl::MsmTask2))))
      return rc;
    if (!d_win_.grow(cdl::msm_tp_scratch_bytes(nterm, subs.size(), nt), ctx_->stream))
      return ctx_->fail(CDL_ERR_CUDA, "MSM scratch allocation failed");
    std::vector<uint32_t> fsubs;  // the chunks of those tasks
    for (uint32_t j : fixed_tasks)
      for (uint32_t c = 0; c < tasks2[j].sub_cnt; c++) fsubs.push_back(tasks2[j].sub_off + c);
    if (!fsubs.empty()) {
      if ((rc = reserve(s_fsub_, fsubs.size() * 4))) return rc;
      memcpy(s_fsub_.h(), fsubs.data(), fsubs.size() * 4);
      CDL_CUDA(ctx_, cudaMemcpyAsync(s_fsub_.d(), s_fsub_.h(), fsubs.size() * 4, cudaMemcpyHostToDevice, ctx_->stream));
    }
    memcpy(s_sub_.h(), subs.data(), subs.size() * sizeof(cdl::MsmSub));
    memcpy(s_t2_.h(), tasks2.data(), tasks2.size() * sizeof(cdl::MsmTask2));
    CDL_CUDA(ctx_, cudaMemcpyAsync(s_sub_.d(), s_sub_.h(), subs.size() * sizeof(cdl::MsmSub), cudaMemcpyHostToDevice, ctx_->stream));
    CDL_CUDA(ctx_, cudaMemcpyAsync(s_t2_.d(), s_t2_.h(), tasks2.size() * sizeof(cdl::MsmTask2), cudaMemcpyHostToDevice, ctx_->stream));
    tick();
    cdl::launch_msm_tp(points, (const uint32_t*)s_idx_.d(), (const cdl::Fr*)s_sc_.d(), (int)nterm, (const cdl::MsmSub*)s_sub_.d(),
                       (int)subs.size(), (const cdl::MsmTask2*)s_t2_.d(), (int)nt, d_pool(), (uint8_t*)s_out_.d(), d_win_.d(),
                       ctx_->stream, fixed_, fsubs.empty() ? nullptr : (const uint32_t*)s_fsub_.d(), (int)fsubs.size());
    tock(0, alg, 128.0 * nterm);
    launches += fsubs.empty() ? 3 : 4;  // recode, bucket warps, chunk sums (+ fixed-base warps); tock counted the combine
  } else {
    tick();
    cdl::launch_msm_small(points, (const uint32_t*)s_idx_.d(), (const cdl::Fr*)s_sc_.d(), (const MsmTask*)s_task_.d(), (int)nt,
                          max_terms, d_pool(), (uint8_t*)s_out_.d(), ctx_->stream);
    tock(0, alg, 128.0 * nterm);
  }
  CDL_CUDA(ctx_, cudaGetLastError());
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_out_.h(), s_out_.d(), nt * 48, cudaMemcpyDeviceToHost, ctx_->stream));
  CDL_CUDA(ctx_, ctx_->sync_stream());
  finish_timing();
  memcpy(st.out48.data(), s_out_.h(), nt * 48);
  return CDL_OK;
}

int32_t Engine::run_elem(const std::vector<ElemOp>& ops, const std::vector<Fr>& sc) {
  ProfScope ps(prof.gpu);
  size_t n = ops.size();
  if (!n) return CDL_OK;
  int32_t rc;
  if ((rc = reserve(s_ops_, n * sizeof(ElemOp))) || (rc = reserve(s_sc_, sc.size() * 32))) return rc;
  memcpy(s_ops_.h(), ops.data(), n * sizeof(ElemOp));
  memcpy(s_sc_.h(), sc.data(), sc.size() * 32);
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_ops_.d(), s_ops_.h(), n * sizeof(ElemOp), cudaMemcpyHostToDevice, ctx_->stream));
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_sc_.d(), s_sc_.h(), sc.size() * 32, cudaMemcpyHostToDevice, ctx_->stream));
  tick();
  cdl::launch_elem_ops(d_pool(), (const ElemOp*)s_ops_.d(), (const cdl::Fr*)s_sc_.d(), (int)n, ctx_->stream, fixed_);
  tock(1, 3193.0 * n, 288.0 * n);  // §8d: 3193 modmul per scalar multiplication; src + add + dst points
  CDL_CUDA(ctx_, cudaGetLastError());
  CDL_CUDA(ctx_, ctx_->sync_stream());
  finish_timing();
  return CDL_OK;
}

// ------------------------------------------------------------------ helpers
namespace {

// a stage with a fixed number of tasks/terms per instance; instance b builds
// into its own slice, so the build parallelises over the batch
struct StageBuilder {
  MsmStage& st;
  uint32_t B, terms_per, tasks_per;
  StageBuilder(MsmStage& s, uint32_t B_, uint32_t terms, uint32_t tasks) : st(s), B(B_), terms_per(terms), tasks_per(tasks) {
    st.idx.assign((size_t)B * terms, 0);
    st.sc.assign((size_t)B * terms, FR_ZERO);
    st.tasks.assign((size_t)B * tasks, MsmTask{0, 0, 0, 0});
    st.extra.assign((size_t)B * tasks, 0);
  }
  MsmSlice slice(uint32_t b) {
    MsmSlice s;
    s.idx = st.idx.data() + (size_t)b * terms_per;
    s.sc = st.sc.data() + (size_t)b * terms_per;
    s.tasks = st.tasks.data() + (size_t)b * tasks_per;
    s.extra = st.extra.data() + (size_t)b * tasks_per;
    s.term_base = b * terms_per;
    return s;
  }
  const uint8_t* out(uint32_t b, uint32_t task) const { return st.out48.data() + ((size_t)b * tasks_per + task) * 48; }
};

inline bool is_inf_enc(const uint8_t* e) { return memcmp(e, kInfEnc, 48) == 0; }

// batches of at least this many proofs derive T_2, U_2, A_2, B_2 from R and S in a second launch
constexpr uint32_t kStep3SplitBatch = 8;

}  // namespace

// ------------------------------------------------------------------ ShufflePermuteCommit
int32_t Engine::shuffle_permute_commit(const Layout& L, uint32_t B, const std::vector<std::vector<uint32_t>>& perms,
                                       const std::vector<Fr>& ks, std::vector<cdl_rand*>& rands,
                                       std::vector<std::vector<Fr>>& rs_m) {
  ProfScope ptot(prof.total);
  const uint32_t ell = L.ell;
  // Ts[i] = k * Rs[perm[i]], Us[i] = k * Ss[perm[i]]   (common/util.go:55-66)
  std::vector<ElemOp> ops((size_t)B * 2 * ell);
  std::vector<Fr> sc(B);
  for (uint32_t b = 0; b < B; b++) {
    uint32_t base = L.base(b);
    sc[b] = ks[b];
    for (uint32_t i = 0; i < ell; i++) {
      ops[(size_t)b * 2 * ell + i] = ElemOp{base + L.Rs + perms[b][i], cdl::kNoPoint, base + L.Ts + i, b};
      ops[(size_t)b * 2 * ell + ell + i] = ElemOp{base + L.Ss + perms[b][i], cdl::kNoPoint, base + L.Us + i, b};
    }
  }
  int32_t rc = run_elem(ops, sc);
  if (rc) return rc;
  // M = <perm(0..ell-1), Gs> + <rs_m, Hs>   (common/util.go:68-85)
  MsmStage st;
  StageBuilder sb(st, B, ell + kBlinders, 1);
  rs_m.assign(B, std::vector<Fr>(kBlinders));
  std::vector<Fr> small(ell);  // fr.NewElement(j), once per call
  for (uint32_t j = 0; j < ell; j++) small[j] = fr_from_u64(j);
  for (uint32_t b = 0; b < B; b++) {
    rands[b]->r.get_frs(rs_m[b].data(), kBlinders);
    MsmSlice s = sb.slice(b);
    s.begin(L.base(b) + L.M);
    for (uint32_t i = 0; i < ell; i++) s.term(L.Gs + i, small[perms[b][i]]);
    for (uint32_t j = 0; j < kBlinders; j++) s.term(L.Hs + j, rs_m[b][j]);
    s.end();
  }
  return run_msm(st);
}

// ------------------------------------------------------------------ Prove
namespace {

struct ProveState {
  Transcript tr{"curdleproofs"};
  bool failed = false;
  std::string err;
  std::vector<Fr> as, perm_as, rs_a, bs, rs_b, cs, ds, r_cs, x, r;
  Fr alpha, beta, p, r_p, z, r_t, r_u, r_a, r_b, r_k, z_k, z_t, z_u;
  Fr beta_ipa;
  // wire pieces (48-byte encodings)
  uint8_t A[48], T1[48], T2[48], U1[48], U2[48], R[48], S[48], Bp[48], C[48], B_c[48], B_d[48];
  uint8_t A1[48], A2[48], B1[48], B2[48], B_a[48], B_t[48], B_u[48];
  std::vector<uint8_t> L_C, R_C, L_D, R_D, L_A, L_T, L_U, R_A, R_T, R_U;
  Fr c0, d0, x0;
  void fail(const std::string& e) { if (!failed) { failed = true; err = e; } }
};

// innerproductargument.go:299-391
bool generate_ipa_blinders(Rand& rand, const std::vector<Fr>& cs, const std::vector<Fr>& ds, std::vector<Fr>& rs,
                           std::vector<Fr>& zs, std::string& err) {
  size_t n = cs.size();
  rs.resize(n);
  zs.resize(n - 2);
  rand.get_frs(rs.data(), n);
  rand.get_frs(zs.data(), n - 2);
  Fr omega = fr_add(fr_inner(rs.data(), ds.data(), n), fr_inner(zs.data(), cs.data(), n - 2));
  Fr delta = fr_inner(rs.data(), zs.data(), n - 2);
  Fr inv_c = fr_inv(cs[n - 2]);
  Fr t1 = fr_sub(fr_mul(fr_mul(rs[n - 2], inv_c), omega), delta);
  Fr t2 = fr_add(fr_mul(fr_mul(fr_neg(rs[n - 2]), inv_c), cs[n - 1]), rs[n - 1]);
  if (fr_is_zero(t2)) { err = "last_z_term2 is zero"; return false; }
  Fr last_z = fr_mul(t1, fr_inv(t2));
  Fr pen_z = fr_mul(fr_neg(inv_c), fr_add(fr_mul(last_z, cs[n - 1]), omega));
  zs.push_back(pen_z);
  zs.push_back(last_z);
  Fr chk = fr_add(fr_inner(rs.data(), ds.data(), n), fr_inner(zs.data(), cs.data(), n));
  if (!fr_is_zero(chk) || !fr_is_zero(fr_inner(rs.data(), zs.data(), n))) {
    err = "failed to generate IPA blinders: constraints not satisfied";
    return false;
  }
  return true;
}

void put_u32_be(std::vector<uint8_t>& v, uint32_t x) {
  v.push_back((uint8_t)(x >> 24)); v.push_back((uint8_t)(x >> 16)); v.push_back((uint8_t)(x >> 8)); v.push_back((uint8_t)x);
}
void put_pt(std::vector<uint8_t>& v, const uint8_t* e) { v.insert(v.end(), e, e + 48); }
void put_slice(std::vector<uint8_t>& v, const std::vector<uint8_t>& pts) {
  put_u32_be(v, (uint32_t)(pts.size() / 48));
  v.insert(v.end(), pts.begin(), pts.end());
}
void put_fr(std::vector<uint8_t>& v, const Fr& s) {
  uint8_t b[32];
  fr_to_bytes_be(b, s);
  v.insert(v.end(), b, b + 32);
}

}  // namespace

int32_t Engine::prove(const Layout& L, uint32_t B, const cdl_crs* crs, const std::vector<std::vector<uint32_t>>& perms,
                      const std::vector<Fr>& ks, const std::vector<std::vector<Fr>>& rs_m_in,
                      std::vector<cdl_rand*>& rands, std::vector<std::vector<uint8_t>>& proofs,
                      std::vector<int32_t>& status, std::vector<std::string>& errs, std::vector<uint8_t>& inst_enc,
                      bool witness_is_ours) {
  ProfScope ptot(prof.total);
  const uint32_t ell = L.ell, n = L.n, m = L.m;
  if (n != (1u << m)) return ctx_->fail(CDL_ERR_PROTOCOL, "cs and ds are not a power of two (ell + 4 = %u)", n);
  int32_t rc;
  std::vector<std::unique_ptr<ProveState>> S(B);
  for (auto& s : S) s.reset(new ProveState());
  const uint8_t* H_enc = crs->enc.data() + 48 * (size_t)L.H;
  MsmStage st;

  // ---- step 1: transcript over the instance (curdleproof.go:50-58)
  std::vector<uint32_t> src;
  src.reserve((size_t)B * (4 * ell + 1));
  for (uint32_t b = 0; b < B; b++) {
    uint32_t base = L.base(b);
    for (uint32_t i = 0; i < 4 * ell; i++) src.push_back(base + L.Rs + i);  // Rs, Ss, Ts, Us are contiguous
    src.push_back(base + L.M);
  }
  if ((rc = compress(src, inst_enc))) return rc;
  const size_t per_inst = (size_t)(4 * ell + 1) * 48;
  par(B, [&](size_t b) {
    ProveState& s = *S[b];
    const uint8_t* e = inst_enc.data() + b * per_inst;
    s.tr.append_points("curdleproofs_step1", e, 4 * ell + 1);
    s.as.resize(ell);
    for (uint32_t i = 0; i < ell; i++) s.as[i] = s.tr.challenge("curdleproofs_vec_a");
    s.rs_a.resize(kBlinders - 2);
    rands[b]->r.get_frs(s.rs_a.data(), kBlinders - 2);  // :61
    s.perm_as.resize(ell);
    for (uint32_t i = 0; i < ell; i++) s.perm_as[i] = s.as[perms[b][i]];
  });

  // ---- A = <perm_as, Gs> + <rs_a', Hs>   (:72-79)
  {
    StageBuilder sb(st, B, ell + 2, 1);
    par(B, [&](size_t b) {
      ProveState& s = *S[b];
      MsmSlice sl = sb.slice((uint32_t)b);
      sl.begin(L.base((uint32_t)b) + L.A);
      for (uint32_t i = 0; i < ell; i++) sl.term(L.Gs + i, s.perm_as[i]);
      for (uint32_t j = 0; j < 2; j++) sl.term(L.Hs + j, s.rs_a[j]);
      sl.end();
    });
    if ((rc = run_msm(st))) return rc;
    for (uint32_t b = 0; b < B; b++) memcpy(S[b]->A, sb.out(b, 0), 48);
  }

  // ---- same-permutation argument, step 1-2 (samepermutationargument.go:44-80)
  par(B, [&](size_t b) {
    ProveState& s = *S[b];
    const uint8_t* M_enc = inst_enc.data() + b * per_inst + (size_t)4 * ell * 48;
    s.tr.append_points("same_perm_step1", s.A, 1);
    s.tr.append_points("same_perm_step1", M_enc, 1);
    s.tr.append_scalars("same_perm_step1", s.as.data(), ell);
    s.alpha = s.tr.challenge("same_perm_alpha");
    s.beta = s.tr.challenge("same_perm_beta");
    s.bs.resize(ell);
    s.p = FR_ONE;
    std::vector<Fr> alpha_times(ell);  // alpha * j for j < ell by repeated addition
    alpha_times[0] = FR_ZERO;
    for (uint32_t j = 1; j < ell; j++) alpha_times[j] = fr_add(alpha_times[j - 1], s.alpha);
    for (uint32_t i = 0; i < ell; i++) {
      s.bs[i] = fr_add(fr_add(alpha_times[perms[b][i]], s.perm_as[i]), s.beta);
      s.p = fr_mul(s.p, s.bs[i]);
    }
    s.rs_b.resize(kBlinders);
    for (uint32_t i = 0; i < kBlinders; i++) {
      Fr ra = i < 2 ? s.rs_a[i] : FR_ZERO;
      s.rs_b[i] = fr_add(fr_mul(s.alpha, rs_m_in[b][i]), ra);
    }
  });
  // B = A + alpha*M + beta*sum(Gs)   (:62-73; sum(Gs) is crs.Gsum: every cdl_crs has Gsum = sum Gs and
  // Hsum = sum Hs, which cdl_crs_from_points checks)
  {
    StageBuilder sb(st, B, 3, 1);
    for (uint32_t b = 0; b < B; b++) {
      ProveState& s = *S[b];
      MsmSlice sl = sb.slice(b);
      uint32_t base = L.base(b);
      sl.begin(base + L.B);
      sl.term(base + L.A, FR_ONE);
      sl.term(base + L.M, s.alpha);
      sl.term(L.Gsum, s.beta);
      sl.end();
    }
    if ((rc = run_msm(st))) return rc;
    for (uint32_t b = 0; b < B; b++) memcpy(S[b]->Bp, sb.out(b, 0), 48);
  }

  // ---- grand-product argument (grandproductargument.go:52-92)
  std::vector<Fr> gp_alpha(B), gp_beta(B), gp_beta_inv(B);
  std::vector<std::vector<Fr>> gp_scale;  // G'[i] = gp_scale[b][i] * (Gs || Hs)[i]
  // With the CRS fixed-base tables at hand (fixed_base.cuh) the CRS-based vectors of the two folding arguments —
  // G and G' of the inner-product argument, Gm of the same-multiscalar argument — are not folded in their first
  // two rounds at all: a folded base is a short linear combination of CRS points,
  //   V1[i] = V[i] + x1 V[i + n/2],   V2[i] = V[i] + x1 V[i + n/2] + x2 V[i + n/4] + x1 x2 V[i + 3n/4],
  // so the second round's MSMs take two CRS terms per base (220 products each, against 700 for a bucket term
  // plus 1 500 for the scalar multiplication that would have produced the base) and V2 is built once, straight
  // from the CRS, by three or four chained table multiplications per element.  Rounds three onwards fold as
  // before.  Small batches (no tables) keep the plain schedule: it has fewer launches.
  const bool lazy = fixed_.tab != nullptr && n >= 8;
  std::vector<std::array<Fr, 4>> ipa_x(B), sm_x(B);  // gamma_0, gamma_0^-1, gamma_1, gamma_1^-1 of the two arguments
  par(B, [&](size_t b) {
    ProveState& s = *S[b];
    s.tr.append_points("gprod_step1", s.Bp, 1);
    s.tr.append_scalar("gprod_step1", s.p);
    gp_alpha[b] = s.tr.challenge("gprod_alpha");
    s.cs.assign(ell, FR_ONE);
    for (uint32_t i = 1; i < ell; i++) s.cs[i] = fr_mul(s.cs[i - 1], s.bs[i - 1]);
    s.r_cs.resize(kBlinders);
    rands[b]->r.get_frs(s.r_cs.data(), kBlinders);
  });
  {
    StageBuilder sb(st, B, n, 1);
    par(B, [&](size_t b) {
      ProveState& s = *S[b];
      MsmSlice sl = sb.slice((uint32_t)b);
      sl.begin(L.base((uint32_t)b) + L.scratch);
      for (uint32_t i = 0; i < ell; i++) sl.term(L.Gs + i, s.cs[i]);
      for (uint32_t j = 0; j < kBlinders; j++) sl.term(L.Hs + j, s.r_cs[j]);
      sl.end();
    });
    if ((rc = run_msm(st))) return rc;
    for (uint32_t b = 0; b < B; b++) memcpy(S[b]->C, sb.out(b, 0), 48);
  }
  std::vector<std::vector<Fr>> r_b_plus_alpha(B);
  std::vector<Fr> beta_l1(B);
  {
    // Gs'[i] = beta^-(i+1) Gs[i], Hs'[i] = beta^-(ell+1) Hs[i]  (:94-103) -> Gp; G = Gs || Hs.
    // Only the LOWER half of G' = Gs' || Hs' is ever materialised: everything the prover does with the upper
    // half before the first fold is linear in it — B_d, the self-check, L_D / R_D of the first round and the
    // first fold G'_L + gamma^-1 G'_R — and is taken on the CRS points themselves with the scale factor
    // gp_scale[i] = beta^-(i+1) (beta^-(ell+1) for the Hs part) multiplied into the scalar, where the
    // fixed-base tables (fixed_base.cuh) apply.
    const uint32_t nh = lazy ? 0 : n / 2;  // lazy: G' is first materialised after the second round, from the CRS
    std::vector<ElemOp> ops((size_t)B * nh);
    std::vector<Fr> sc((size_t)B * (ell + 1));
    gp_scale.assign(B, std::vector<Fr>());
    par(B, [&](size_t b) {
      ProveState& s = *S[b];
      r_b_plus_alpha[b].resize(kBlinders);
      for (uint32_t i = 0; i < kBlinders; i++) r_b_plus_alpha[b][i] = fr_add(s.rs_b[i], gp_alpha[b]);
      s.r_p = fr_inner(r_b_plus_alpha[b].data(), s.r_cs.data(), kBlinders);
      s.tr.append_points("gprod_step2", s.C, 1);
      s.tr.append_scalar("gprod_step2", s.r_p);
      gp_beta[b] = s.tr.challenge("gprod_beta");
      if (fr_is_zero(gp_beta[b])) { s.fail("beta is zero"); }
      Fr beta_inv = fr_inv(gp_beta[b]);
      gp_beta_inv[b] = beta_inv;
      uint32_t base = L.base((uint32_t)b);
      Fr t = beta_inv;
      Fr* scb = sc.data() + b * (ell + 1);
      std::vector<Fr>& scale = gp_scale[b];
      scale.resize(n);
      for (uint32_t i = 0; i < ell; i++) {
        scb[i] = t;
        scale[i] = t;
        if (i < nh) ops[b * nh + i] = ElemOp{L.Gs + i, cdl::kNoPoint, base + L.Gp + i, (uint32_t)(b * (ell + 1) + i)};
        t = fr_mul(t, beta_inv);
      }
      scb[ell] = t;
      for (uint32_t j = 0; j < kBlinders; j++) {
        scale[ell + j] = t;
        if (ell + j < nh)  // only for ell < 4
          ops[b * nh + ell + j] = ElemOp{L.Hs + j, cdl::kNoPoint, base + L.Gp + ell + j, (uint32_t)(b * (ell + 1) + ell)};
      }
    });
    if ((rc = run_elem(ops, sc))) return rc;
    std::vector<cdl::CopyRange> cr(B);
    for (uint32_t b = 0; b < B; b++) cr[b] = cdl::CopyRange{L.Gs, L.base(b) + L.G, n, 0};  // Gs and Hs are adjacent in the CRS image
    if ((rc = copy_ranges(cr))) return rc;
  }
  // D, the self-check on D, B_c, B_d  (:105-177, innerproductargument.go:59-72).
  // D = B - <beta^i, Gs'> + <alpha*beta^(ell+1), Hs'> (:132-138) with Gs'[i] = beta^-(i+1) Gs[i] and
  // Hs'[j] = beta^-(ell+1) Hs[j] is B - beta^-1 * Gsum + alpha * Hsum term by term - the very formula
  // the verifier uses (:243-246) - so it is computed as that three-term MSM (same point, same bytes).  Term by
  // term only because every cdl_crs has Gsum = sum Gs and Hsum = sum Hs (checked by cdl_crs_from_points).
  // The reference's self-check msm(Gs||Hs, cs||r_cs) == C (:164-170) recomputes C = <cs, Gs> + <r_cs, Hs>
  // (:66-73) from the very same operands: it cannot fail, so it is not launched.  msm(G', d) == D
  // (:171-177) depends on the caller's M and rs_m and is the reference's error path for a witness that
  // does not match the commitment: it is kept whenever the caller supplied them (cdl_prove), and
  // skipped when this library computed M from rs_m itself a moment ago (the Whisk wrapper).
  std::vector<std::vector<Fr>> rs_c(B), rs_d(B);
  std::vector<std::array<uint8_t, 48>> D_enc(B);
  {
    StageBuilder sb(st, B, 3 + (witness_is_ours ? 0 : n) + 2 * n, 4);
    par(B, [&](size_t b) {
      ProveState& s = *S[b];
      const Fr& beta = gp_beta[b];
      const Fr& alpha = gp_alpha[b];
      // ds[i] = bs[i]*beta^(i+1) - beta^i
      s.ds.resize(ell);
      Fr tb = FR_ONE;
      for (uint32_t i = 0; i < ell; i++) {
        Fr nx = fr_mul(tb, beta);
        s.ds[i] = fr_sub(fr_mul(s.bs[i], nx), tb);
        tb = nx;
      }
      Fr beta_l = tb;  // beta^ell
      beta_l1[b] = fr_mul(beta_l, beta);
      std::vector<Fr> r_ds(kBlinders);
      for (uint32_t i = 0; i < kBlinders; i++) r_ds[i] = fr_mul(beta_l1[b], r_b_plus_alpha[b][i]);
      s.z = fr_sub(fr_add(fr_mul(s.r_p, beta_l1[b]), fr_mul(s.p, beta_l)), FR_ONE);
      s.cs.insert(s.cs.end(), s.r_cs.begin(), s.r_cs.end());
      s.ds.insert(s.ds.end(), r_ds.begin(), r_ds.end());
      if (!fr_eq(fr_inner(s.cs.data(), s.ds.data(), n), s.z)) s.fail("IPA(C, D) != z");
      std::string e;
      if (!s.failed && !generate_ipa_blinders(rands[b]->r, s.cs, s.ds, rs_c[b], rs_d[b], e)) s.fail("generate IPA blinders: " + e);
      if (s.failed) { rs_c[b].assign(n, FR_ZERO); rs_d[b].assign(n, FR_ZERO); }
      uint32_t base = L.base((uint32_t)b);
      MsmSlice sl = sb.slice((uint32_t)b);
      // D = B - beta^-1 * Gsum + alpha * Hsum
      sl.begin(base + L.scratch + 1);
      sl.term(base + L.B, FR_ONE);
      sl.term(L.Gsum, fr_neg(gp_beta_inv[b]));
      sl.term(L.Hsum, alpha);
      sl.end();
      sl.begin(base + L.scratch + 3);  // msm(G', d) must equal D
      if (!witness_is_ours)
        for (uint32_t i = 0; i < n; i++) sl.term(L.Gs + i, fr_mul(s.ds[i], gp_scale[b][i]));  // G'[i] = scale[i] * (Gs || Hs)[i]
      sl.end();
      sl.begin(base + L.scratch + 4);  // B_c: G is still the unfolded Gs || Hs, named by its CRS-image indices
      for (uint32_t i = 0; i < n; i++) sl.term(L.Gs + i, rs_c[b][i]);  // (fixed-base tables, fixed_base.cuh)
      sl.end();
      sl.begin(base + L.scratch + 5);  // B_d
      for (uint32_t i = 0; i < n; i++) sl.term(L.Gs + i, fr_mul(rs_d[b][i], gp_scale[b][i]));
      sl.end();
    });
    if ((rc = run_msm(st))) return rc;
    for (uint32_t b = 0; b < B; b++) {
      ProveState& s = *S[b];
      memcpy(D_enc[b].data(), sb.out(b, 0), 48);
      if (!witness_is_ours && memcmp(sb.out(b, 1), D_enc[b].data(), 48) != 0) s.fail("msm(G', d) != D");
      memcpy(s.B_c, sb.out(b, 2), 48);
      memcpy(s.B_d, sb.out(b, 3), 48);
    }
  }
  // ---- inner-product argument (innerproductargument.go:74-188)
  par(B, [&](size_t b) {
    ProveState& s = *S[b];
    s.tr.append_points("ipa_step1", s.C, 1);
    s.tr.append_points("ipa_step1", D_enc[b].data(), 1);
    s.tr.append_scalar("ipa_step1", s.z);
    s.tr.append_points("ipa_step1", s.B_c, 1);
    s.tr.append_points("ipa_step1", s.B_d, 1);
    Fr alpha = s.tr.challenge("ipa_alpha");
    s.beta_ipa = s.tr.challenge("ipa_beta");
    for (uint32_t i = 0; i < n; i++) {
      s.cs[i] = fr_add(rs_c[b][i], fr_mul(alpha, s.cs[i]));
      s.ds[i] = fr_add(rs_d[b][i], fr_mul(alpha, s.ds[i]));
    }
  });
  uint32_t ipa_round = 0;
  for (uint32_t half = n / 2; half >= 1; half /= 2, ipa_round++) {
    const uint32_t round = ipa_round;
    const bool expand = lazy && round == 1;  // bases of this round are pairs of CRS points
    StageBuilder sb(st, B, (expand ? 8 : 4) * half + 2, 4);
    par(B, [&](size_t b) {
      ProveState& s = *S[b];
      uint32_t base = L.base((uint32_t)b);
      const Fr *c_L = s.cs.data(), *c_R = s.cs.data() + half, *d_L = s.ds.data(), *d_R = s.ds.data() + half;
      MsmSlice sl = sb.slice((uint32_t)b);
      const std::vector<Fr>& scale = gp_scale[b];
      const uint32_t len1 = n / 2;
      // term a * G[e] / a * G'[e] of the current (possibly virtual) vectors.  First round: G is the unfolded
      // Gs || Hs (adjacent in the CRS image) and G'[e] = scale[e] * (Gs || Hs)[e]: naming the CRS points themselves
      // lets the launch use their fixed-base tables.
      auto g_term = [&](uint32_t e, const Fr& a) {
        if (round == 0) sl.term(L.Gs + e, a);
        else if (expand) { sl.term(L.Gs + e, a); sl.term_more(L.Gs + e + len1, fr_mul(a, ipa_x[b][0])); }
        else sl.term(base + L.G + e, a);
      };
      auto gp_term = [&](uint32_t e, const Fr& a) {
        if (round == 0) sl.term(L.Gs + e, fr_mul(a, scale[e]));
        else if (expand) {
          sl.term(L.Gs + e, fr_mul(a, scale[e]));
          sl.term_more(L.Gs + e + len1, fr_mul(fr_mul(a, ipa_x[b][1]), scale[e + len1]));
        } else sl.term(base + L.Gp + e, a);
      };
      sl.begin(base + L.scratch);  // L_C = <c_L, G_R> + <c_L, d_R> * (beta*H)
      for (uint32_t i = 0; i < half; i++) g_term(half + i, c_L[i]);
      sl.term(L.H, fr_mul(s.beta_ipa, fr_inner(c_L, d_R, half)));
      sl.end();
      sl.begin(base + L.scratch + 1);  // L_D = <d_R, G'_L>
      for (uint32_t i = 0; i < half; i++) gp_term(i, d_R[i]);
      sl.end();
      sl.begin(base + L.scratch + 2);  // R_C = <c_R, G_L> + <c_R, d_L> * (beta*H)
      for (uint32_t i = 0; i < half; i++) g_term(i, c_R[i]);
      sl.term(L.H, fr_mul(s.beta_ipa, fr_inner(c_R, d_L, half)));
      sl.end();
      sl.begin(base + L.scratch + 3);  // R_D = <d_L, G'_R>
      for (uint32_t i = 0; i < half; i++) gp_term(half + i, d_L[i]);
      sl.end();
    });
    if ((rc = run_msm(st))) return rc;
    // folds after this round: none after the first when lazy; V2 from the CRS after the second (below)
    const bool plain_fold = half > 1 && !(lazy && round <= 1);
    const bool first_fold = round == 0;
    std::vector<ElemOp> ops(plain_fold ? (size_t)B * 2 * (half) : 0);
    // first fold of G' (plain schedule): the right half is not materialised (see the Gs' stage); its source is the
    // CRS point with the per-element scalar gamma^-1 * scale[half + i]
    std::vector<Fr> sc((size_t)B * 2 + (first_fold && plain_fold ? (size_t)B * half : 0));
    par(B, [&](size_t b) {
      ProveState& s = *S[b];
      const uint8_t *lc = sb.out((uint32_t)b, 0), *ld = sb.out((uint32_t)b, 1), *rcc = sb.out((uint32_t)b, 2), *rd = sb.out((uint32_t)b, 3);
      s.L_C.insert(s.L_C.end(), lc, lc + 48);
      s.L_D.insert(s.L_D.end(), ld, ld + 48);
      s.R_C.insert(s.R_C.end(), rcc, rcc + 48);
      s.R_D.insert(s.R_D.end(), rd, rd + 48);
      s.tr.append_points("ipa_loop", lc, 1);
      s.tr.append_points("ipa_loop", ld, 1);
      s.tr.append_points("ipa_loop", rcc, 1);
      s.tr.append_points("ipa_loop", rd, 1);
      Fr gamma = s.tr.challenge("ipa_gamma");
      if (fr_is_zero(gamma)) s.fail("ipa gamma challenge is zero");
      Fr gamma_inv = fr_inv(gamma);
      for (uint32_t i = 0; i < half; i++) {
        s.cs[i] = fr_add(s.cs[i], fr_mul(gamma_inv, s.cs[half + i]));
        s.ds[i] = fr_add(s.ds[i], fr_mul(gamma, s.ds[half + i]));
      }
      sc[2 * b] = gamma;
      sc[2 * b + 1] = gamma_inv;
      if (round <= 1) { ipa_x[b][2 * round] = gamma; ipa_x[b][2 * round + 1] = gamma_inv; }
      if (plain_fold) {  // the folded bases of the last round are never read again
        uint32_t base = L.base((uint32_t)b);
        ElemOp* o = ops.data() + b * 2 * half;
        const uint32_t g0 = first_fold ? L.Gs : base + L.G;  // first fold: sources are the CRS points
        for (uint32_t i = 0; i < half; i++) {
          o[i] = ElemOp{g0 + half + i, g0 + i, base + L.G + i, (uint32_t)(2 * b)};
          if (first_fold) {
            const uint32_t si = (uint32_t)(2 * B + b * half + i);
            sc[si] = fr_mul(gamma_inv, gp_scale[b][half + i]);
            o[half + i] = ElemOp{L.Gs + half + i, base + L.Gp + i, base + L.Gp + i, si};
          } else {
            o[half + i] = ElemOp{base + L.Gp + half + i, base + L.Gp + i, base + L.Gp + i, (uint32_t)(2 * b + 1)};
          }
        }
      }
    });
    if ((rc = run_elem(ops, sc))) return rc;
    if (lazy && round == 1 && half > 1) {
      // G2[i] = C[i] + x1 C[i+2q] + x2 C[i+q] + x1 x2 C[i+3q] with x = gamma, C = Gs || Hs, q = half;
      // G'2[i] = s[i] C[i] + y1 s[i+2q] C[i+2q] + y2 s[i+q] C[i+q] + y1 y2 s[i+3q] C[i+3q] with y = gamma^-1,
      // s = gp_scale: four chained launches of table multiplications (the last one for G' only).
      const uint32_t q = half;
      for (int pass = 0; pass < 4; pass++) {
        const uint32_t per = pass < 3 ? 2 * q : q;
        std::vector<ElemOp> o2((size_t)B * per);
        std::vector<Fr> s2((size_t)B * (q + 1));  // per proof: q per-element scalars for G', one shared scalar for G
        par(B, [&](size_t b) {
          const uint32_t base = L.base((uint32_t)b);
          const std::vector<Fr>& scale = gp_scale[b];
          const Fr x1 = ipa_x[b][0], y1 = ipa_x[b][1], x2 = ipa_x[b][2], y2 = ipa_x[b][3];
          ElemOp* o = o2.data() + b * per;
          Fr* sv = s2.data() + b * (q + 1);
          const uint32_t sbase = (uint32_t)(b * (q + 1));
          // offsets of the CRS point each pass adds, for G (first pass: add C[i] as the plain summand) and G'
          static const uint32_t g_off[3] = {2, 1, 3}, gp_off[4] = {0, 2, 1, 3};
          if (pass < 3) {
            sv[q] = pass == 0 ? x1 : pass == 1 ? x2 : fr_mul(x1, x2);
            for (uint32_t i = 0; i < q; i++)
              o[i] = ElemOp{L.Gs + i + g_off[pass] * q, pass == 0 ? L.Gs + i : base + L.G + i, base + L.G + i, sbase + q};
          }
          const Fr yc = pass == 0 ? FR_ONE : pass == 1 ? y1 : pass == 2 ? y2 : fr_mul(y1, y2);
          ElemOp* op = o + (pass < 3 ? q : 0);
          for (uint32_t i = 0; i < q; i++) {
            const uint32_t e = i + gp_off[pass] * q;
            sv[i] = pass == 0 ? scale[e] : fr_mul(yc, scale[e]);
            op[i] = ElemOp{L.Gs + e, pass == 0 ? cdl::kNoPoint : base + L.Gp + i, base + L.Gp + i, sbase + i};
          }
        });
        if ((rc = run_elem(o2, s2))) return rc;
      }
    }
  }
  for (uint32_t b = 0; b < B; b++) { S[b]->c0 = S[b]->cs[0]; S[b]->d0 = S[b]->ds[0]; }

  // ---- step 3: R, S, T, U, same-scalar commitments, A', B_a/B_t/B_u
  // (curdleproof.go:101-122,146-148; samescalarargument.go:46-64; samemultiscalarargument.go:58-72)
  {
    // T_2 = k*R + r_t*H, U_2, A_2 = r_k*R + r_a*H, B_2 (groupcommitment.go:17-52) are linear in R and S.
    // One proof at a time they are folded into the same launch as <k*as, Rs> + r_t*H (no dependent
    // stage on the latency path); a batch computes R and S once and derives the four points in a
    // second, tiny launch of two-term MSMs over (R, H) / (S, H): 2 instead of 6 MSMs of ell terms.
    const bool split = B >= kStep3SplitBatch;
    const uint32_t terms = (split ? 2 * ell : 6 * (ell + 1)) + 4 + 3 + (n) + (ell + 1) + (ell + 1);
    StageBuilder sb(st, B, terms, 14);
    // working vectors of the same-multiscalar argument
    {
      std::vector<cdl::CopyRange> cr;
      cr.reserve((size_t)B * 8);
      for (uint32_t b = 0; b < B; b++) {
        uint32_t base = L.base(b);
        cr.push_back({L.Gs, base + L.Gm, ell + 2, 0});                 // Gs || Hs[0..2)
        cr.push_back({L.Gt, base + L.Gm + ell + 2, 2, 0});             // Gt, Gu
        cr.push_back({base + L.Ts, base + L.Tp, ell, 0});
        cr.push_back({base + L.Us, base + L.Up, ell, 0});
        cr.push_back({cdl::kNoPoint, base + L.Tp + ell, 2, 0});        // T' = Ts || 0 || 0 || H || 0
        cr.push_back({L.H, base + L.Tp + ell + 2, 1, 0});
        cr.push_back({cdl::kNoPoint, base + L.Tp + ell + 3, 1, 0});
        cr.push_back({cdl::kNoPoint, base + L.Up + ell, 3, 0});        // U' = Us || 0 || 0 || 0 || H
        cr.push_back({L.H, base + L.Up + ell + 3, 1, 0});
      }
      if ((rc = copy_ranges(cr))) return rc;
    }
    par(B, [&](size_t b) {
      ProveState& s = *S[b];
      Rand& rand = rands[b]->r;
      s.r_t = rand.get_fr();
      s.r_u = rand.get_fr();
      s.r_a = rand.get_fr();  // samescalarargument.go:46-57
      s.r_b = rand.get_fr();
      s.r_k = rand.get_fr();
      s.r.resize(n);
      rand.get_frs(s.r.data(), n);  // samemultiscalarargument.go:58
      const Fr& k = ks[b];
      uint32_t base = L.base((uint32_t)b);
      MsmSlice sl = sb.slice((uint32_t)b);
      uint32_t o = base + L.scratch;
      auto lin = [&](uint32_t out, uint32_t pts, const Fr* mulby, uint32_t extra_pt, const Fr* extra_sc) {
        sl.begin(out);
        if (!split || !mulby)
          for (uint32_t i = 0; i < ell; i++) sl.term(base + pts + i, mulby ? fr_mul(*mulby, s.as[i]) : s.as[i]);
        if (extra_sc && !split) sl.term(extra_pt, *extra_sc);
        sl.end();  // split: the four derived points are empty tasks here and are filled by the next launch
      };
      lin(o + 0, L.Rs, nullptr, 0, nullptr);        // R = <as, Rs>
      lin(o + 1, L.Ss, nullptr, 0, nullptr);        // S = <as, Ss>
      sl.begin(o + 2); sl.term(L.Gt, s.r_t); sl.end();  // T_1 = r_t * Gt
      lin(o + 3, L.Rs, &k, L.H, &s.r_t);            // T_2 = k*R + r_t*H
      sl.begin(o + 4); sl.term(L.Gu, s.r_u); sl.end();  // U_1
      lin(o + 5, L.Ss, &k, L.H, &s.r_u);            // U_2
      sl.begin(o + 6); sl.term(L.Gt, s.r_a); sl.end();  // A_1 = r_a * Gt
      lin(o + 7, L.Rs, &s.r_k, L.H, &s.r_a);        // A_2 = r_k*R + r_a*H
      sl.begin(o + 8); sl.term(L.Gu, s.r_b); sl.end();  // B_1
      lin(o + 9, L.Ss, &s.r_k, L.H, &s.r_b);        // B_2
      sl.begin(o + 10);                              // A' = A + T_1 + U_1
      sl.term(base + L.A, FR_ONE); sl.term(L.Gt, s.r_t); sl.term(L.Gu, s.r_u);
      sl.end();
      sl.begin(o + 11);                              // B_a = <r, G>
      for (uint32_t i = 0; i < n; i++) sl.term(i < ell + 2 ? L.Gs + i : L.Gt + (i - ell - 2), s.r[i]);  // Gm = Gs || Hs[0..2) || Gt || Gu
      sl.end();
      sl.begin(o + 12);                              // B_t = <r, T'>
      for (uint32_t i = 0; i < ell; i++) sl.term(base + L.Ts + i, s.r[i]);
      sl.term(L.H, s.r[ell + 2]);
      sl.end();
      sl.begin(o + 13);                              // B_u = <r, U'>
      for (uint32_t i = 0; i < ell; i++) sl.term(base + L.Us + i, s.r[i]);
      sl.term(L.H, s.r[ell + 3]);
      sl.end();
    });
    if ((rc = run_msm(st))) return rc;
    MsmStage st2;
    StageBuilder sb2(st2, split ? B : 0, 8, 4);
    if (split) {
      par(B, [&](size_t b) {
        ProveState& s = *S[b];
        uint32_t base = L.base((uint32_t)b), o = base + L.scratch;
        MsmSlice sl = sb2.slice((uint32_t)b);
        auto two = [&](uint32_t out, uint32_t pt, const Fr& a, const Fr& h) {
          sl.begin(out); sl.term(pt, a); sl.term(L.H, h); sl.end();
        };
        two(o + 3, o + 0, ks[b], s.r_t);   // T_2 = k*R + r_t*H
        two(o + 5, o + 1, ks[b], s.r_u);   // U_2 = k*S + r_u*H
        two(o + 7, o + 0, s.r_k, s.r_a);   // A_2 = r_k*R + r_a*H
        two(o + 9, o + 1, s.r_k, s.r_b);   // B_2 = r_k*S + r_b*H
      });
      if ((rc = run_msm(st2))) return rc;
    }
    par(B, [&](size_t b) {
      ProveState& s = *S[b];
      auto out = [&](uint32_t t) {
        if (split && (t == 3 || t == 5 || t == 7 || t == 9)) return sb2.out((uint32_t)b, (t - 3) / 2);
        return sb.out((uint32_t)b, t);
      };
      memcpy(s.R, out(0), 48); memcpy(s.S, out(1), 48);
      memcpy(s.T1, out(2), 48); memcpy(s.T2, out(3), 48); memcpy(s.U1, out(4), 48); memcpy(s.U2, out(5), 48);
      memcpy(s.A1, out(6), 48); memcpy(s.A2, out(7), 48); memcpy(s.B1, out(8), 48); memcpy(s.B2, out(9), 48);
      memcpy(s.B_a, out(11), 48); memcpy(s.B_t, out(12), 48); memcpy(s.B_u, out(13), 48);
      // same-scalar argument transcript (samescalarargument.go:66-80)
      const uint8_t* seq[10] = {s.R, s.S, s.T1, s.T2, s.U1, s.U2, s.A1, s.A2, s.B1, s.B2};
      for (auto e : seq) s.tr.append_points("sameexp_points", e, 1);
      Fr a = s.tr.challenge("sameexp_alpha");
      s.z_k = fr_add(s.r_k, fr_mul(ks[b], a));
      s.z_t = fr_add(s.r_a, fr_mul(s.r_t, a));
      s.z_u = fr_add(s.r_b, fr_mul(s.r_u, a));
      // same-multiscalar argument, step 1 (samemultiscalarargument.go:74-83)
      const uint8_t* ie = inst_enc.data() + b * per_inst;
      s.tr.append_points("same_msm_step1", out(10), 1);
      s.tr.append_points("same_msm_step1", s.T2, 1);
      s.tr.append_points("same_msm_step1", s.U2, 1);
      s.tr.append_points("same_msm_step1", ie + (size_t)2 * ell * 48, ell);  // Ts
      s.tr.append_points("same_msm_step1", kInfEnc, 1);
      s.tr.append_points("same_msm_step1", kInfEnc, 1);
      s.tr.append_points("same_msm_step1", H_enc, 1);
      s.tr.append_points("same_msm_step1", kInfEnc, 1);
      s.tr.append_points("same_msm_step1", ie + (size_t)3 * ell * 48, ell);  // Us
      s.tr.append_points("same_msm_step1", kInfEnc, 1);
      s.tr.append_points("same_msm_step1", kInfEnc, 1);
      s.tr.append_points("same_msm_step1", kInfEnc, 1);
      s.tr.append_points("same_msm_step1", H_enc, 1);
      s.tr.append_points("same_msm_step1", s.B_a, 1);
      s.tr.append_points("same_msm_step1", s.B_t, 1);
      s.tr.append_points("same_msm_step1", s.B_u, 1);
      Fr alpha = s.tr.challenge("same_msm_alpha");
      // x = perm_as || rs_a || r_t || r_u ; x = r + alpha*x   (curdleproof.go:167-170, :80-83)
      s.x.resize(n);
      for (uint32_t i = 0; i < ell; i++) s.x[i] = s.perm_as[i];
      s.x[ell] = s.rs_a[0]; s.x[ell + 1] = s.rs_a[1]; s.x[ell + 2] = s.r_t; s.x[ell + 3] = s.r_u;
      for (uint32_t i = 0; i < n; i++) s.x[i] = fr_add(s.r[i], fr_mul(s.x[i], alpha));
    });
  }
  // ---- same-multiscalar rounds (samemultiscalarargument.go:85-140)
  // Gm = Gs || Hs[0..2) || Gt || Gu in CRS-image indices
  auto cm = [&](uint32_t i) { return i < ell + 2 ? L.Gs + i : L.Gt + (i - ell - 2); };
  uint32_t sm_round = 0;
  for (uint32_t half = n / 2; half >= 1; half /= 2, sm_round++) {
    const uint32_t round = sm_round;
    const bool expand = lazy && round == 1;  // Gm's bases of this round are pairs of CRS points (see `lazy`)
    StageBuilder sb(st, B, (expand ? 8 : 6) * half, 6);
    par(B, [&](size_t b) {
      ProveState& s = *S[b];
      uint32_t base = L.base((uint32_t)b);
      const Fr *x_L = s.x.data(), *x_R = s.x.data() + half;
      MsmSlice sl = sb.slice((uint32_t)b);
      const uint32_t vec[3] = {L.Gm, L.Tp, L.Up};
      const uint32_t len1 = n / 2;
      // first round: Gm is still Gs || Hs[0..2) || Gt || Gu, named by its CRS-image indices (fixed-base tables)
      auto term = [&](int v, uint32_t e, const Fr& a) {
        if (v == 0 && round == 0) sl.term(cm(e), a);
        else if (v == 0 && expand) { sl.term(cm(e), a); sl.term_more(cm(e + len1), fr_mul(a, sm_x[b][0])); }
        else sl.term(base + vec[v] + e, a);
      };
      for (int v = 0; v < 3; v++) {  // L_A, L_T, L_U over the right halves with x_L
        sl.begin(base + L.scratch + v);
        for (uint32_t i = 0; i < half; i++) term(v, half + i, x_L[i]);
        sl.end();
      }
      for (int v = 0; v < 3; v++) {  // R_A, R_T, R_U over the left halves with x_R
        sl.begin(base + L.scratch + 3 + v);
        for (uint32_t i = 0; i < half; i++) term(v, i, x_R[i]);
        sl.end();
      }
    });
    if ((rc = run_msm(st))) return rc;
    // T' and U' fold every round; Gm as well, except in the first two rounds of the lazy schedule
    const bool fold_gm = !(lazy && round <= 1);
    const uint32_t nvec = fold_gm ? 3 : 2;
    std::vector<ElemOp> ops(half > 1 ? (size_t)B * nvec * half : 0);
    std::vector<Fr> sc(B);
    par(B, [&](size_t b) {
      ProveState& s = *S[b];
      std::vector<uint8_t>* dstv[6] = {&s.L_A, &s.L_T, &s.L_U, &s.R_A, &s.R_T, &s.R_U};
      for (int t = 0; t < 6; t++) {
        const uint8_t* e = sb.out((uint32_t)b, t);
        dstv[t]->insert(dstv[t]->end(), e, e + 48);
        s.tr.append_points("same_msm_loop", e, 1);
      }
      Fr gamma = s.tr.challenge("same_msm_gamma");
      if (fr_is_zero(gamma)) s.fail("gamma is zero");
      Fr gamma_inv = fr_inv(gamma);
      for (uint32_t i = 0; i < half; i++) s.x[i] = fr_add(s.x[i], fr_mul(gamma_inv, s.x[half + i]));
      sc[b] = gamma;
      if (round <= 1) { sm_x[b][2 * round] = gamma; sm_x[b][2 * round + 1] = gamma_inv; }
      if (half > 1) {
        uint32_t base = L.base((uint32_t)b);
        const uint32_t vec[3] = {L.Tp, L.Up, L.Gm};
        const bool first = round == 0;  // first fold of Gm: sources are the CRS points
        ElemOp* o = ops.data() + b * nvec * half;
        for (uint32_t v = 0; v < nvec; v++)
          for (uint32_t i = 0; i < half; i++) {
            uint32_t src = base + vec[v] + half + i, add = base + vec[v] + i;
            if (v == 2 && first) {
              src = cm(half + i);
              add = cm(i);
            }
            o[v * half + i] = ElemOp{src, add, base + vec[v] + i, (uint32_t)b};
          }
      }
    });
    if ((rc = run_elem(ops, sc))) return rc;
    if (lazy && round == 1 && half > 1) {
      // Gm2[i] = C[i] + x1 C[i+2q] + x2 C[i+q] + x1 x2 C[i+3q], x = gamma, C = Gm in CRS indices, q = half
      const uint32_t q = half;
      for (int pass = 0; pass < 3; pass++) {
        std::vector<ElemOp> o2((size_t)B * q);
        std::vector<Fr> s2(B);
        par(B, [&](size_t b) {
          const uint32_t base = L.base((uint32_t)b);
          static const uint32_t off[3] = {2, 1, 3};
          s2[b] = pass == 0 ? sm_x[b][0] : pass == 1 ? sm_x[b][2] : fr_mul(sm_x[b][0], sm_x[b][2]);
          ElemOp* o = o2.data() + b * q;
          for (uint32_t i = 0; i < q; i++)
            o[i] = ElemOp{cm(i + off[pass] * q), pass == 0 ? cm(i) : base + L.Gm + i, base + L.Gm + i, (uint32_t)b};
        });
        if ((rc = run_elem(o2, s2))) return rc;
      }
    }
  }

  // ---- serialize (curdleproof.go:358-387 and the sub-proof Serialize methods)
  proofs.assign(B, {});
  status.assign(B, CDL_OK);
  errs.assign(B, "");
  for (uint32_t b = 0; b < B; b++) {
    ProveState& s = *S[b];
    if (s.failed) { status[b] = CDL_ERR_PROTOCOL; errs[b] = s.err; continue; }
    std::vector<uint8_t>& v = proofs[b];
    put_pt(v, s.A); put_pt(v, s.T1); put_pt(v, s.T2); put_pt(v, s.U1); put_pt(v, s.U2); put_pt(v, s.R); put_pt(v, s.S);
    put_pt(v, s.Bp);                      // same-permutation proof
    put_pt(v, s.C); put_fr(v, s.r_p);     // grand-product proof
    put_pt(v, s.B_c); put_pt(v, s.B_d);   // inner-product proof
    put_slice(v, s.L_C); put_slice(v, s.R_C); put_slice(v, s.L_D); put_slice(v, s.R_D);
    put_fr(v, s.c0); put_fr(v, s.d0);
    put_pt(v, s.A1); put_pt(v, s.A2); put_pt(v, s.B1); put_pt(v, s.B2);  // same-scalar proof
    put_fr(v, s.z_k); put_fr(v, s.z_t); put_fr(v, s.z_u);
    put_pt(v, s.B_a); put_pt(v, s.B_t); put_pt(v, s.B_u);                // same-multiscalar proof
    put_slice(v, s.L_A); put_slice(v, s.L_T); put_slice(v, s.L_U);
    put_slice(v, s.R_A); put_slice(v, s.R_T); put_slice(v, s.R_U);
    put_fr(v, s.x[0]);
  }
  return CDL_OK;
}

// ------------------------------------------------------------------ wire walker
std::string parse_wire_proof(const uint8_t* buf, size_t len, bool with_m, WireProof& out, size_t* used) {
  size_t pos = 0;
  out.points.clear();
  int nsc = 0, nlen = 0;
  auto point = [&]() -> const char* {
    if (pos + 48 > len) return "unexpected EOF";
    uint8_t f = buf[pos] & 0xe0;
    if (f == 0xe0 || f == 0x60 || f == 0x20) return "invalid encoding";
    if (!(f & 0x80)) return "uncompressed point encodings are not supported by this build";
    out.points.push_back(buf + pos);
    pos += 48;
    return nullptr;
  };
  auto slice = [&]() -> const char* {
    if (pos + 4 > len) return "unexpected EOF";
    uint32_t c = ((uint32_t)buf[pos] << 24) | ((uint32_t)buf[pos + 1] << 16) | ((uint32_t)buf[pos + 2] << 8) | buf[pos + 3];
    pos += 4;
    if ((size_t)c * 48 > len - pos) return "unexpected EOF";
    out.lens[nlen++] = c;
    for (uint32_t i = 0; i < c; i++)
      if (const char* e = point()) return e;
    return nullptr;
  };
  auto scalar = [&]() -> const char* {
    if (pos + 32 > len) return "unexpected EOF";
    out.scalars[nsc++] = buf + pos;
    pos += 32;
    return nullptr;
  };
#define CDL_TRY(x) do { if (const char* e__ = (x)) return e__; } while (0)
  if (with_m) CDL_TRY(point());
  for (int i = 0; i < 7; i++) CDL_TRY(point());  // A, T_1, T_2, U_1, U_2, R, S
  CDL_TRY(point());                               // B
  CDL_TRY(point()); CDL_TRY(scalar());            // C, Rp
  CDL_TRY(point()); CDL_TRY(point());             // B_c, B_d
  for (int i = 0; i < 4; i++) CDL_TRY(slice());   // L_Cs, R_Cs, L_Ds, R_Ds
  CDL_TRY(scalar()); CDL_TRY(scalar());           // c0, d0
  for (int i = 0; i < 4; i++) CDL_TRY(point());   // A_1, A_2, B_1, B_2
  for (int i = 0; i < 3; i++) CDL_TRY(scalar());  // Z_k, Z_t, Z_u
  for (int i = 0; i < 3; i++) CDL_TRY(point());   // B_a, B_t, B_u
  for (int i = 0; i < 6; i++) CDL_TRY(slice());   // L_A, L_T, L_U, R_A, R_T, R_U
  CDL_TRY(scalar());                              // x
#undef CDL_TRY
  if (used) *used = pos;
  return "";
}

}  // namespace cdlh
