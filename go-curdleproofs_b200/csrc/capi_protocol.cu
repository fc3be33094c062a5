// Protocol-level C ABI: common.Rand, CRS, ShufflePermuteCommit, Prove, Verify and
// the Whisk wrappers (single and batched), on top of the batched engine.
#include <cstring>
#include <memory>
#include <algorithm>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "host/engine.hpp"

using cdlh::affine_to_jac;
using cdlh::Engine;
using cdlh::engine_of;
using cdlh::Fr;
using cdlh::kMinLaneBatch;
using cdlh::Layout;
using cdlh::run_split;
using cdlh::slots_for;

static_assert(sizeof(Fr) == sizeof(cdl_fr), "host fr layout");

extern "C" cdl_ctx* cdl_lane_(cdl_ctx* root, size_t slot, size_t i);  // capi.cu

namespace {

// BLS12-381 G1 generator, affine Montgomery form (gnark bls12381.Generators())
const uint32_t kGenX[12] = {0xfd530c16u, 0x5cb38790u, 0x9976fff5u, 0x7817fc67u, 0x143ba1c1u, 0x154f95c7u,
                            0xf3d0e747u, 0xf0ae6acdu, 0x21dbf440u, 0xedce6eccu, 0x9e0bfb75u, 0x12017741u};
const uint32_t kGenY[12] = {0x0ce72271u, 0xbaac93d5u, 0x7918fd8eu, 0x8c22631au, 0x570725ceu, 0xdd595f13u,
                            0x50405194u, 0x51ac5829u, 0xad0059c0u, 0x0e1c8c3fu, 0x5008a26au, 0x0bbc3efcu};
const uint64_t kFpOne[6] = {0x760900000002fffdull, 0xebf4000bc40c0002ull, 0x5f48985753c758baull,
                            0x77ce585370525745ull, 0x5c071a97a256ec6dull, 0x15f65ec3fa80e493ull};

}  // namespace

Engine* cdlh::engine_of(cdl_ctx* c) {
  if (!c->engine) c->engine = new Engine(c);
  Engine* E = static_cast<Engine*>(c->engine);
  E->clear_fixed();  // begin_call selects the tables of its CRS; every other call runs without
  return E;
}

const cdl::G1Affine* cdl_crs::points_on(size_t s) const {
  Replica& r = rep[s];
  if (r.d_points) return r.d_points;
  const size_t bytes = host.size() * sizeof(cdl::G1Affine);
  if (cudaMalloc(&r.d_points, bytes) != cudaSuccess) {
    cudaGetLastError();
    r.d_points = nullptr;
    return nullptr;
  }
  if (cudaMemcpy(r.d_points, host.data(), bytes, cudaMemcpyHostToDevice) != cudaSuccess) {
    cudaFree(r.d_points);
    r.d_points = nullptr;
  }
  return r.d_points;
}

void cdlh::affine_to_jac(cdl_g1_jac* out, const cdl_g1_affine& a) {
  bool inf = true;
  for (int i = 0; i < 6; i++) inf = inf && a.x.l[i] == 0 && a.y.l[i] == 0;
  if (inf) {
    memcpy(out->x.l, kFpOne, 48);
    memcpy(out->y.l, kFpOne, 48);
    memset(out->z.l, 0, 48);
  } else {
    out->x = a.x;
    out->y = a.y;
    memcpy(out->z.l, kFpOne, 48);
  }
}

namespace {

// n draws a_i from r, points a_i * G (rand.go:72-95), written to pool[dst..]
int32_t rand_points_to_pool(Engine* E, cdl_rand* r, uint32_t gen_slot, uint32_t dst, size_t n) {
  if (!n) return CDL_OK;
  std::vector<Fr> sc(n);
  r->r.get_frs(sc.data(), n);
  std::vector<cdl::ElemOp> ops(n);
  for (size_t i = 0; i < n; i++) ops[i] = cdl::ElemOp{gen_slot, cdl::kNoPoint, (uint32_t)(dst + i), (uint32_t)i};
  return E->run_elem(ops, sc);
}

cdl_g1_affine generator() {
  cdl_g1_affine g;
  memcpy(g.x.l, kGenX, 48);
  memcpy(g.y.l, kGenY, 48);
  return g;
}

int32_t put_generator(Engine* E, uint32_t slot) {
  const cdl_g1_affine g = generator();
  return E->upload_points(slot, &g, 1);
}

// finish a CRS object from pool[0 .. ell+9): keeps the host image, copies it to slot 0's device buffer (the
// other slots upload theirs on first use), caches encodings
int32_t crs_finish(cdl_ctx* c, Engine* E, const Layout& L, cdl_crs** out) {
  std::unique_ptr<cdl_crs> crs(new cdl_crs());
  crs->ctx = c;
  crs->ell = L.ell;
  crs->rep.resize(c->slots.size());
  int32_t rc = E->set_infinity(L.INF, 1);
  if (rc) return rc;
  std::vector<uint32_t> src(L.crs_size);
  for (uint32_t i = 0; i < L.crs_size; i++) src[i] = i;
  if ((rc = E->compress(src, crs->enc))) return rc;
  crs->host.resize(L.crs_size);
  if ((rc = E->download_points(0, crs->host.data(), L.crs_size))) return rc;
  if (!crs->points_on(0)) return c->fail(CDL_ERR_CUDA, "crs upload failed");
  *out = crs.release();
  return CDL_OK;
}

struct Prep {
  Engine* E;
  Layout L;
};

constexpr size_t kPoolIndexLimit = (size_t)1 << 30;  // MSM term indices carry flags in bits 30 and 31

// common prologue of the protocol calls; `intake`: room behind the instance regions for Engine::load_instances
int32_t begin_call(cdl_ctx* c, const cdl_crs* crs, size_t B, Engine** E, Layout* L, bool intake = false) {
  if (crs->ctx != c->root()) return c->fail(CDL_ERR_INVALID_ARG, "crs belongs to another context");
  *L = Layout(crs->ell);
  const size_t need = (size_t)L->crs_size + B * (size_t)L->inst_size + (intake ? Engine::intake_points(*L, B) : 0);
  if (need >= kPoolIndexLimit)
    return c->fail(CDL_ERR_TOO_LARGE, "%zu instances of ell = %u need %zu pool points; pool indices are below 2^30", B,
                   L->ell, need);
  CDL_CUDA(c, cudaSetDevice(c->device));
  *E = engine_of(c);
  c->spin_wait = B < 8 && c->parent == nullptr;  // latency regime: see cdl_ctx::sync_stream
  int32_t rc = (*E)->ensure_pool(need);
  if (rc) return rc;
  (*E)->select_fixed(*L, crs, B);
  return (*E)->load_crs(*L, crs);
}

// number of lanes a slot's block of n instances is cut into
size_t lanes_for(cdl_ctx* c, size_t n) {
  if (c->n_lanes <= 1) return 1;
  return std::max<size_t>(1, std::min<size_t>((size_t)c->n_lanes, n / kMinLaneBatch));
}

}  // namespace

size_t cdlh::slots_for(cdl_ctx* c, size_t B, size_t min_block) {
  if (c->parent) return 1;
  return std::max<size_t>(1, std::min<size_t>(c->slots.size(), B / min_block));
}

// first unit of block s when B units are dealt to D slots in contiguous blocks (sharding.shard_bounds)
static size_t shard_lo(size_t B, size_t D, size_t s) { return s * (B / D) + std::min(s, B % D); }

int32_t cdlh::run_split(cdl_ctx* c, size_t B, const std::function<int32_t(cdl_ctx*, size_t, size_t)>& fn, bool lanes,
                        size_t align, size_t min_block) {
  std::lock_guard<std::mutex> lk(c->mu);
  return run_split_locked(c, B, fn, lanes, align, min_block);
}

int32_t cdlh::run_split_locked(cdl_ctx* c, size_t B, const std::function<int32_t(cdl_ctx*, size_t, size_t)>& fn,
                               bool lanes, size_t align, size_t min_block) {
  struct Piece { cdl_ctx* ctx; size_t lo, hi; };
  std::vector<Piece> pieces;
  const size_t D = slots_for(c, B, min_block);
  auto bound = [&](size_t s) {
    if (s == D) return B;
    return std::min(B, (shard_lo(B, D, s) + align / 2) / align * align);
  };
  for (size_t s = 0; s < D; s++) {
    const size_t lo = bound(s), n = bound(s + 1) - lo;
    if (!n) continue;
    const size_t G = lanes ? lanes_for(c, n) : 1;
    for (size_t g = 0; g < G; g++) {
      cdl_ctx* l = cdl_lane_(c, s, g);
      if (!l) return c->fail(CDL_ERR_CUDA, "lane context creation failed");
      pieces.push_back(Piece{l, lo + n * g / G, lo + n * (g + 1) / G});
    }
  }
  CDL_CUDA(c, cudaSetDevice(c->device));
  std::vector<int32_t> rc(pieces.size(), CDL_OK);
  std::vector<std::thread> th;
  for (size_t i = 0; i < pieces.size(); i++)
    th.emplace_back([&, i] { rc[i] = fn(pieces[i].ctx, pieces[i].lo, pieces[i].hi); });
  for (auto& t : th) t.join();
  for (size_t i = 0; i < pieces.size(); i++)
    if (rc[i] != CDL_OK) return c->fail(rc[i], "%s", pieces[i].ctx->err.c_str());
  return CDL_OK;
}

namespace {

// whether a batched protocol call of B instances on c is cut into pieces (run_split) rather than run on c itself
bool split_lanes(cdl_ctx* c, size_t B) { return !c->parent && (cdlh::slots_for(c, B) > 1 || lanes_for(c, B) > 1); }

// f(engine, slot) for every engine of a root context: its own (slot 0) and its lanes'
template <class F>
void for_each_engine(cdl_ctx* c, F f) {
  if (c->engine) f(static_cast<Engine*>(c->engine), (size_t)0);
  for (size_t s = 0; s < c->slots.size(); s++)
    for (cdl_ctx* l : c->slots[s].lanes)
      if (l->engine) f(static_cast<Engine*>(l->engine), s);
}

// length of the union of the kernel intervals of slot s's engines
double slot_busy_ms(cdl_ctx* c, size_t s) {
  std::vector<std::pair<float, float>> iv;
  for_each_engine(c, [&](Engine* E, size_t es) {
    if (es == s) iv.insert(iv.end(), E->intervals.begin(), E->intervals.end());
  });
  std::sort(iv.begin(), iv.end());
  double busy = 0, cur_lo = 0, cur_hi = -1;
  for (auto& p : iv) {
    if (cur_hi < 0 || p.first > cur_hi) {
      if (cur_hi >= 0) busy += cur_hi - cur_lo;
      cur_lo = p.first;
      cur_hi = p.second;
    } else if (p.second > cur_hi) {
      cur_hi = p.second;
    }
  }
  if (cur_hi >= 0) busy += cur_hi - cur_lo;
  return busy;
}

}  // namespace

extern "C" {

void cdl_engine_free_(void* engine) { delete static_cast<Engine*>(engine); }

uint64_t cdl_launch_count(cdl_ctx* c) {
  if (!c) return 0;
  std::lock_guard<std::mutex> lk(c->mu);
  uint64_t n = 0;
  for_each_engine(c, [&](Engine* E, size_t) { n += E->launches; });
  return n;
}

int32_t cdl_engine_stats(cdl_ctx* c, uint64_t* launches, double* ms, double* modmul, double* bytes, int reset) {
  if (!c) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  for (int i = 0; i < 4; i++) {
    if (launches) launches[i] = 0;
    if (ms) ms[i] = 0;
    if (modmul) modmul[i] = 0;
    if (bytes) bytes[i] = 0;
  }
  for_each_engine(c, [&](Engine* E, size_t) {
    for (int i = 0; i < 4; i++) {
      if (launches) launches[i] += E->stats.n[i];
      if (ms) ms[i] += E->stats.ms[i];
      if (modmul) modmul[i] += E->stats.modmul[i];
      if (bytes) bytes[i] += E->stats.bytes[i];
    }
    if (reset) { E->stats = Engine::Stats(); E->intervals.clear(); }
  });
  return CDL_OK;
}

int32_t cdl_engine_busy_ms(cdl_ctx* c, double* busy_ms) {
  if (!c || !busy_ms) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  double busy = 0;
  for (size_t s = 0; s < c->slots.size(); s++) busy = std::max(busy, slot_busy_ms(c, s));
  *busy_ms = busy;
  return CDL_OK;
}

int32_t cdl_engine_busy_ms_device(cdl_ctx* c, size_t slot, double* busy_ms) {
  if (!c || !busy_ms || slot >= c->slots.size()) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  *busy_ms = slot_busy_ms(c, slot);
  return CDL_OK;
}

int32_t cdl_host_selftest(uint8_t* out32, const cdl_fr* a, const cdl_fr* b, cdl_fr* fr_out) {
  if (!out32 || !a || !b || !fr_out) return CDL_ERR_INVALID_ARG;
  cdlh::Transcript t("test protocol");
  t.append_message("some label", reinterpret_cast<const uint8_t*>("some data"), 9);
  t.challenge_bytes("challenge", out32, 32);
  Fr x, y;
  memcpy(&x, a, 32);
  memcpy(&y, b, 32);
  Fr t1 = cdlh::fr_sub(cdlh::fr_add(cdlh::fr_mul(x, y), x), y);
  Fr r = cdlh::fr_mul(cdlh::fr_inv(t1), cdlh::fr_pow_u64(x, 5));
  memcpy(fr_out, &r, 32);
  // the batched inversion must agree with the single one and keep zeros
  std::vector<Fr> bi = cdlh::fr_batch_inv({x, t1, cdlh::FR_ZERO, y, t1});
  if (!cdlh::fr_eq(bi[1], cdlh::fr_inv(t1)) || !cdlh::fr_eq(bi[4], bi[1]) || !cdlh::fr_is_zero(bi[2]) ||
      !cdlh::fr_eq(bi[0], cdlh::fr_inv(x)) || !cdlh::fr_eq(bi[3], cdlh::fr_inv(y)))
    return CDL_ERR_INTERNAL;
  if (!cdlh::fr_is_zero(t1) && !cdlh::fr_eq(cdlh::fr_mul(t1, cdlh::fr_inv(t1)), cdlh::FR_ONE)) return CDL_ERR_INTERNAL;
  return CDL_OK;
}

int32_t cdl_host_selftest_fibers(uint32_t n, uint32_t rounds, uint8_t* digest32, int32_t* used_x8) {
  if (!digest32 || !used_x8 || n == 0 || n > (1u << 16)) return CDL_ERR_INVALID_ARG;
  auto work = [&](size_t i, uint8_t* out) {  // out: rounds * 32 + 32 bytes
    cdlh::Transcript t("curdleproofs");
    cdlh::Rand rnd(1000 + i);
    uint8_t msg[200];
    for (uint32_t r = 0; r < rounds; r++) {
      size_t len = 1 + (i * 7 + r * 13) % sizeof msg;
      for (size_t k = 0; k < len; k++) msg[k] = (uint8_t)(i + 31 * r + k);
      t.append_message("selftest_msg", msg, len);
      Fr c = t.challenge("selftest_challenge");
      Fr x = rnd.get_fr();
      t.append_scalar("selftest_rand", x);
      cdlh::fr_to_bytes_be(out + 32 * r, cdlh::fr_add(c, x));
    }
    t.challenge_bytes("selftest_final", out + 32 * rounds, 32);
  };
  const size_t per = (size_t)rounds * 32 + 32;
  std::vector<uint8_t> plain(n * per), fib(n * per);
  for (size_t i = 0; i < n; i++) work(i, plain.data() + i * per);
  *used_x8 = cdlh::fibers_available() ? 1 : 0;
  cdlh::ThreadPool pool(3);
  std::function<void(size_t)> fn([&](size_t i) { work(i, fib.data() + i * per); });
  pool.parallel_for((n + 7) / 8, std::function<void(size_t)>([&](size_t g) {
    cdlh::run_fiber_group(fn, 8 * g, n - 8 * g < 8 ? n - 8 * g : 8);
  }));
  cdlh::Shake256 h;
  h.absorb(fib.data(), fib.size());
  h.read(digest32, 32);
  return plain == fib ? CDL_OK : CDL_ERR_INTERNAL;
}

// ------------------------------------------------------------------ Rand
int32_t cdl_rand_new(uint64_t seed, cdl_rand** out) {
  if (!out) return CDL_ERR_INVALID_ARG;
  *out = new cdl_rand(seed);
  return CDL_OK;
}
void cdl_rand_free(cdl_rand* r) { delete r; }
int32_t cdl_rand_get_frs(cdl_rand* r, size_t n, cdl_fr* out) {
  if (!r || (n && !out)) return CDL_ERR_INVALID_ARG;
  r->r.get_frs(reinterpret_cast<Fr*>(out), n);
  return CDL_OK;
}
int32_t cdl_rand_generate_permutation(cdl_rand* r, size_t n, uint32_t* out) {
  if (!r || (n && !out)) return CDL_ERR_INVALID_ARG;
  std::vector<uint32_t> p = r->r.generate_permutation(n);
  memcpy(out, p.data(), n * 4);
  return CDL_OK;
}
int32_t cdl_rand_get_g1_affines(cdl_ctx* c, cdl_rand* r, size_t n, cdl_g1_affine* out) {
  if (!c || !r || (n && !out)) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  Engine* E = engine_of(c);
  int32_t rc;
  if ((rc = E->ensure_pool(n + 1)) || (rc = put_generator(E, 0)) || (rc = rand_points_to_pool(E, r, 0, 1, n))) return rc;
  return E->download_points(1, out, n);
}

// ------------------------------------------------------------------ CRS
int32_t cdl_crs_generate(cdl_ctx* c, size_t ell, cdl_rand* r, cdl_crs** out) {
  if (!c || !r || !out || ell == 0 || ell > (1u << 24)) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  Engine* E = engine_of(c);
  Layout L((uint32_t)ell);
  int32_t rc;
  if ((rc = E->ensure_pool(L.crs_size + 1))) return rc;
  const uint32_t gen = L.crs_size;  // scratch slot after the CRS image
  if ((rc = put_generator(E, gen))) return rc;
  // draw order: Gs (ell), Hs (4), H, Gt, Gu   (crs.go:21-40); these are contiguous in the image
  if ((rc = rand_points_to_pool(E, r, gen, L.Gs, ell + 7))) return rc;
  // Gsum = sum Gs, Hsum = sum Hs   (crs.go:41-48)
  cdlh::MsmStage st;
  st.idx.resize(ell + 4);
  st.sc.assign(ell + 4, cdlh::FR_ONE);
  for (uint32_t i = 0; i < ell + 4; i++) st.idx[i] = i;
  st.tasks.push_back(cdl::MsmTask{0, (uint32_t)ell, L.Gsum, 0});
  st.tasks.push_back(cdl::MsmTask{(uint32_t)ell, 4, L.Hsum, 0});
  if ((rc = E->run_msm(st))) return rc;
  return crs_finish(c, E, L, out);
}

int32_t cdl_crs_from_points(cdl_ctx* c, size_t ell, const cdl_g1_affine* points, cdl_crs** out) {
  if (!c || !points || !out || ell == 0 || ell > (1u << 24)) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  Engine* E = engine_of(c);
  Layout L((uint32_t)ell);
  int32_t rc;
  if ((rc = E->ensure_pool(L.crs_size + 1)) || (rc = E->upload_points(0, points, ell + 9))) return rc;
  return crs_finish(c, E, L, out);
}

int32_t cdl_crs_export(cdl_ctx* c, const cdl_crs* crs, cdl_g1_affine* points) {
  if (!c || !crs || !points) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  CDL_CUDA(c, cudaMemcpy(points, crs->rep[0].d_points, (size_t)(crs->ell + 9) * sizeof(cdl::G1Affine), cudaMemcpyDeviceToHost));
  return CDL_OK;
}

size_t cdl_crs_ell(const cdl_crs* crs) { return crs ? crs->ell : 0; }

int32_t cdl_set_fixed_base_min_batch(cdl_ctx* c, int32_t instances) {
  if (!c || instances < -1) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  c->root()->fixed_min_batch = instances;
  return CDL_OK;
}

int32_t cdl_set_batch_verify_min(cdl_ctx* c, int32_t proofs) {
  if (!c || proofs < -1) return CDL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(c->mu);
  c->root()->batch_verify_min = proofs;
  return CDL_OK;
}

void cdl_crs_free(cdl_crs* crs) {
  if (!crs) return;
  for (size_t s = 0; s < crs->rep.size(); s++) {
    const cdl_crs::Replica& r = crs->rep[s];
    cudaSetDevice(crs->ctx->slots[s].device);
    if (r.d_points) cudaFree(r.d_points);
    if (r.d_fixed) cudaFree(r.d_fixed);
  }
  delete crs;
}

}  // extern "C"

// ------------------------------------------------------------------ ShufflePermuteCommit / Prove / Verify
// The batched forms take B caller-supplied instances (instance-major arrays) and give every instance what
// the single call gives it; the single calls are their B = 1 front ends.
namespace {

bool rands_present(cdl_rand* const* rands, size_t B) {
  for (size_t b = 0; b < B; b++)
    if (!rands[b]) return false;
  return true;
}

// the instances whose permutation is in range; the others fail with CDL_ERR_INVALID_ARG before any draw
std::vector<uint32_t> valid_instances(cdl_ctx* c, uint32_t ell, size_t B, const uint32_t* perms, int32_t* status) {
  std::vector<uint32_t> sel;
  sel.reserve(B);
  for (size_t b = 0; b < B; b++) {
    const uint32_t* p = perms + b * ell;
    status[b] = CDL_OK;
    for (uint32_t i = 0; i < ell && status[b] == CDL_OK; i++)
      if (p[i] >= ell) status[b] = c->fail(CDL_ERR_INVALID_ARG, "permutation entry out of range");
    if (status[b] == CDL_OK) sel.push_back((uint32_t)b);
  }
  return sel;
}

}  // namespace

extern "C" {

int32_t cdl_shuffle_permute_commit_batch(cdl_ctx* c, const cdl_crs* crs, size_t B, const cdl_g1_affine* Rs,
                                         const cdl_g1_affine* Ss, const uint32_t* perms, const cdl_fr* ks,
                                         cdl_rand* const* rands, cdl_g1_affine* Ts, cdl_g1_affine* Us, cdl_g1_jac* M,
                                         cdl_fr* rs_m, int32_t* status) {
  if (!c || !crs || B == 0 || !Rs || !Ss || !perms || !ks || !rands || !Ts || !Us || !M || !rs_m || !status ||
      !rands_present(rands, B))
    return CDL_ERR_INVALID_ARG;
  if (split_lanes(c, B)) {
    const size_t e = crs->ell;
    return run_split(c, B, [&](cdl_ctx* lane, size_t lo, size_t hi) {
      return cdl_shuffle_permute_commit_batch(lane, crs, hi - lo, Rs + lo * e, Ss + lo * e, perms + lo * e, ks + lo,
                                              rands + lo, Ts + lo * e, Us + lo * e, M + lo, rs_m + 4 * lo, status + lo);
    });
  }
  std::lock_guard<std::mutex> lk(c->mu);
  Engine* E;
  Layout L(1);
  int32_t rc = begin_call(c, crs, B, &E, &L, true);
  if (rc) return rc;
  const uint32_t ell = L.ell;
  const std::vector<uint32_t> sel = valid_instances(c, ell, B, perms, status);
  const uint32_t Bn = (uint32_t)sel.size();
  if (!Bn) return CDL_OK;
  const cdl_g1_affine* in[2] = {Rs, Ss};
  if ((rc = E->load_instances(L, sel, in, 2, nullptr))) return rc;
  std::vector<std::vector<uint32_t>> pv(Bn);
  std::vector<Fr> kv(Bn);
  std::vector<cdl_rand*> rv(Bn);
  for (uint32_t j = 0; j < Bn; j++) {
    pv[j].assign(perms + (size_t)sel[j] * ell, perms + ((size_t)sel[j] + 1) * ell);
    memcpy(&kv[j], ks + sel[j], 32);
    rv[j] = rands[sel[j]];
  }
  std::vector<std::vector<Fr>> rsm;
  if ((rc = E->shuffle_permute_commit(L, Bn, pv, kv, rv, rsm))) return rc;
  // Ts | Us | M of every instance, gathered behind the instance regions and downloaded in one copy
  const uint32_t tail = L.base(Bn), per = 2 * ell + 1;
  std::vector<cdl::CopyRange> ranges;
  for (uint32_t j = 0; j < Bn; j++) {
    ranges.push_back(cdl::CopyRange{L.base(j) + L.Ts, tail + j * per, 2 * ell, 0});
    ranges.push_back(cdl::CopyRange{L.base(j) + L.M, tail + j * per + 2 * ell, 1, 0});
  }
  std::vector<cdl_g1_affine> out((size_t)Bn * per);
  if ((rc = E->copy_ranges(ranges)) || (rc = E->download_points(tail, out.data(), out.size()))) return rc;
  for (uint32_t j = 0; j < Bn; j++) {
    const size_t b = sel[j];
    const cdl_g1_affine* o = out.data() + (size_t)j * per;
    memcpy(Ts + b * ell, o, (size_t)ell * sizeof(cdl_g1_affine));
    memcpy(Us + b * ell, o + ell, (size_t)ell * sizeof(cdl_g1_affine));
    affine_to_jac(M + b, o[2 * ell]);
    memcpy(rs_m + 4 * b, rsm[j].data(), 4 * 32);
  }
  return CDL_OK;
}

int32_t cdl_shuffle_permute_commit(cdl_ctx* c, const cdl_crs* crs, const cdl_g1_affine* Rs, const cdl_g1_affine* Ss,
                                   const uint32_t* perm, const cdl_fr* k, cdl_rand* r, cdl_g1_affine* Ts,
                                   cdl_g1_affine* Us, cdl_g1_jac* M, cdl_fr* rs_m) {
  int32_t status = CDL_OK;
  cdl_rand* rr[1] = {r};
  int32_t rc = cdl_shuffle_permute_commit_batch(c, crs, 1, Rs, Ss, perm, k, rr, Ts, Us, M, rs_m, &status);
  return rc ? rc : status;
}

int32_t cdl_prove_batch(cdl_ctx* c, const cdl_crs* crs, size_t B, const cdl_g1_affine* Rs, const cdl_g1_affine* Ss,
                        const cdl_g1_affine* Ts, const cdl_g1_affine* Us, const cdl_g1_jac* M, const uint32_t* perms,
                        const cdl_fr* ks, const cdl_fr* rs_m, cdl_rand* const* rands, uint8_t* proofs,
                        size_t proof_cap, size_t* proof_lens, int32_t* status) {
  if (!c || !crs || B == 0 || !Rs || !Ss || !Ts || !Us || !M || !perms || !ks || !rs_m || !rands || !proofs ||
      !proof_lens || !status || !rands_present(rands, B))
    return CDL_ERR_INVALID_ARG;
  if (split_lanes(c, B)) {
    const size_t e = crs->ell;
    return run_split(c, B, [&](cdl_ctx* lane, size_t lo, size_t hi) {
      return cdl_prove_batch(lane, crs, hi - lo, Rs + lo * e, Ss + lo * e, Ts + lo * e, Us + lo * e, M + lo,
                             perms + lo * e, ks + lo, rs_m + 4 * lo, rands + lo, proofs + lo * proof_cap, proof_cap,
                             proof_lens + lo, status + lo);
    });
  }
  std::lock_guard<std::mutex> lk(c->mu);
  Engine* E;
  Layout L(1);
  int32_t rc = begin_call(c, crs, B, &E, &L, true);
  if (rc) return rc;
  const uint32_t ell = L.ell;
  const std::vector<uint32_t> sel = valid_instances(c, ell, B, perms, status);
  const uint32_t Bn = (uint32_t)sel.size();
  if (!Bn) return CDL_OK;
  const cdl_g1_affine* in[4] = {Rs, Ss, Ts, Us};
  if ((rc = E->load_instances(L, sel, in, 4, M))) return rc;
  std::vector<std::vector<uint32_t>> pv(Bn);
  std::vector<Fr> kv(Bn);
  std::vector<std::vector<Fr>> rsm(Bn, std::vector<Fr>(4));
  std::vector<cdl_rand*> rv(Bn);
  for (uint32_t j = 0; j < Bn; j++) {
    pv[j].assign(perms + (size_t)sel[j] * ell, perms + ((size_t)sel[j] + 1) * ell);
    memcpy(&kv[j], ks + sel[j], 32);
    memcpy(rsm[j].data(), rs_m + 4 * (size_t)sel[j], 4 * 32);
    rv[j] = rands[sel[j]];
  }
  std::vector<std::vector<uint8_t>> out;
  std::vector<int32_t> st;
  std::vector<std::string> errs;
  std::vector<uint8_t> inst_enc;
  if (L.n != (1u << L.m)) {  // Engine::prove refuses the whole call; here it is every instance's error
    for (uint32_t b : sel) status[b] = c->fail(CDL_ERR_PROTOCOL, "cs and ds are not a power of two (ell + 4 = %u)", L.n);
    return CDL_OK;
  }
  if ((rc = E->prove(L, Bn, crs, pv, kv, rsm, rv, out, st, errs, inst_enc, false))) return rc;
  for (uint32_t j = 0; j < Bn; j++) {
    const size_t b = sel[j];
    if (st[j] != CDL_OK) { status[b] = c->fail(st[j], "%s", errs[j].c_str()); continue; }
    proof_lens[b] = out[j].size();
    if (out[j].size() > proof_cap) {
      status[b] = c->fail(CDL_ERR_INVALID_ARG, "proof buffer too small: need %zu bytes", out[j].size());
      continue;
    }
    memcpy(proofs + b * proof_cap, out[j].data(), out[j].size());
  }
  return CDL_OK;
}

int32_t cdl_prove(cdl_ctx* c, const cdl_crs* crs, const cdl_g1_affine* Rs, const cdl_g1_affine* Ss,
                  const cdl_g1_affine* Ts, const cdl_g1_affine* Us, const cdl_g1_jac* M, const uint32_t* perm,
                  const cdl_fr* k, const cdl_fr* rs_m, cdl_rand* r, uint8_t* proof, size_t proof_cap,
                  size_t* proof_len) {
  int32_t status = CDL_OK;
  cdl_rand* rr[1] = {r};
  int32_t rc = cdl_prove_batch(c, crs, 1, Rs, Ss, Ts, Us, M, perm, k, rs_m, rr, proof, proof_cap, proof_len, &status);
  return rc ? rc : status;
}

}  // extern "C"

// ------------------------------------------------------------------ Verify helpers
namespace {

// Decode B serialized proofs (+ optional leading M) and their instance encodings into
// the pool: fills pp[b] (indices, encodings, scalars) and marks decode failures.
// inst_enc[b] must hold Rs | Ss | Ts | Us encodings (4*ell*48 B) when decode_instance.
int32_t load_proofs(Engine* E, const Layout& L, uint32_t B, const uint8_t* const* proof_ptr, const size_t* proof_len,
                    bool with_m, const uint8_t* const* m_enc, const std::vector<const uint8_t*>& inst_enc,
                    bool decode_instance, std::vector<Engine::ParsedProof>& pp) {
  const uint32_t ell = L.ell;
  pp.assign(B, Engine::ParsedProof());
  std::vector<uint8_t> enc;
  std::vector<uint32_t> dst;
  std::vector<uint32_t> owner;  // instance of each queued point
  for (uint32_t b = 0; b < B; b++) {
    Engine::ParsedProof& q = pp[b];
    q.inst_enc = inst_enc[b];
    cdlh::WireProof w;
    size_t used = 0;
    std::string e = cdlh::parse_wire_proof(proof_ptr[b], proof_len[b], with_m, w, &used);
    if (!e.empty()) { q.err = "decoding proof: " + e; continue; }
    q.sc.resize(7);
    bool sc_ok = true;
    for (int i = 0; i < 7; i++) sc_ok = sc_ok && cdlh::fr_from_bytes_be_canonical(q.sc[i], w.scalars[i]);
    if (!sc_ok) { q.err = "decoding proof: scalar is not canonical"; continue; }
    memcpy(q.lens, w.lens, sizeof q.lens);
    if (w.points.size() + (with_m ? 0 : 1) > 19 + 10 * 32) { q.err = "decoding proof: too many points"; continue; }
    const uint32_t base = L.base(b);
    uint32_t slot = base + L.PP;
    if (!with_m) {  // M comes from the caller (already in the pool at L.M)
      q.pt.push_back(base + L.M);
      q.enc.push_back(m_enc[b]);
    }
    for (const uint8_t* p : w.points) {
      q.pt.push_back(slot);
      q.enc.push_back(p);
      enc.insert(enc.end(), p, p + 48);
      dst.push_back(slot++);
      owner.push_back(b);
    }
    if (decode_instance) {
      enc.insert(enc.end(), inst_enc[b], inst_enc[b] + (size_t)4 * ell * 48);
      for (uint32_t i = 0; i < 4 * ell; i++) { dst.push_back(base + L.Rs + i); owner.push_back(b); }
    }
    q.ok = true;
  }
  std::vector<uint8_t> st;
  int32_t rc = E->decompress(enc.data(), dst, st);
  if (rc) return rc;
  for (size_t i = 0; i < st.size(); i++)
    if (st[i] && pp[owner[i]].ok) {
      pp[owner[i]].ok = false;
      pp[owner[i]].err = "decoding point: rejected encoding (reason " + std::to_string((int)st[i]) + ")";
    }
  return CDL_OK;
}

}  // namespace

extern "C" {

int32_t cdl_verify_batch(cdl_ctx* c, const cdl_crs* crs, size_t B, const uint8_t* proofs, size_t proof_stride,
                         const size_t* proof_lens, const cdl_g1_affine* Rs, const cdl_g1_affine* Ss,
                         const cdl_g1_affine* Ts, const cdl_g1_affine* Us, const cdl_g1_jac* M,
                         cdl_rand* const* rands, int32_t* ok, int32_t* status) {
  if (!c || !crs || B == 0 || !proofs || !proof_lens || !Rs || !Ss || !Ts || !Us || !M || !rands || !ok || !status ||
      !rands_present(rands, B))
    return CDL_ERR_INVALID_ARG;
  for (size_t b = 0; b < B; b++) {
    if (proof_lens[b] > proof_stride) return c->fail(CDL_ERR_INVALID_ARG, "proof %zu is longer than the proof stride", b);
    ok[b] = 0;
  }
  if (split_lanes(c, B)) {
    const size_t e = crs->ell;
    return run_split(c, B, [&](cdl_ctx* lane, size_t lo, size_t hi) {
      return cdl_verify_batch(lane, crs, hi - lo, proofs + lo * proof_stride, proof_stride, proof_lens + lo,
                              Rs + lo * e, Ss + lo * e, Ts + lo * e, Us + lo * e, M + lo, rands + lo, ok + lo,
                              status + lo);
    });
  }
  std::lock_guard<std::mutex> lk(c->mu);
  Engine* E;
  Layout L(1);
  int32_t rc = begin_call(c, crs, B, &E, &L, true);
  if (rc) return rc;
  const uint32_t ell = L.ell;
  std::vector<uint32_t> sel(B);
  for (size_t b = 0; b < B; b++) sel[b] = (uint32_t)b;
  const cdl_g1_affine* in[4] = {Rs, Ss, Ts, Us};
  if ((rc = E->load_instances(L, sel, in, 4, M))) return rc;
  // transcript encodings Rs | Ss | Ts | Us | M of every instance, in one launch
  const size_t per = (size_t)4 * ell + 1;
  std::vector<uint32_t> src(B * per);
  for (size_t b = 0; b < B; b++) {
    const uint32_t base = L.base((uint32_t)b);
    for (uint32_t i = 0; i < 4 * ell; i++) src[b * per + i] = base + L.Rs + i;
    src[b * per + 4 * ell] = base + L.M;
  }
  std::vector<uint8_t> inst;
  if ((rc = E->compress(src, inst))) return rc;
  std::vector<const uint8_t*> inst_ptr(B), m_enc(B), proof_ptr(B);
  for (size_t b = 0; b < B; b++) {
    inst_ptr[b] = inst.data() + b * per * 48;
    m_enc[b] = inst_ptr[b] + (size_t)4 * ell * 48;
    proof_ptr[b] = proofs + b * proof_stride;
  }
  std::vector<Engine::ParsedProof> pp;
  if ((rc = load_proofs(E, L, (uint32_t)B, proof_ptr.data(), proof_lens, false, m_enc.data(), inst_ptr, false, pp)))
    return rc;
  // a proof that fails to decode is the reference's decode error: Engine::verify makes no draws for it
  std::vector<uint8_t> decode_failed(B);
  for (size_t b = 0; b < B; b++) decode_failed[b] = !pp[b].ok;
  std::vector<cdl_rand*> rv(rands, rands + B);
  std::vector<int32_t> verdict, st;
  std::vector<std::string> errs;
  if ((rc = E->verify(L, (uint32_t)B, crs, pp, rv, verdict, st, errs))) return rc;
  for (size_t b = 0; b < B; b++) {
    status[b] = decode_failed[b] ? CDL_ERR_DECODE : st[b];
    if (status[b] != CDL_OK) c->fail(status[b], "%s", errs[b].c_str());
    else ok[b] = verdict[b];
  }
  return CDL_OK;
}

int32_t cdl_verify(cdl_ctx* c, const cdl_crs* crs, const uint8_t* proof, size_t proof_len,
                   const cdl_g1_affine* Rs, const cdl_g1_affine* Ss, const cdl_g1_affine* Ts,
                   const cdl_g1_affine* Us, const cdl_g1_jac* M, cdl_rand* r, int32_t* ok) {
  int32_t status = CDL_OK;
  cdl_rand* rr[1] = {r};
  int32_t rc = cdl_verify_batch(c, crs, 1, proof, proof_len, &proof_len, Rs, Ss, Ts, Us, M, rr, ok, &status);
  return rc ? rc : status;
}

// ------------------------------------------------------------------ Whisk
int32_t cdl_whisk_generate_shuffle_proof_batch(cdl_ctx* c, const cdl_crs* crs, size_t B, const uint8_t* pre_trackers,
                                               cdl_rand* const* rands_in, uint8_t* post_trackers, uint8_t* proofs_out,
                                               size_t proof_cap, int32_t* status_out) {
  if (!c || !crs || !pre_trackers || !rands_in || !post_trackers || !proofs_out || !status_out || B == 0)
    return CDL_ERR_INVALID_ARG;
  if (split_lanes(c, B)) {
    const size_t tb = (size_t)crs->ell * 96;
    return run_split(c, B, [&](cdl_ctx* lane, size_t lo, size_t hi) {
      return cdl_whisk_generate_shuffle_proof_batch(lane, crs, hi - lo, pre_trackers + lo * tb, rands_in + lo,
                                                    post_trackers + lo * tb, proofs_out + lo * proof_cap, proof_cap,
                                                    status_out + lo);
    });
  }
  std::lock_guard<std::mutex> lk(c->mu);
  Engine* E;
  Layout L(1);
  int32_t rc = begin_call(c, crs, B, &E, &L);
  if (rc) return rc;
  const uint32_t ell = L.ell;
  std::vector<cdl_rand*> rands(rands_in, rands_in + B);
  // whisk.go:64-71: permutation, then k
  std::vector<std::vector<uint32_t>> perms(B);
  std::vector<Fr> ks(B);
  for (size_t b = 0; b < B; b++) {
    perms[b] = rands[b]->r.generate_permutation(ell);
    ks[b] = rands[b]->r.get_fr();
  }
  // whisk.go:73-80: trackers -> points (SetBytes with subgroup check), rG -> Rs, krG -> Ss
  std::vector<uint32_t> dst((size_t)B * 2 * ell);
  for (size_t b = 0; b < B; b++)
    for (uint32_t i = 0; i < ell; i++) {
      dst[(b * ell + i) * 2] = L.base((uint32_t)b) + L.Rs + i;
      dst[(b * ell + i) * 2 + 1] = L.base((uint32_t)b) + L.Ss + i;
    }
  std::vector<uint8_t> st;
  if ((rc = E->decompress(pre_trackers, dst, st))) return rc;
  bool any_bad = false;
  for (size_t b = 0; b < B; b++) {
    status_out[b] = CDL_OK;
    for (uint32_t i = 0; i < 2 * ell; i++)
      if (st[b * 2 * ell + i]) { status_out[b] = CDL_ERR_DECODE; any_bad = true; }
  }
  std::vector<std::vector<Fr>> rsm;
  if ((rc = E->shuffle_permute_commit(L, (uint32_t)B, perms, ks, rands, rsm))) return rc;
  std::vector<std::vector<uint8_t>> proofs;
  std::vector<int32_t> status;
  std::vector<std::string> errs;
  std::vector<uint8_t> inst_enc;
  if ((rc = E->prove(L, (uint32_t)B, crs, perms, ks, rsm, rands, proofs, status, errs, inst_enc, true))) return rc;
  const size_t per_inst = (size_t)(4 * ell + 1) * 48;
  for (size_t b = 0; b < B; b++) {
    uint8_t* po = proofs_out + b * proof_cap;
    memset(po, 0, proof_cap);
    uint8_t* post = post_trackers + b * (size_t)ell * 96;
    if (status_out[b] != CDL_OK) { memset(post, 0, (size_t)ell * 96); continue; }
    if (status[b] != CDL_OK) { status_out[b] = status[b]; c->fail(status[b], "generating proof: %s", errs[b].c_str()); any_bad = true; continue; }
    const uint8_t* ie = inst_enc.data() + b * per_inst;
    if (48 + proofs[b].size() > proof_cap) { status_out[b] = CDL_ERR_INVALID_ARG; any_bad = true; continue; }
    memcpy(po, ie + (size_t)4 * ell * 48, 48);  // M   (whisk/types.go:57-61)
    memcpy(po + 48, proofs[b].data(), proofs[b].size());
    for (uint32_t i = 0; i < ell; i++) {  // NewWhiskTracker(Ts[i], Us[i])  (whisk.go:108-111)
      memcpy(post + 96 * i, ie + ((size_t)2 * ell + i) * 48, 48);
      memcpy(post + 96 * i + 48, ie + ((size_t)3 * ell + i) * 48, 48);
    }
  }
  (void)any_bad;
  return CDL_OK;
}

int32_t cdl_whisk_generate_shuffle_proof(cdl_ctx* c, const cdl_crs* crs, const uint8_t* pre_trackers, cdl_rand* r,
                                         uint8_t* post_trackers, uint8_t* proof, size_t proof_cap) {
  int32_t status = CDL_OK;
  cdl_rand* rr[1] = {r};
  int32_t rc = cdl_whisk_generate_shuffle_proof_batch(c, crs, 1, pre_trackers, rr, post_trackers, proof, proof_cap, &status);
  if (rc) return rc;
  if (status == CDL_ERR_DECODE) return c->fail(status, "getting points: a pre-shuffle tracker failed to decode");
  if (status == CDL_ERR_INVALID_ARG) return c->fail(status, "proof buffer too small");
  return status;
}

int32_t cdl_whisk_is_valid_shuffle_proof_batch(cdl_ctx* c, const cdl_crs* crs, size_t B, const uint8_t* pre_trackers,
                                               const uint8_t* post_trackers, const uint8_t* proofs, size_t proof_len,
                                               cdl_rand* const* rands_in, int32_t* ok, int32_t* status_out) {
  if (!c || !crs || !pre_trackers || !post_trackers || !proofs || !rands_in || !ok || !status_out || B == 0)
    return CDL_ERR_INVALID_ARG;
  if (split_lanes(c, B)) {
    const size_t tb = (size_t)crs->ell * 96;
    return run_split(c, B, [&](cdl_ctx* lane, size_t lo, size_t hi) {
      return cdl_whisk_is_valid_shuffle_proof_batch(lane, crs, hi - lo, pre_trackers + lo * tb, post_trackers + lo * tb,
                                                    proofs + lo * proof_len, proof_len, rands_in + lo, ok + lo,
                                                    status_out + lo);
    });
  }
  std::lock_guard<std::mutex> lk(c->mu);
  Engine* E;
  Layout L(1);
  int32_t rc = begin_call(c, crs, B, &E, &L);
  if (rc) return rc;
  const uint32_t ell = L.ell;
  // instance encodings in transcript order Rs | Ss | Ts | Us   (whisk.go:31-44)
  std::vector<uint8_t> inst((size_t)B * 4 * ell * 48);
  std::vector<const uint8_t*> inst_ptr(B), proof_ptr(B);
  std::vector<size_t> plen(B, proof_len);
  for (size_t b = 0; b < B; b++) {
    uint8_t* ie = inst.data() + b * (size_t)4 * ell * 48;
    const uint8_t* pre = pre_trackers + b * (size_t)ell * 96;
    const uint8_t* post = post_trackers + b * (size_t)ell * 96;
    for (uint32_t i = 0; i < ell; i++) {
      memcpy(ie + (size_t)i * 48, pre + 96 * i, 48);
      memcpy(ie + ((size_t)ell + i) * 48, pre + 96 * i + 48, 48);
      memcpy(ie + ((size_t)2 * ell + i) * 48, post + 96 * i, 48);
      memcpy(ie + ((size_t)3 * ell + i) * 48, post + 96 * i + 48, 48);
    }
    inst_ptr[b] = ie;
    proof_ptr[b] = proofs + b * proof_len;
  }
  std::vector<Engine::ParsedProof> pp;
  if ((rc = load_proofs(E, L, (uint32_t)B, proof_ptr.data(), plen.data(), true, nullptr, inst_ptr, true, pp))) return rc;
  std::vector<cdl_rand*> rands(rands_in, rands_in + B);
  std::vector<int32_t> verdict, status;
  std::vector<std::string> errs;
  // decode failures are the reference's (false, err) with a decode error
  std::vector<uint8_t> decode_failed(B, 0);
  for (size_t b = 0; b < B; b++) decode_failed[b] = !pp[b].ok;
  if ((rc = E->verify(L, (uint32_t)B, crs, pp, rands, verdict, status, errs))) return rc;
  for (size_t b = 0; b < B; b++) {
    ok[b] = verdict[b];
    status_out[b] = decode_failed[b] ? CDL_ERR_DECODE : status[b];
    if (status_out[b] != CDL_OK) { ok[b] = 0; c->fail(status_out[b], "%s", errs[b].c_str()); }
  }
  return CDL_OK;
}

int32_t cdl_whisk_is_valid_shuffle_proof(cdl_ctx* c, const cdl_crs* crs, const uint8_t* pre_trackers,
                                         const uint8_t* post_trackers, size_t n_pre, size_t n_post,
                                         const uint8_t* proof, size_t proof_len, cdl_rand* r, int32_t* ok) {
  if (!c || !crs || !ok) return CDL_ERR_INVALID_ARG;
  *ok = 0;
  if (n_pre != n_post) return c->fail(CDL_ERR_PROTOCOL, "pre and post shuffle trackers must be the same length");
  if (n_pre != crs->ell) return c->fail(CDL_ERR_INVALID_ARG, "tracker count %zu does not match the CRS (ell = %u)", n_pre, crs->ell);
  int32_t status = CDL_OK;
  cdl_rand* rr[1] = {r};
  int32_t rc = cdl_whisk_is_valid_shuffle_proof_batch(c, crs, 1, pre_trackers, post_trackers, proof, proof_len, rr, ok, &status);
  if (rc) return rc;
  return status;
}


// ------------------------------------------------------------------ Whisk tracker opening proofs
// whisk.GenerateWhiskTrackerProof / IsValidWhiskTrackerProof (whisk/whisk.go:116-176): a Schnorr-style
// proof that the tracker (rG, krG) and the commitment kG share k.  Constant work per tracker (3 / 4
// scalar multiplications), so it is only worth a launch when batched over validators; the layout in
// the point pool is [G | per instance: rG krG kG A B A' B'].
namespace {
constexpr uint32_t kTpStride = 7;
const uint8_t kGenEnc[48] = {0x97, 0xf1, 0xd3, 0xa7, 0x31, 0x97, 0xd7, 0x94, 0x26, 0x95, 0x63, 0x8c, 0x4f, 0xa9, 0xac, 0x0f,
                             0xc3, 0x68, 0x8c, 0x4f, 0x97, 0x74, 0xb9, 0x05, 0xa1, 0x4e, 0x3a, 0x3f, 0x17, 0x1b, 0xac, 0x58,
                             0x6c, 0x55, 0xe8, 0x3f, 0xf9, 0x7a, 0x1a, 0xef, 0xfb, 0x3a, 0xf0, 0x0a, 0xdb, 0x22, 0xc6, 0xbb};

cdlh::Fr tracker_challenge(const uint8_t* kG, const uint8_t* krG, const uint8_t* rG, const uint8_t* A, const uint8_t* B) {
  cdlh::Transcript tr("whisk_opening_proof");
  tr.append_points("tracker_opening_proof", kG, 1);
  tr.append_points("tracker_opening_proof", kGenEnc, 1);
  tr.append_points("tracker_opening_proof", krG, 1);
  tr.append_points("tracker_opening_proof", rG, 1);
  tr.append_points("tracker_opening_proof", A, 1);
  tr.append_points("tracker_opening_proof", B, 1);
  return tr.challenge("tracker_opening_proof_challenge");
}

// the end of whisk.GenerateWhiskTrackerProof (whisk/whisk.go:149-176) once kG, A = blinder*G and B = blinder*rG
// are encoded: the challenge and the 128-byte proof A | B | s with s = blinder - challenge*k
void write_tracker_proof(uint8_t* out, const uint8_t* tracker, const uint8_t* kG, const uint8_t* A, const uint8_t* B,
                         const Fr& k, const Fr& blinder) {
  const Fr ch = tracker_challenge(kG, tracker + 48, tracker, A, B);
  memcpy(out, A, 48);
  memcpy(out + 48, B, 48);
  cdlh::fr_to_bytes_be(out + 96, cdlh::fr_sub(blinder, cdlh::fr_mul(ch, k)));
}

// scalars of one validator's registration, all multiples of G: r, k*r, k, blinder, blinder*r
constexpr size_t kRegScalars = 5;
}  // namespace

int32_t cdl_whisk_generate_tracker_proof_batch(cdl_ctx* c, size_t B, const uint8_t* trackers, const cdl_fr* ks,
                                               cdl_rand* const* rands, uint8_t* proofs, int32_t* status_out) {
  if (!c || !trackers || !ks || !rands || !proofs || !status_out || B == 0 || B > (1u << 24)) return CDL_ERR_INVALID_ARG;
  if (slots_for(c, B) > 1)
    return run_split(c, B, [&](cdl_ctx* lane, size_t lo, size_t hi) {
      return cdl_whisk_generate_tracker_proof_batch(lane, hi - lo, trackers + 96 * lo, ks + lo, rands + lo,
                                                    proofs + 128 * lo, status_out + lo);
    }, false);
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  Engine* E = engine_of(c);
  int32_t rc;
  if ((rc = E->ensure_pool(1 + B * kTpStride)) || (rc = put_generator(E, 0))) return rc;
  // tracker.getPoints(): rG, krG with curve + subgroup checks
  std::vector<uint32_t> dst(2 * B);
  for (size_t b = 0; b < B; b++) { dst[2 * b] = (uint32_t)(1 + b * kTpStride); dst[2 * b + 1] = dst[2 * b] + 1; }
  std::vector<uint8_t> st;
  if ((rc = E->decompress(trackers, dst, st))) return rc;
  // kG = k*G, A = blinder*G, B = blinder*rG
  std::vector<Fr> sc(2 * B);
  std::vector<cdl::ElemOp> ops(3 * B);
  for (size_t b = 0; b < B; b++) {
    status_out[b] = (st[2 * b] || st[2 * b + 1]) ? CDL_ERR_DECODE : CDL_OK;
    uint32_t base = (uint32_t)(1 + b * kTpStride);
    memcpy(&sc[2 * b], &ks[b], 32);
    sc[2 * b + 1] = rands[b]->r.get_fr();  // blinder (whisk.go:157)
    ops[3 * b] = cdl::ElemOp{0, cdl::kNoPoint, base + 2, (uint32_t)(2 * b)};
    ops[3 * b + 1] = cdl::ElemOp{0, cdl::kNoPoint, base + 3, (uint32_t)(2 * b + 1)};
    ops[3 * b + 2] = cdl::ElemOp{base, cdl::kNoPoint, base + 4, (uint32_t)(2 * b + 1)};
  }
  if ((rc = E->run_elem(ops, sc))) return rc;
  std::vector<uint32_t> src(3 * B);
  for (size_t b = 0; b < B; b++)
    for (uint32_t j = 0; j < 3; j++) src[3 * b + j] = (uint32_t)(1 + b * kTpStride + 2 + j);
  std::vector<uint8_t> enc;
  if ((rc = E->compress(src, enc))) return rc;
  E->par(B, [&](size_t b) {
    uint8_t* out = proofs + 128 * b;
    if (status_out[b] != CDL_OK) { memset(out, 0, 128); return; }
    const uint8_t* kG = enc.data() + 48 * (3 * b);
    write_tracker_proof(out, trackers + 96 * b, kG, kG + 48, kG + 96, sc[2 * b], sc[2 * b + 1]);
  });
  return CDL_OK;
}

// The composition "draw r; rG = r*G; krG = k*rG; kG = k*G; cdl_whisk_generate_tracker_proof_batch" with every point
// written as a multiple of G: k*r and blinder*r are taken mod q on the host, so the five points of every validator
// come from one Engine::base_mul of G (DESIGN §5e).
int32_t cdl_whisk_generate_registration_batch(cdl_ctx* c, size_t B, const cdl_fr* ks, cdl_rand* const* rands,
                                              uint8_t* trackers, uint8_t* k_comms, uint8_t* proofs, int32_t* status) {
  if (!c || !ks || !rands || !trackers || !k_comms || !proofs || !status || B == 0) return CDL_ERR_INVALID_ARG;
  if (B > CDL_WHISK_REGISTER_MAX) {
    std::lock_guard<std::mutex> lk(c->mu);
    return c->fail(CDL_ERR_TOO_LARGE, "whisk registration: %zu validators exceed 2^21", B);
  }
  if (!rands_present(rands, B)) return CDL_ERR_INVALID_ARG;
  const size_t min_block = cdlh::base_mul_min_block(kRegScalars);
  if (slots_for(c, B, min_block) > 1)
    return run_split(c, B, [&](cdl_ctx* lane, size_t lo, size_t hi) {
      return cdl_whisk_generate_registration_batch(lane, hi - lo, ks + lo, rands + lo, trackers + 96 * lo,
                                                   k_comms + 48 * lo, proofs + 128 * lo, status + lo);
    }, false, 1, min_block);
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  Engine* E = engine_of(c);
  std::vector<Fr> sc(kRegScalars * B);
  E->par(B, [&](size_t v) {
    Fr* s = &sc[kRegScalars * v];
    const Fr r = rands[v]->r.get_fr();
    if (cdlh::fr_is_zero(r) || cdlh::fr_eq(r, cdlh::FR_ONE)) {  // refused: s stays zero, the blinder is not drawn
      status[v] = CDL_ERR_PROTOCOL;
      return;
    }
    Fr k;
    memcpy(&k, ks + v, 32);
    const Fr blinder = rands[v]->r.get_fr();
    s[0] = r;
    s[1] = cdlh::fr_mul(r, k);  // r < q first: k may have limbs >= q
    s[2] = k;
    s[3] = blinder;
    s[4] = cdlh::fr_mul(blinder, r);
    status[v] = CDL_OK;
  });
  for (size_t v = 0; v < B; v++)
    if (status[v] != CDL_OK) c->fail(status[v], "whisk registration: validator %zu drew r = 0 or 1", v);
  // rG krG kG A B of every validator
  std::vector<uint8_t> enc(48 * sc.size());
  int32_t rc = E->base_mul(generator(), sc.data(), sc.size(), nullptr, enc.data());
  if (rc) return rc;
  E->par(B, [&](size_t v) {
    if (status[v] != CDL_OK) return;
    const uint8_t* e = enc.data() + 48 * kRegScalars * v;
    const Fr* s = &sc[kRegScalars * v];
    memcpy(trackers + 96 * v, e, 96);
    memcpy(k_comms + 48 * v, e + 96, 48);
    write_tracker_proof(proofs + 128 * v, e, e + 96, e + 144, e + 192, s[2], s[3]);
  });
  return CDL_OK;
}

int32_t cdl_whisk_is_valid_tracker_proof_batch(cdl_ctx* c, size_t B, const uint8_t* trackers, const uint8_t* k_comms,
                                               const uint8_t* proofs, int32_t* ok, int32_t* status_out) {
  if (!c || !trackers || !k_comms || !proofs || !ok || !status_out || B == 0 || B > (1u << 24)) return CDL_ERR_INVALID_ARG;
  if (slots_for(c, B) > 1)
    return run_split(c, B, [&](cdl_ctx* lane, size_t lo, size_t hi) {
      return cdl_whisk_is_valid_tracker_proof_batch(lane, hi - lo, trackers + 96 * lo, k_comms + 48 * lo,
                                                    proofs + 128 * lo, ok + lo, status_out + lo);
    }, false);
  std::lock_guard<std::mutex> lk(c->mu);
  CDL_CUDA(c, cudaSetDevice(c->device));
  Engine* E = engine_of(c);
  int32_t rc;
  if ((rc = E->ensure_pool(1 + B * kTpStride)) || (rc = put_generator(E, 0))) return rc;
  // decode: proof (A, B, s), tracker (rG, krG), commitment kG
  std::vector<uint8_t> enc(B * 5 * 48);
  std::vector<uint32_t> dst(5 * B);
  std::vector<Fr> S(B);
  for (size_t b = 0; b < B; b++) {
    uint32_t base = (uint32_t)(1 + b * kTpStride);
    uint8_t* e = enc.data() + b * 5 * 48;
    memcpy(e, trackers + 96 * b, 96);          // rG, krG
    memcpy(e + 96, k_comms + 48 * b, 48);      // kG
    memcpy(e + 144, proofs + 128 * b, 96);     // A, B
    for (uint32_t j = 0; j < 5; j++) dst[5 * b + j] = base + j;
    status_out[b] = cdlh::fr_from_bytes_be_canonical(S[b], proofs + 128 * b + 96) ? CDL_OK : CDL_ERR_DECODE;
  }
  std::vector<uint8_t> st;
  if ((rc = E->decompress(enc.data(), dst, st))) return rc;
  cdlh::MsmStage stage;
  stage.idx.resize(4 * B);
  stage.sc.resize(4 * B);
  stage.tasks.resize(2 * B);
  E->par(B, [&](size_t b) {
    for (uint32_t j = 0; j < 5; j++)
      if (st[5 * b + j]) status_out[b] = CDL_ERR_DECODE;
    uint32_t base = (uint32_t)(1 + b * kTpStride);
    const uint8_t* e = enc.data() + b * 5 * 48;
    Fr ch = status_out[b] == CDL_OK ? tracker_challenge(e + 96, e + 48, e, e + 144, e + 192) : cdlh::FR_ZERO;
    // A' = s*G + c*kG ; B' = s*rG + c*krG
    stage.idx[4 * b] = 0;            stage.sc[4 * b] = S[b];
    stage.idx[4 * b + 1] = base + 2; stage.sc[4 * b + 1] = ch;
    stage.idx[4 * b + 2] = base;     stage.sc[4 * b + 2] = S[b];
    stage.idx[4 * b + 3] = base + 1; stage.sc[4 * b + 3] = ch;
    stage.tasks[2 * b] = cdl::MsmTask{(uint32_t)(4 * b), 2, base + 5, 0};
    stage.tasks[2 * b + 1] = cdl::MsmTask{(uint32_t)(4 * b + 2), 2, base + 6, 0};
  });
  if ((rc = E->run_msm(stage))) return rc;
  for (size_t b = 0; b < B; b++) {
    const uint8_t* e = enc.data() + b * 5 * 48;
    bool good = status_out[b] == CDL_OK && memcmp(stage.out48.data() + 48 * (2 * b), e + 144, 48) == 0 &&
                memcmp(stage.out48.data() + 48 * (2 * b + 1), e + 192, 48) == 0;
    ok[b] = good ? 1 : 0;
  }
  return CDL_OK;
}

}  // extern "C"
