// Batched curdleproof.Verify (curdleproof.go:199-318) — see host/engine.hpp.
//
// The reference defers every verifier relation C_k == <x_k, v_k> into one
// random linear combination (msmaccumulator.go:23-64) and tests
// MSM(all bases) == A_c.  Here the accumulated points C_k are themselves
// expanded over proof / instance points, so the whole accumulator collapses to
// ONE multi-scalar multiplication per proof whose result must be the point at
// infinity (the same group equation, hence the same verdict).  The same-scalar
// argument's four direct equalities (samescalarargument.go:92-99) are four more
// tiny MSMs in the same launch.  One earlier launch produces the two points
// the verifier must feed to its transcript: A' = A + T_1 + U_1 and
// D = B - beta^-1 Gsum + alpha Hsum (both depend only on proof bytes and on
// challenges drawn before either is hashed).
//
// A lane with enough proofs first checks all the tasks of that second launch at once (batch_check): one large
// MSM over a random linear combination of them, which is the point at infinity when every proof passes.  Only
// when it is not does the per-proof launch run, on the same stage, to find which proofs fail.
#include <algorithm>
#include <array>
#include <cstring>

#include "host/engine.hpp"

using cdl::MsmTask;

namespace cdlh {

namespace {

const uint8_t kInfEncV[48] = {0xc0};

// lanes with at least this many proofs in the second launch try the combined check first
// (cdl_set_batch_verify_min).  On a B200 (1 000 W) it costs 0.90x the per-proof launch's device time at 32 proofs
// and 0.56-0.67x from 64 on (tools/batch_verify.py, profiles/r5_batch_verify.txt)
constexpr uint32_t kBatchVerifyMinDefault = 64;

struct VState {
  Transcript tr{"curdleproofs"};
  bool failed = false;      // reference returns (false, err)
  std::string err;
  bool late_failed = false;  // an error the reference would only reach after the same-scalar check
  std::string late_err;
  std::vector<Fr> as;
  Fr sp_alpha, sp_beta, p, gp_alpha, gp_beta, gp_beta_inv, z;
  Rand snapshot{0};
  bool have_snapshot = false;
  Fr aw[8] = {};           // the accumulator's random weights a1..a8 (drawn from the caller's Rand)
  uint8_t digest[32] = {};  // this proof's input to the combined check's weights
  void fail(const std::string& e) { if (!failed) { failed = true; err = e; } }
};

// indices into ParsedProof::pt / enc in wire order (M first)
struct Wire {
  uint32_t M = 0, A = 1, T1 = 2, T2 = 3, U1 = 4, U2 = 5, R = 6, S = 7, B = 8, C = 9, B_c = 10, B_d = 11;
  uint32_t L_C, R_C, L_D, R_D, A1, A2, B1, B2, B_a, B_t, B_u, L_A, L_T, L_U, R_A, R_T, R_U, total;
  explicit Wire(const uint32_t* lens) {
    uint32_t o = 12;
    L_C = o; o += lens[0];
    R_C = o; o += lens[1];
    L_D = o; o += lens[2];
    R_D = o; o += lens[3];
    A1 = o++; A2 = o++; B1 = o++; B2 = o++;
    B_a = o++; B_t = o++; B_u = o++;
    L_A = o; o += lens[4];
    L_T = o; o += lens[5];
    L_U = o; o += lens[6];
    R_A = o; o += lens[7];
    R_T = o; o += lens[8];
    R_U = o; o += lens[9];
    total = o;
  }
};

inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace

int32_t Engine::batch_check(const MsmStage& st, const std::vector<Fr>& rho, uint32_t crs_size, const uint32_t* d_idx,
                            const cdl::Fr* d_sc, const MsmTask* d_tasks, bool* all_inf) {
  *all_inf = false;
  const uint32_t nterm = (uint32_t)st.idx.size(), nt = (uint32_t)st.tasks.size();
  const size_t nc = (size_t)nterm + crs_size;
  const cdl::BigMsmDims d = cdl::big_msm_dims(nc, cdl::big_msm_pick_c(nc), 0, 1);
  // sorted entries, bucket offsets and point indices of the large MSM are 32-bit; such a lane keeps the
  // per-proof launch (same verdicts)
  if (!nterm || nc >= ((size_t)1 << 30) || cdl::big_msm_entries(d) >= ((uint64_t)1 << 32)) return CDL_OK;
  // stage positions of the terms on CRS bases, grouped by base (counting sort)
  std::vector<uint32_t> off(crs_size + 1, 0);
  for (uint32_t j = 0; j < nterm; j++)
    if (st.idx[j] < crs_size) off[st.idx[j] + 1]++;
  for (uint32_t b = 0; b < crs_size; b++) off[b + 1] += off[b];
  const uint32_t npos = off[crs_size];
  // staging: rho | off | pos, then the downloaded flag
  const size_t h_off = al256((size_t)nt * 32), h_pos = h_off + al256(((size_t)crs_size + 1) * 4),
               h_flag = h_pos + al256((size_t)npos * 4);
  int32_t rc;
  if ((rc = reserve(s_bv_, h_flag + 4))) return rc;
  uint8_t* hb = (uint8_t*)s_bv_.h();
  memcpy(hb, rho.data(), (size_t)nt * 32);
  memcpy(hb + h_off, off.data(), off.size() * 4);
  uint32_t* pos = (uint32_t*)(hb + h_pos);
  for (uint32_t j = 0; j < nterm; j++)
    if (st.idx[j] < crs_size) pos[off[st.idx[j]]++] = j;
  // device: combined indices | scalars | result | flag | large-MSM scratch (grow-only)
  const size_t d_csc = al256(nc * 4), d_res = d_csc + al256(nc * 32), d_flag = d_res + al256(sizeof(cdl::G1Jac)),
               d_scr = d_flag + 256, need = d_scr + cdl::big_msm_scratch_bytes(d);
  if (!d_bv_.grow(need, ctx_->stream)) return CDL_OK;  // the per-proof launch needs no more memory
  uint8_t* db = (uint8_t*)d_bv_.d();
  const uint8_t* sb = (const uint8_t*)s_bv_.d();
  uint32_t* cidx = (uint32_t*)db;
  cdl::Fr* csc = (cdl::Fr*)(db + d_csc);
  cdl::G1Jac* res = (cdl::G1Jac*)(db + d_res);
  uint32_t* flag = (uint32_t*)(db + d_flag);
  CDL_CUDA(ctx_, cudaMemcpyAsync(s_bv_.d(), s_bv_.h(), h_flag, cudaMemcpyHostToDevice, ctx_->stream));
  tick();
  cdl::launch_bv_assemble(d_idx, d_sc, d_tasks, nt, (const cdl::Fr*)sb, nterm, (const uint32_t*)(sb + h_off),
                          (const uint32_t*)(sb + h_pos), crs_size, cidx, csc, ctx_->stream);
  // the other lanes' bucket warps rely on the persisting-L2 window: leave it in place
  int nk = 0;
  cudaError_t e = cdl::launch_big_msm(d_pool(), csc, d, 0, db + d_scr, ctx_->sm_count, res, ctx_->stream, cidx,
                                      /*release_l2=*/false, &nk);
  cdl::launch_bv_is_inf(res, flag, ctx_->stream);
  tock(0, msm_algorithmic_modmul(nc), 128.0 * nc);
  launches += 2 + nk;  // two assembly kernels, the large MSM's and the flag kernel; tock counted one
  CDL_CUDA(ctx_, e);
  CDL_CUDA(ctx_, cudaGetLastError());
  CDL_CUDA(ctx_, cudaMemcpyAsync(hb + h_flag, flag, 4, cudaMemcpyDeviceToHost, ctx_->stream));
  CDL_CUDA(ctx_, ctx_->sync_stream());
  finish_timing();
  *all_inf = *(const uint32_t*)(hb + h_flag) == 1;
  return CDL_OK;
}

int32_t Engine::verify(const Layout& L, uint32_t B, const cdl_crs* crs, std::vector<ParsedProof>& pp,
                       std::vector<cdl_rand*>& rands, std::vector<int32_t>& verdict, std::vector<int32_t>& status,
                       std::vector<std::string>& errs) {
  struct Tot { double& a; double t0; ~Tot() { a += Engine::now() - t0; } } ptot{prof.total, now()};
  const uint32_t ell = L.ell, n = L.n;
  int32_t rc;
  verdict.assign(B, 0);
  status.assign(B, CDL_OK);
  errs.assign(B, "");
  std::vector<std::unique_ptr<VState>> S(B);
  for (auto& s : S) s.reset(new VState());
  const uint8_t* H_enc = crs->enc.data() + 48 * (size_t)L.H;
  MsmStage st;

  for (uint32_t b = 0; b < B; b++)
    if (!pp[b].ok) S[b]->fail(pp[b].err);

  std::vector<std::array<uint8_t, 48>> Aprime(B), Denc(B);

  // ---- transcript up to the grand-product challenges (curdleproof.go:213-223,
  // samepermutationargument.go:118-130, grandproductargument.go:219-232)
  par(B, [&](size_t b) {
    VState& s = *S[b];
    if (s.failed) return;
    const ParsedProof& q = pp[b];
    Wire w(q.lens);
    const uint8_t* ie = q.inst_enc;
    if (memcmp(ie + (size_t)2 * ell * 48, kInfEncV, 48) == 0) { s.fail("randomizer is zero"); return; }
    s.tr.append_points("curdleproofs_step1", ie, 4 * ell);
    s.tr.append_points("curdleproofs_step1", q.enc[w.M], 1);
    s.as.resize(ell);
    for (uint32_t i = 0; i < ell; i++) s.as[i] = s.tr.challenge("curdleproofs_vec_a");
    s.tr.append_points("same_perm_step1", q.enc[w.A], 1);
    s.tr.append_points("same_perm_step1", q.enc[w.M], 1);
    s.tr.append_scalars("same_perm_step1", s.as.data(), ell);
    s.sp_alpha = s.tr.challenge("same_perm_alpha");
    s.sp_beta = s.tr.challenge("same_perm_beta");
    s.p = FR_ONE;
    Fr i_alpha = FR_ZERO;  // i * alpha
    for (uint32_t i = 0; i < ell; i++) {
      s.p = fr_mul(s.p, fr_add(fr_add(i_alpha, s.sp_beta), s.as[i]));
      i_alpha = fr_add(i_alpha, s.sp_alpha);
    }
    s.tr.append_points("gprod_step1", q.enc[w.B], 1);
    s.tr.append_scalar("gprod_step1", s.p);
    s.gp_alpha = s.tr.challenge("gprod_alpha");
    s.tr.append_points("gprod_step2", q.enc[w.C], 1);
    s.tr.append_scalar("gprod_step2", q.sc[0]);  // Rp
    s.gp_beta = s.tr.challenge("gprod_beta");
    if (fr_is_zero(s.gp_beta)) { s.fail("beta is zero"); return; }
    s.gp_beta_inv = fr_inv(s.gp_beta);
  });

  // ---- launch 1: the two points the verifier must hash, in one launch.
  //   D = B - beta^-1 * Gsum + alpha * Hsum   (grandproductargument.go:243-246)
  //   A' = A + T_1 + U_1                      (curdleproof.go:268-269; hashed by the same-multiscalar argument)
  {
    st.clear();
    std::vector<int> slot(B, -1);
    for (uint32_t b = 0; b < B; b++) {
      VState& s = *S[b];
      if (s.failed) continue;
      const ParsedProof& q = pp[b];
      Wire w(q.lens);
      slot[b] = (int)st.tasks.size();
      st.tasks.push_back(MsmTask{(uint32_t)st.idx.size(), 3, L.base(b) + L.scratch + 1, 0});
      st.idx.push_back(q.pt[w.B]); st.sc.push_back(FR_ONE);
      st.idx.push_back(L.Gsum); st.sc.push_back(fr_neg(s.gp_beta_inv));
      st.idx.push_back(L.Hsum); st.sc.push_back(s.gp_alpha);
      st.tasks.push_back(MsmTask{(uint32_t)st.idx.size(), 3, L.base(b) + L.scratch, 0});
      st.idx.push_back(q.pt[w.A]); st.sc.push_back(FR_ONE);
      st.idx.push_back(q.pt[w.T1]); st.sc.push_back(FR_ONE);
      st.idx.push_back(q.pt[w.U1]); st.sc.push_back(FR_ONE);
    }
    if ((rc = run_msm(st))) return rc;
    for (uint32_t b = 0; b < B; b++)
      if (slot[b] >= 0) {
        memcpy(Denc[b].data(), st.out48.data() + 48 * (size_t)slot[b], 48);
        memcpy(Aprime[b].data(), st.out48.data() + 48 * ((size_t)slot[b] + 1), 48);
      }
  }

  // ---- rest of the transcript; build the final launch
  // per instance: up to 5 tasks; the big one has at most 5*ell + 8 + 13 + 10*m terms
  std::vector<std::vector<uint32_t>> t_idx(B);
  std::vector<std::vector<Fr>> t_sc(B);
  std::vector<std::vector<uint32_t>> t_cnt(B);  // term count of each of the instance's tasks
  std::vector<uint8_t> have_big(B, 0);
  // The scalars of the 5*ell + 7 structurally shared bases are computed on the device from a small per-proof
  // block (k_verify_scalars.cu); CDL_VERIFY_SCALARS=host keeps the host computation (cross-check, A/B).
  static const bool device_scalars = [] {
    const char* e = getenv("CDL_VERIFY_SCALARS");
    return !(e && e[0] == 'h');
  }();
  const bool dev_sc = device_scalars && L.m <= (uint32_t)cdl::kVsMaxM;
  std::vector<cdl::VsParams> vsp(dev_sc ? B : 0);
  std::vector<uint32_t> merged_at(B, 0);  // position of the first merged-base term inside the instance's big task
  const int32_t bv_set = ctx_->root()->batch_verify_min;
  const uint32_t bv_min = bv_set >= 0 ? (uint32_t)bv_set : kBatchVerifyMinDefault;
  const bool bv_maybe = bv_min > 0 && B >= bv_min;
  par(B, [&](size_t b) {
    VState& s = *S[b];
    if (s.failed) return;
    const ParsedProof& q = pp[b];
    Wire w(q.lens);
    Rand& rand = rands[b]->r;
    const uint32_t base = L.base((uint32_t)b);
    const Fr &Rp = q.sc[0], &c0 = q.sc[1], &d0 = q.sc[2], &Zk = q.sc[3], &Zt = q.sc[4], &Zu = q.sc[5], &xf = q.sc[6];
    // merged base scalars of the accumulator (msmaccumulator.go:37-43 merges by base)
    std::vector<Fr> sGs(ell, FR_ZERO), sTs(ell, FR_ZERO), sUs(ell, FR_ZERO), sRs(ell, FR_ZERO), sSs(ell, FR_ZERO);
    Fr sHs[4] = {FR_ZERO, FR_ZERO, FR_ZERO, FR_ZERO}, sH = FR_ZERO, sGt = FR_ZERO, sGu = FR_ZERO;
    // -A_c as extra terms: (pool index, scalar)
    std::vector<uint32_t>& idx = t_idx[b];
    std::vector<Fr>& sc = t_sc[b];
    auto neg_term = [&](uint32_t point, const Fr& coeff) { idx.push_back(point); sc.push_back(fr_neg(coeff)); };

    // -- same-permutation: C = B - A - alpha*M ; <beta.., Gs>   (samepermutationargument.go:132-142)
    Fr a1 = s.aw[0] = rand.get_fr();
    const Fr a1b = fr_mul(a1, s.sp_beta);
    if (!dev_sc)
      for (uint32_t i = 0; i < ell; i++) sGs[i] = a1b;
    neg_term(q.pt[w.B], a1);
    neg_term(q.pt[w.A], fr_neg(a1));
    neg_term(q.pt[w.M], fr_neg(fr_mul(a1, s.sp_alpha)));

    // -- grand product -> inner product (grandproductargument.go:234-283, innerproductargument.go:201-294)
    std::vector<Fr> us(dev_sc ? 0 : n);
    if (!dev_sc) {
      Fr t = s.gp_beta_inv;
      for (uint32_t i = 0; i < ell; i++) { us[i] = t; t = fr_mul(t, s.gp_beta_inv); }
      for (uint32_t i = ell; i < n; i++) us[i] = t;
    }
    Fr beta_l = fr_pow_u64(s.gp_beta, ell);
    Fr beta_l1 = fr_mul(beta_l, s.gp_beta);
    s.z = fr_sub(fr_add(fr_mul(s.p, beta_l), fr_mul(Rp, beta_l1)), FR_ONE);
    s.tr.append_points("ipa_step1", q.enc[w.C], 1);
    s.tr.append_points("ipa_step1", Denc[b].data(), 1);
    s.tr.append_scalar("ipa_step1", s.z);
    s.tr.append_points("ipa_step1", q.enc[w.B_c], 1);
    s.tr.append_points("ipa_step1", q.enc[w.B_d], 1);
    Fr ipa_alpha = s.tr.challenge("ipa_alpha");
    Fr ipa_beta = s.tr.challenge("ipa_beta");
    if (n & (n - 1)) { s.fail("ipa n is not a power of two"); return; }
    const uint32_t m = L.m;
    // the reference indexes the four slices for i < m unchecked (would panic) and its MultiExp
    // rejects a length mismatch: both are errors at this boundary
    if (q.lens[0] < m || q.lens[1] < m || q.lens[2] < m || q.lens[3] < m) { s.fail("ipa proof has too few rounds"); return; }
    std::vector<Fr> gamma(m);
    for (uint32_t i = 0; i < m; i++) {
      s.tr.append_points("ipa_loop", q.enc[w.L_C + i], 1);
      s.tr.append_points("ipa_loop", q.enc[w.L_D + i], 1);
      s.tr.append_points("ipa_loop", q.enc[w.R_C + i], 1);
      s.tr.append_points("ipa_loop", q.enc[w.R_D + i], 1);
      gamma[i] = s.tr.challenge("ipa_gamma");
    }
    if (q.lens[0] != m || q.lens[1] != m || q.lens[2] != m || q.lens[3] != m) { s.fail("ipa multiexp: length mismatch"); return; }
    std::vector<Fr> gamma_inv = fr_batch_inv(gamma);
    // s[i] = prod over the set bits j of i of gamma[m-j-1] (innerproductargument.go:223-234), built by
    // doubling: one product per entry instead of one per set bit
    std::vector<Fr> sv(dev_sc ? 0 : n), svp(dev_sc ? 0 : n);
    if (!dev_sc) {
      sv[0] = svp[0] = FR_ONE;
      for (uint32_t j = 0; j < m; j++)
        for (uint32_t i = 0; i < (1u << j); i++) {
          sv[i + (1u << j)] = fr_mul(sv[i], gamma[m - j - 1]);
          svp[i + (1u << j)] = fr_mul(svp[i], gamma_inv[m - j - 1]);
        }
    }
    // AC1 = <gamma, L_C> + B_c + alpha*C + (alpha^2 z)*(beta*H) + <gamma^-1, R_C>  vs  c0*s on Gs||Hs, beta*d0*c0 on H
    Fr a2 = s.aw[1] = rand.get_fr();
    const Fr a2c0 = fr_mul(a2, c0);
    if (!dev_sc) {
      for (uint32_t i = 0; i < ell; i++) sGs[i] = fr_add(sGs[i], fr_mul(a2c0, sv[i]));
      for (uint32_t j = 0; j < 4; j++) sHs[j] = fr_add(sHs[j], fr_mul(a2c0, sv[ell + j]));
    }
    sH = fr_add(sH, fr_mul(a2, fr_mul(fr_mul(ipa_beta, d0), c0)));
    for (uint32_t i = 0; i < m; i++) {
      neg_term(q.pt[w.L_C + i], fr_mul(a2, gamma[i]));
      neg_term(q.pt[w.R_C + i], fr_mul(a2, gamma_inv[i]));
    }
    neg_term(q.pt[w.B_c], a2);
    neg_term(q.pt[w.C], fr_mul(a2, ipa_alpha));
    sH = fr_sub(sH, fr_mul(a2, fr_mul(fr_mul(fr_mul(ipa_alpha, ipa_alpha), s.z), ipa_beta)));
    // AC2 = <gamma, L_D> + B_d + alpha*D + <gamma^-1, R_D>  vs  s'*us*d0 on Gs||Hs;  D = B - beta^-1 Gsum + alpha_gp Hsum
    Fr a3 = s.aw[2] = rand.get_fr();
    const Fr a3d0 = fr_mul(a3, d0);
    if (!dev_sc) {
      for (uint32_t i = 0; i < ell; i++) sGs[i] = fr_add(sGs[i], fr_mul(a3d0, fr_mul(svp[i], us[i])));
      for (uint32_t j = 0; j < 4; j++) sHs[j] = fr_add(sHs[j], fr_mul(a3d0, fr_mul(svp[ell + j], us[ell + j])));
    }
    for (uint32_t i = 0; i < m; i++) {
      neg_term(q.pt[w.L_D + i], fr_mul(a3, gamma[i]));
      neg_term(q.pt[w.R_D + i], fr_mul(a3, gamma_inv[i]));
    }
    neg_term(q.pt[w.B_d], a3);
    neg_term(base + L.scratch + 1, fr_mul(a3, ipa_alpha));  // D from launch 1
    s.snapshot = rand;  // state the reference leaves behind when the same-scalar check fails
    s.have_snapshot = true;

    // -- same-scalar argument: direct equalities (samescalarargument.go:83-100), tasks 0..3
    const uint8_t* seq[10] = {q.enc[w.R], q.enc[w.S], q.enc[w.T1], q.enc[w.T2], q.enc[w.U1], q.enc[w.U2],
                              q.enc[w.A1], q.enc[w.A2], q.enc[w.B1], q.enc[w.B2]};
    for (auto e : seq) s.tr.append_points("sameexp_points", e, 1);
    Fr ss_alpha = s.tr.challenge("sameexp_alpha");
    std::vector<uint32_t> small_idx;
    std::vector<Fr> small_sc;
    auto eq_task = [&](std::initializer_list<std::pair<uint32_t, Fr>> terms) {
      for (auto& t : terms) { small_idx.push_back(t.first); small_sc.push_back(t.second); }
      t_cnt[b].push_back((uint32_t)terms.size());
    };
    // A.T_1 + alpha*T.T_1 - z_t*Gt == 0 ;  A.T_2 + alpha*T.T_2 - z_k*R - z_t*H == 0 ; same for B / U / Gu / S / z_u
    eq_task({{q.pt[w.A1], FR_ONE}, {q.pt[w.T1], ss_alpha}, {L.Gt, fr_neg(Zt)}});
    eq_task({{q.pt[w.A2], FR_ONE}, {q.pt[w.T2], ss_alpha}, {q.pt[w.R], fr_neg(Zk)}, {L.H, fr_neg(Zt)}});
    eq_task({{q.pt[w.B1], FR_ONE}, {q.pt[w.U1], ss_alpha}, {L.Gu, fr_neg(Zu)}});
    eq_task({{q.pt[w.B2], FR_ONE}, {q.pt[w.U2], ss_alpha}, {q.pt[w.S], fr_neg(Zk)}, {L.H, fr_neg(Zu)}});

    // -- same-multiscalar argument (samemultiscalarargument.go:159-235, 239-280)
    auto late = [&](const char* e) { s.late_failed = true; s.late_err = e; };
    s.tr.append_points("same_msm_step1", Aprime[b].data(), 1);
    s.tr.append_points("same_msm_step1", q.enc[w.T2], 1);
    s.tr.append_points("same_msm_step1", q.enc[w.U2], 1);
    const uint8_t* ie = q.inst_enc;
    s.tr.append_points("same_msm_step1", ie + (size_t)2 * ell * 48, ell);
    s.tr.append_points("same_msm_step1", kInfEncV, 1);
    s.tr.append_points("same_msm_step1", kInfEncV, 1);
    s.tr.append_points("same_msm_step1", H_enc, 1);
    s.tr.append_points("same_msm_step1", kInfEncV, 1);
    s.tr.append_points("same_msm_step1", ie + (size_t)3 * ell * 48, ell);
    s.tr.append_points("same_msm_step1", kInfEncV, 1);
    s.tr.append_points("same_msm_step1", kInfEncV, 1);
    s.tr.append_points("same_msm_step1", kInfEncV, 1);
    s.tr.append_points("same_msm_step1", H_enc, 1);
    s.tr.append_points("same_msm_step1", q.enc[w.B_a], 1);
    s.tr.append_points("same_msm_step1", q.enc[w.B_t], 1);
    s.tr.append_points("same_msm_step1", q.enc[w.B_u], 1);
    Fr sm_alpha = s.tr.challenge("same_msm_alpha");
    const uint32_t lg_n = q.lens[4];
    if (lg_n >= 32) late("recursive steps greater than expected");
    else if (n != (1u << lg_n)) late("must by log2(L_a)");
    else if (q.lens[5] != lg_n || q.lens[6] != lg_n || q.lens[7] != lg_n || q.lens[8] != lg_n || q.lens[9] != lg_n)
      late("same msm proof: inconsistent round counts");
    if (!s.late_failed) {
      std::vector<Fr> ch(lg_n);
      for (uint32_t i = 0; i < lg_n; i++) {
        s.tr.append_points("same_msm_loop", q.enc[w.L_A + i], 1);
        s.tr.append_points("same_msm_loop", q.enc[w.L_T + i], 1);
        s.tr.append_points("same_msm_loop", q.enc[w.L_U + i], 1);
        s.tr.append_points("same_msm_loop", q.enc[w.R_A + i], 1);
        s.tr.append_points("same_msm_loop", q.enc[w.R_T + i], 1);
        s.tr.append_points("same_msm_loop", q.enc[w.R_U + i], 1);
        ch[i] = s.tr.challenge("same_msm_gamma");
      }
      std::vector<Fr> ch_inv = fr_batch_inv(ch);
      // xs[i] = x * prod over the set bits j of i of ch[lg_n-1-j] (samemultiscalarargument.go:267-277), by doubling
      std::vector<Fr> xs(dev_sc ? 0 : n);
      if (!dev_sc) {
        xs[0] = xf;
        for (uint32_t j = 0; j < lg_n; j++)
          for (uint32_t i = 0; i < (1u << j); i++) xs[i + (1u << j)] = fr_mul(xs[i], ch[lg_n - 1 - j]);
      }
      // over G = Gs || Hs[0..2) || Gt || Gu with point B_a + alpha*A' + <ch, L_A> + <ch^-1, R_A>
      Fr a4 = s.aw[3] = rand.get_fr();
      if (!dev_sc) {
        for (uint32_t i = 0; i < ell; i++) sGs[i] = fr_add(sGs[i], fr_mul(a4, xs[i]));
        sHs[0] = fr_add(sHs[0], fr_mul(a4, xs[ell]));
        sHs[1] = fr_add(sHs[1], fr_mul(a4, xs[ell + 1]));
        sGt = fr_add(sGt, fr_mul(a4, xs[ell + 2]));
        sGu = fr_add(sGu, fr_mul(a4, xs[ell + 3]));
      }
      neg_term(q.pt[w.B_a], a4);
      neg_term(base + L.scratch, fr_mul(a4, sm_alpha));  // A' from launch 1
      for (uint32_t i = 0; i < lg_n; i++) {
        neg_term(q.pt[w.L_A + i], fr_mul(a4, ch[i]));
        neg_term(q.pt[w.R_A + i], fr_mul(a4, ch_inv[i]));
      }
      // over T' = Ts || 0 || 0 || H || 0 with point B_t + alpha*T_2 + ...
      Fr a5 = s.aw[4] = rand.get_fr();
      if (!dev_sc) {
        for (uint32_t i = 0; i < ell; i++) sTs[i] = fr_add(sTs[i], fr_mul(a5, xs[i]));
        sH = fr_add(sH, fr_mul(a5, xs[ell + 2]));
      }
      neg_term(q.pt[w.B_t], a5);
      neg_term(q.pt[w.T2], fr_mul(a5, sm_alpha));
      for (uint32_t i = 0; i < lg_n; i++) {
        neg_term(q.pt[w.L_T + i], fr_mul(a5, ch[i]));
        neg_term(q.pt[w.R_T + i], fr_mul(a5, ch_inv[i]));
      }
      // over U' = Us || 0 || 0 || 0 || H with point B_u + alpha*U_2 + ...
      Fr a6 = s.aw[5] = rand.get_fr();
      if (!dev_sc) {
        for (uint32_t i = 0; i < ell; i++) sUs[i] = fr_add(sUs[i], fr_mul(a6, xs[i]));
        sH = fr_add(sH, fr_mul(a6, xs[ell + 3]));
      }
      neg_term(q.pt[w.B_u], a6);
      neg_term(q.pt[w.U2], fr_mul(a6, sm_alpha));
      for (uint32_t i = 0; i < lg_n; i++) {
        neg_term(q.pt[w.L_U + i], fr_mul(a6, ch[i]));
        neg_term(q.pt[w.R_U + i], fr_mul(a6, ch_inv[i]));
      }
      // R == <as, Rs>, S == <as, Ss>   (curdleproof.go:306-311)
      Fr a7 = s.aw[6] = rand.get_fr();
      if (!dev_sc)
        for (uint32_t i = 0; i < ell; i++) sRs[i] = fr_mul(a7, s.as[i]);
      neg_term(q.pt[w.R], a7);
      Fr a8 = s.aw[7] = rand.get_fr();
      if (!dev_sc)
        for (uint32_t i = 0; i < ell; i++) sSs[i] = fr_mul(a8, s.as[i]);
      neg_term(q.pt[w.S], a8);
      if (dev_sc) {  // the inputs of k_verify_scalars; sH holds the host part of H's scalar at this point
        cdl::VsParams& P = vsp[b];
        auto put = [](cdl::Fr& d, const Fr& v) { memcpy(&d, &v, 32); };
        put(P.a1b, a1b); put(P.a2c0, a2c0); put(P.a3d0, a3d0);
        put(P.a4xf, fr_mul(a4, xf)); put(P.a5xf, fr_mul(a5, xf)); put(P.a6xf, fr_mul(a6, xf));
        put(P.a7, a7); put(P.a8, a8); put(P.beta_inv, s.gp_beta_inv); put(P.sH_host, sH);
        for (uint32_t i = 0; i < m; i++) { put(P.gamma[i], gamma[i]); put(P.gamma_inv[i], gamma_inv[i]); put(P.ch[i], ch[i]); }
        P.sc_base = 0;  // set when the stage is assembled
        P.as_base = (uint32_t)(b * ell);
        P.pad[0] = P.pad[1] = 0;
      }
      merged_at[b] = (uint32_t)idx.size();
      // the merged bases
      for (uint32_t i = 0; i < ell; i++) { idx.push_back(L.Gs + i); sc.push_back(sGs[i]); }
      for (uint32_t j = 0; j < 4; j++) { idx.push_back(L.Hs + j); sc.push_back(sHs[j]); }
      idx.push_back(L.H); sc.push_back(sH);
      idx.push_back(L.Gt); sc.push_back(sGt);
      idx.push_back(L.Gu); sc.push_back(sGu);
      for (uint32_t i = 0; i < ell; i++) { idx.push_back(base + L.Ts + i); sc.push_back(sTs[i]); }
      for (uint32_t i = 0; i < ell; i++) { idx.push_back(base + L.Us + i); sc.push_back(sUs[i]); }
      for (uint32_t i = 0; i < ell; i++) { idx.push_back(base + L.Rs + i); sc.push_back(sRs[i]); }
      for (uint32_t i = 0; i < ell; i++) { idx.push_back(base + L.Ss + i); sc.push_back(sSs[i]); }
      have_big[b] = 1;
    }
    // layout of this instance's slice: the four small tasks first, then the big one
    uint32_t big_terms = have_big[b] ? (uint32_t)idx.size() : 0;
    std::vector<uint32_t> all_idx(small_idx);
    std::vector<Fr> all_sc(small_sc);
    if (have_big[b]) {
      all_idx.insert(all_idx.end(), idx.begin(), idx.end());
      all_sc.insert(all_sc.end(), sc.begin(), sc.end());
      t_cnt[b].push_back(big_terms);
    }
    idx.swap(all_idx);
    sc.swap(all_sc);
    if (bv_maybe) {  // binds the combined check's weights to everything this proof's equations depend on
      Transcript t = s.tr;
      uint8_t c[32];
      t.challenge_bytes("batch_verify_weights", c, 32);
      Shake256 h;
      h.absorb(c, 32);
      h.absorb(reinterpret_cast<const uint8_t*>(s.aw), sizeof s.aw);
      h.read(s.digest, 32);
    }
  });

  // ---- launch 2: the four same-scalar equalities + the collapsed accumulator per proof
  st.clear();
  std::vector<int> first_task(B, -1);
  std::vector<cdl::VsParams> vs_launch;
  vs_launch.reserve(dev_sc ? B : 0);
  for (uint32_t b = 0; b < B; b++) {
    if (S[b]->failed) continue;
    first_task[b] = (int)st.tasks.size();
    uint32_t off = (uint32_t)st.idx.size();
    st.idx.insert(st.idx.end(), t_idx[b].begin(), t_idx[b].end());
    st.sc.insert(st.sc.end(), t_sc[b].begin(), t_sc[b].end());
    if (dev_sc && have_big[b]) {  // small tasks (14 terms) come first in the slice, then the big task
      uint32_t small_terms = 0;
      for (size_t t = 0; t + 1 < t_cnt[b].size(); t++) small_terms += t_cnt[b][t];
      vsp[b].sc_base = off + small_terms + merged_at[b];
      vs_launch.push_back(vsp[b]);
    }
    uint32_t k = 0;
    for (uint32_t cnt : t_cnt[b]) {
      st.tasks.push_back(MsmTask{off, cnt, L.base(b) + L.scratch + 2 + k, 0});
      off += cnt;
      k++;
    }
  }
  const size_t np = vs_launch.size();
  if (np) {
    // per-proof parameter blocks and the vector challenges `as` go up once; the kernel runs on the stream
    // between the stage's uploads and its MSM kernels
    if ((rc = reserve(s_vs_, np * sizeof(cdl::VsParams))) || (rc = reserve(s_as_, (size_t)B * ell * 32))) return rc;
    memcpy(s_vs_.h(), vs_launch.data(), np * sizeof(cdl::VsParams));
    Fr* as_h = (Fr*)s_as_.h();
    par(B, [&](size_t b) {
      if (have_big[b]) memcpy(as_h + b * ell, S[b]->as.data(), (size_t)ell * 32);
    });
    CDL_CUDA(ctx_, cudaMemcpyAsync(s_vs_.d(), s_vs_.h(), np * sizeof(cdl::VsParams), cudaMemcpyHostToDevice, ctx_->stream));
    CDL_CUDA(ctx_, cudaMemcpyAsync(s_as_.d(), s_as_.h(), (size_t)B * ell * 32, cudaMemcpyHostToDevice, ctx_->stream));
  }
  // Combined check: one weight per task, 128 bits from SHAKE256 over every included proof's digest (never
  // from the caller's Rand, whose position the caller observes); deterministic, so runs are reproducible.
  uint32_t nin = 0;
  for (uint32_t b = 0; b < B; b++) nin += first_task[b] >= 0;
  const bool combined = bv_maybe && nin >= bv_min;
  std::vector<Fr> rho;
  if (combined) {
    static const char kLabel[] = "curdleproofs_b200 batch verify";
    Shake256 h;
    h.absorb(reinterpret_cast<const uint8_t*>(kLabel), sizeof kLabel - 1);
    for (uint32_t b = 0; b < B; b++)
      if (first_task[b] >= 0) h.absorb(S[b]->digest, 32);
    rho.resize(st.tasks.size());
    for (Fr& r : rho) {
      uint64_t w[4] = {0, 0, 0, 0};
      h.read(reinterpret_cast<uint8_t*>(w), 16);
      if (!w[0] && !w[1]) w[0] = 1;
      r = fr_from_canonical(w);
    }
  }
  bool all_pass = false;  // the combined sum is infinity: every task of the stage is
  rc = run_msm(st, [&](const uint32_t* d_idx, cdl::Fr* d_sc, const MsmTask* d_tasks, bool& done) -> int32_t {
    if (np) {
      cdl::launch_verify_scalars((const cdl::VsParams*)s_vs_.d(), (const cdl::Fr*)s_as_.d(), d_sc, (uint32_t)np, ell, n, L.m,
                                 ctx_->stream);
      launches++;
    }
    if (!combined) return CDL_OK;
    int32_t r = batch_check(st, rho, L.crs_size, d_idx, d_sc, d_tasks, &all_pass);
    done = all_pass;
    return r;
  });
  if (rc) return rc;
  for (uint32_t b = 0; b < B; b++) {
    VState& s = *S[b];
    if (s.failed) { status[b] = CDL_ERR_PROTOCOL; errs[b] = s.err; continue; }
    const uint8_t* o = st.out48.data() + 48 * (size_t)first_task[b];
    bool same_scalar_ok = true;
    for (int t = 0; t < 4 && !all_pass; t++) same_scalar_ok = same_scalar_ok && memcmp(o + 48 * t, kInfEncV, 48) == 0;
    if (!same_scalar_ok) {  // curdleproof.go:250-265: returns (false, nil) before the same-multiscalar step
      verdict[b] = 0;
      if (s.have_snapshot) rands[b]->r = s.snapshot;
      continue;
    }
    if (s.late_failed) {
      status[b] = CDL_ERR_PROTOCOL;
      errs[b] = "verifying same multiscalar: " + s.late_err;
      if (s.have_snapshot) rands[b]->r = s.snapshot;
      continue;
    }
    verdict[b] = all_pass || memcmp(o + 48 * 4, kInfEncV, 48) == 0 ? 1 : 0;  // msmaccumulator.go:63
  }
  return CDL_OK;
}

}  // namespace cdlh
